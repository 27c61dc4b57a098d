"""CPU: the C-ABI library builds, loads, and exports every symbol include/mbpls_b200.h declares."""
import ctypes
import os
import re
import subprocess
import sys

from mbpls_b200 import _cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "mbpls_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\bint\s+(mbpls_[a-z0-9_]+)\s*\(", src)
    return sorted(set(n for n in names if n != "mbpls_red_elems"))


def test_header_declares_what_python_binds():
    assert declared_symbols() == sorted(_cabi.SIGNATURES)


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(lib, name), name
    assert _cabi.load().mbpls_abi_version() == _cabi.ABI_VERSION


def test_product_path_fails_loudly_without_gpu():
    # in a child process that sees no CUDA device, so that this also runs on a machine with a GPU
    code = ("import numpy as np\n"
            "from mbpls_b200 import MBPLS, _cabi\n"
            "try:\n"
            "    MBPLS(n_components=1).fit(np.random.rand(5, 3), np.random.rand(5))\n"
            "except _cabi.MbplsCudaError:\n"
            "    raise SystemExit(0)\n"
            "raise SystemExit('fit did not raise MbplsCudaError without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mbpls_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            assert "oracle" not in open(os.path.join(pkg, fn)).read().replace("no CPU fallback", ""), fn


def test_symmetric_crossprod_split_count_fills_whole_rounds():
    """mbpls_crossprod_splits_syrk is integer arithmetic on (M, Kdim, SM count; 148 without a device): the CTAs on / above the
    diagonal times the split count must fill whole rounds of the SMs on the BASELINE shapes, within the caps."""
    import math
    from mbpls_b200 import _cabi
    for M, K, min_eff in ((2000, 1_000_000, 0.98), (2000, 125_000, 0.98), (5000, 50_000, 0.98), (8192, 8192, 0.95)):
        s = _cabi.call("mbpls_crossprod_splits_syrk", M, K)
        nb = -(-M // 128)
        working = nb * (nb + 1) // 2 * s
        assert 1 <= s <= 64 and s * 8 * M * (-(-M // 16) * 16) <= 1 << 30
        assert working / 148 / math.ceil(working / 148) >= min_eff, (M, K, s)
    assert _cabi.call("mbpls_crossprod_splits_syrk", 1, 1) == 1 and _cabi.call("mbpls_crossprod_splits_syrk", 0, 0) == 1
