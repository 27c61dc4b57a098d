"""GPU: NIPALS where the one-pass kernels do not go, and missing data that is not i.i.d., against the live numpy oracle.

A. Features longer than 20,480 samples run the two-pass trip (xtu_kernel + xw_kernel, which form the NaN-mode denominators
   themselves), deflate through loadings_deflate_global_kernel, and beyond 98,304 samples (or with more than 8 blocks) leave
   the superlevel step spread over all CTAs.  one_pass=False at 1,024 < n <= 16,384 picks a register-resident deflation
   variant by feature length.  Every fit here reads back, through torch.profiler, which kernels ran, and asserts its route.
B. Structured holes (heavy-hole features, block-wise missing rows, holes at mask-word and tile edges, holes in Y) reach the
   branches of csrc/nanmask.cu that i.i.d. holes at <= 10 % never do.
C. The NaN side kernels of csrc/nanmask.cu through the C ABI, against exact sums (math.fsum).

Convergence: a PLS1 second trip's diff_t is rounding noise that grows with the length and number of the features, and at
these lengths it can reach the default max_tol of 1e-14; so these fits use max_tol = 1e-12, where the exits have margin
over that noise, and assert_trips judges the exits that graze the threshold.
"""
import math
import re
import warnings

import numpy as np
import pytest

from helpers import assert_trips, compare, snapshot_model

pytestmark = pytest.mark.gpu
TOL = 1e-8
MAX_TOL = 1e-12
EDGE_ROWS = (0, 31, 32, 63, 1023, 1024)  # first / last sample of mask words and of the 1,024-sample tiles of masked_rowden


# --------------------------------------------------------------------------------------------- #
# helpers
# --------------------------------------------------------------------------------------------- #
def _fit_profiled(kw, X, Y, **rt):
    """Our fit under torch.profiler: (model, names of the CUDA kernels that ran)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from mbpls_b200 import MBPLS
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            m = MBPLS(**kw).set_runtime(**rt).fit([x.copy() for x in X], Y.copy())
            torch.cuda.synchronize()
    return m, {e.key for e in prof.key_averages()}


def _assert_route(kernels, ran=(), not_ran=(), what=""):
    for pat in ran:
        assert any(re.search(pat, k) for k in kernels), f"{what}: no kernel matching {pat!r} ran: {sorted(kernels)}"
    for pat in not_ran:
        hit = [k for k in kernels if re.search(pat, k)]
        assert not hit, f"{what}: {pat!r} should not have run: {hit}"


def _oracle(kw, X, Y):
    from oracle import OracleMBPLS
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return OracleMBPLS(**kw).fit([x.copy() for x in X], Y.copy())


def _check(m, o, X_test, Y_test, kw, what):
    """Everything compare() compares (census and n_samples_seen_ exactly), transform / predict on held-out rows, trips."""
    ref = snapshot_model(o, [x.copy() for x in X_test], Y_test.copy())
    ours = snapshot_model(m, [x.copy() for x in X_test], Y_test.copy())
    compare(ours, ref, TOL, what)
    assert_trips(list(m.n_iter_), list(o.n_iter_), o.diff_trace_, kw["max_tol"], what)
    for key, r in ref.items():  # a NaN anywhere would make the relative errors above meaningless
        assert np.all(np.isfinite(np.asarray(r, float))), f"{what}: oracle {key} is not finite"


def _rejects_one_pass(kw, X, Y):
    from mbpls_b200 import MBPLS
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with pytest.raises(ValueError, match="one_pass=True"):
            MBPLS(**kw).set_runtime(one_pass=True).fit([x.copy() for x in X], Y.copy())


def _two_pass_route(n, nan, B, q):
    """Kernels of a two-pass fit of n samples (csrc/nipals.cu: mbpls_loadings_deflate_f64, mbpls_nipals_xchg_epilogue_f64):
    n > 16,384 deflates through the global kernel; the superlevel step runs on all CTAs only for dense data with B <= 8,
    q <= 16 and ceil(n / 96) rounded up to 32 <= 1,024 (n <= 98,304)."""
    t = "true" if nan else "false"
    ran = [rf"xtu_kernel<{t}>", rf"xw_kernel<{t}>"]
    not_ran = [r"fused_", r"masked_colden", r"masked_rowden"]
    if n > 16384:
        ran.append(r"loadings_deflate_global_kernel")
    mc = not nan and B <= 8 and q <= 16 and (-(-n // 96) + 31) // 32 * 32 <= 1024
    (ran if mc else not_ran).append(r"xchg_epilogue_mc_kernel")
    if not mc:
        ran.append(r"xchg_epilogue_kernel")
    return ran, not_ran


def _heldout(sizes, q, seed, nan_frac=0.0, n=41):
    from oracle.cases import latent_blocks
    Xt, Yt = latent_blocks(n, sizes, q, 4, seed=seed)
    if nan_frac > 0:
        rng = np.random.default_rng(seed + 7)
        for b, x in enumerate(Xt):
            if x.shape[1] > 1:
                hole = rng.random(x.shape) < nan_frac
                hole[:, 0] = False  # every held-out row keeps an observed feature in every block
                x[hole] = np.nan
    return Xt, (Yt if q > 1 else Yt.reshape(-1, 1))


# --------------------------------------------------------------------------------------------- #
# structured missingness
# --------------------------------------------------------------------------------------------- #
def structured_holes(X, Y, seed, *, heavy=None, blockwise=None, edges=False, y_holes=False, iid=0.0):
    """NaN patterns of real multiblock data over latent_blocks output (copies; the inputs are not touched).

    Feature 0 of every block is an anchor that is never missing, so no sample loses a whole block (the reference divides
    0/0 there and the whole fit turns NaN).
    heavy=b       features 2..6 of block b miss 55 %, 80 %, 95 %, all samples but one, and all samples but two.
    blockwise=(b, frac, keep)
                  for `frac` of the samples every feature of block b except the first `keep` (1 or 2) is missing.
    edges         the last two features of every block miss the samples at mask-word and tile edges and sample n - 1.
    y_holes       Y column 0 misses some of the sparse rows of the LAST X block; column 1 stays fully observed, so the
                  first Y score is a real column.  The reference's Y-score step (mbpls.py:903) divides exactly those rows by
                  the masked v'v and every other row by the plain v'v; a Y hole outside them would turn its fit NaN.
    iid           i.i.d. holes in every non-anchor feature.
    """
    rng = np.random.default_rng(seed)
    n = Y.shape[0]
    miss = [np.zeros(x.shape, dtype=bool) for x in X]
    if iid > 0:
        for mb in miss:
            mb[:, 1:] = rng.random((n, mb.shape[1] - 1)) < iid
    if heavy is not None:
        mb = miss[heavy]
        assert mb.shape[1] >= 7
        for j, cnt in zip(range(2, 7), (round(0.55 * n), round(0.80 * n), round(0.95 * n), n - 1, n - 2)):
            mb[:, j] = False
            mb[rng.choice(n, cnt, replace=False), j] = True
    if edges:
        rows = [r for r in EDGE_ROWS if r < n] + [n - 1]
        for mb in miss:
            for j in range(max(1, mb.shape[1] - 2), mb.shape[1]):
                mb[rows, j] = True
    if blockwise is not None:
        b, frac, keep = blockwise
        rows = rng.choice(n, int(frac * n), replace=False)
        miss[b][np.ix_(rows, np.arange(keep, miss[b].shape[1]))] = True
        miss[b][np.ix_(rows, np.arange(1, keep))] = False
    for mb in miss:
        mb[:, 0] = False
    Xh = [x.copy() for x in X]
    for x, mb in zip(Xh, miss):
        x[mb] = np.nan
    Yh = Y.copy()
    if y_holes:
        assert Y.shape[1] >= 2
        last_sparse = np.flatnonzero(miss[-1].any(axis=1))
        rows = rng.choice(last_sparse, len(last_sparse) // 3, replace=False)
        Yh[rows, 0] = np.nan
        assert 0 < len(rows) < len(last_sparse)  # sparse rows of the last block with and without a Y hole
    for x in Xh:
        assert not np.isnan(x).all(axis=1).any() and not np.isnan(x).all(axis=0).any()
    return Xh, Yh


def _share_under_holes(x, u):
    """Per feature: the share of u'u that sits under the holes of x (masked_colden switches to a direct sum above 1/2)."""
    hole = np.isnan(x)
    return (hole * (u ** 2)[:, None]).sum(axis=0) / float(u @ u)


# --------------------------------------------------------------------------------------------- #
# A. long features: the two-pass kernels
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("n,sizes,q,K", [
    (20481, (40, 1, 37), 1, 3),             # first length past the one-pass kernels, PLS1
    (24575, (30, 1, 25, 14), 3, 4),         # odd n: the padding of ld
    (65537, (50, 1, 20), 3, 3),
    (100003, (45, 30, 1), 1, 3),            # superlevel step on one CTA (n > 98,304), PLS1
    (100003, (25, 1, 40), 3, 4),            # and PLS2
    (30001, (9, 1, 7, 12, 5, 8, 3, 10, 6), 3, 3),  # 9 blocks: superlevel step on one CTA at any n
])
def test_long_features_dense_match_oracle(n, sizes, q, K):
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(n, sizes, q, K, seed=n % 101 + q)
    if q == 1:
        Y = Y.ravel()
    kw = dict(n_components=K, method="NIPALS", max_tol=MAX_TOL)
    Xt, Yt = _heldout(sizes, q, seed=n % 53 + 1)
    if q == 1:
        Yt = Yt.ravel()
    m, kernels = _fit_profiled(kw, X, Y)
    ran, not_ran = _two_pass_route(n, False, len(sizes), q)
    _assert_route(kernels, ran, not_ran, f"dense n={n}")
    _check(m, _oracle(kw, X, Y), Xt, Yt, kw, f"two-pass dense n={n} B={len(sizes)} q={q}")
    _rejects_one_pass(kw, X, Y)


@pytest.mark.parametrize("n,q,pattern", [
    (24575, 2, dict(iid=0.06)),
    (24575, 2, dict(heavy=0, blockwise=(2, 0.25, 1), edges=True, y_holes=True)),
    (24575, 1, dict(heavy=1, blockwise=(0, 0.3, 2), edges=True, iid=0.02)),
    (100003, 1, dict(iid=0.05)),
    (100003, 1, dict(heavy=2, blockwise=(0, 0.2, 1), edges=True)),
])
def test_long_features_nan_match_oracle(n, q, pattern):
    """xtu_kernel<true> / xw_kernel<true> form every masked denominator themselves (no bit matrix) and the deflation kernels
    divide masked loadings by their own masked ts'ts."""
    from oracle.cases import latent_blocks
    sizes = (12, 9, 10)
    X, Y = latent_blocks(n, sizes, max(q, 2), 3, seed=n % 89 + len(pattern))
    Y = Y[:, :max(q, 2)] if pattern.get("y_holes") else Y[:, :q]
    X, Y = structured_holes(X, Y, seed=n % 13, **pattern)
    kw = dict(n_components=3, method="NIPALS", sparse_data=True, max_tol=MAX_TOL)
    Xt, Yt = _heldout(sizes, Y.shape[1], seed=n % 31 + 2, nan_frac=0.15)
    m, kernels = _fit_profiled(kw, X, Y)
    ran, not_ran = _two_pass_route(n, True, len(sizes), Y.shape[1])
    _assert_route(kernels, ran, not_ran, f"NaN n={n}")
    o = _oracle(kw, X, Y)
    _check(m, o, Xt, Yt, kw, f"two-pass NaN n={n} {sorted(pattern)}")
    for b in range(len(sizes)):
        for a, r in zip(m.sparse_X_info_[b], o.sparse_X_info_[b]):
            assert np.array_equal(a, r)
        assert np.array_equal(np.asarray(m.x_scalers_[b].n_samples_seen_), np.asarray(o.x_scalers_[b].n_samples_seen_))
    for a, r in zip(m.sparse_Y_info_["Y"], o.sparse_Y_info_["Y"]):
        assert np.array_equal(a, r)
    _rejects_one_pass(kw, X, Y)


# one_pass=False below the one-pass limit: the deflation variant by feature length (B200: 227 KB of opt-in shared memory per
# block, so ts and u0 fit twice in shared memory up to ld = 14,464; register-resident variants up to n = 16,384)
@pytest.mark.parametrize("n,nan,deflate", [
    (5000, False, r"loadings_deflate_regs2_kernel<12>"),
    (7000, False, r"loadings_deflate_regs2_kernel<16>"),
    (7000, True, r"loadings_deflate_regs2_kernel<16>"),
    (11000, False, r"loadings_deflate_regs2_kernel<24>"),
    (14000, False, r"loadings_deflate_regs2_kernel<32>"),
    (15000, False, r"loadings_deflate_regs_kernel<32>"),    # ld = 15,008 > 14,464: ts and u0 through L1
    (15000, True, r"loadings_deflate_regs_kernel<32>"),
    (18000, False, r"loadings_deflate_global_kernel"),
])
def test_two_pass_deflation_variants_match_oracle(n, nan, deflate):
    from oracle.cases import latent_blocks
    sizes = (33, 1, 20)
    X, Y = latent_blocks(n, sizes, 2, 3, seed=n % 97 + nan)
    if nan:
        X, Y = structured_holes(X, Y, seed=n % 17, iid=0.05, edges=True)
    kw = dict(n_components=3, method="NIPALS", sparse_data=nan, max_tol=MAX_TOL)
    Xt, Yt = _heldout(sizes, 2, seed=n % 29 + 3, nan_frac=0.1 if nan else 0.0)
    m, kernels = _fit_profiled(kw, X, Y, one_pass=False)
    t = "true" if nan else "false"
    _assert_route(kernels, [deflate, rf"xtu_kernel<{t}>", rf"xw_kernel<{t}>"], [r"fused_"], f"one_pass=False n={n}")
    _check(m, _oracle(kw, X, Y), Xt, Yt, kw, f"two-pass deflation n={n} nan={nan}")


# --------------------------------------------------------------------------------------------- #
# B. structured missingness through the one-pass kernels (and once through the two-pass ones)
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("n,q,pattern,also_two_pass", [
    # n % 32 == 31; masked_colden with the products in shared memory (n <= 12,800)
    (3007, 2, dict(heavy=0, blockwise=(2, 0.25, 1), edges=True, y_holes=True), True),
    (3007, 1, dict(heavy=1, blockwise=(0, 0.22, 2), edges=True, iid=0.03), False),
    # n % 32 == 1; masked_colden from global memory, features split over the CTA pair of a cluster
    (15009, 2, dict(heavy=0, blockwise=(2, 0.28, 2), edges=True, y_holes=True), False),
    (15009, 1, dict(heavy=2, blockwise=(1, 0.25, 1), edges=True, iid=0.02), True),
])
def test_structured_holes_one_pass_match_oracle(n, q, pattern, also_two_pass):
    from oracle.cases import latent_blocks
    sizes = (12, 9, 10)
    X, Y = latent_blocks(n, sizes, max(q, 2), 3, seed=n % 83 + len(pattern))
    Y = Y[:, :max(q, 2)] if pattern.get("y_holes") else Y[:, :q]
    X, Y = structured_holes(X, Y, seed=n % 11 + q, **pattern)
    kw = dict(n_components=3, method="NIPALS", sparse_data=True, max_tol=MAX_TOL)
    Xt, Yt = _heldout(sizes, Y.shape[1], seed=n % 37 + 4, nan_frac=0.15)
    o = _oracle(kw, X, Y)
    # the first Y score is a fully observed Y column: its share under the heavy-hole features is above one half, so the
    # direct-sum branch of masked_colden runs (for u0, and for u on the first trip)
    u0 = o.y_scaler_.transform(Y)[:, o.sparse_Y_info_["Y"][3][0]]
    assert np.max(_share_under_holes(X[pattern["heavy"]], u0)) > 0.9
    smem = n * 8 <= 100 * 1024
    m, kernels = _fit_profiled(kw, X, Y)
    _assert_route(kernels, [r"fused_trip_kernel", r"fused_deflate_kernel", r"nan_bitmask_kernel", r"masked_rowden_kernel",
                            rf"masked_colden_kernel<{'true' if smem else 'false'}>"],
                  [r"xw_kernel"], f"one-pass structured n={n}")
    _check(m, o, Xt, Yt, kw, f"one-pass structured n={n} {sorted(pattern)}")
    for b in range(len(sizes)):
        assert np.array_equal(np.asarray(m.x_scalers_[b].n_samples_seen_), np.asarray(o.x_scalers_[b].n_samples_seen_))
    if also_two_pass:
        m2, kernels = _fit_profiled(kw, X, Y, one_pass=False)
        _assert_route(kernels, [r"xtu_kernel<true>", r"xw_kernel<true>"], [r"fused_", r"masked_colden"], "two-pass")
        _check(m2, o, Xt, Yt, kw, f"two-pass structured n={n} {sorted(pattern)}")


# --------------------------------------------------------------------------------------------- #
# C. the NaN side kernels through the C ABI
# --------------------------------------------------------------------------------------------- #
EPS = np.finfo(np.float64).eps


def _dev():
    import torch
    return torch.device("cuda", torch.cuda.current_device())


def _packed(hole, ldw):
    """p x ldw uint32 words, bit (i & 31) of word i >> 5 set where sample i is missing; zero words beyond the samples."""
    p, n = hole.shape
    nw = (n + 31) // 32
    padded = np.zeros((p, ldw * 32), dtype=bool)
    padded[:, :n] = hole
    return np.packbits(padded, axis=1, bitorder="little").view("<u4")[:, :ldw].copy()


@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000, 1025, 12801])
def test_nan_bitmask_is_bit_exact(n):
    import torch
    from mbpls_b200 import _cabi
    from mbpls_b200.engine import ptr, stream_ptr
    rng = np.random.default_rng(n)
    p = 37
    ld = -(-n // 16) * 16 + 16
    x = rng.standard_normal((p, ld))
    x[:, n:] = np.nan                                      # the padding must give clear bits
    hole = rng.random((p, n)) < 0.3
    hole[1] = True                                         # every sample missing
    hole[2] = False                                        # none
    hole[3] = False
    hole[3, [i for i in (0, 31, 32, 63, n - 1) if i < n]] = True
    x[:, :n][hole] = np.nan
    lib_ldw = _cabi.call("mbpls_nan_bitmask_ldw", n)
    assert lib_ldw % 4 == 0 and lib_ldw >= (n + 31) // 32
    for ldw in (lib_ldw, lib_ldw + 9):
        xd = torch.from_numpy(x).to(_dev())
        bits = torch.full((p, ldw), -1, dtype=torch.int32, device=_dev())  # every word the kernel must write starts non-zero
        _cabi.call("mbpls_nan_bitmask_f64", ptr(xd), ld, n, p, ptr(bits), ldw, stream_ptr(_dev()))
        torch.cuda.synchronize()
        got = bits.cpu().numpy().view(np.uint32)
        assert np.array_equal(got, _packed(hole, ldw)), (n, ldw)


def _holes_with_share(v2, share, rng):
    """A hole set whose share of sum(v2) is just past `share`, with observed samples left over: samples are added in random
    order, except that the 1 % with the smallest v2 come last (they carry far less than 0.1 % of the sum, so even a share
    of 0.999 is reached before them)."""
    n = len(v2)
    small = np.argsort(v2)[:max(1, n // 100)]
    order = rng.permutation(n)
    order = np.concatenate((order[~np.isin(order, small)], rng.permutation(small)))
    c = np.cumsum(v2[order]) / v2.sum()
    k = int(np.searchsorted(c, share)) + 1
    return order[:min(k, n - 1)]


@pytest.mark.parametrize("n", [3001, 12800, 12801, 20011])
@pytest.mark.parametrize("with_v2", [False, True])
def test_masked_colden_against_exact_sums(n, with_v2):
    """Both forms (products staged in shared memory for n <= 12,800, global gathers above); missing shares on either side of
    the one-half switch between "total minus missing" and a direct sum over the observed samples, down to one observed
    sample with a tiny product (total minus missing would cancel to nothing there); the tail word of n % 32 != 0."""
    import torch
    from mbpls_b200 import _cabi
    from mbpls_b200.engine import ptr, stream_ptr
    rng = np.random.default_rng(n + with_v2)
    dev, st = _dev(), stream_ptr(_dev())
    nbuf = -(-n // 32) * 32 + 64
    v = np.full(nbuf, 1e3)                                 # beyond n: values that would show if a tail bit were read
    v[:n] = rng.standard_normal(n)
    v2 = np.full(nbuf, 1e3)
    v2[:n] = np.abs(v[:n]) * rng.uniform(0.5, 2.0, n) * np.sign(v[:n]) if with_v2 else v[:n]
    prod = v[:n] * v2[:n]                                  # >= 0
    shares = [0.0, 0.3, 0.49, 0.51, 0.9, 0.999]
    holes = [_holes_with_share(prod, s, rng) if s > 0 else np.array([], dtype=int) for s in shares]
    tiny = int(np.argmin(prod))                            # all but one missing, and the one left has the smallest product
    holes.append(np.setdiff1d(np.arange(n), [tiny]))
    holes.append(np.setdiff1d(np.arange(n), [int(np.argmax(prod))]))
    holes.append(np.array([n - 1]))
    holes.append(np.arange(1, n))                          # only sample 0 observed
    labels = [f"share {s}" for s in shares] + ["all but the smallest", "all but the largest", "last", "all but the first"]
    p = len(holes) + 2                                     # + two fully observed features (col_nan = 0)
    labels += ["dense", "dense"]
    hole = np.zeros((p, n), dtype=bool)
    for j, h in enumerate(holes):
        hole[j, h] = True
    col_nan = hole.sum(axis=1).astype(np.int32)
    ldw = _cabi.call("mbpls_nan_bitmask_ldw", n)
    vv = math.fsum(prod)
    obs = np.array([math.fsum(prod[~hole[j]]) for j in range(p)])
    assert np.all(obs > 0) and np.all(col_nan < n)  # every feature keeps an observed sample (all-NaN features are not fitted)
    want = {0: np.where(col_nan > 0, 1.0 / obs, 1.0), 1: 1.0 / obs, 2: obs}
    bits = torch.from_numpy(_packed(hole, ldw).view(np.int32)).to(dev)
    vd, v2d = torch.from_numpy(v).to(dev), torch.from_numpy(v2).to(dev)
    vvd = torch.tensor([vv], dtype=torch.float64, device=dev)
    cnd = torch.from_numpy(col_nan).to(dev)
    zero, one = torch.zeros(1, dtype=torch.int32, device=dev), torch.ones(1, dtype=torch.int32, device=dev)
    for mode in (0, 1, 2):
        for done in (None, zero):
            out = torch.full((p,), np.nan, dtype=torch.float64, device=dev)
            _cabi.call("mbpls_masked_colden_f64", ptr(bits), ldw, n, p, ptr(cnd), ptr(vd), ptr(v2d) if with_v2 else None,
                       ptr(vvd), mode, ptr(out), ptr(done), st)
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            err = np.abs(got - want[mode]) / np.abs(want[mode])
            bad = np.flatnonzero(~(err <= 8 * n * EPS))
            assert bad.size == 0, (mode, done is not None, [labels[j] for j in bad], err.max())
        out = torch.full((p,), np.nan, dtype=torch.float64, device=dev)
        _cabi.call("mbpls_masked_colden_f64", ptr(bits), ldw, n, p, ptr(cnd), ptr(vd), ptr(v2d) if with_v2 else None,
                   ptr(vvd), mode, ptr(out), ptr(one), st)
        torch.cuda.synchronize()
        assert torch.isnan(out).all(), "done = 1 must leave the output untouched"


@pytest.mark.parametrize("n", [1000, 2500, 4097])
def test_masked_rowden_against_exact_sums(n):
    """Splits of 1 ... 100 features: the 4-, 2- and 1-feature loops of every warp and their remainders; rows with one observed
    feature in a split, and with none."""
    import torch
    from mbpls_b200 import _cabi
    from mbpls_b200.engine import ptr, stream_ptr
    rng = np.random.default_rng(n)
    dev, st = _dev(), stream_ptr(_dev())
    lens = [1, 7, 8, 9, 24, 25, 31, 32, 33, 57, 100]
    f1 = np.cumsum(lens).astype(np.int32)
    f0 = np.concatenate(([0], f1[:-1])).astype(np.int32)
    p, S = int(f1[-1]), len(lens)
    w = rng.standard_normal(p) * rng.uniform(0.1, 10.0, p)
    hole = rng.random((p, n)) < 0.5
    for s in range(S):  # rows whose split keeps one observed feature, and a row that keeps none
        a, b = f0[s], f1[s]
        for i in rng.choice(n, 5, replace=False):
            hole[a:b, i] = True
            hole[rng.integers(a, b), i] = False
        hole[a:b, (7 * s + 3) % n] = True
        hole[a:b, [r for r in EDGE_ROWS + (n - 1,) if r < n]] = rng.random((b - a, 1)) < 0.5
    ldw = _cabi.call("mbpls_nan_bitmask_ldw", n)
    ldt = -(-n // 16) * 16 + 16
    want = np.array([[math.fsum(w[a:b][~hole[a:b, i]] ** 2) for i in range(n)] for a, b in zip(f0, f1)])
    bits = torch.from_numpy(_packed(hole, ldw).view(np.int32)).to(dev)
    wd, f0d, f1d = torch.from_numpy(w).to(dev), torch.from_numpy(f0).to(dev), torch.from_numpy(f1).to(dev)
    zero, one = torch.zeros(1, dtype=torch.int32, device=dev), torch.ones(1, dtype=torch.int32, device=dev)
    for done in (None, zero):
        Tden = torch.full((S, ldt), np.nan, dtype=torch.float64, device=dev)
        _cabi.call("mbpls_masked_rowden_f64", ptr(bits), ldw, n, ptr(wd), ptr(f0d), ptr(f1d), S, ptr(Tden), ldt, ptr(done), st)
        torch.cuda.synchronize()
        got = Tden.cpu().numpy()
        assert np.isnan(got[:, n:]).all(), "samples beyond n must not be written"
        got = got[:, :n]
        for s in range(S):
            zero_rows = want[s] == 0
            assert np.all(got[s][zero_rows] == 0.0), (lens[s], np.flatnonzero(got[s][zero_rows]))
            err = np.abs(got[s] - want[s])[~zero_rows] / want[s][~zero_rows]
            assert np.all(err <= 8 * lens[s] * EPS), (lens[s], err.max())
    Tden = torch.full((S, ldt), np.nan, dtype=torch.float64, device=dev)
    _cabi.call("mbpls_masked_rowden_f64", ptr(bits), ldw, n, ptr(wd), ptr(f0d), ptr(f1d), S, ptr(Tden), ldt, ptr(one), st)
    torch.cuda.synchronize()
    assert torch.isnan(Tden).all(), "done = 1 must leave the output untouched"
