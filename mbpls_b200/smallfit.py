"""Whole NIPALS fits in one kernel launch (csrc/smallfit.cu): the launch-latency regime of the reference.  Dense fits, and for
cross-validation, permutation tests and bootstrap also fits with missing values (sparse_data=True, nanmode).

The reference's README quickstart (README.rst:82-95) and the leave-one-out loops of its notebooks
(``cross_val_predict(MBPLS(n_components=k), X, y, cv=len(X))``, examples/real_world_applications/*.ipynb) fit matrices of
a few hundred kilobytes.  Through the streaming kernels such a fit is ~150 launches plus a host readback per component;
here one persistent CTA per fit runs the whole loop of mbpls/mbpls.py:821-983 on the device, and a grid of CTAs runs all
folds of a cross-validation at once.  This module packs the inputs (one host->device copy), launches, and unpacks the
results (one device->host copy).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _cabi
from . import engine as E
from ._cabi import call
from .engine import F64, ptr, stream_ptr

# a fit runs in one CTA when its matrix has at most this many elements (1 MB of fp64): beyond it the single SM's L2
# bandwidth costs more than the launches it saves
SMALL_ELEMS = 1 << 17
# cross-validation: all folds at once when their private copies of the training data fit this many bytes; permutation
# tests and bootstrap (slot mode): the per-fit outputs of one launch
CV_WORKSPACE_BYTES = 4 << 30


def eligible(method: str, sparse: bool, group, n: int, p: int, force) -> bool:
    """force: the runtime option small_path (None = automatic by size; MBPLS_SMALL_PATH=0 in the environment turns the
    automatic choice off, which the test-suite uses to keep exercising the streaming kernels on small fixtures)."""
    if force is False or method != 'NIPALS' or sparse or group is not None or p < 1 or n < 1:
        return False
    if force is None and os.environ.get("MBPLS_SMALL_PATH", "1") == "0":
        return False
    return bool(force) or n * p <= SMALL_ELEMS


def batch_eligible(estimator, ntr_max: int, p: int) -> bool:
    """Slot-mode batches (permutation tests, bootstrap) of NIPALS fits, dense or NaN mode (sparse_data=True fits NIPALS
    whatever the method, as MBPLS.fit does): the workspace is bounded by the slots, so only the size of one fit decides
    (small_path None: automatic, False: never, True: always)."""
    rt = estimator._runtime()
    force = rt["small_path"]
    if force is False or (estimator.method != 'NIPALS' and not estimator.sparse_data) or rt["group"] is not None:
        return False
    if force is None:
        return os.environ.get("MBPLS_SMALL_PATH", "1") != "0" and ntr_max * p <= 8 * SMALL_ELEMS
    return True


def nan_fits_eligible(x_obs: np.ndarray, y_obs: np.ndarray, x_rows: Sequence, y_rows: Sequence,
                      block_cols: Optional[Sequence] = None, block_rows: Optional[Sequence] = None) -> np.ndarray:
    """Per fit, whether the NaN-mode batch runs it (True) or it goes to MBPLS.fit (False).

    x_obs (n, p) / y_obs (n, q): True where the source holds a value (not NaN); x_rows[f] / y_rows[f]: the X rows of fit f and
    the Y rows paired with them (repeats allowed).  block_cols[f] None, or a column range (lo, hi) of X that fit f reads on the
    rows block_rows[f] instead of x_rows[f] (a block-permuted fit).  A fit needs an observed value of every feature and every Y
    column on its rows, and a Y column observed on all of its Y rows to start the Y scores from (mbpls.py:832-836; without one
    the reference draws np.random.rand)."""
    def counts(obs, rows):  # (fits, columns): observed values on each fit's rows, with multiplicity
        n = obs.shape[0]
        lens = np.fromiter((len(r) for r in rows), dtype=np.int64, count=len(rows))
        flat = np.concatenate([np.asarray(r, dtype=np.int64) for r in rows]) if len(rows) else np.zeros(0, np.int64)
        mult = np.bincount(np.repeat(np.arange(len(rows)), lens) * n + flat, minlength=len(rows) * n).reshape(len(rows), n)
        return mult.astype(np.float64) @ obs.astype(np.float64), lens  # exact counts, through BLAS
    x_obs = np.asarray(x_obs, dtype=bool)
    xc, _ = counts(x_obs, x_rows)
    if block_cols is not None:
        groups = {}
        for f, c in enumerate(block_cols):
            if c is not None:
                groups.setdefault((int(c[0]), int(c[1])), []).append(f)
        for (lo, hi), fs in groups.items():
            xc[fs, lo:hi] = counts(x_obs[:, lo:hi], [block_rows[f] for f in fs])[0]
    yc, ylen = counts(np.asarray(y_obs, dtype=bool), y_rows)
    return (xc > 0).all(axis=1) & (yc > 0).all(axis=1) & (yc == ylen[:, None]).any(axis=1)


def observed(a) -> np.ndarray:
    """(n, m) host mask of the entries of a source array (numpy or torch) that are not NaN."""
    if isinstance(a, torch.Tensor):
        return (~torch.isnan(a)).cpu().numpy()
    return ~np.isnan(np.asarray(a, dtype=np.float64))


def slot_count(device, nfits: int) -> int:
    """Persistent CTAs of a slot-mode launch: one 1024-thread CTA per SM, no more than there are fits."""
    return max(1, min(nfits, torch.cuda.get_device_properties(device).multi_processor_count))


def unit_batches(n_units: int, fits_per_unit: int, bytes_per_fit: int) -> list:
    """[u0, u1) ranges of whole units (a permutation's folds, a resample) whose per-fit outputs fit CV_WORKSPACE_BYTES each:
    one range, i.e. one launch, unless the request is larger than that."""
    per = max(1, CV_WORKSPACE_BYTES // max(1, fits_per_unit * bytes_per_fit))
    return [(u, min(n_units, u + per)) for u in range(0, n_units, per)]


def pack_source(blocks: Sequence, Y, device):
    """Feature-major source matrix [X_1' ; ... ; X_B' ; Y'] ((p + q) x ldx, raw values) on the device in ONE copy, with the
    block offset table (B + 1 int32) behind it in the same buffer.  Host arrays are transposed into one pinned staging
    buffer; device tensors are concatenated on the device.  Returns (flat device buffer, n, sizes, p, q, ldx)."""
    n = int(blocks[0].shape[0])
    sizes = [int(b.shape[1]) for b in blocks]
    p, q = sum(sizes), int(Y.shape[1])
    ldx = (n + 1) // 2 * 2
    off = np.concatenate(([0], np.cumsum(sizes))).astype(np.int32)
    tail = (len(off) + 1) // 2  # doubles that hold the int32 table
    if all(isinstance(b, torch.Tensor) and b.is_cuda for b in blocks):
        Yd = Y if isinstance(Y, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(Y, dtype=np.float64))
        parts = [b.to(F64).t() for b in blocks] + [Yd.to(device=device, dtype=F64).t()]
        D = torch.zeros((p + q) * ldx + tail, dtype=F64, device=device)
        D[:(p + q) * ldx].view(p + q, ldx)[:, :n] = torch.cat(parts, dim=0)
        D[(p + q) * ldx:].view(torch.int32)[:len(off)] = torch.from_numpy(off).to(device)
        return D, n, sizes, p, q, ldx
    H = torch.empty((p + q) * ldx + tail, dtype=F64, pin_memory=True)
    Hn = H.numpy()
    M = Hn[:(p + q) * ldx].reshape(p + q, ldx)
    o = 0
    for b in blocks:
        a = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
        M[o:o + a.shape[1], :n] = a.T
        o += a.shape[1]
    Ya = Y.detach().cpu().numpy() if isinstance(Y, torch.Tensor) else np.asarray(Y)
    M[p:p + q, :n] = Ya.T
    if ldx > n:
        M[:, n:] = 0.0
    Hn[(p + q) * ldx:].view(np.int32)[:len(off)] = off
    return H.to(device, non_blocking=True), n, sizes, p, q, ldx


PER_FIT = ("small", "beta")  # sections indexed by fit in slot mode too; the others are indexed by slot


@dataclass
class Layout:
    """Offsets (in doubles) of the result sections inside the packed output buffer: one entry per fit, or in slot mode
    (nslots > 0) one per slot for every section but `small` and `beta` (no `beta` section without want_beta)."""
    nfits: int
    p: int
    q: int
    B: int
    K: int
    ldw: int
    nslots: int = 0
    want_beta: bool = True

    def __post_init__(self):
        p, q, B, K, ldw, F = self.p, self.q, self.B, self.K, self.ldw, self.nfits
        self.sizes = dict(stats=4 * p + 4 * q, Wt=K * p, W=K * p, P=K * p, Ts=K * ldw, U=K * ldw, Tb=B * K * ldw,
                          small=K * (q + 2 * B + 4) + B + 2, R=K * p, beta=q * p if self.want_beta else 0)
        self.off, o = {}, 0
        for name, sz in self.sizes.items():
            self.off[name] = o
            o += sz * (F if name in PER_FIT or not self.nslots else self.nslots)
        self.total = o

    def section(self, buf, name):
        """Every entry of a section, one row each."""
        n = self.nfits if name in PER_FIT or not self.nslots else self.nslots
        return buf[self.off[name]:self.off[name] + n * self.sizes[name]].reshape(n, self.sizes[name])

    def view(self, buf, name, f=0):
        sz = self.sizes[name]
        o = self.off[name] + f * sz
        return buf[o:o + sz]


def launch(D: torch.Tensor, n_src: int, p: int, q: int, ldx: int, block_off: Sequence[int], K: int, standardize: bool,
           norm_kind: int, max_tol: float, max_iter: int, train_sets: Optional[List[np.ndarray]],
           test_sets: Optional[List[np.ndarray]] = None, *, y_sets: Optional[List[np.ndarray]] = None, nslots: int = 0,
           fit_preds: bool = False, want_beta: bool = True, nanmode: bool = False, block_perm=None):
    """Run ``len(train_sets)`` fits concurrently (train_sets None: one fit on all samples).  ``D`` is pack_source's buffer.
    y_sets: per fit, the Y rows paired with its X rows train_sets[f] (None: the same rows).  nslots > 0: slot mode, that many
    persistent CTAs work through the fits, workspace per slot (nslots 0: one CTA and one workspace per fit).  fit_preds: the
    held-out predictions per fit, (nfits, K, max test size, q), instead of by sample (K, n_src, q; not in slot mode).
    want_beta False: no beta section (slot mode only).  nanmode: the NaN-mode fit of sparse_data=True (K <= 64); a fit the
    kernel cannot run (see nan_fits_eligible) comes back flagged like a singular one.  block_perm: (perm_table (R, n_src) row
    permutations, pairs (nfits, 2)): a fit with pairs[f] = (r, b), r >= 0, reads every X row i of block b (training and held-out
    rows) from row perm_table[r, i]; r = -1 permutes nothing (not with train_sets None).
    Returns (layout, packed device result buffer, predictions device tensor or None, buffers to keep alive)."""
    dev = D.device
    B = len(block_off) - 1
    if block_perm is not None and train_sets is None:
        raise ValueError("block_perm needs train_sets")
    boff_ptr = C.c_void_p(D.data_ptr() + 8 * (p + q) * ldx)  # the table pack_source put behind the matrix
    packed = None
    if train_sets is None:  # one fit on every sample of the source: no index tables at all
        F, ld_idx, ldw, ld_t = 1, n_src, (n_src + 1) // 2 * 2, 0
        iptr = lambda i: None
    else:
        F = len(train_sets)
        ld_idx = max(len(t) for t in train_sets)
        ldw = (ld_idx + 1) // 2 * 2

        def table(sets, ld):
            idx = np.zeros((F, ld), dtype=np.int32)
            cnt = np.zeros(F, dtype=np.int32)
            for f, t in enumerate(sets):
                idx[f, :len(t)] = t
                cnt[f] = len(t)
            return idx.ravel(), cnt

        ints = list(table(train_sets, ld_idx))
        ld_t = 0
        if test_sets is not None:
            ld_t = max(1, max(len(t) for t in test_sets))
            ints += table(test_sets, ld_t)
        if y_sets is not None:
            ints.append(table(y_sets, ld_idx)[0])
        if block_perm is not None:
            ints += [np.ascontiguousarray(block_perm[0], dtype=np.int32).ravel(),
                     np.ascontiguousarray(block_perm[1], dtype=np.int32).ravel()]
        if nslots:
            ints.append(np.zeros(1, dtype=np.int32))  # the ticket counter (zeroed again on the stream by the entry point)
        packed = torch.from_numpy(np.concatenate(ints)).to(dev, non_blocking=True)  # every index table in one copy
        offs = np.cumsum([0] + [len(a) for a in ints])
        iptr = lambda i: C.c_void_p(packed.data_ptr() + 4 * int(offs[i]))
    nt = 4 if test_sets is not None else 2  # tables before the Y rows, the block permutations and the ticket
    npm = nt + (y_sets is not None)  # the permutation table, then the (r, b) pairs
    S = nslots or F  # workspaces
    lay = Layout(F, p, q, B, K, ldw, nslots, want_beta)
    out = torch.empty(lay.total, dtype=F64, device=dev)
    work = torch.empty(S * (p + q) * ldw, dtype=F64, device=dev)
    sstride = call("mbpls_smallfit_nan_scratch_doubles", p, q, B, K, ldw) if nanmode else \
        call("mbpls_smallfit_scratch_doubles", p, B, ldw)
    scratch = torch.empty(S * sstride, dtype=F64, device=dev)
    preds = None
    if test_sets is not None:
        shape = (F, K, ld_t, q) if fit_preds else (K, n_src, q)
        preds = torch.full(shape, float("nan"), dtype=F64, device=dev)
    base = out.data_ptr()
    sec = lambda name: C.c_void_p(base + 8 * lay.off[name])
    args = _cabi.SmallFitArgs(
        n_src=n_src, p=p, B=B, q=q, K=K, nfits=F, ldx=ldx, Xsrc=D.data_ptr(), Ysrc=D.data_ptr() + 8 * p * ldx, block_off=boff_ptr,
        standardize=1 if standardize else 0, norm_kind=norm_kind, max_iter=int(min(max_iter, 2**31 - 1)), max_tol=float(max_tol),
        train_idx=iptr(0), train_cnt=iptr(1), ld_idx=ld_idx,
        test_idx=iptr(2) if test_sets is not None else None, test_cnt=iptr(3) if test_sets is not None else None, ld_tidx=ld_t,
        ldw=ldw, Xw=work.data_ptr(), Yw=work.data_ptr() + 8 * S * p * ldw, stats=sec("stats"), Wt=sec("Wt"), W=sec("W"), P=sec("P"),
        Ts=sec("Ts"), U=sec("U"), Tb=sec("Tb"), small=sec("small"), R=sec("R"), beta=sec("beta") if want_beta else None,
        preds=preds.data_ptr() if preds is not None and not fit_preds else None, scratch=scratch.data_ptr(), scratch_stride=sstride,
        ytrain_idx=iptr(nt) if y_sets is not None else None, fit_preds=preds.data_ptr() if fit_preds and preds is not None else None,
        nslots=int(nslots), ticket=iptr(len(ints) - 1) if nslots else None, nanmode=1 if nanmode else 0,
        perm_rows=iptr(npm) if block_perm is not None else None,
        n_perm=int(np.shape(block_perm[0])[0]) if block_perm is not None else 0,
        fit_perm=iptr(npm + 1) if block_perm is not None else None)
    call("mbpls_smallfit_nipals_f64", C.byref(args), stream_ptr(dev))
    return lay, out, preds, (packed, work, scratch)


def unpack_small(small: np.ndarray, K: int, q: int, B: int):
    """Sections of the per-fit `small` block (see include/mbpls_b200.h)."""
    o = 0
    def take(sz):
        nonlocal o
        v = small[o:o + sz]
        o += sz
        return v
    return dict(V=take(K * q).reshape(K, q), A=take(K * B).reshape(K, B), pssb=take(K * B).reshape(K, B), tt=take(K), vv=take(K),
                diff=take(K), trips=take(K), varxb=take(B), vary=float(take(1)[0]), singular=bool(take(1)[0] != 0.0))
