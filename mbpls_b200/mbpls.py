"""Drop-in for ``mbpls.mbpls.MBPLS`` (reference: mbpls/mbpls.py:22-1437) whose fit / predict /
transform bodies run on a B200 through the hand-written sm_100a kernels of ``csrc/``.

The surface is the reference's: same constructor signature and defaults (mbpls.py:243-253), same
methods (fit :273, transform :1052, predict :1337, fit_transform :1412, fit_predict :1418, r2_score
:1424, explained_variance_score :1431, inherited score/get_params/set_params), same fitted
attributes with the same shapes and list-vs-array conventions (SURVEY.md section 8a contract table),
same warnings and exception types.  Inputs may be numpy arrays / array-likes (as in the reference) or
torch tensors, including CUDA tensors that are already column-major (feature-major), which are
consumed without a layout change.

Extras that are *not* in the reference (none of them constructor parameters, so ``sklearn.clone``
and ``get_params`` behave identically): ``n_iter_`` (NIPALS trips per component), ``set_runtime``.
"""
from __future__ import annotations

import warnings
import weakref
from typing import List, Optional

import numpy as np
import torch
from sklearn import metrics
from sklearn.base import BaseEstimator, MultiOutputMixin, RegressorMixin, TransformerMixin
from sklearn.exceptions import NotFittedError
from sklearn.preprocessing import StandardScaler

from . import _cabi
from . import engine as E
from .engine import F64, ShardMap, call, ptr, stream_ptr

__all__ = ["MBPLS"]

_SPARSITY_MSG = ("The sparsity of your data is likely to high for this algorithm. This can cause either convergence"
                 "problems or crash the algorithm.")

_LAZY_NAMES = ("Ts_", "U_", "V_", "T_", "W_", "W_non_normal_", "W_concat_", "P_", "R_", "beta_", "x_scalers_", "y_scaler_")

_RUNTIME_DEFAULTS = dict(
    device=None,          # torch device (default: current CUDA device)
    group=None,           # torch.distributed process group: shard the feature axis over its ranks
    materialize=True,     # copy fitted attributes to numpy at the end of fit (False: on first access)
    fuse_next_xtu=True,   # loadings+deflation pass also emits the next component's first weights
    fuse_first_trip=False,  # dense NIPALS: the standardisation pass also runs the first component's first trip (csrc/fused.cu).
                          # Opt-in: saves 6 ms of the 835 ms headline fit, but its statistics are summed in another order than
                          # the standalone pass, which moves noise-floor exits of deep PLS1 components by a trip
    deflate_mode=0,       # 0 auto (smem-resident pipeline), 1 force global-memory fallback
    standardize_mode=0,   # idem for the standardisation pass
    trips_per_sync=None,  # NIPALS trips enqueued per convergence-flag readback (None: auto)
    max_iter=1_000_000,   # safety cap on NIPALS trips; the reference loop is unbounded (mbpls.py:841)
    global_sizes=None,    # multi-GPU: the blocks passed in are this rank's column ranges of blocks of these sizes
    profile=None,         # dict collecting CUDA-event pairs per kernel (bench.py roofline)
    deflate_last=False,   # also deflate X after the last component (the reference does; the result is never read)
    one_pass=None,        # NIPALS trip as ONE read of X (csrc/fused.cu): None auto (n <= 20480), False two-pass kernels
    one_pass_deflate=None,  # loadings+deflation also runs the next component's whole first trip (None auto, False off)
    small_path=None,      # dense single-GPU NIPALS: the whole fit as ONE kernel launch (csrc/smallfit.cu).  None: when the matrix has
                          # at most smallfit.SMALL_ELEMS elements; True / False force it on / off
    unipals_route=None,   # UNIPALS with n >= p: "gram" = everything in p-space from X'X / X'Y (crossmethods._fit_unipals_gram),
                          # "stream" = the reference's per-component passes over X; None: whichever a cost model says is cheaper
    timings=None,         # dict: wall-clock seconds per phase of fit (ingest / standardize / solve / materialize), measured with a
                          # device synchronisation at every phase boundary (diagnostics; bench.py --verbose)
    gather=None,          # multi-GPU, per-feature attributes (W_, P_, R_, beta_, x_scalers_): "all" = every rank materialises the
                          # full p x K arrays (all-gather), "local" = every rank its own rows, sharded like the input it passed.
                          # None: "local" when the input was pre-sharded (global_sizes), else "all"
)


# Small dense steps (pinv(P'W), the q x q eigen-problems, the superlevel epilogue) run in single-CTA device kernels whose
# shared-memory tiles are sized for 64 (csrc/smalllin.cu SL_MAX, csrc/nipals.cu EPI_MAXB / EPI_MAXQ).  The reference has no such
# limits; they are checked before any data is uploaded or modified.
MAX_COMPONENTS = MAX_RESPONSES = MAX_BLOCKS = 64


def _check_limits(n_components, q: int, B: int) -> int:
    try:
        K = int(n_components)
    except (TypeError, ValueError) as exc:
        raise ValueError(f"n_components must be an integer, got {n_components!r}") from exc
    if K < 1:
        raise ValueError(f"n_components must be >= 1, got {K}")
    for what, val, cap in (("n_components", K, MAX_COMPONENTS), ("Y columns", q, MAX_RESPONSES), ("X blocks", B, MAX_BLOCKS)):
        if val > cap:
            raise NotImplementedError(f"mbpls_b200 supports at most {cap} {what} (got {val}): the K x K / q x q / B-wide "
                                      "steps of the fit run in fixed-size single-CTA kernels")
    return K


def _is_block_list(X) -> bool:
    return isinstance(X, list) and not isinstance(X[0], list)  # mbpls.py:301


def _shape2(a):
    if isinstance(a, torch.Tensor):
        return tuple(a.shape)
    return tuple(np.shape(a))


def _as_2d_source(a, what: str, allow_empty: bool = False):
    """Array-like -> numpy float64 view / torch tensor with 2 dims (no copy when already float64)."""
    if isinstance(a, torch.Tensor):
        t = a
    else:
        t = np.asarray(a)  # pandas DataFrames included (a view when the frame is one float block)
        if t.dtype not in (np.float64, np.float32):  # float32 is widened on the device, after the upload (engine.ingest_feature_major)
            try:
                t = t.astype(np.float64)
            except (TypeError, ValueError) as exc:
                raise ValueError(f"could not convert {what} to float64") from exc
    if t.ndim != 2:
        raise ValueError(f"Expected 2D array, got {t.ndim}D array instead ({what}).")
    if t.shape[0] < 1 or (t.shape[1] < 1 and not allow_empty):
        raise ValueError(f"Found array with {t.shape[0]} sample(s) and {t.shape[1]} feature(s) while a minimum of 1 is required.")
    return t


class MBPLS(TransformerMixin, RegressorMixin, MultiOutputMixin, BaseEstimator):
    """(Multiblock) PLS regression on a B200; see the module docstring and the reference docstring
    (mbpls/mbpls.py:23-241) for parameter and attribute semantics."""

    def __init__(self, n_components=2, full_svd=False, method='NIPALS', standardize=True, max_tol=1e-14,
                 nipals_convergence_norm=2, calc_all=True, sparse_data=False, copy=True):
        self.n_components = n_components
        self.full_svd = full_svd
        self.method = method
        self.standardize = standardize
        self.max_tol = max_tol
        self.nipals_convergence_norm = nipals_convergence_norm
        self.calc_all = calc_all
        self.sparse_data = sparse_data
        self.copy = copy

    # ------------------------------------------------------------------ runtime plumbing
    def set_runtime(self, **kw) -> "MBPLS":
        rt = self._runtime()
        for k, v in kw.items():
            if k not in _RUNTIME_DEFAULTS:
                raise TypeError(f"unknown runtime option {k!r}")
            rt[k] = v
        return self

    def _runtime(self) -> dict:
        rt = self.__dict__.get("_rt")
        if rt is None:
            rt = dict(_RUNTIME_DEFAULTS)
            self.__dict__["_rt"] = rt
        return rt

    def __getstate__(self):
        self._materialize_all()
        state = dict(self.__dict__)
        for k in ("_rt", "_dev", "_lazy", "_dev_scalers", "_cv_weights", "_rows", "_col_nan", "_exchange"):
            state.pop(k, None)
        return state

    def __getattr__(self, name):
        # only called when normal lookup fails: lazily materialised fitted attributes
        lazy = self.__dict__.get("_lazy")
        if lazy and name in lazy:
            self._materialize_all()
            return self.__dict__[name]
        raise AttributeError(f"{type(self).__name__!r} object has no attribute {name!r}")

    def _materialize_all(self):
        lazy = self.__dict__.get("_lazy")
        if lazy:
            self.__dict__["_lazy"] = None
            for name, fn in lazy.items():
                self.__dict__[name] = fn()

    def _group_info(self):
        group = self._runtime()["group"]
        if group is None:
            return None, 0, 1
        import torch.distributed as dist
        return group, dist.get_rank(group), dist.get_world_size(group)

    def _gather_mode(self) -> str:
        rt = self._runtime()
        mode = rt["gather"]
        if mode is None:
            mode = "local" if rt["global_sizes"] is not None else "all"
        if mode not in ("all", "local"):
            raise ValueError("runtime option gather must be 'all', 'local' or None")
        return mode

    def _gather_features_dev(self, t_local: torch.Tensor, shard: ShardMap, force_all: bool = False) -> torch.Tensor:
        """K x p_local device tensor -> K x p_global device tensor (same on every rank); in "local" gather mode the
        rank's own K x p_local rows (no collective: a rank that passed its column ranges gets their attributes back)."""
        group, rank, world = self._group_info()
        if world == 1 or shard.world == 1:  # single GPU, or feature axis replicated (row-sharded fit)
            return t_local[:, :shard.p_local]
        if not force_all and self._gather_mode() == "local":
            return t_local[:, :shard.p_local]
        import torch.distributed as dist
        per = -(-shard.p_global // world)
        K = t_local.shape[0]
        pad = torch.zeros((K, per), dtype=t_local.dtype, device=t_local.device)
        pad[:, :shard.p_local] = t_local[:, :shard.p_local]
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad, group=group)
        return torch.cat(parts, dim=1)[:, :shard.p_global]

    def _gather_features(self, t_local: torch.Tensor, shard: ShardMap, force_all: bool = False) -> np.ndarray:
        """K x p_local device tensor -> K x p_global (or, "local" gather mode, K x p_local) numpy array."""
        return E.to_host(self._gather_features_dev(t_local, shard, force_all))

    def _local_attrs(self, shard: ShardMap) -> bool:
        """True when per-feature attributes hold this rank's rows only ("local" gather mode of a feature-sharded fit)."""
        _, _, world = self._group_info()
        return world > 1 and shard.world > 1 and self._gather_mode() == "local"

    def _feature_bounds(self, shard: ShardMap):
        """Column boundaries of the blocks inside a gathered (global) or local per-feature result."""
        if self._local_attrs(shard):
            return np.asarray(shard.block_off)
        return np.concatenate(([0], np.cumsum(shard.sizes)))

    def _features_T(self, t_local: torch.Tensor, shard: ShardMap, split: bool):
        """Component-major K x p_local device result -> the reference's layout: one p x K numpy array, or (split) the list
        of per-block p_b x K arrays (p = all features, or this rank's in "local" gather mode).  The transposition runs on the
        device and the copies land in pinned memory (engine.to_host)."""
        full = self._gather_features_dev(t_local, shard)
        if not split:
            return E.to_host(full, transpose=True)
        bounds = self._feature_bounds(shard)
        return [E.to_host(full[:, int(bounds[b]):int(bounds[b + 1])], transpose=True) for b in range(len(shard.sizes))]

    def _gather_samples(self, t: torch.Tensor, n_local: int) -> np.ndarray:
        """K x ld device tensor of per-sample results -> n x K numpy array; concatenates the row shards when the
        sample axis is sharded (row-sharded KERNEL fit), plain copy otherwise."""
        rows = self.__dict__.get("_rows")
        if rows is None:
            return E.to_host(t[:, :n_local], transpose=True)
        import torch.distributed as dist
        group, counts = rows
        K, mx = t.shape[0], max(counts)
        pad = torch.zeros((K, mx), dtype=t.dtype, device=t.device)
        pad[:, :n_local] = t[:, :n_local]
        parts = [torch.empty_like(pad) for _ in counts]
        dist.all_gather(parts, pad, group=group)
        full = torch.cat([pt[:, :c] for pt, c in zip(parts, counts)], dim=1)
        return E.to_host(full, transpose=True)

    # ------------------------------------------------------------------ NaN census (mbpls.py:255-271)
    def check_sparsity_level(self, data):
        """Reference-compatible census of one array (mbpls.py:255-271), computed by the device census kernel."""
        device = E.require_cuda(self._runtime()["device"])
        src = _as_2d_source(data, "data")
        n, p = int(src.shape[0]), int(src.shape[1])
        with torch.cuda.device(device):
            Xt = E.alloc_feature_major(p, n, device)
            E.ingest_feature_major(src, n, 0, p, Xt, device)
            col_nan, row_flag, _ = E.nan_census(Xt, n, E._i32([0, p], device), 1)
            return self._census_from_flags(row_flag[0, :n].cpu().numpy().astype(bool), (col_nan > 0).cpu().numpy())

    @staticmethod
    def _census_from_flags(row_has: np.ndarray, col_has: np.ndarray):
        if col_has.sum() / col_has.size > 0.5:
            warnings.warn(_SPARSITY_MSG)
        if row_has.sum() / row_has.size > 0.5:
            warnings.warn(_SPARSITY_MSG)
        return (np.where(row_has)[0], np.where(col_has)[0], np.where(~row_has)[0], np.where(~col_has)[0])

    # ------------------------------------------------------------------ ingest shared by fit / predict / transform
    def _ingest(self, X, n_expected: Optional[int], shard: Optional[ShardMap], device, what="X", adopt=False,
                adopt_writable=True):
        gs = self._runtime()["global_sizes"]
        blocks = X if _is_block_list(X) else [X]
        blocks = [_as_2d_source(b, what, allow_empty=gs is not None) for b in blocks]
        n = blocks[0].shape[0]
        want = n if n_expected is None else int(n_expected)
        for b in blocks:
            if int(b.shape[0]) != want:  # check_consistent_length, mbpls.py:309,322
                raise ValueError("Found input variables with inconsistent numbers of samples: %r"
                                 % [int(b.shape[0]), want])
        sizes = [int(b.shape[1]) for b in blocks]
        _, rank, world = self._group_info()
        if gs is not None:  # pre-sharded input
            want_shard = ShardMap.build(gs, rank, world)
            local = [c1 - c0 for c0, c1 in want_shard.local_ranges]
            if sizes != local:
                raise ValueError("pre-sharded blocks have widths %r, expected %r" % (sizes, local))
            if shard is not None and list(shard.sizes) != list(gs):
                raise ValueError("X has %r features per block, but MBPLS was fitted with %r" % (list(gs), list(shard.sizes)))
            shard = want_shard
        elif shard is None:
            shard = ShardMap.build(sizes, rank, world)
        elif list(shard.sizes) != sizes:
            raise ValueError("X has %r features per block, but MBPLS was fitted with %r" % (sizes, list(shard.sizes)))
        Xt = E.ingest_blocks(blocks, n, shard, device, presharded=gs is not None, adopt=adopt, adopt_writable=adopt_writable)
        return Xt, n, shard

    # ------------------------------------------------------------------ fit (mbpls.py:273-1050)
    def fit(self, X, Y):
        if self.sparse_data is True and self.method != 'NIPALS':  # mbpls.py:286-290
            warnings.warn("The parameter sparse data was set to 'True', but the chosen method is not 'NIPALS'."
                          "The method will be set to 'NIPALS'")
            self.method = 'NIPALS'
        if self.method not in ('NIPALS', 'UNIPALS', 'KERNEL', 'SIMPLS'):
            raise NameError('Method you called is unknown')  # mbpls.py:1050
        rt = self._runtime()
        device = E.require_cuda(rt["device"])
        group, rank, world = self._group_info()
        sparse = bool(self.sparse_data)
        self.__dict__["_lazy"] = None
        self.__dict__["_dev"] = None
        self.__dict__["_dev_scalers"] = None
        self.__dict__["_rows"] = None
        self.__dict__["_attrs_local_sizes"] = None
        for name in _LAZY_NAMES:  # results of an earlier fit must not shadow the lazily materialised ones of this fit
            self.__dict__.pop(name, None)

        # (explicit choices among the streaming kernels keep the fit on them)
        tuned = any(rt[k] != _RUNTIME_DEFAULTS[k] for k in ("one_pass", "one_pass_deflate", "deflate_mode", "standardize_mode",
                                                            "fuse_next_xtu", "fuse_first_trip", "trips_per_sync", "deflate_last"))
        if self.method == 'NIPALS' and not sparse and group is None and rt["global_sizes"] is None and rt["small_path"] is not False \
                and rt["profile"] is None and (rt["small_path"] is True or not tuned):
            with torch.cuda.device(device):
                if self._try_fit_small(X, Y, device):
                    if rt["materialize"]:
                        self._materialize_all()
                    return self

        if self.method in ('KERNEL', 'UNIPALS') and world > 1:
            blocks0 = X if _is_block_list(X) else [X]
            n0, p0 = int(_shape2(blocks0[0])[0]), sum(int(_shape2(b)[1]) for b in blocks0)
            if n0 >= p0 and rt["global_sizes"] is None:
                with torch.cuda.device(device):
                    self._fit_kernel_row_sharded(X, Y, group, rank, world, device)
                if rt["materialize"]:
                    self._materialize_all()
                return self

        import time as _time
        tm = rt["timings"]

        def mark(name, _t=[_time.perf_counter()]):
            if tm is not None:
                torch.cuda.synchronize(device)
                now = _time.perf_counter()
                tm[name] = tm.get(name, 0.0) + now - _t[0]
                _t[0] = now

        with torch.cuda.device(device):
            # ---- Y (mbpls.py:293-298)
            Ysrc = Y if isinstance(Y, torch.Tensor) else np.asarray(Y)
            if Ysrc.ndim == 1:
                Ysrc = Ysrc.reshape(-1, 1)
            Ysrc = _as_2d_source(Ysrc, "Y")
            n, q = int(Ysrc.shape[0]), int(Ysrc.shape[1])
            _check_limits(self.n_components, q, len(X) if _is_block_list(X) else 1)
            # ---- X blocks (mbpls.py:299-347)
            Xt, n_x, shard = self._ingest(X, n, None, device, adopt=not self.copy)
            B = len(shard.sizes)
            ld = Xt.shape[1]
            self.__dict__["_attrs_local_sizes"] = tuple(shard.sizes) if self._local_attrs(shard) else None
            Yt = E.alloc_feature_major(q, n, device)
            E.ingest_feature_major(Ysrc, n, 0, q, Yt, device)
            boff_dev = E._i32(shard.block_off, device)
            mark("ingest")

            row_flag = ycol_flag = None
            if sparse:
                row_flag, ycol_flag = self._fit_census(Xt, Yt, n, q, shard, boff_dev, group)
            elif not self.standardize:
                self._require_finite(Xt, Yt, n)

            # ---- standardisation (mbpls.py:299-326)
            zss = None
            pre_lazy = None
            first_trip = None
            if self.standardize:
                prof = rt["profile"]
                ys = E.standardize_fit(Yt, n, rt["standardize_mode"])
                if prof is not None:
                    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                    ev[0].record(torch.cuda.current_stream(device))
                xs = None
                if self.method == 'NIPALS' and not sparse and rt["one_pass"] is not False and rt["standardize_mode"] == 0 \
                        and rt["fuse_first_trip"] and rt["one_pass_deflate"] is not False and rt["deflate_mode"] == 0:
                    # dense NIPALS: the standardisation pass also runs the first trip of the first component (u = Y[:, 0])
                    fused = E.standardize_fit_first_trip(Xt, n, shard.block_off, Yt[0])
                    if fused is not None:
                        xs, first_trip = fused
                if xs is None:
                    xs = E.standardize_fit(Xt, n, rt["standardize_mode"])
                if prof is not None:
                    ev[1].record(torch.cuda.current_stream(device))
                    prof.setdefault("standardize", []).append(ev)
                if not sparse:
                    # NaN shows up as seen < n, +-inf as a non-finite column mean / variance: no extra pass over X
                    # (one flag on the device, one read-back -- or none: between GPUs the flag itself is all-reduced)
                    pl = shard.p_local
                    ok = (xs.seen[:pl] == n).all() & torch.isfinite(xs.mean[:pl]).all() & torch.isfinite(xs.var[:pl]).all() \
                        & (ys.seen[:q] == n).all() & torch.isfinite(ys.mean[:q]).all() & torch.isfinite(ys.var[:q]).all()
                    self._raise_if_any_rank(~ok, "Input contains NaN or infinity.", group)
                pre_lazy = self._lazy_scalers(xs, ys, shard, q)
                zss = xs.zss
                self.__dict__["_dev_scalers"] = (xs.mean[:shard.p_local], xs.scale[:shard.p_local], ys.mean[:q], ys.scale[:q])
            self.num_blocks_ = B
            mark("standardize")

            if self.method == 'NIPALS':
                self._fit_nipals(Xt, Yt, n, q, shard, boff_dev, zss, row_flag, ycol_flag, group, device, first_trip)
            else:
                from . import crossmethods
                crossmethods.fit(self, Xt, Yt, n, q, shard, boff_dev, zss, group, device)
            if pre_lazy:
                self.__dict__["_lazy"].update(pre_lazy)
            mark("solve")
        if rt["materialize"]:
            self._materialize_all()
            mark("materialize")
        return self

    # ---- KERNEL / UNIPALS with n >= p on several GPUs: shard the SAMPLE axis (SURVEY.md 8e)
    def _fit_kernel_row_sharded(self, X, Y, group, rank, world, device):
        """Every rank ingests its contiguous range of samples of all blocks; column statistics and the sums over samples
        (KERNEL: the p x p / p x q cross-products, once; UNIPALS: X'Y, X'ts and Y'ts per component) are all-reduced;
        everything indexed by features runs replicated; scores stay row-local."""
        from . import crossmethods as CM
        blocks = X if _is_block_list(X) else [X]
        blocks = [_as_2d_source(b, "X") for b in blocks]
        Ysrc = Y if isinstance(Y, torch.Tensor) else np.asarray(Y)
        if Ysrc.ndim == 1:
            Ysrc = Ysrc.reshape(-1, 1)
        Ysrc = _as_2d_source(Ysrc, "Y")
        n, q = int(Ysrc.shape[0]), int(Ysrc.shape[1])
        _check_limits(self.n_components, q, len(blocks))
        for b in blocks:
            if int(b.shape[0]) != n:
                raise ValueError("Found input variables with inconsistent numbers of samples: %r" % [int(b.shape[0]), n])
        per = -(-n // world)
        counts = [max(0, min(n, (r + 1) * per) - min(n, r * per)) for r in range(world)]
        r0 = min(n, rank * per)
        nl = counts[rank]
        if min(counts) < 1:
            raise ValueError("fewer samples than GPUs")
        sizes = [int(b.shape[1]) for b in blocks]
        shard = ShardMap.build(sizes, 0, 1)  # the feature axis is replicated
        Xt = E.ingest_blocks([b[r0:r0 + nl] for b in blocks], nl, shard, device)
        Yt = E.alloc_feature_major(q, nl, device)
        E.ingest_feature_major(Ysrc[r0:r0 + nl], nl, 0, q, Yt, device)
        B, p, ld = len(sizes), shard.p_local, Xt.shape[1]
        boff_dev = E._i32(shard.block_off, device)
        self.__dict__["_rows"] = (group, counts)
        ones = torch.zeros(ld, dtype=F64, device=device)
        ones[:nl] = 1.0

        def standardize_rows(Mt, feats, one_off):
            """StandardScaler.fit_transform with the sums over samples all-reduced (two-pass, like sklearn)."""
            tot = CM.xt_vec(Mt, nl, ones, one_off, 1).clone()
            E.allreduce_(tot, group)
            cnt = torch.full((1,), float(n), dtype=F64, device=device)
            mean = tot.clone()
            CM.scale_rows_(mean.view(1, -1), feats, cnt, True)
            CM.rank1_update_(Mt, nl, ones, mean)  # x <- x - mean
            corr = CM.xt_vec(Mt, nl, ones, one_off, 1).clone()
            ssq = E.feature_sumsq(Mt, nl)[:feats].clone()
            E.allreduce_(corr, group)
            E.allreduce_(ssq, group)
            var, scale = torch.empty_like(mean), torch.empty_like(mean)
            call("mbpls_scaler_finish_f64", ptr(corr), ptr(ssq), ptr(mean), float(n), ptr(var), ptr(scale), feats,
                 stream_ptr(device))
            E.standardize_apply(Mt, nl, torch.zeros_like(mean), scale)
            return mean, var, scale

        zss = None
        ok = E.all_finite(Xt, nl) and E.all_finite(Yt, nl)
        self._raise_if_any_rank(not ok, "Input contains NaN or infinity.", group)
        if self.standardize:
            xm, xv, xs = standardize_rows(Xt, p, E._i32([0, p], device))
            ym, yv, ys = standardize_rows(Yt, q, E._i32([0, q], device))
            seen = np.full(p, n, dtype=np.int64)
            xm_h, xv_h, xs_h = xm.cpu().numpy(), xv.cpu().numpy(), xs.cpu().numpy()
            self.x_scalers_, g0 = [], 0
            for pb in sizes:
                self.x_scalers_.append(_make_scaler(xm_h[g0:g0 + pb], xv_h[g0:g0 + pb], xs_h[g0:g0 + pb], seen[g0:g0 + pb]))
                g0 += pb
            self.y_scaler_ = _make_scaler(ym.cpu().numpy(), yv.cpu().numpy(), ys.cpu().numpy(), np.full(q, n, dtype=np.int64))
            self.__dict__["_dev_scalers"] = (xm, xs, ym, ys)
        self.num_blocks_ = B
        fit_rows = CM._fit_kernel if self.method == 'KERNEL' else CM._fit_unipals
        fit_rows(self, Xt, Yt, nl, q, shard, boff_dev, zss, None, device, rows_group=group, n_global=n)

    # ---- small problems: the whole NIPALS fit in one kernel launch (csrc/smallfit.cu)
    def _try_fit_small(self, X, Y, device) -> bool:
        """Dense NIPALS on a matrix of at most smallfit.SMALL_ELEMS elements (README quickstart, CV folds): one packed
        host->device copy, ONE kernel that runs mbpls.py:303-326 and :821-989 with the while loop on the device, one packed
        device->host copy.  Returns False (nothing done) when the problem is not eligible."""
        from . import smallfit as SF
        rt = self._runtime()
        blocks = X if _is_block_list(X) else [X]
        shapes = [_shape2(b) for b in blocks]
        if any(len(sh) != 2 for sh in shapes):
            return False  # let the general path raise the reference's error
        n, p = int(shapes[0][0]), sum(int(sh[1]) for sh in shapes)
        if not SF.eligible(self.method, bool(self.sparse_data), rt["group"], n, p, rt["small_path"]):
            return False
        Ysrc = Y if isinstance(Y, torch.Tensor) else np.asarray(Y)
        if Ysrc.ndim == 1:
            Ysrc = Ysrc.reshape(-1, 1)
        Ysrc = _as_2d_source(Ysrc, "Y")
        blocks = [_as_2d_source(b, "X") for b in blocks]
        q = int(Ysrc.shape[1])
        for b in blocks:
            if int(b.shape[0]) != int(Ysrc.shape[0]):  # check_consistent_length, mbpls.py:309,322
                raise ValueError("Found input variables with inconsistent numbers of samples: %r" % [int(b.shape[0]), int(Ysrc.shape[0])])
        B = len(blocks)
        K = _check_limits(self.n_components, q, B)
        for a in blocks + [Ysrc]:  # check_array(force_all_finite=True), :293,:310
            ok = bool(torch.isfinite(a).all()) if isinstance(a, torch.Tensor) else bool(np.isfinite(a).all())
            if not ok:
                raise ValueError("Input contains NaN or infinity.")
        D, n, sizes, p, q, ldx = SF.pack_source(blocks, Ysrc, device)
        shard = ShardMap.build(sizes, 0, 1)
        lay, out, _, keep = SF.launch(D, n, p, q, ldx, shard.block_off, K, bool(self.standardize),
                                      E.norm_kind_of(self.nipals_convergence_norm), self.max_tol, rt["max_iter"], None)
        host = E.to_host(out)  # one copy: every result of the fit
        ldw = lay.ldw
        sm = SF.unpack_small(lay.view(host, "small"), K, q, B)
        trips = [int(t) for t in sm["trips"]]
        self.n_iter_ = trips
        if any(t >= rt["max_iter"] for t in trips):
            warnings.warn("NIPALS hit the max_iter safety cap before diff_t <= max_tol")
        dv = lambda name, *shape: lay.view(out, name).view(*shape)   # device views (kept for predict / transform / CV)
        hv = lambda name, *shape: lay.view(host, name).reshape(*shape)
        Wt_d, W_d, P_d, V_d = dv("Wt", K, p), dv("W", K, p), dv("P", K, p), lay.view(out, "small")[:K * q].view(K, q)
        if sm["singular"]:  # more components than the data has rank: R = W pinv(P'W) exactly like the reference (:988)
            colnorm = torch.sqrt(E.rows_sumsq(Wt_d, p))
            M = E.small_pinv(E.gram(P_d, Wt_d, p) / colnorm.view(1, -1))
            R_d = E.right_multiply(Wt_d, p, 1.0 / colnorm, M)
            beta_d = E.right_multiply(R_d, p, None, V_d.contiguous())
            R_h, beta_h = E.to_host(R_d, transpose=True), E.to_host(beta_d, transpose=True)
        else:
            R_d, beta_d = dv("R", K, p), dv("beta", q, p)
            R_h, beta_h = np.ascontiguousarray(hv("R", K, p).T), np.ascontiguousarray(hv("beta", q, p).T)
        self.num_blocks_ = B
        self.__dict__["_exchange"] = None
        self.__dict__["_dev"] = dict(shard=shard, R=R_d, beta=beta_d, W=W_d, P=P_d, V=V_d, _keep=(out, keep))
        self.__dict__["_cv_weights"] = Wt_d
        st_d, st_h = lay.view(out, "stats"), lay.view(host, "stats")
        lazy = {}
        if self.standardize:
            self.__dict__["_dev_scalers"] = (st_d[0:p], st_d[2 * p:3 * p], st_d[4 * p:4 * p + q], st_d[4 * p + 2 * q:4 * p + 3 * q])
            off_ = shard.block_off
            seen = np.full(p, n, dtype=np.int64)
            # scikit-learn scaler objects on first access (constructing B + 1 estimators is a tenth of this path's time)
            lazy["x_scalers_"] = lambda: [_make_scaler(st_h[off_[b]:off_[b + 1]], st_h[p + off_[b]:p + off_[b + 1]],
                                                       st_h[2 * p + off_[b]:2 * p + off_[b + 1]], seen[off_[b]:off_[b + 1]])
                                          for b in range(B)]
            lazy["y_scaler_"] = lambda: _make_scaler(st_h[4 * p:4 * p + q], st_h[4 * p + q:4 * p + 2 * q],
                                                     st_h[4 * p + 2 * q:4 * p + 3 * q], np.full(q, n, dtype=np.int64))
        for name, v in _small_attributes(sm, shard.sizes, self.calc_all).items():
            setattr(self, name, v)
        self.W_concat_ = np.empty((p, 0))
        off = shard.block_off
        split = lambda M_: [np.ascontiguousarray(M_[:, off[b]:off[b + 1]].T) for b in range(B)]
        Tb = hv("Tb", B, K, ldw)
        self.Ts_ = np.ascontiguousarray(hv("Ts", K, ldw)[:, :n].T)
        self.U_ = np.ascontiguousarray(hv("U", K, ldw)[:, :n].T)
        self.V_ = np.ascontiguousarray(sm["V"].T)
        self.T_ = [np.ascontiguousarray(Tb[b][:, :n].T) for b in range(B)]
        self.W_, self.W_non_normal_, self.P_ = split(hv("W", K, p)), split(hv("Wt", K, p)), split(hv("P", K, p))
        self.R_, self.beta_ = R_h, beta_h
        self.__dict__["_lazy"] = lazy or None
        return True

    # ---- helpers of fit
    def _raise_if_any_rank(self, bad, msg: str, group):
        """bad: a Python bool or a 0-d boolean tensor on the device (then there is a single read-back)."""
        if group is not None:
            import torch.distributed as dist
            if isinstance(bad, torch.Tensor):
                flag = bad.to(torch.int32).reshape(1)
            else:
                flag = torch.tensor([1 if bad else 0], dtype=torch.int32, device=torch.device("cuda", torch.cuda.current_device()))
            dist.all_reduce(flag, group=group)
            bad = bool(flag.item())
        if bool(bad):
            raise ValueError(msg)

    def _require_finite(self, Xt, Yt, n):
        ok = E.all_finite(Xt, n) and E.all_finite(Yt, n)
        self._raise_if_any_rank(not ok, "Input contains NaN or infinity.", self._runtime()["group"])

    def _fit_census(self, Xt, Yt, n, q, shard, boff_dev, group):
        """sparse_X_info_ / sparse_Y_info_ (mbpls.py:294-296, 304-313) from the device census."""
        B = len(shard.sizes)
        col_nan, row_flag, xinf = E.nan_census(Xt, n, boff_dev, B)
        if group is not None:
            import torch.distributed as dist
            rf = row_flag.to(torch.int32)
            dist.all_reduce(rf, op=dist.ReduceOp.MAX, group=group)
            row_flag.copy_(rf.to(torch.uint8))
        one = E._i32([0, q], Yt.device)
        ycol_nan, yrow_flag, yinf = E.nan_census(Yt, n, one, 1)
        self._raise_if_any_rank(bool(xinf.item()) or bool(yinf.item()),
                                "Input contains infinity or a value too large for dtype('float64').", group)
        col_full = self._gather_features(col_nan.view(1, -1).to(F64), shard, force_all=True)[0] > 0  # census lists global columns
        rows = row_flag[:, :n].cpu().numpy().astype(bool)
        self.sparse_Y_info_ = {'Y': self._census_from_flags(yrow_flag[0, :n].cpu().numpy().astype(bool),
                                                            (ycol_nan[:q] > 0).cpu().numpy())}
        self.sparse_X_info_ = {}
        g0 = 0
        for b, pb in enumerate(shard.sizes):
            self.sparse_X_info_[b] = self._census_from_flags(rows[b], col_full[g0:g0 + pb])
            g0 += pb
        self.__dict__["_col_nan"] = col_nan  # per local feature, for the masked denominators of the one-pass kernels
        return row_flag, (ycol_nan[:q] > 0).to(torch.uint8).contiguous()

    def _lazy_scalers(self, xs, ys, shard, q):
        """x_scalers_ / y_scaler_ as lazily materialised attributes: the statistics stay on the device (predict / transform
        use them there) and are gathered into scikit-learn StandardScaler objects on first access (32 MB of D2H per
        million features that a fit should not wait for)."""
        box = {}
        me = weakref.proxy(self)  # no cycle self -> _lazy -> closure -> self: an unmaterialised model frees its device buffers at once

        def build():
            if not box:
                mean = me._gather_features(xs.mean.view(1, -1), shard)[0]
                var = me._gather_features(xs.var.view(1, -1), shard)[0]
                scale = me._gather_features(xs.scale.view(1, -1), shard)[0]
                seen = me._gather_features(xs.seen.view(1, -1).to(F64), shard)[0].astype(np.int64)
                bounds = me._feature_bounds(shard)
                box["x"] = [_make_scaler(mean[a:b], var[a:b], scale[a:b], seen[a:b]) for a, b in zip(bounds[:-1], bounds[1:])]
                box["y"] = _make_scaler(ys.mean[:q].cpu().numpy(), ys.var[:q].cpu().numpy(), ys.scale[:q].cpu().numpy(),
                                        ys.seen[:q].cpu().numpy())
            return box

        return {"x_scalers_": lambda: build()["x"], "y_scaler_": lambda: build()["y"]}

    def _block_sums(self, per_feature: torch.Tensor, boff_dev, B, group) -> np.ndarray:
        s = E.segsum(per_feature, boff_dev, B).clone()
        E.allreduce_(s, group)
        return s.cpu().numpy()

    # ---- NIPALS (mbpls.py:809-993)
    def _fit_nipals(self, Xt, Yt, n, q, shard, boff_dev, zss, row_flag, ycol_flag, group, device, first_trip=None):
        rt = self._runtime()
        B, K = len(shard.sizes), int(self.n_components)
        sparse = bool(self.sparse_data)
        p_loc = shard.p_local
        varxb = vary = None
        if self.calc_all:  # mbpls.py:822-830, :938-945
            if zss is None:
                zss = E.feature_sumsq(Xt, n)
            varxb = self._block_sums(zss, boff_dev, B, group)
            vary = float(E.segsum(E.feature_sumsq(Yt, n), E._i32([0, q], device), 1).item())
        # initial Y-score vector (mbpls.py:832-838)
        if sparse:
            dense_cols = self.sparse_Y_info_['Y'][3]
            if len(dense_cols) == 0:
                u0 = torch.zeros(Xt.shape[1], dtype=F64, device=device)
                u0[:n] = torch.from_numpy(np.random.rand(n)).to(device)
                if group is not None:
                    import torch.distributed as dist
                    dist.broadcast(u0, src=dist.get_global_rank(group, 0), group=group)
            else:
                u0 = Yt[int(dense_cols[0])]
        else:
            u0 = Yt[0]
        res = E.nipals_fit(Xt, Yt, n, shard.block_off, K, u0=u0, nanmode=sparse, row_flag=row_flag, ycol_flag=ycol_flag,
                           max_tol=self.max_tol, norm_kind=E.norm_kind_of(self.nipals_convergence_norm),
                           max_iter=rt["max_iter"], group=group, fuse_next_xtu=rt["fuse_next_xtu"],
                           deflate_mode=rt["deflate_mode"], trips_per_sync=rt["trips_per_sync"], profile=rt["profile"],
                           deflate_last=rt["deflate_last"], one_pass=rt["one_pass"],
                           one_pass_deflate=rt["one_pass_deflate"], first_trip=first_trip, col_nan=self.__dict__.pop("_col_nan", None) if sparse else None,
                           p_widest=-(-shard.p_global // max(shard.world, 1)))
        self.n_iter_ = list(res.n_iter)
        self.__dict__["_exchange"] = res.exchange
        if any(it >= rt["max_iter"] for it in res.n_iter):
            warnings.warn("NIPALS hit the max_iter safety cap before diff_t <= max_tol")
        # ---- finalise (mbpls.py:985-989): W = concat(W_non_normal_)/colnorm, R = W pinv(P'W), beta = R V'
        Wt, P = res.Wt[:, :p_loc], res.P[:, :p_loc]
        colnorm = torch.sqrt(E.rows_sumsq(Wt, p_loc, group))
        PtW = E.gram(P, Wt, p_loc, group) / colnorm.view(1, -1)
        M = E.small_pinv(PtW)  # pinv(P'W), K x K, one-sided Jacobi SVD on the device (:988)
        R = E.right_multiply(Wt, p_loc, 1.0 / colnorm, M)
        beta = E.right_multiply(R, p_loc, None, res.V[:, :q].contiguous())
        self.__dict__["_dev"] = dict(shard=shard, R=R, beta=beta, W=res.W[:, :p_loc], P=P, V=res.V[:, :q])
        self.__dict__["_cv_weights"] = Wt  # un-normalised weights: prefix models for model_selection.cross_val_predict

        # ---- small host-side bookkeeping
        A = res.A[:, :B].cpu().numpy().T.copy()  # B x K
        self.A_ = A
        if self.calc_all:
            pssb = res.pssb[:, :B].clone()
            E.allreduce_(pssb, group)
            pssb = pssb.cpu().numpy()  # K x B
            tt, vv = np.asarray(res.tt), np.asarray(res.vv)
            self.explained_var_x_ = [float(tt[k] * pssb[k].sum() / varxb.sum()) for k in range(K)]
            self.explained_var_y_ = [float(tt[k] * vv[k] / vary) for k in range(K)]
            self.explained_var_xblocks_ = (tt[None, :] * pssb.T) / varxb[:, None]
            self.A_corrected_ = np.stack([_bip_corrected(A[:, k], shard.sizes) for k in range(K)], axis=1)
        else:
            self.explained_var_x_, self.explained_var_y_ = [], []
            self.explained_var_xblocks_ = np.empty((B, 0))
            self.A_corrected_ = np.empty((B, 0))
        self.W_concat_ = np.empty((shard.p_global, 0))

        me = weakref.proxy(self)  # (see _lazy_scalers)
        lazy = {
            "Ts_": lambda: E.to_host(res.Ts[:, :n], transpose=True),
            "U_": lambda: E.to_host(res.U[:, :n], transpose=True),
            "V_": lambda: E.to_host(res.V[:, :q], transpose=True),
            "T_": lambda: [E.to_host(res.Tb[b, :, :n], transpose=True) for b in range(B)],
            "W_": lambda: me._features_T(res.W, shard, True),
            "W_non_normal_": lambda: me._features_T(res.Wt, shard, True),
            "P_": lambda: me._features_T(res.P, shard, True),
            "R_": lambda: me._features_T(R, shard, False),
            "beta_": lambda: me._features_T(beta, shard, False),
        }
        self.__dict__["_lazy"] = lazy

    # ------------------------------------------------------------------ new-data paths
    def _check_is_fitted(self):
        lazy = self.__dict__.get("_lazy")
        if "beta_" not in self.__dict__ and not (lazy and "beta_" in lazy):
            raise NotFittedError("This MBPLS instance is not fitted yet. Call 'fit' with appropriate arguments "
                                 "before using this estimator.")

    def _device_model(self, device):
        """Fitted matrices on the device (kept from fit, or rebuilt from the numpy attributes)."""
        dev = self.__dict__.get("_dev")
        if dev is not None and dev["R"].device == device:
            return dev
        _, rank, world = self._group_info()
        if self.__dict__.get("_rows") is not None:
            rank, world = 0, 1
        P_ = self.P_
        local = self.__dict__.get("_attrs_local_sizes")  # attributes hold this rank's rows only: (global block sizes)
        if local is not None:
            shard = ShardMap.build(list(local), rank, world)
            if [int(pb.shape[0]) for pb in P_] != [c1 - c0 for c0, c1 in shard.local_ranges]:
                raise ValueError("this model holds rank-local attributes of a different rank / world size")
        else:
            shard = ShardMap.build([int(pb.shape[0]) for pb in P_], rank, world)

        def up(full_pk):  # p x K numpy (global, or already this rank's rows) -> K x p_local device
            rows = full_pk if local is not None else full_pk[shard.lo:shard.hi]
            return torch.from_numpy(np.ascontiguousarray(rows.T)).to(device)

        dev = dict(shard=shard, R=up(self.R_), beta=up(self.beta_), P=up(np.concatenate(P_, axis=0)),
                   V=torch.from_numpy(np.ascontiguousarray(self.V_.T)).to(device))
        if isinstance(self.W_, list):
            dev["W"] = up(np.concatenate(self.W_, axis=0))
        self.__dict__["_dev"] = dev
        return dev

    def _device_scalers(self, shard, device):
        sc = self.__dict__.get("_dev_scalers")
        if sc is not None and sc[0].device == device:
            return sc
        mean = np.concatenate([np.atleast_1d(s.mean_) for s in self.x_scalers_])
        scale = np.concatenate([np.atleast_1d(s.scale_) for s in self.x_scalers_])
        if self.__dict__.get("_attrs_local_sizes") is None:
            mean, scale = mean[shard.lo:shard.hi], scale[shard.lo:shard.hi]
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(device)
        sc = (t(mean), t(scale), t(np.atleast_1d(self.y_scaler_.mean_)), t(np.atleast_1d(self.y_scaler_.scale_)))
        self.__dict__["_dev_scalers"] = sc
        return sc

    def _prepare_new_X(self, X, device, scaled_copy: bool):
        """Ingest new data.  scaled_copy=False: X is left untouched (device views are adopted zero-copy) and the
        scaler statistics are returned for on-the-fly standardisation inside the product kernel;
        scaled_copy=True: a private, standardised copy (needed by the sequential block-score deflation)."""
        dev = self._device_model(device)
        shard = dev["shard"]
        Xt, m, _ = self._ingest(X, None, shard, device, adopt=not scaled_copy, adopt_writable=False)
        mean = scale = None
        if self.standardize:
            mean, scale, _, _ = self._device_scalers(shard, device)
            if scaled_copy:
                E.standardize_apply(Xt, m, mean, scale)
                mean = scale = None
        return dev, shard, Xt, m, mean, scale

    def _check_flag(self, flag, group):
        bad = bool(flag.item())
        if self.sparse_data:
            return
        self._raise_if_any_rank(bad, "Input contains NaN or infinity.", group)

    def predict(self, X, copy=True):
        """y_hat = inverse_scale(scale(X) . beta_)  (mbpls.py:1337-1410); NaN entries count as zero after
        scaling (:1379-1383).  One pass over X: standardisation and the finiteness check are fused into the product."""
        self._check_is_fitted()
        device = E.require_cuda(self._runtime()["device"])
        group, _, _ = self._group_info()
        with torch.cuda.device(device):
            dev, shard, Xt, m, mean, scale = self._prepare_new_X(X, device, scaled_copy=False)
            if shard.world == 1:
                group = None  # model replicated on every rank (single GPU or row-sharded fit): no collective
            q = dev["beta"].shape[0]
            flag = torch.zeros(1, dtype=torch.int32, device=device)
            Yh = E.skinny_gemm(Xt, m, dev["beta"], shard.block_off, group, mean, scale, flag)
            self._check_flag(flag, group)
            if self.standardize:
                _, _, ymean, yscale = self._device_scalers(shard, device)
                call("mbpls_scaler_inverse_f64", ptr(Yh), Yh.shape[1], m, q, ptr(ymean), ptr(yscale), stream_ptr(device))
            return E.to_host(Yh[:, :m], transpose=True)

    def transform(self, X, Y=None, return_block_scores=False, copy=True):
        """Superscores (and block scores / Y scores) of new data (mbpls.py:1052-1335)."""
        self._check_is_fitted()
        device = E.require_cuda(self._runtime()["device"])
        group, _, _ = self._group_info()
        with torch.cuda.device(device):
            want_blocks = self.method != 'SIMPLS' and return_block_scores
            # only the NaN-mode block scores deflate the new data in place and need a private standardised copy
            dev, shard, Xt, m, mean, scale = self._prepare_new_X(X, device, scaled_copy=want_blocks and bool(self.sparse_data))
            if shard.world == 1:
                group = None
            if want_blocks and "W" not in dev:
                raise AttributeError("block scores need W_ (fit with calc_all=True)")
            K = dev["R"].shape[0]
            flag = torch.zeros(1, dtype=torch.int32, device=device)
            Ts_dev = E.skinny_gemm(Xt, m, dev["R"], shard.block_off, group, mean, scale, flag)  # K x ld   (:1110-1117)
            self._check_flag(flag, group)
            Ts = E.to_host(Ts_dev[:, :m], transpose=True)
            out = [Ts]
            if want_blocks and not self.sparse_data:
                # Dense data: the K sequential deflations of :1131-1155 collapse to one product and a K x K
                # triangular correction,  T_b = X_b W_b - Ts striu(P_b' W_b)  (SURVEY.md 8f-3): X is read once.
                from . import crossmethods as CM
                B = len(shard.sizes)
                T = []
                for b in range(B):
                    o0, o1 = shard.block_off[b], shard.block_off[b + 1]
                    Wb, Pb = dev["W"][:, o0:o1], dev["P"][:, o0:o1]
                    full = E.skinny_gemm(Xt[o0:o1], m, Wb, [0, o1 - o0], group,
                                         None if mean is None else mean[o0:o1], None if scale is None else scale[o0:o1])  # X_b W_b
                    Cb = torch.triu(E.gram(Pb, Wb, o1 - o0, group), diagonal=1).contiguous()  # striu(P_b' W_b)
                    cols = [CM.lincomb_sub(full[k].contiguous(), Ts_dev, k, Cb[:k, k].contiguous(), m)[:m] if k > 0
                            else full[0, :m] for k in range(K)]
                    T.append(E.to_host(torch.stack(cols, dim=1)))
                out.append(T)
            elif want_blocks:  # NaN mode: sequential deflation, NaNs stay NaN and count as zero (:1126-1155)
                B = len(shard.sizes)
                T = []
                for b in range(B):
                    o0, o1 = shard.block_off[b], shard.block_off[b + 1]
                    Xb = Xt[o0:o1]
                    cols = []
                    for k in range(K):
                        if k > 0 and o1 > o0:
                            call("mbpls_rank1_update_f64", ptr(Xb), Xb.shape[1], m, o1 - o0, ptr(Ts_dev[k - 1]),
                                 ptr(dev["P"][k - 1, o0:o1]), stream_ptr(device))
                        tk = E.skinny_gemm(Xb, m, dev["W"][k:k + 1, o0:o1], [0, o1 - o0], group)
                        cols.append(tk[0, :m])
                    T.append(E.to_host(torch.stack(cols, dim=1)))
                out.append(T)
            if Y is not None:  # :1119-1125, :1156-1166
                Ysrc = Y if isinstance(Y, torch.Tensor) else np.asarray(Y)
                if Ysrc.ndim == 1:
                    Ysrc = Ysrc.reshape(-1, 1)
                Ysrc = _as_2d_source(Ysrc, "Y")
                q = int(Ysrc.shape[1])
                Yt = E.alloc_feature_major(q, m, device)
                E.ingest_feature_major(Ysrc, m, 0, q, Yt, device)
                ymean = yscale = None
                if self.standardize:
                    _, _, ymean, yscale = self._device_scalers(shard, device)
                yflag = torch.zeros(1, dtype=torch.int32, device=device)
                Ur = E.skinny_gemm(Yt, m, dev["V"], [0, q], None, ymean, yscale, yflag)  # K x ld
                self._check_flag(yflag, None)
                nrm = torch.sqrt(E.rows_sumsq(Ur, m))
                call("mbpls_rows_scale_f64", ptr(Ur), Ur.shape[1], K, m, ptr(nrm), 1, stream_ptr(device))
                out.append(E.to_host(Ur[:, :m], transpose=True))
        return out[0] if len(out) == 1 else tuple(out)

    # ------------------------------------------------------------------ convenience (mbpls.py:1412-1437)
    def fit_transform(self, X, y=None, **fit_params):
        return self.fit(X, y, **fit_params).transform(X, y)

    def fit_predict(self, X, Y, **fit_params):
        return self.fit(X, Y, **fit_params).predict(X)

    def r2_score(self, X, Y):
        if self.standardize:
            return metrics.r2_score(Y, self.predict(X))
        return metrics.r2_score(Y, self.predict(X), sample_weight=None, multioutput='variance_weighted')

    def explained_variance_score(self, X, Y):
        if self.standardize:
            return metrics.explained_variance_score(Y, self.predict(X))
        return metrics.explained_variance_score(Y, self.predict(X), sample_weight=None,
                                                multioutput='variance_weighted')


    # ------------------------------------------------------------------ reporting (mbpls.py:1439-1556)
    def _component_indices(self, num_components):
        """The reference's argument convention (:1454-1473): an int N means the first N components, a sequence
        holds 1-based component numbers; requests beyond the fitted model are truncated with a printed note."""
        if isinstance(num_components, (int, np.integer)):
            comps = np.arange(int(num_components))
        else:
            comps = np.asarray(list(num_components), dtype=int) - 1
        if len(comps) > self.n_components:
            print("You requested more components to be plotted than your fitted model has.")
            print("The requested list will be shortened to the maximum amount of components possible")
            comps = comps[:self.n_components]
        if len(comps) and (comps.max() + 1 > self.n_components or comps.min() < 0):
            raise ValueError("You requested not existing indices.")
        return comps

    def plot_data(self, num_components=2):
        """Everything ``plot`` draws, as arrays: per requested component the block importances (%), the explained
        Y variance (%), the loadings of every block mapped back to the original variable scale through
        ``x_scalers_[b].inverse_transform`` (:1494-1498) and the block scores."""
        self._check_is_fitted()
        T = getattr(self, "T_", None)
        if self.method == 'SIMPLS' or not isinstance(T, list) or len(T) == 0 or T[0].shape[1] == 0:
            raise AttributeError("plot needs block scores and importances (NIPALS / UNIPALS, or KERNEL with calc_all=True)")
        out = []
        for comp in self._component_indices(num_components):
            loadings = []
            for b in range(self.num_blocks_):
                pb = self.P_[b][:, comp]
                loadings.append(self.x_scalers_[b].inverse_transform(pb.reshape(1, -1)).ravel() if self.standardize else pb)
            ev_y = float(100 * self.explained_var_y_[comp]) if len(self.explained_var_y_) > comp else float("nan")
            out.append(dict(component=int(comp) + 1, explained_var_y_percent=ev_y,
                            importance_percent=100 * np.ravel(self.A_[:, comp]), loadings=loadings,
                            block_scores=[self.T_[b][:, comp] for b in range(self.num_blocks_)]))
        return out

    def plot(self, num_components=2):
        """Per component: block importances, loadings (original scale) and block scores of every block; then a bar
        chart of the block importances (mbpls.py:1439-1556).  Needs matplotlib, like the reference."""
        data = self.plot_data(num_components)
        from matplotlib import pyplot as plt
        from matplotlib.gridspec import GridSpec
        B = self.num_blocks_

        def quarter_ticks(length):
            step = max(1, length // 4)
            plt.xticks(np.arange(0, length, step), np.arange(1, length + 1, step))

        for d in data:
            plt.figure()
            plt.suptitle("Component {}: {}% expl. var. in Y".format(d["component"], round(d["explained_var_y_percent"], 2)),
                         fontsize=12, fontweight='bold')
            head = GridSpec(1, B, top=0.875, bottom=0.85, right=0.95)
            body = GridSpec(2, B, top=0.8, hspace=0.45, wspace=0.45, right=0.95)
            for b in range(B):
                plt.subplot(head[0, b])
                plt.text(0.5, 0, "X-Block {:d}\nImportance: {:.0f}%".format(b + 1, d["importance_percent"][b]),
                         fontsize=12, horizontalalignment='center')
                plt.axis('off')
                for row, series, xlabel, ylabel in ((0, d["loadings"][b], "Variable", "Loading"),
                                                    (1, d["block_scores"][b], "Sample", "Block Score")):
                    plt.subplot(body[row, b])
                    plt.plot(series)
                    quarter_ticks(len(series))
                    plt.xlabel(xlabel)
                    if b == 0:
                        plt.ylabel(ylabel)
                    plt.grid()
            plt.show()
        plt.figure()
        plt.suptitle("Block importances", fontsize=14, fontweight='bold')
        ax = plt.subplot(GridSpec(1, 1, top=0.825, right=0.7, hspace=0.45, wspace=0.4)[0, 0])
        width = 0.8 / max(1, len(data))
        for i, d in enumerate(data):
            ax.bar(np.arange(B) + 1 - 0.4 + (i + 0.5) * width, d["importance_percent"], width=width,
                   label="Component {}".format(d["component"]))
        ax.set_xticks(np.arange(B) + 1)
        ax.legend(bbox_to_anchor=(1.04, 1), loc="upper left")
        ax.set_xlabel("Block")
        ax.set_ylabel("Block importance in %")
        plt.show()


def _make_scaler(mean, var, scale, seen) -> StandardScaler:
    """A scikit-learn StandardScaler carrying statistics computed on the device, so that
    ``x_scalers_[b].transform / inverse_transform`` work exactly as with the reference (notebooks use them)."""
    sc = StandardScaler(with_mean=True, with_std=True)
    sc.mean_ = np.array(mean, dtype=np.float64)
    sc.var_ = np.array(var, dtype=np.float64)
    sc.scale_ = np.array(scale, dtype=np.float64)
    seen = np.array(seen, dtype=np.int64)
    sc.n_samples_seen_ = seen[0] if seen.size and np.ptp(seen) == 0 else seen
    sc.n_features_in_ = int(sc.mean_.shape[0])
    return sc


def _small_attributes(sm: dict, sizes, calc_all: bool) -> dict:
    """A_, and with calc_all A_corrected_ and the explained variances (mbpls.py:932-964), of one fit of the one-kernel path
    from the reduced scalars of its `small` block (smallfit.unpack_small)."""
    A = np.ascontiguousarray(sm["A"].T)
    B, K = A.shape
    if not calc_all:
        return dict(A_=A, explained_var_x_=[], explained_var_y_=[], explained_var_xblocks_=np.empty((B, 0)),
                    A_corrected_=np.empty((B, 0)))
    tt, vv, pssb, varxb = sm["tt"], sm["vv"], sm["pssb"], sm["varxb"]
    return dict(A_=A,
                explained_var_x_=[float(tt[k] * pssb[k].sum() / varxb.sum()) for k in range(K)],
                explained_var_y_=[float(tt[k] * vv[k] / sm["vary"]) for k in range(K)],
                explained_var_xblocks_=(tt[None, :] * pssb.T) / varxb[:, None],
                A_corrected_=np.stack([_bip_corrected(A[:, k], sizes) for k in range(K)], axis=1))


def _bip_corrected(a, sizes):
    """Block importances corrected for block size (mbpls.py:950-963): O(B) host bookkeeping."""
    a = np.asarray(a, dtype=np.float64).ravel()
    if a.size == 1:
        return np.array([1.0])
    sizes = np.asarray(sizes, dtype=np.float64)
    corrected = a * (1.0 - sizes / sizes.sum())
    return corrected / corrected.sum()
