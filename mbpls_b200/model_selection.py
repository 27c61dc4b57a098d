"""Device-resident cross-validation driver (SURVEY.md section 8f, rank 1).

Every real-world notebook of the reference runs
``sklearn.model_selection.cross_val_predict(MBPLS(n_components=k), X, y, cv=len(X))`` for a range of ``k``
(``examples/real_world_applications/*.ipynb``): n refits per k, each of which re-validates, copies and -- with a
GPU estimator -- would re-upload X.  Here X and Y are uploaded once (feature-major); each fold gathers its training
samples on the device, runs the normal fit kernels on them, and predicts its held-out samples; with
``n_components_list`` the predictions for every smaller model are read off the *same* fit, because a K-component
NIPALS / UNIPALS / SIMPLS / KERNEL fit contains all of its prefixes (``beta_k = R_k V_k'`` with
``R_k = W_k pinv(P_k' W_k)``, mbpls/mbpls.py:986-989).

The result equals ``cross_val_predict(clone(estimator), X, y, cv=cv)`` (tests/test_gpu_cv.py).

Validation of a fitted model's reported quantities: ``permutation_test_score`` (does the model predict better than chance?
the cross-validation re-run on permutations of ``y``) and ``bootstrap`` (how stable are ``A_`` / ``beta_``? refits on
resamples of the rows).  Both need 10^3 - 10^5 fits; for NIPALS, dense or with missing values (``sparse_data=True``), they
all run in one slot-mode launch of ``smallfit_kernel`` (persistent CTAs that claim fit after fit, X rows paired with permuted /
resampled Y rows on the device).  ``block_permutation_test`` asks whether each block adds anything given the others: it
permutes the rows of one block at a time and re-runs the cross-validation and the fit on all rows, for null distributions of
the score and of the block's importance ``A_``; in the batch, a fit reads the permuted block's columns through a row map.
"""
from __future__ import annotations

import warnings
from typing import Iterable, Optional, Sequence

import numpy as np
import torch
from sklearn.base import clone

from . import engine as E
from . import smallfit as SF
from .engine import F64
from .mbpls import MBPLS, _as_2d_source, _is_block_list

__all__ = ["cross_val_predict", "permutation_test_score", "bootstrap", "block_permutation_test"]


def _folds(n: int, cv) -> list:
    if isinstance(cv, (int, np.integer)):
        from sklearn.model_selection import KFold
        return [(tr, te) for tr, te in KFold(n_splits=int(cv)).split(np.arange(n))]
    if hasattr(cv, "split"):
        return [(tr, te) for tr, te in cv.split(np.arange(n))]
    return [(np.asarray(tr), np.asarray(te)) for tr, te in cv]


def _prefix_betas(model: MBPLS, ks: Sequence[int], device) -> list:
    """beta for the first k components, k in ks, from one fitted model (device tensors q x p each)."""
    dev = model._device_model(device)
    shard = dev["shard"]
    p = shard.p_local
    group, _, _ = model._group_info()
    P, V = dev["P"], dev["V"]
    if model.method == 'SIMPLS':
        # SIMPLS: R and Q columns do not depend on later components (mbpls.py:1004-1013, :1044)
        return [E.right_multiply(dev["R"][:k], p, None, V[:k].contiguous()) for k in ks]
    Wfull = model.__dict__.get("_cv_weights")  # K x p un-normalised / concatenated weights kept by fit for CV
    out = []
    for k in ks:
        Wk, Pk = Wfull[:k], P[:k]
        if model.method == 'NIPALS':
            coln = torch.sqrt(E.rows_sumsq(Wk, p, group))
            M = E.small_pinv(E.gram(Pk, Wk, p, group) / coln.view(1, -1))
            R = E.right_multiply(Wk, p, 1.0 / coln, M)
        else:
            M = E.small_pinv(E.gram(Pk, Wk, p, group))
            R = E.right_multiply(Wk, p, None, M)
        out.append(E.right_multiply(R, p, None, V[:k].contiguous()))
    return out


def _fold_predictions(estimator, Xraw, Yraw, shard, q, K, ks, fits, device) -> list:
    """One refit through ``MBPLS.fit`` per (X train rows, Y train rows, test rows) of ``fits``, on the feature-major device
    copies Xraw / Yraw.  A fit may carry a fourth entry (b, pi): the columns of block b then come from rows pi[train rows] and
    pi[test rows] (a block permutation test).  Returns, per fit, {k: (len(test rows), q) array} of held-out predictions (k in
    ks, or K)."""
    off = shard.block_off
    out = []
    rows = lambda idx: torch.as_tensor(np.asarray(idx), device=device, dtype=torch.long)
    for fit in fits:
        tr, ytr, te = fit[:3]
        tr_d = rows(tr)
        ytr_d = tr_d if ytr is tr else rows(ytr)
        te_d = rows(te)
        ntr, nte = len(tr), len(te)
        Xtr = E.alloc_feature_major(shard.p_local, ntr, device)
        Xtr[:, :ntr] = Xraw.index_select(1, tr_d)              # gather of the training samples (device copy)
        Ytr = Yraw.index_select(1, ytr_d).t().contiguous()     # ntr x q
        Xte = E.alloc_feature_major(shard.p_local, nte, device)
        Xte[:, :nte] = Xraw.index_select(1, te_d)
        if len(fit) > 3:                                       # block b's columns on the permuted rows
            b, pi = fit[3]
            Xtr[off[b]:off[b + 1], :ntr] = Xraw[off[b]:off[b + 1]].index_select(1, rows(pi[tr]))
            Xte[off[b]:off[b + 1], :nte] = Xraw[off[b]:off[b + 1]].index_select(1, rows(pi[te]))
        m = clone(estimator)
        m.set_params(n_components=K, copy=False)
        m.set_runtime(device=device, materialize=False)
        pred = {}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m.fit([Xtr[off[b]:off[b + 1], :ntr].t() for b in range(len(shard.sizes))], Ytr)
            te_blocks = [Xte[off[b]:off[b + 1], :nte].t() for b in range(len(shard.sizes))]
            if ks is None:
                pred[K] = np.asarray(m.predict(te_blocks)).reshape(nte, q)
            else:
                dev, sh, Xt_new, mm, mean, scale = m._prepare_new_X(te_blocks, device, scaled_copy=False)
                for k, beta_k in zip(ks, _prefix_betas(m, ks, device)):
                    Yh = E.skinny_gemm(Xt_new, mm, beta_k, sh.block_off, None, mean, scale)
                    if m.standardize:
                        _, _, ymean, yscale = m._device_scalers(sh, device)
                        E.call("mbpls_scaler_inverse_f64", E.ptr(Yh), Yh.shape[1], mm, q, E.ptr(ymean), E.ptr(yscale),
                               E.stream_ptr(device))
                    pred[k] = Yh[:, :mm].cpu().numpy().T
        out.append(pred)
    return out


def _sources(X, y):
    """Blocks and a 2-D y as numpy arrays / tensors: (blocks, Y, y was 1-D, n, q, block sizes)."""
    blocks = X if _is_block_list(X) else [X]
    blocks = [_as_2d_source(b, "X") for b in blocks]
    Ysrc = y if isinstance(y, torch.Tensor) else np.asarray(y)
    y1d = Ysrc.ndim == 1
    if y1d:
        Ysrc = Ysrc.reshape(-1, 1)
    Ysrc = _as_2d_source(Ysrc, "y")
    return blocks, Ysrc, y1d, int(Ysrc.shape[0]), int(Ysrc.shape[1]), [int(b.shape[1]) for b in blocks]


def _require_finite(arrays, allow_nan: bool = False):
    """check_array's finiteness test (mbpls.py:310): NaN is accepted with sparse_data=True, +-inf never (as MBPLS.fit)."""
    for a in arrays:
        if allow_nan:
            bad = bool(torch.isinf(a).any()) if isinstance(a, torch.Tensor) else bool(np.isinf(a).any())
            if bad:
                raise ValueError("Input contains infinity or a value too large for dtype('float64').")
            continue
        ok = bool(torch.isfinite(a).all()) if isinstance(a, torch.Tensor) else bool(np.isfinite(a).all())
        if not ok:
            raise ValueError("Input contains NaN or infinity.")


def _nan_eligible(blocks, Ysrc, x_rows, y_rows, block_cols=None, block_rows=None) -> np.ndarray:
    """smallfit.nan_fits_eligible on the source arrays: per fit, True if the NaN-mode batch can run it."""
    x_obs = np.hstack([SF.observed(b) for b in blocks])
    return SF.nan_fits_eligible(x_obs, SF.observed(Ysrc), x_rows, y_rows, block_cols, block_rows)


def _upload(blocks, Ysrc, n, q, shard, device):
    """Feature-major device copies of X (p x ld) and Y (q x ld) for the refit loop."""
    Xraw = E.ingest_blocks(blocks, n, shard, device)
    Yraw = E.alloc_feature_major(q, n, device)
    E.ingest_feature_major(Ysrc, n, 0, q, Yraw, device)
    return Xraw, Yraw


def _batched_small_cv(estimator, blocks, Ysrc, n, q, sizes, shard, K, ks, folds, device):
    """All folds of a NIPALS cross-validation in ONE kernel launch (csrc/smallfit.cu): one CTA per fold gathers its training
    samples from the shared source, fits K components with the loop on the device, and predicts its held-out samples for
    every prefix 1..K of the model.  sparse_data=True runs the NaN-mode fit (any method: MBPLS.fit fits NIPALS then too).
    Returns {k: (n, q) array}, or None when the problem is not eligible, a fold's training rows are not
    (smallfit.nan_fits_eligible) or a fold comes back flagged (-> fold loop)."""
    rt = estimator._runtime()
    p = sum(sizes)
    force = rt["small_path"]
    sparse = bool(estimator.sparse_data)
    if force is False or (estimator.method != 'NIPALS' and not sparse) or not folds:
        return None
    ntr_max = max(len(tr) for tr, _ in folds)
    if force is None:
        import os
        if os.environ.get("MBPLS_SMALL_PATH", "1") == "0":
            return None
        if ntr_max * p > 8 * SF.SMALL_ELEMS or len(folds) * (p + q) * ntr_max * 8 > SF.CV_WORKSPACE_BYTES:
            return None
    from .mbpls import _check_limits
    _check_limits(K, q, len(sizes))
    _require_finite(blocks + [Ysrc], allow_nan=sparse)
    if sparse and not _nan_eligible(blocks, Ysrc, [tr for tr, _ in folds], [tr for tr, _ in folds]).all():
        return None
    D, n, sizes, p, q, ldx = SF.pack_source(blocks, Ysrc, device)
    lay, out, preds_d, keep = SF.launch(D, n, p, q, ldx, shard.block_off, K, bool(estimator.standardize),
                                        E.norm_kind_of(estimator.nipals_convergence_norm), estimator.max_tol, rt["max_iter"],
                                        [np.asarray(tr, dtype=np.int32) for tr, _ in folds],
                                        [np.asarray(te, dtype=np.int32) for _, te in folds], nanmode=sparse)
    sm_all = E.to_host(out[lay.off["small"]:lay.off["small"] + lay.sizes["small"] * len(folds)]).reshape(len(folds), -1)
    if np.any(sm_all[:, -1] != 0.0):  # some fold has more components than rank: the fold loop applies the pseudo-inverse
        return None
    Pm = E.to_host(preds_d)  # K x n x q
    return {k: np.ascontiguousarray(Pm[k - 1]) for k in (ks or [K])}


def cross_val_predict(estimator: MBPLS, X, y, cv=5, n_components_list: Optional[Iterable[int]] = None):
    """Out-of-fold predictions of ``estimator`` (an unfitted ``mbpls_b200.MBPLS``) with the data kept on the GPU.

    Returns an (n, q) array like ``sklearn.model_selection.cross_val_predict``; with ``n_components_list`` a dict
    ``{k: (n, q) array}`` obtained from one fit per fold with ``max(k)`` components.
    With a process group in the estimator's runtime options the FOLDS are spread over the ranks (rank r fits folds r, r + world,
    ...; the data is replicated, every fit runs on one GPU) and the out-of-fold predictions are summed across the ranks, so every
    rank returns the complete result.
    """
    rt = estimator._runtime()
    group = rt["group"]
    device = E.require_cuda(rt["device"])
    blocks, Ysrc, y1d, n, q, sizes = _sources(X, y)
    ks = None if n_components_list is None else sorted(set(int(k) for k in n_components_list))
    K = estimator.n_components if ks is None else max(ks)
    folds = _folds(n, cv)
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        folds = folds[rank::world]

    def finish(preds):
        """dict k -> (n, q) with NaN outside this rank's folds -> the complete arrays on every rank"""
        if group is not None:
            keys = sorted(preds)
            stack = torch.from_numpy(np.stack([preds[k] for k in keys])).to(device)
            seen = (~torch.isnan(stack)).to(F64)
            stack = torch.nan_to_num(stack, nan=0.0)
            dist.all_reduce(stack, group=group)
            dist.all_reduce(seen, group=group)
            stack = torch.where(seen > 0, stack / seen.clamp(min=1.0), torch.full_like(stack, float("nan")))
            host = stack.cpu().numpy()
            preds = {k: host[i] for i, k in enumerate(keys)}
        if ks is None:
            return preds[K].ravel() if y1d else preds[K]
        return {k: (v.ravel() if y1d else v) for k, v in preds.items()}

    with torch.cuda.device(device):
        shard = E.ShardMap.build(sizes, 0, 1)
        batched = _batched_small_cv(estimator, blocks, Ysrc, n, q, sizes, shard, K, ks, folds, device) if folds else None
        if batched is not None:
            return finish(batched)
        Xraw, Yraw = _upload(blocks, Ysrc, n, q, shard, device)  # uploaded once
        preds = {k: np.full((n, q), np.nan) for k in (ks or [K])}
        per_fold = _fold_predictions(estimator, Xraw, Yraw, shard, q, K, ks, [(tr, tr, te) for tr, te in folds], device)
        for (tr, te), pred in zip(folds, per_fold):
            for k, v in pred.items():
                preds[k][te] = v
    return finish(preds)


# ---------------------------------------------------------------------------------------------------------------- resampling
_SCORINGS = (None, "r2", "explained_variance", "neg_mean_squared_error", "neg_root_mean_squared_error", "neg_mean_absolute_error")


def _check_scoring(scoring):
    if not (scoring is None or isinstance(scoring, str)) or scoring not in _SCORINGS:
        raise ValueError(f"scoring must be one of {_SCORINGS}, got {scoring!r}")


def _scores(scoring, y_true: np.ndarray, y_pred: np.ndarray) -> np.ndarray:
    """sklearn.metrics scores (multioutput='uniform_average') of many predictions at once: arrays (..., m samples, q outputs)
    -> scores (...).  Same values as the scikit-learn function on each (m, q) slice, edge cases included (r2 of fewer than two
    samples is NaN; a zero denominator follows force_finite).  scoring None is the estimator's inherited score, r2."""
    y_true, y_pred = np.broadcast_arrays(np.asarray(y_true, dtype=np.float64), np.asarray(y_pred, dtype=np.float64))
    m = y_true.shape[-2]
    if scoring in ("neg_mean_squared_error", "neg_root_mean_squared_error"):
        mse = np.mean((y_true - y_pred) ** 2, axis=-2)
        return -np.mean(mse if scoring == "neg_mean_squared_error" else np.sqrt(mse), axis=-1)
    if scoring == "neg_mean_absolute_error":
        return -np.mean(np.mean(np.abs(y_pred - y_true), axis=-2), axis=-1)
    if scoring in (None, "r2"):
        if m < 2:
            return np.full(y_true.shape[:-2], np.nan)
        num = np.sum((y_true - y_pred) ** 2, axis=-2)
        den = np.sum((y_true - np.mean(y_true, axis=-2, keepdims=True)) ** 2, axis=-2)
    else:  # explained_variance
        d = y_true - y_pred
        num = np.mean((d - np.mean(d, axis=-2, keepdims=True)) ** 2, axis=-2)
        den = np.mean((y_true - np.mean(y_true, axis=-2, keepdims=True)) ** 2, axis=-2)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = np.where((num != 0) & (den != 0), 1.0 - num / den, np.where(num != 0, 0.0, 1.0))
    return np.mean(out, axis=-1)


def _permutations(n: int, n_permutations: int, random_state) -> np.ndarray:
    """(1 + n_permutations) x n row orders: the identity, then rs.permutation(n) in order as scikit-learn draws them."""
    from sklearn.utils import check_random_state
    rs = check_random_state(random_state)
    return np.stack([np.arange(n)] + [rs.permutation(n) for _ in range(n_permutations)])


def _resamples(n: int, n_resamples: int, random_state) -> np.ndarray:
    """n_resamples x n bootstrap row sets: sklearn.utils.resample(np.arange(n)) with one shared random state."""
    from sklearn.utils import check_random_state, resample
    rs = check_random_state(random_state)
    return np.stack([resample(np.arange(n), random_state=rs) for _ in range(n_resamples)]).reshape(n_resamples, n)


def _host(a) -> np.ndarray:
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def permutation_test_score(estimator: MBPLS, X, y, cv=5, n_permutations: int = 100, random_state=0, scoring=None,
                           n_components_list: Optional[Iterable[int]] = None):
    """Significance of a cross-validated score by permutation of ``y``, as ``sklearn.model_selection.permutation_test_score``,
    for an unfitted ``mbpls_b200.MBPLS`` and ``X`` one array or a list of blocks.

    Returns ``(score, permutation_scores, pvalue)``: the mean over the folds of the score of the unpermuted cross-validation,
    the same for each of ``n_permutations`` permutations of the rows of ``y``, and ``(#{permutation_scores >= score} + 1) /
    (n_permutations + 1)``.  With ``n_components_list`` a dict ``{k: (score, permutation_scores, pvalue)}`` from one
    ``max(k)``-component fit per fold and permutation.

    Permutations are drawn as scikit-learn draws them (``check_random_state(random_state)``, then ``permutation(n)`` once per
    permutation), so on a single array with a deterministic ``cv`` the result equals scikit-learn's function run with this
    estimator.  The folds are taken from ``cv`` once and reused for every permutation: a splitter whose ``split`` differs from
    call to call needs a fixed ``random_state``.  ``scoring``: None (the estimator's ``score``, r2), "r2",
    "explained_variance", "neg_mean_squared_error", "neg_root_mean_squared_error" or "neg_mean_absolute_error".

    NIPALS problems small enough for one CTA, dense or with ``sparse_data=True``, run every fit of every permutation in one
    kernel launch; other methods and larger problems refit through ``MBPLS.fit``, and so do the fits the batch cannot run
    (more components than rank; with missing values, training rows that leave a feature or Y column unobserved or no Y column
    fully observed).
    """
    _check_scoring(scoring)
    rt = estimator._runtime()
    if rt["group"] is not None:
        raise NotImplementedError("permutation_test_score runs on one GPU: no process group in the runtime options")
    device = E.require_cuda(rt["device"])
    blocks, Ysrc, _, n, q, sizes = _sources(X, y)
    ks = None if n_components_list is None else sorted(set(int(k) for k in n_components_list))
    K = estimator.n_components if ks is None else max(ks)
    kk = ks or [K]
    folds = _folds(n, cv)
    perms = _permutations(n, int(n_permutations), random_state)
    R, nf = perms.shape[0], len(folds)
    fits = [(r, i) for r in range(R) for i in range(nf)]  # (permutation, fold)
    ld_t = max(1, max(len(te) for _, te in folds))
    preds = np.full((R, nf, len(kk), ld_t, q), np.nan)  # held-out predictions by position in the fold's test list

    with torch.cuda.device(device):
        shard = E.ShardMap.build(sizes, 0, 1)
        redo = fits
        if SF.batch_eligible(estimator, max(len(tr) for tr, _ in folds), sum(sizes)):
            redo = _permutation_batches(estimator, blocks, Ysrc, n, q, shard, K, kk, folds, perms, preds, device)
        if redo:  # every fit (generic path), or the fits the batch flagged or could not run, one by one through MBPLS.fit
            Xraw, Yraw = _upload(blocks, Ysrc, n, q, shard, device)
            todo = [(folds[i][0], perms[r][folds[i][0]], folds[i][1]) for r, i in redo]
            for (r, i), pred in zip(redo, _fold_predictions(estimator, Xraw, Yraw, shard, q, K, kk, todo, device)):
                for j, k in enumerate(kk):
                    preds[r, i, j, :len(folds[i][1])] = pred[k]

    Yh = _host(Ysrc)
    S = np.zeros((R, len(kk)))
    for i, (_, te) in enumerate(folds):
        yt = Yh[perms[:, te]]                                       # R x nte x q: y[pi_r[te]]
        S += _scores(scoring, yt[:, None], preds[:, i, :, :len(te)])
    S /= nf
    res = {}
    for j, k in enumerate(kk):
        score, perm_scores = float(S[0, j]), S[1:, j].copy()
        res[k] = (score, perm_scores, (np.sum(perm_scores >= score) + 1.0) / (n_permutations + 1.0))
    return res[K] if ks is None else res


def _permutation_batches(estimator, blocks, Ysrc, n, q, shard, K, kk, folds, perms, preds, device) -> list:
    """Every (permutation, fold) fit in slot-mode launches of smallfit_kernel (one unless the per-fit outputs exceed
    CV_WORKSPACE_BYTES): fit (r, i) gathers X rows tr_i and Y rows pi_r[tr_i] and predicts X rows te_i for every prefix
    model.  Fills preds; returns the (permutation, fold) pairs of the fits flagged singular (more components than rank) or,
    with sparse_data=True, not eligible (smallfit.nan_fits_eligible) or flagged by the kernel, which the caller refits."""
    from .mbpls import _check_limits
    rt = estimator._runtime()
    sparse = bool(estimator.sparse_data)
    _check_limits(K, q, len(shard.sizes))
    _require_finite(blocks + [Ysrc], allow_nan=sparse)
    R, nf = perms.shape[0], len(folds)
    redo = set()
    if sparse:
        ok = _nan_eligible(blocks, Ysrc, [tr for _ in range(R) for tr, _ in folds], [perms[r][tr] for r in range(R) for tr, _ in folds])
        redo.update(divmod(int(f), nf) for f in np.flatnonzero(~ok))
    D, n, sizes, p, q, ldx = SF.pack_source(blocks, Ysrc, device)
    B = len(sizes)
    ld_t = preds.shape[3]
    kidx = [k - 1 for k in kk]
    small_sz = K * (q + 2 * B + 4) + B + 2
    for r0, r1 in SF.unit_batches(R, nf, 8 * (small_sz + K * ld_t * q)):
        F = (r1 - r0) * nf
        lay, out, fp, keep = SF.launch(
            D, n, p, q, ldx, shard.block_off, K, bool(estimator.standardize), E.norm_kind_of(estimator.nipals_convergence_norm),
            estimator.max_tol, rt["max_iter"],
            [np.asarray(tr, dtype=np.int32) for _ in range(r0, r1) for tr, _ in folds],
            [np.asarray(te, dtype=np.int32) for _ in range(r0, r1) for _, te in folds],
            y_sets=[perms[r][tr].astype(np.int32) for r in range(r0, r1) for tr, _ in folds],
            nslots=SF.slot_count(device, F), fit_preds=True, want_beta=False, nanmode=sparse)
        flags = E.to_host(lay.section(out, "small")[:, -1])
        host = E.to_host(fp)                                        # F x K x ld_t x q
        preds[r0:r1] = host[:, kidx].reshape(r1 - r0, nf, len(kk), ld_t, q)
        redo.update(divmod(r0 * nf + int(f), nf) for f in np.nonzero(flags != 0.0)[0])
    return sorted(redo)


def bootstrap(estimator: MBPLS, X, y, n_resamples: int = 100, random_state=0) -> dict:
    """Refits of an unfitted ``mbpls_b200.MBPLS`` on bootstrap resamples of the rows, for the spread of the block importances
    and coefficients (``np.percentile`` over the returned arrays gives confidence intervals).

    Resample r uses the rows ``sklearn.utils.resample(np.arange(n), random_state=rs)`` with one ``rs =
    check_random_state(random_state)`` drawn in order.  Returns a dict of arrays stacked over the resamples: ``indices``
    (R x n), ``A_`` (R x B x K), ``beta_`` (R x p x q), ``n_iter_`` (R x K, NIPALS) and, with ``calc_all``, ``A_corrected_``
    (R x B x K), ``explained_var_x_`` / ``explained_var_y_`` (R x K) and ``explained_var_xblocks_`` (R x B x K).  Entry r is
    the attribute of ``clone(estimator).fit([x[idx] for x in X], y[idx])``.

    NIPALS problems small enough for one CTA, dense or with ``sparse_data=True``, fit every resample in one kernel launch;
    other methods, larger problems and the resamples the batch cannot run (more components than rank; with missing values,
    rows that leave a feature or Y column unobserved or no Y column fully observed) refit through ``MBPLS.fit``.
    """
    from .mbpls import _check_limits, _small_attributes
    rt = estimator._runtime()
    if rt["group"] is not None:
        raise NotImplementedError("bootstrap runs on one GPU: no process group in the runtime options")
    device = E.require_cuda(rt["device"])
    blocks, Ysrc, y1d, n, q, sizes = _sources(X, y)
    idx = _resamples(n, int(n_resamples), random_state)
    R, K, B, p = idx.shape[0], int(estimator.n_components), len(sizes), sum(sizes)
    names = ["A_", "beta_"] + (["n_iter_"] if estimator.method == 'NIPALS' else []) + \
        (["A_corrected_", "explained_var_x_", "explained_var_y_", "explained_var_xblocks_"] if estimator.calc_all else [])
    res = {name: [None] * R for name in names}
    redo = list(range(R))
    sparse = bool(estimator.sparse_data)
    with torch.cuda.device(device):
        shard = E.ShardMap.build(sizes, 0, 1)
        if SF.batch_eligible(estimator, n, p):
            _check_limits(K, q, B)
            _require_finite(blocks + [Ysrc], allow_nan=sparse)
            ok = _nan_eligible(blocks, Ysrc, idx, idx) if sparse else np.ones(R, dtype=bool)
            D, n, sizes, p, q, ldx = SF.pack_source(blocks, Ysrc, device)
            redo = []
            for r0, r1 in SF.unit_batches(R, 1, 8 * (K * (q + 2 * B + 4) + B + 2 + q * p)):
                lay, out, _, keep = SF.launch(
                    D, n, p, q, ldx, shard.block_off, K, bool(estimator.standardize),
                    E.norm_kind_of(estimator.nipals_convergence_norm), estimator.max_tol, rt["max_iter"],
                    [idx[r].astype(np.int32) for r in range(r0, r1)], nslots=SF.slot_count(device, r1 - r0), nanmode=sparse)
                small, beta = E.to_host(lay.section(out, "small")), E.to_host(lay.section(out, "beta"))
                for r in range(r0, r1):
                    sm = SF.unpack_small(small[r - r0], K, q, B)
                    if sm["singular"] or not ok[r]:  # R = W pinv(P'W) like the reference, or a NaN fit the batch cannot run
                        redo.append(r)
                        continue
                    attrs = _small_attributes(sm, sizes, estimator.calc_all)
                    attrs["beta_"] = beta[r - r0].reshape(q, p).T
                    attrs["n_iter_"] = sm["trips"]
                    for name in names:
                        res[name][r] = attrs[name]
    for r in redo:
        m = _refit(estimator, rt, blocks, Ysrc, y1d, idx[r])
        for name in names:
            res[name][r] = getattr(m, name)
    out = {"indices": idx}
    out.update({name: np.stack([np.asarray(v, dtype=np.float64) for v in vals]) for name, vals in res.items()})
    if "n_iter_" in out:
        out["n_iter_"] = out["n_iter_"].astype(np.int64)
    return out


def _refit(estimator, rt, blocks, Ysrc, y1d, rows, block_perm=None, n_components=None) -> MBPLS:
    """``clone(estimator)`` with the runtime options ``rt`` fitted through ``MBPLS.fit`` on rows ``rows`` of every block and of
    y.  block_perm (b, pi): block b takes the rows pi[rows] instead."""
    m = clone(estimator)
    if n_components is not None:
        m.set_params(n_components=n_components)
    m.set_runtime(**rt)
    t = lambda a, r: a[torch.as_tensor(r, device=a.device)] if isinstance(a, torch.Tensor) else a[r]
    Xb = [t(x, block_perm[1][rows] if block_perm is not None and b == block_perm[0] else rows) for b, x in enumerate(blocks)]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.fit(Xb, t(Ysrc, rows).reshape(-1) if y1d else t(Ysrc, rows))
    return m


def block_permutation_test(estimator: MBPLS, X, y, cv=5, n_permutations: int = 100, random_state=0, scoring=None,
                           n_components_list: Optional[Iterable[int]] = None) -> dict:
    """Does block b add anything, given the other blocks?  A permutation test of each block of a multiblock model: the rows of
    block b alone are permuted, which breaks its link with ``y`` and with the other blocks and leaves everything else as it
    is; the cross-validation is run again, and the model refitted on all rows.

    ``estimator`` is an unfitted ``mbpls_b200.MBPLS`` and ``X`` a list of B >= 2 blocks (one array: see
    ``permutation_test_score``).  The R = ``n_permutations`` row orders are drawn as ``permutation_test_score`` draws them
    (``check_random_state(random_state)``, then ``permutation(n)`` R times), and the same R orders permute every block, so the
    blocks' null distributions are paired.  The folds are taken from ``cv`` once; ``scoring`` takes the values of
    ``permutation_test_score``.  Returns a dict:

    - ``score``: the mean over the folds of the unpermuted cross-validated score;
    - ``permutation_scores`` (B, R): the same with the rows of block b permuted by permutation r;
    - ``pvalue`` (B,): ``(#{permutation_scores[b] >= score} + 1) / (R + 1)``;
    - ``A_`` (B, K): ``A_`` of the unpermuted fit on all rows (block b's importance in component k);
    - ``A_permuted`` (B, R, K): block b's row of ``A_`` in the fits on all rows with block b permuted by permutation r;
    - ``A_pvalue`` (B, K): ``(#{A_permuted[b, :, k] >= A_[b, k]} + 1) / (R + 1)``.

    With ``n_components_list``, ``score``, ``permutation_scores`` and ``pvalue`` are dicts keyed by k from one ``max(k)``-component
    fit per fold, permutation and block, and the ``A_*`` entries are those of the ``max(k)`` fit (``A_[:, :k]`` is the
    k-component model's: a NIPALS component does not depend on later ones).  SIMPLS computes no ``A_``: the ``A_*`` keys are
    absent then.

    NIPALS problems small enough for one CTA, dense or with ``sparse_data=True``, run every fit (the cross-validations, the
    unpermuted fit on all rows and the B x R block-permuted ones) in one kernel launch; other methods, larger problems and the
    fits the batch cannot run (more components than rank; with missing values, rows that leave a feature or Y column
    unobserved or no Y column fully observed) refit through ``MBPLS.fit``.
    """
    _check_scoring(scoring)
    rt = estimator._runtime()
    if rt["group"] is not None:
        raise NotImplementedError("block_permutation_test runs on one GPU: no process group in the runtime options")
    if not (isinstance(X, list) and len(X) >= 2 and _is_block_list(X)):
        raise ValueError("block_permutation_test needs X as a list of at least two blocks; permutation_test_score tests a "
                         "single array")
    device = E.require_cuda(rt["device"])
    blocks, Ysrc, y1d, n, q, sizes = _sources(X, y)
    ks = None if n_components_list is None else sorted(set(int(k) for k in n_components_list))
    K = estimator.n_components if ks is None else max(ks)
    kk, B = ks or [K], len(sizes)
    folds = _folds(n, cv)
    perms = _permutations(n, int(n_permutations), random_state)[1:]  # R x n, without the identity
    R, nf = perms.shape[0], len(folds)
    units = [None] + [(b, r) for b in range(B) for r in range(R)]   # unit 0 permutes nothing, unit 1 + b R + r block b by r
    has_A = estimator.method != 'SIMPLS' or bool(estimator.sparse_data)
    ld_t = max(1, max(len(te) for _, te in folds))
    preds = np.full((len(units), nf, len(kk), ld_t, q), np.nan)      # held-out predictions by position in the fold's test list
    A_all = np.full((len(units), B, K), np.nan)                      # A_ of the fits on all rows

    with torch.cuda.device(device):
        shard = E.ShardMap.build(sizes, 0, 1)
        redo_cv, redo_full = [(u, i) for u in range(len(units)) for i in range(nf)], list(range(len(units)) if has_A else [])
        if SF.batch_eligible(estimator, n, sum(sizes)):
            redo_cv, redo_full = _block_permutation_batches(estimator, blocks, Ysrc, n, q, shard, K, kk, folds, perms, units,
                                                            preds, A_all, device)
        if redo_cv:  # every CV fit (generic path), or those the batch flagged or could not run, one by one through MBPLS.fit
            Xraw, Yraw = _upload(blocks, Ysrc, n, q, shard, device)
            todo = []
            for u, i in redo_cv:
                tr, te = folds[i]
                todo.append((tr, tr, te) if units[u] is None else (tr, tr, te, (units[u][0], perms[units[u][1]])))
            for (u, i), pred in zip(redo_cv, _fold_predictions(estimator, Xraw, Yraw, shard, q, K, kk, todo, device)):
                for j, k in enumerate(kk):
                    preds[u, i, j, :len(folds[i][1])] = pred[k]
    for u in redo_full:
        bp = None if units[u] is None else (units[u][0], perms[units[u][1]])
        A_all[u] = _refit(estimator, rt, blocks, Ysrc, y1d, np.arange(n), bp, n_components=K).A_

    Yh = _host(Ysrc)
    S = np.zeros((len(units), len(kk)))
    for i, (_, te) in enumerate(folds):
        S += _scores(scoring, Yh[te][None, None], preds[:, i, :, :len(te)])
    return _block_permutation_result(S / nf, A_all if has_A else None, B, R, ks)


def _block_permutation_result(S: np.ndarray, A_all: Optional[np.ndarray], B: int, R: int, ks) -> dict:
    """block_permutation_test's dict from the mean fold scores S ((1 + B R) units x prefix models, unit 0 unpermuted, unit
    1 + b R + r block b permuted by permutation r) and the A_ of the fits on all rows (units x B x K, None: no A_)."""
    res = {}
    for j, k in enumerate(ks or [None]):
        score, perm_scores = float(S[0, j]), S[1:, j].reshape(B, R)
        res[k] = (score, perm_scores, (np.sum(perm_scores >= score, axis=1) + 1.0) / (R + 1.0))
    out = {name: (res[None][i] if ks is None else {k: v[i] for k, v in res.items()})
           for i, name in enumerate(("score", "permutation_scores", "pvalue"))}
    if A_all is not None:
        A0 = A_all[0]
        Ap = np.stack([A_all[1 + b * R:1 + (b + 1) * R, b] for b in range(B)])  # B x R x K
        out.update(A_=A0, A_permuted=Ap, A_pvalue=(np.sum(Ap >= A0[:, None, :], axis=1) + 1.0) / (R + 1.0))
    return out


def _block_permutation_batches(estimator, blocks, Ysrc, n, q, shard, K, kk, folds, perms, units, preds, A_all, device):
    """Every fit of a block permutation test in slot-mode launches of smallfit_kernel (one unless the per-fit outputs exceed
    CV_WORKSPACE_BYTES).  Per unit (no permutation, or block b permuted by permutation r): the fold fits, which gather X rows
    tr_i (block b's columns through the row map) and predict X rows te_i for every prefix model, then one fit on all rows.
    Fills preds and A_all; returns the (unit, fold) pairs and the units of the fits on all rows that were flagged or, with
    sparse_data=True, not eligible (smallfit.nan_fits_eligible), which the caller refits through MBPLS.fit."""
    from .mbpls import _check_limits
    rt = estimator._runtime()
    sparse = bool(estimator.sparse_data)
    _check_limits(K, q, len(shard.sizes))
    _require_finite(blocks + [Ysrc], allow_nan=sparse)
    nf, U, off = len(folds), len(units), shard.block_off
    per = nf + 1                                                     # fits per unit: the folds, then all rows
    trs = [np.asarray(tr, dtype=np.int32) for tr, _ in folds] + [np.arange(n, dtype=np.int32)]
    tes = [np.asarray(te, dtype=np.int32) for _, te in folds] + [np.zeros(0, dtype=np.int32)]
    pair = lambda u: (-1, 0) if units[u] is None else (units[u][1], units[u][0])  # (r, b) as the kernel takes it
    redo = set()
    if sparse:
        cols = [None if v is None else (off[v[0]], off[v[0] + 1]) for v in units for _ in trs]
        prow = [None if v is None else perms[v[1]][t] for v in units for t in trs]
        ok = _nan_eligible(blocks, Ysrc, [t for _ in units for t in trs], [t for _ in units for t in trs], cols, prow)
        redo.update(divmod(int(f), per) for f in np.flatnonzero(~ok))
    D, n, sizes, p, q, ldx = SF.pack_source(blocks, Ysrc, device)
    B, ld_t = len(sizes), preds.shape[3]
    kidx = [k - 1 for k in kk]
    small_sz = K * (q + 2 * B + 4) + B + 2
    for u0, u1 in SF.unit_batches(U, per, 8 * (small_sz + K * ld_t * q)):
        F = (u1 - u0) * per
        lay, out, fp, keep = SF.launch(
            D, n, p, q, ldx, off, K, bool(estimator.standardize), E.norm_kind_of(estimator.nipals_convergence_norm),
            estimator.max_tol, rt["max_iter"], [t for _ in range(u0, u1) for t in trs], [t for _ in range(u0, u1) for t in tes],
            nslots=SF.slot_count(device, F), fit_preds=True, want_beta=False, nanmode=sparse,
            block_perm=(perms if len(perms) else np.zeros((1, n), np.int32), [pair(u) for u in range(u0, u1) for _ in trs]))
        small = E.to_host(lay.section(out, "small")).reshape(u1 - u0, per, -1)
        host = E.to_host(fp).reshape(u1 - u0, per, K, -1, q)         # fits x K x ld_t x q
        preds[u0:u1] = host[:, :nf][:, :, kidx]
        A_all[u0:u1] = small[:, nf, K * q:K * q + K * B].reshape(u1 - u0, K, B).transpose(0, 2, 1)
        redo.update((u0 + int(u), int(i)) for u, i in zip(*np.nonzero(small[:, :, -1] != 0.0)))
    return sorted((u, i) for u, i in redo if i < nf), sorted(u for u, i in redo if i == nf)
