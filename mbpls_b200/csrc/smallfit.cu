// Whole NIPALS fits inside ONE kernel: one persistent CTA per fit, loop control on the device; dense data, or missing values
// (NaN mode, smallfit_kernel<true>: see sf_fit).
//
// The reference's quickstart (README.rst:82-95: 40 x (200 + 250), 3 components) and the leave-one-out loops of its
// notebooks (cross_val_predict(MBPLS(k), X, y, cv=len(X)) for 15 values of k; examples/real_world_applications/*.ipynb) live
// where a fit is microseconds of arithmetic: through the streaming kernels such a fit is ~150 launches and a host readback per
// component, i.e. launch latency.  Here the `while diff_t > max_tol` loop of mbpls/mbpls.py:841 runs on the device: a CTA of
// 1024 threads gathers its training samples from the shared source matrix, standardises them (sklearn StandardScaler
// semantics, as csrc/ingest.cu), and runs the multiblock NIPALS of :821-983 -- weights, block scores, superlevel step,
// convergence test, loadings, rank-1 deflation, bookkeeping -- on its private L2-resident copy; no host synchronisation, no
// other launch.  The grid holds one CTA per fit, so all folds of a cross-validation run concurrently (SURVEY.md 8f-1); with
// test indices the CTA also predicts its held-out samples for EVERY prefix of the model (1..K components) from one fit:
// for NIPALS P'W is upper triangular, so R = W (P'W)^-1 follows column by column, r_k = (w_k - sum_{j<k} r_j (p_j.w_k)) /
// (p_k.w_k), and beta_k = beta_{k-1} + r_k v_k' (:986-989 for every leading block at once).
//
// Reductions have fixed shapes (warp shuffles + fixed-order block sums), so results are bitwise reproducible.
//
// Slot mode (nslots > 0, permutation tests and bootstrap: 10^4 - 10^5 fits): a grid of nslots persistent CTAs, each claiming
// the next fit from a ticket counter until none is left, so the workspace is bounded by the slots instead of the fits and a
// slot whose fit converged early (trip counts vary a lot under a permuted PLS2 y) takes the next one.  The arithmetic of a fit
// reads only its own inputs and workspace, so its results are bitwise the same whichever slot runs it, and in either mode.
//
// Block permutation tests (perm_rows / fit_perm): a fit may read the features of one block from permuted source rows, in its
// training gather and in its held-out predictions; Y and the other blocks keep their rows.
#include <vector>
#include "launch.cuh"
#include "../../include/mbpls_b200.h"

using namespace mbpls;

namespace {

constexpr int SF_THREADS = 1024;
constexpr int SF_WARPS = SF_THREADS / 32;
constexpr int SF_MAXB = 64, SF_MAXQ = 64, SF_MAXK = 64;  // SF_MAXK: components of a NaN-mode fit

__device__ __forceinline__ double sf_scale_from(double cnt, double mean, double corr, double ssq, double& var) {
  ssq -= corr * corr / cnt;  // corrected two-pass variance (sklearn _incremental_mean_and_var)
  var = ssq / cnt;
  const double eps = 2.220446049250313e-16;
  const double bound = cnt * eps * var + (cnt * mean * eps) * (cnt * mean * eps);
  return (var <= bound) ? 1.0 : sqrt(var);  // _is_constant_feature -> scale 1
}

// gather the training samples of one source feature, standardise, store; returns sum of squares of what was stored.
// rmap != NULL (a block-permuted fit, the feature in the permuted block): training sample t reads source row rmap[tr[t]].
// NANMODE: the nan-aware StandardScaler of csrc/ingest.cu (statistics over the observed values, NaN stored as NaN, nansum of
// z^2) and the observed count in *cnt_out.
template <bool NANMODE>
__device__ __forceinline__ double sf_ingest_feature(const double* __restrict__ src, const int* __restrict__ tr,
                                                     const int* __restrict__ rmap, int ntr, double* __restrict__ dst,
                                                     int standardize, double* mean_out, double* var_out, double* scale_out,
                                                     double* cnt_out, int lane) {
  const auto at = [&](int t) {
    const int i = tr ? tr[t] : t;
    return src[rmap ? rmap[i] : i];
  };
  double mean = 0.0, var = 0.0, scale = 1.0, cnt = ntr;
  if constexpr (NANMODE) {
    double o = 0.0;
    for (int t = lane; t < ntr; t += 32) o += isnan(at(t)) ? 0.0 : 1.0;
    cnt = warp_sum(o);
  }
  if (standardize) {
    double s = 0.0;
    for (int t = lane; t < ntr; t += 32) {
      const double x = at(t);
      if (!NANMODE || !isnan(x)) s += x;
    }
    s = warp_sum(s);
    mean = NANMODE ? s / cnt : s / ntr;
    double c = 0.0, ss = 0.0;
    for (int t = lane; t < ntr; t += 32) {
      const double d = at(t) - mean;
      if (!NANMODE || !isnan(d)) {
        c += d;
        ss += d * d;
      }
    }
    c = warp_sum(c);
    ss = warp_sum(ss);
    scale = sf_scale_from(NANMODE ? cnt : static_cast<double>(ntr), mean, c, ss, var);
  }
  double z2 = 0.0;
  for (int t = lane; t < ntr; t += 32) {
    double z = at(t);
    if (standardize) {
      z = z - mean;
      z = z / scale;
    }
    dst[t] = z;
    if (!NANMODE || !isnan(z)) z2 = fma(z, z, z2);
  }
  z2 = warp_sum(z2);
  if (lane == 0) {
    *mean_out = mean;
    *var_out = var;
    *scale_out = scale;
    if constexpr (NANMODE) *cnt_out = cnt;
  }
  return z2;
}

__shared__ int s_fit;   // slot mode: the fit thread 0 claimed for the CTA
__shared__ int s_ycol;  // NaN mode: the Y column the Y scores start from (mbpls.py:832-836)
__shared__ double s_cn[SF_MAXK], s_fac[SF_MAXK];  // NaN mode: |w~_k|; Gauss-Jordan row factors
__shared__ int s_piv;                             // NaN mode: pivot row
__shared__ int s_prow[3];  // block permutation, held-out sample: the permuted block's features [lo, hi) and their row

// The fit the calling CTA runs, and its workspace: the fit in per-fit mode, the CTA's slot in slot mode.  Derived again where
// needed rather than held in registers through the component loop (the kernel has none to spare).
__device__ __forceinline__ int sf_cur_fit(const mbpls_smallfit_args& a) { return a.nslots > 0 ? s_fit : static_cast<int>(blockIdx.x); }
__device__ __forceinline__ size_t sf_cur_ws(const mbpls_smallfit_args& a) { return a.nslots > 0 ? blockIdx.x : sf_cur_fit(a); }

// The fit's refit / singular flag, the last entry of its `small` block, derived afresh where needed (NaN mode: no register
// holds it through the fit).
__device__ __forceinline__ double* sf_flag(const mbpls_smallfit_args& a) {
  return a.small + (static_cast<size_t>(sf_cur_fit(a)) + 1) * (static_cast<size_t>(a.K) * (a.q + 2 * a.B + 4) + a.B + 2) - 1;
}

// Block permutation: the row map of fit f (perm_rows row r for fit_perm[f] = (r, b)) and the feature range [*lo, *hi) of
// block b, read through off (the block offsets); NULL and an empty range for a fit that permutes nothing.  Derived where it is
// used, like sf_cur_fit.
__device__ __forceinline__ const int* sf_block_map(const mbpls_smallfit_args& a, int f, const int* off, int* lo, int* hi) {
  *lo = *hi = 0;
  if (!a.fit_perm || a.fit_perm[2 * f] < 0) return nullptr;
  const int b = a.fit_perm[2 * f + 1];
  *lo = off[b];
  *hi = off[b + 1];
  return a.perm_rows + static_cast<size_t>(a.fit_perm[2 * f]) * a.n_src;
}

// One whole fit by the calling CTA: inputs and outputs (small, beta, fit_preds) of fit sf_cur_fit, workspace sf_cur_ws.
// NANMODE (sparse_data=True, mbpls.py:832-930): NaN entries stay NaN in the workspace copy and count as zero in every
// numerator; features / Y columns with a hole on the fit's rows, and samples with a hole in a block, divide by masked sums
// that the pass reading the element accumulates alongside (as xtu_kernel<true> / xw_kernel<true> / the NaN-mode epilogue).
template <bool NANMODE>
__device__ __forceinline__ void sf_fit(const mbpls_smallfit_args& a) {
  __shared__ double scratch[32 * 4];
  __shared__ __align__(16) double s_part[SF_THREADS];  // partial block scores [group][sample]
  __shared__ double s_nb[SF_MAXB], s_a[SF_MAXB], s_v[SF_MAXQ];
  __shared__ double s_sc[8];
  __shared__ int s_off[SF_MAXB + 1];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = a.p, B = a.B, q = a.q, K = a.K;
  const long ldw = a.ldw;
  const int f = sf_cur_fit(a);
  const size_t ws = sf_cur_ws(a);
  const int ntr = a.train_cnt ? a.train_cnt[f] : a.n_src;  // train_idx == NULL: every sample of the source, in order
  const int* __restrict__ tr = a.train_idx ? a.train_idx + static_cast<size_t>(f) * a.ld_idx : nullptr;
  const int* __restrict__ ytr = a.ytrain_idx ? a.ytrain_idx + static_cast<size_t>(f) * a.ld_idx : tr;

  double* Xw = a.Xw + ws * p * ldw;
  double* Yw = a.Yw + ws * q * ldw;
  double* stats = a.stats + ws * (4 * static_cast<size_t>(p) + 4 * q);
  double *xmean = stats, *xvar = stats + p, *xscale = stats + 2 * static_cast<size_t>(p), *xzss = stats + 3 * static_cast<size_t>(p);
  double *ymean = stats + 4 * static_cast<size_t>(p), *yvar = ymean + q, *yscale = ymean + 2 * q, *yzss = ymean + 3 * q;
  double* Wt = a.Wt + ws * K * p;
  double* W = a.W + ws * K * p;
  double* P = a.P + ws * K * p;
  double* Ts = a.Ts + ws * K * ldw;
  double* U = a.U + ws * K * ldw;
  double* Tb = a.Tb + ws * B * K * ldw;
  // small: V (K*q) | A (K*B) | pssb (K*B) | tt (K) | vv (K) | diff (K) | trips (K) | varxb (B) | vary (1) | singular (1)
  double* small = a.small + static_cast<size_t>(f) * (static_cast<size_t>(K) * (q + 2 * B + 4) + B + 2);
  double *V = small, *A = V + static_cast<size_t>(K) * q, *pssb = A + static_cast<size_t>(K) * B, *ttv = pssb + static_cast<size_t>(K) * B,
         *vvv = ttv + K, *diffv = vvv + K, *tripsv = diffv + K, *varxb = tripsv + K, *vary = varxb + B, *singular = vary + 1;
  // scratch vectors: u | ts | ts_old | T (B*ldw) | w (p)
  double* sv = a.scratch + ws * a.scratch_stride;
  double *u = sv, *ts = u + ldw, *ts_old = ts + ldw, *T = ts_old + ldw, *w = T + static_cast<size_t>(B) * ldw;
  // NaN mode, behind them: xobs (p) | yobs (q): observed counts on the fit's rows | rowhole (B*ldw: sample i has a hole in
  // block b) | G (K*K) | Gauss-Jordan workspace (K*2K) | prefix coefficients C_k (k*q for k = 1..K)
  double *xobs = w + p, *yobs = xobs + p, *rowhole = yobs + q;

  for (int b = tid; b <= B; b += SF_THREADS) s_off[b] = a.block_off[b];
  __syncthreads();

  // ---- prologue: gather + StandardScaler (mbpls.py:303-326), varx / vary (:822-830); the features of a permuted block
  // read their rows through its map (the census of NaN mode below is taken on this copy, so the holes move with the rows)
  {
    int plo, phi;
    const int* pmap = sf_block_map(a, f, s_off, &plo, &phi);
    for (int j = warp; j < p; j += SF_WARPS) {
      const double z2 = sf_ingest_feature<NANMODE>(a.Xsrc + static_cast<size_t>(j) * a.ldx, tr, j >= plo && j < phi ? pmap : nullptr,
                                                   ntr, Xw + static_cast<size_t>(j) * ldw, a.standardize, xmean + j, xvar + j,
                                                   xscale + j, xobs + j, lane);
      if (lane == 0) xzss[j] = z2;
    }
  }
  for (int c = warp; c < q; c += SF_WARPS) {
    const double z2 = sf_ingest_feature<NANMODE>(a.Ysrc + static_cast<size_t>(c) * a.ldx, ytr, nullptr, ntr,
                                                 Yw + static_cast<size_t>(c) * ldw, a.standardize, ymean + c, yvar + c,
                                                 yscale + c, yobs + c, lane);
    if (lane == 0) yzss[c] = z2;
  }
  for (int i = tid; i < ntr; i += SF_THREADS) ts_old[i] = 0.0;
  __syncthreads();
  for (int b = warp; b < B; b += SF_WARPS) {
    double s = 0.0;
    for (int j = s_off[b] + lane; j < s_off[b + 1]; j += 32) s += xzss[j];
    s = warp_sum(s);
    if (lane == 0) varxb[b] = s;
  }
  if (warp == SF_WARPS - 1) {
    double s = 0.0;
    for (int c = lane; c < q; c += 32) s += yzss[c];
    s = warp_sum(s);
    if (lane == 0) *vary = s;
  }
  if constexpr (NANMODE) {
    // census of the fit's rows: samples with a hole per block (the last block's also pick the masked Y-score rows, :903)
    for (int e = tid; e < B * ntr; e += SF_THREADS) {
      const int b = e / ntr, i = e - b * ntr;
      double hole = 0.0;
      for (int j = s_off[b]; j < s_off[b + 1]; ++j)
        if (isnan(Xw[static_cast<size_t>(j) * ldw + i])) hole = 1.0;
      rowhole[static_cast<size_t>(b) * ldw + i] = hole;
    }
    // the host refits through MBPLS.fit a fit with no fully observed Y column (the reference draws np.random.rand) or with
    // a feature / Y column that has no observed value on the fit's rows
    bool bad = false;
    for (int j = tid; j < p; j += SF_THREADS) bad |= !(xobs[j] > 0.0);
    for (int c = tid; c < q; c += SF_THREADS) bad |= !(yobs[c] > 0.0);
    if (tid == 0) {
      int c0 = -1;
      for (int c = q - 1; c >= 0; --c)
        if (yobs[c] == static_cast<double>(ntr)) c0 = c;
      s_ycol = c0;
      bad |= c0 < 0;
    }
    if (__syncthreads_or(bad)) {
      if (tid == 0) *sf_flag(a) = 1.0;
      return;
    }
  }

  // thread layout of the block-score pass: group g of samples-wide thread rows walks every G-th feature of a block
  int npad = 32;
  while (npad < ntr && npad < SF_THREADS) npad <<= 1;
  const int G = SF_THREADS / npad;          // >= 1
  const int gi = tid % npad, gg = tid / npad;  // sample lane, feature group

  for (int k = 0; k < K; ++k) {
    // u = first Y column (dense data, :838; NaN mode: the first one without a hole, :832-836), u'u
    double uu;
    {
      double acc = 0.0;
      const double* y0 = Yw;
      if constexpr (NANMODE) y0 += static_cast<size_t>(s_ycol) * ldw;
      for (int i = tid; i < ntr; i += SF_THREADS) {
        const double v0 = y0[i];
        u[i] = v0;
        acc = fma(v0, v0, acc);
      }
      uu = block_sum1(acc, scratch);
    }
    int trips = 0;
    double diff = 1.0, tt = 0.0, vv = 0.0;
    while (true) {  // :841
      // ---- block weights w~_j = x_j . u / u'u (:847-856) and their squared block norms (:860)
      for (int j = warp; j < p; j += SF_WARPS) {
        const double* x = Xw + static_cast<size_t>(j) * ldw;
        double s = 0.0;
        if constexpr (NANMODE) {  // masked u'u of a feature with a hole (:848-852)
          double d = 0.0;
          bool hole = false;
          for (int i = lane; i < ntr; i += 32) {
            const double xi = x[i];
            hole |= isnan(xi);
            if (!isnan(xi)) {
              s = fma(xi, u[i], s);
              d = fma(u[i], u[i], d);
            }
          }
          s = warp_sum(s);
          d = warp_sum(d);
          hole = __any_sync(0xffffffffu, hole);
          if (lane == 0) w[j] = hole ? s / d : s / uu;
        } else {
          for (int i = lane; i < ntr; i += 32) s = fma(x[i], u[i], s);
          s = warp_sum(s);
          if (lane == 0) w[j] = s / uu;
        }
      }
      __syncthreads();
      for (int b = warp; b < B; b += SF_WARPS) {
        double s = 0.0;
        for (int j = s_off[b] + lane; j < s_off[b + 1]; j += 32) s = fma(w[j], w[j], s);
        s = warp_sum(s);
        if (lane == 0) s_nb[b] = sqrt(s);
      }
      __syncthreads();
      // ---- block scores t_b = X_b w_b (:863-875); T'u (:879)
      for (int b = 0; b < B; ++b) {
        const double nb = s_nb[b];
        for (int i0 = 0; i0 < ntr; i0 += npad) {
          const int i = i0 + gi;
          double acc = 0.0;
          if constexpr (NANMODE) {  // masked sum of w~_j^2 of a sample with a hole in the block (:867-872)
            __shared__ double s_den[SF_THREADS];
            double den = 0.0;
            if (i < ntr)
              for (int j = s_off[b] + gg; j < s_off[b + 1]; j += G) {
                const double x = Xw[static_cast<size_t>(j) * ldw + i];
                if (!isnan(x)) {
                  acc = fma(x, w[j], acc);
                  den = fma(w[j], w[j], den);
                }
              }
            s_part[tid] = acc;
            s_den[tid] = den;
            __syncthreads();
            if (gg == 0 && i < ntr) {
              double t = 0.0, d = 0.0;
              for (int g = 0; g < G; ++g) {
                t += s_part[g * npad + gi];
                d += s_den[g * npad + gi];
              }
              // w_b = w~_b / nb, so sum_obs x w / sum_obs w^2 = nb * num / den (as the NaN-mode epilogue)
              T[static_cast<size_t>(b) * ldw + i] = rowhole[static_cast<size_t>(b) * ldw + i] != 0.0 ? nb * t / d : t / nb;
            }
          } else {
            if (i < ntr)
              for (int j = s_off[b] + gg; j < s_off[b + 1]; j += G) acc = fma(Xw[static_cast<size_t>(j) * ldw + i], w[j], acc);
            s_part[tid] = acc;
            __syncthreads();
            if (gg == 0 && i < ntr) {
              double t = 0.0;
              for (int g = 0; g < G; ++g) t += s_part[g * npad + gi];
              T[static_cast<size_t>(b) * ldw + i] = t / nb;
            }
          }
          __syncthreads();
        }
      }
      for (int b = warp; b < B; b += SF_WARPS) {
        double s = 0.0;
        for (int i = lane; i < ntr; i += 32) s = fma(T[static_cast<size_t>(b) * ldw + i], u[i], s);
        s = warp_sum(s);
        if (lane == 0) s_a[b] = s / uu;
      }
      __syncthreads();
      if (tid == 0) {  // superweights to unit length (:880)
        double s = 0.0;
        for (int b = 0; b < B; ++b) s = fma(s_a[b], s_a[b], s);
        s = sqrt(s);
        for (int b = 0; b < B; ++b) s_a[b] /= s;
      }
      __syncthreads();
      // ---- superscore ts = T a, unit length (:882-883); convergence metric (:884-888)
      double ss = 0.0;
      for (int i = tid; i < ntr; i += SF_THREADS) {
        double t = 0.0;
        for (int b = 0; b < B; ++b) t = fma(T[static_cast<size_t>(b) * ldw + i], s_a[b], t);
        ts[i] = t;
        ss = fma(t, t, ss);
      }
      ss = block_sum1(ss, scratch);
      const double tsn = sqrt(ss);
      double v4[4] = {0.0, 0.0, 0.0, 0.0};
      double dmax = 0.0, dmin = INFINITY;
      for (int i = tid; i < ntr; i += SF_THREADS) {
        const double t = ts[i] / tsn;
        const double d = ts_old[i] - t;
        ts[i] = t;
        ts_old[i] = t;
        v4[0] = fma(d, d, v4[0]);
        v4[1] += fabs(d);
        dmax = fmax(dmax, fabs(d));
        dmin = fmin(dmin, fabs(d));
        v4[3] = fma(t, t, v4[3]);
      }
      block_sum<4>(v4, scratch);
      dmax = warp_max(dmax);
      dmin = warp_min(dmin);
      __syncthreads();
      if (lane == 0) {
        scratch[warp] = dmax;
        scratch[32 + warp] = dmin;
      }
      __syncthreads();
      if (tid == 0) {
        double mx = 0.0, mn = INFINITY;
        for (int wv = 0; wv < SF_WARPS; ++wv) {
          mx = fmax(mx, scratch[wv]);
          mn = fmin(mn, scratch[32 + wv]);
        }
        double d;
        switch (a.norm_kind) {  // matrix norms of an n x 1 array (np.linalg.norm semantics, SURVEY.md a6')
          case MBPLS_NORM_L1: d = v4[1]; break;
          case MBPLS_NORM_MAX: d = mx; break;
          case MBPLS_NORM_MIN: d = mn; break;
          default: d = sqrt(v4[0]);
        }
        s_sc[0] = d;
      }
      __syncthreads();
      tt = v4[3];
      // ---- Y weights v = Y'ts / ts'ts (:899), Y scores u = Y v / v'v to unit length (:911-913)
      for (int c = warp; c < q; c += SF_WARPS) {
        double s = 0.0;
        if constexpr (NANMODE) {  // masked ts'ts of a Y column with a hole (:890-897)
          double d = 0.0;
          bool hole = false;
          for (int i = lane; i < ntr; i += 32) {
            const double yi = Yw[static_cast<size_t>(c) * ldw + i];
            hole |= isnan(yi);
            if (!isnan(yi)) {
              s = fma(yi, ts[i], s);
              d = fma(ts[i], ts[i], d);
            }
          }
          s = warp_sum(s);
          d = warp_sum(d);
          hole = __any_sync(0xffffffffu, hole);
          if (lane == 0) s_v[c] = hole ? s / d : s / tt;
        } else {
          for (int i = lane; i < ntr; i += 32) s = fma(Yw[static_cast<size_t>(c) * ldw + i], ts[i], s);
          s = warp_sum(s);
          if (lane == 0) s_v[c] = s / tt;
        }
      }
      __syncthreads();
      if (tid == 0) {
        double s = 0.0;
        for (int c = 0; c < q; ++c) s = fma(s_v[c], s_v[c], s);
        s_sc[1] = s;
      }
      __syncthreads();
      vv = s_sc[1];
      double un = 0.0;
      for (int i = tid; i < ntr; i += SF_THREADS) {
        double num = 0.0, val;
        if (NANMODE && rowhole[static_cast<size_t>(B - 1) * ldw + i] != 0.0) {
          // samples with a hole in the LAST X block use the observed Y columns only (the reference indexes
          // sparse_X_info_[block] with the block left over from :863, at :903); every other sample divides by v'v
          double den = 0.0;
          for (int c = 0; c < q; ++c) {
            const double yi = Yw[static_cast<size_t>(c) * ldw + i];
            if (!isnan(yi)) {
              num = fma(yi, s_v[c], num);
              den = fma(s_v[c], s_v[c], den);
            }
          }
          val = num / den;
        } else {
          for (int c = 0; c < q; ++c) num = fma(Yw[static_cast<size_t>(c) * ldw + i], s_v[c], num);
          val = num / vv;
        }
        u[i] = val;
        un = fma(val, val, un);
      }
      un = block_sum1(un, scratch);
      const double unorm = sqrt(un);
      double uun = 0.0;
      for (int i = tid; i < ntr; i += SF_THREADS) {
        const double val = u[i] / unorm;
        u[i] = val;
        uun = fma(val, val, uun);
      }
      uu = block_sum1(uun, scratch);
      ++trips;
      if (trips > 1) {  // the first trip has nothing to compare with (:884-885)
        diff = s_sc[0];
        if (!(diff > a.max_tol)) break;
      }
      if (trips >= a.max_iter) break;
      __syncthreads();
    }
    __syncthreads();
    // ---- loadings p_j = x_j . ts (:920), rank-1 deflation x_j -= ts p_j (:969), bookkeeping (:975-983)
    for (int j = warp; j < p; j += SF_WARPS) {
      double* x = Xw + static_cast<size_t>(j) * ldw;
      double s = 0.0, pj;
      if constexpr (NANMODE) {  // a feature with a hole divides by its masked ts'ts (:923-925); NaN stays NaN below
        double d = 0.0;
        bool hole = false;
        for (int i = lane; i < ntr; i += 32) {
          const double xi = x[i];
          hole |= isnan(xi);
          if (!isnan(xi)) {
            s = fma(xi, ts[i], s);
            d = fma(ts[i], ts[i], d);
          }
        }
        s = warp_sum(s);
        d = warp_sum(d);
        pj = __any_sync(0xffffffffu, hole) ? s / d : s;
      } else {
        for (int i = lane; i < ntr; i += 32) s = fma(x[i], ts[i], s);
        pj = warp_sum(s);
      }
      for (int i = lane; i < ntr; i += 32) x[i] = __dsub_rn(x[i], __dmul_rn(ts[i], pj));  // ts*p is rounded first (:969)
      if (lane == 0) {
        P[static_cast<size_t>(k) * p + j] = pj;
        const double wt = w[j];
        Wt[static_cast<size_t>(k) * p + j] = wt;
        int b = 0;
        while (b + 1 < B && j >= s_off[b + 1]) ++b;
        W[static_cast<size_t>(k) * p + j] = wt / s_nb[b];
      }
    }
    for (int i = tid; i < ntr; i += SF_THREADS) {
      Ts[static_cast<size_t>(k) * ldw + i] = ts[i];
      U[static_cast<size_t>(k) * ldw + i] = u[i];
      for (int b = 0; b < B; ++b) Tb[(static_cast<size_t>(b) * K + k) * ldw + i] = T[static_cast<size_t>(b) * ldw + i];
    }
    if (tid < q) V[static_cast<size_t>(k) * q + tid] = s_v[tid];
    if (tid < B) A[static_cast<size_t>(k) * B + tid] = s_a[tid] * s_a[tid];
    if (tid == 0) {
      ttv[k] = tt;
      vvv[k] = vv;
      diffv[k] = diff;
      tripsv[k] = static_cast<double>(trips);
    }
    __syncthreads();
    for (int b = warp; b < B; b += SF_WARPS) {
      double s = 0.0;
      for (int j = s_off[b] + lane; j < s_off[b + 1]; j += 32) {
        const double pj = P[static_cast<size_t>(k) * p + j];
        s = fma(pj, pj, s);
      }
      s = warp_sum(s);
      if (lane == 0) pssb[static_cast<size_t>(k) * B + b] = s;
    }
    __syncthreads();
  }

  // ---- R = W (P'W)^-1 and beta = R V' (:986-989): W = concat(W_non_normal) / column norm; P'W is upper triangular for
  // NIPALS, so r_k follows by substitution over k (and the leading blocks give every prefix model).  A (near-)singular P'W --
  // more components than the data has rank -- is flagged instead: the host then applies the pseudo-inverse like the reference.
  double* R = a.R + sf_cur_ws(a) * K * p;
  double* beta = a.beta ? a.beta + static_cast<size_t>(sf_cur_fit(a)) * q * p : nullptr;
  double dmin_abs = INFINITY, dmax_abs = 0.0;
  // NaN mode: the superscores are not orthogonal, so P'W is a full matrix and the leading block of R does not give the prefix
  // models.  Every prefix k inverts its own k x k block G_k = P_k'W_k (Gauss-Jordan, partial pivoting) and keeps the
  // coefficients C_k = G_k^-1 V_k (k x q) of y_hat_k(z) = sum_{i<k} (z . w_i) C_k[i]; R = W G_K^-1.  The pivots take the place
  // of the diagonal in the singularity test.
  double* PW = rowhole + static_cast<size_t>(B) * ldw;  // G = P'W, K x K
  double* M = PW + static_cast<size_t>(K) * K;          // [G_k | I] -> [I | G_k^-1], k rows of stride 2K
  double* Cs = M + 2 * static_cast<size_t>(K) * K;      // C_k at k (k - 1) / 2 * q
  if constexpr (NANMODE) {
    const int ldm = 2 * K;
    for (int k = 0; k < K; ++k) {
      double s = 0.0;
      for (int j = tid; j < p; j += SF_THREADS) {
        const double wt = Wt[static_cast<size_t>(k) * p + j];
        s = fma(wt, wt, s);
      }
      s = block_sum1(s, scratch);
      if (tid == 0) s_cn[k] = sqrt(s);
    }
    __syncthreads();
    for (int e = warp; e < K * K; e += SF_WARPS) {  // G[i][j] = p_i . w~_j / |w~_j|
      const int i = e / K, j = e - i * K;
      double s = 0.0;
      for (int l = lane; l < p; l += 32) s = fma(P[static_cast<size_t>(i) * p + l], Wt[static_cast<size_t>(j) * p + l], s);
      s = warp_sum(s);
      if (lane == 0) PW[e] = s / s_cn[j];
    }
    __syncthreads();
    for (int k = 1; k <= K; ++k) {
      for (int e = tid; e < 2 * k * k; e += SF_THREADS) {
        const int r = e / (2 * k), c = e - r * 2 * k;
        M[r * ldm + c] = c < k ? PW[r * K + c] : (c - k == r ? 1.0 : 0.0);
      }
      __syncthreads();
      for (int col = 0; col < k; ++col) {
        if (tid == 0) {
          int best_r = col;
          double best = fabs(M[col * ldm + col]);
#pragma unroll 1  // (unrolled, the search is where the NaN instantiation runs out of its 64 registers)
          for (int r = col + 1; r < k; ++r) {
            const double v = fabs(M[r * ldm + col]);
            if (v > best) {
              best = v;
              best_r = r;
            }
          }
          s_piv = best_r;
          dmin_abs = fmin(dmin_abs, best);
          dmax_abs = fmax(dmax_abs, best);
        }
        __syncthreads();
        const int pr = s_piv;
        if (pr != col)
          for (int c = tid; c < 2 * k; c += SF_THREADS) {
            const double t = M[col * ldm + c];
            M[col * ldm + c] = M[pr * ldm + c];
            M[pr * ldm + c] = t;
          }
        __syncthreads();
        const double pv = M[col * ldm + col];
        for (int r = tid; r < k; r += SF_THREADS) s_fac[r] = M[r * ldm + col];
        __syncthreads();
        for (int c = tid; c < 2 * k; c += SF_THREADS) M[col * ldm + c] /= pv;
        __syncthreads();
        for (int e = tid; e < 2 * k * k; e += SF_THREADS) {
          const int r = e / (2 * k), c = e - r * 2 * k;
          if (r != col) M[r * ldm + c] -= s_fac[r] * M[col * ldm + c];
        }
        __syncthreads();
      }
      double* Ck = Cs + static_cast<size_t>(k) * (k - 1) / 2 * q;
      for (int e = tid; e < k * q; e += SF_THREADS) {
        const int i = e / q, c = e - i * q;
        double s = 0.0;
        for (int j = 0; j < k; ++j) s = fma(M[i * ldm + k + j], V[static_cast<size_t>(j) * q + c], s);
        Ck[e] = s;
      }
      __syncthreads();
    }
    for (int j = tid; j < p; j += SF_THREADS)  // M holds G_K^-1
      for (int c = 0; c < K; ++c) {
        double acc = 0.0;
        for (int i = 0; i < K; ++i) acc = fma(Wt[static_cast<size_t>(i) * p + j] / s_cn[i], M[i * ldm + K + c], acc);
        R[static_cast<size_t>(c) * p + j] = acc;
      }
    __syncthreads();
  } else {
    for (int k = 0; k < K; ++k) {
      double s = 0.0;
      for (int j = tid; j < p; j += SF_THREADS) {
        const double wt = Wt[static_cast<size_t>(k) * p + j];
        s = fma(wt, wt, s);
      }
      s = block_sum1(s, scratch);
      const double cn = sqrt(s);
      for (int j = tid; j < p; j += SF_THREADS) R[static_cast<size_t>(k) * p + j] = Wt[static_cast<size_t>(k) * p + j] / cn;
      __syncthreads();
      for (int jj = 0; jj < k; ++jj) {  // r_k -= r_jj (p_jj . w_k);  w_k is still intact in R[k] only before the updates: use Wt/cn
        double d = 0.0;
        for (int j = tid; j < p; j += SF_THREADS) d = fma(P[static_cast<size_t>(jj) * p + j], Wt[static_cast<size_t>(k) * p + j] / cn, d);
        d = block_sum1(d, scratch);
        for (int j = tid; j < p; j += SF_THREADS) R[static_cast<size_t>(k) * p + j] -= R[static_cast<size_t>(jj) * p + j] * d;
        __syncthreads();
      }
      double d = 0.0;
      for (int j = tid; j < p; j += SF_THREADS) d = fma(P[static_cast<size_t>(k) * p + j], Wt[static_cast<size_t>(k) * p + j] / cn, d);
      d = block_sum1(d, scratch);
      dmin_abs = fmin(dmin_abs, fabs(d));
      dmax_abs = fmax(dmax_abs, fabs(d));
      for (int j = tid; j < p; j += SF_THREADS) R[static_cast<size_t>(k) * p + j] /= d;
      __syncthreads();
    }
  }
  for (int j = tid; beta && j < p; j += SF_THREADS) {
    for (int c = 0; c < q; ++c) {
      double acc = 0.0;
      for (int k = 0; k < K; ++k) acc = fma(R[static_cast<size_t>(k) * p + j], V[static_cast<size_t>(k) * q + c], acc);
      beta[static_cast<size_t>(c) * p + j] = acc;
    }
  }
  if (tid == 0) *(NANMODE ? sf_flag(a) : singular) = (!(dmin_abs > 1e-10 * dmax_abs) || !isfinite(dmax_abs)) ? 1.0 : 0.0;

  // ---- held-out predictions for every prefix of the model (cross-validation)
  if ((!a.preds && !a.fit_preds) || !a.test_idx) return;
  __syncthreads();
  const int fit = sf_cur_fit(a);
  const int nte = a.test_cnt[fit];
  const int* __restrict__ te = a.test_idx + static_cast<size_t>(fit) * a.ld_tidx;
  // y_hat_k(x) = sum_{j<=k} (z . r_j) v_j, z the standardised sample; back to the Y scale (:1386)
  for (int t = 0; t < nte; ++t) {
    const int idx = te[t];
    if (a.fit_perm) {  // a permuted block's features of the held-out sample come from its mapped row (kept in shared memory:
                       // the NaN instantiation has no register to spare here)
      if (tid == 0) {
        int lo, hi;
        const int* m = sf_block_map(a, fit, s_off, &lo, &hi);
        s_prow[0] = lo;
        s_prow[1] = hi;
        s_prow[2] = m ? m[idx] : idx;
      }
      __syncthreads();
    }
    for (int k = warp; k < K; k += SF_WARPS) {
      double s = 0.0;
      for (int j = lane; j < p; j += 32) {
        double z = a.Xsrc[static_cast<size_t>(j) * a.ldx + (a.fit_perm && j >= s_prow[0] && j < s_prow[1] ? s_prow[2] : idx)];
        if (a.standardize) z = (z - xmean[j]) / xscale[j];
        if constexpr (NANMODE) {  // NaN counts as zero after scaling (:1379-1384); s_part[k] = z . w_k
          if (isnan(z)) z = 0.0;
          s = fma(z, Wt[static_cast<size_t>(k) * p + j], s);
        } else {
          s = fma(z, R[static_cast<size_t>(k) * p + j], s);
        }
      }
      s = warp_sum(s);
      if (lane == 0) s_part[k] = NANMODE ? s / s_cn[k] : s;
    }
    __syncthreads();
    // preds[k][idx][c] (by sample) or fit_preds[f][k][t][c] (by position in the fit's test list)
    double* dst = a.preds ? a.preds + static_cast<size_t>(idx) * q : a.fit_preds + (static_cast<size_t>(fit) * K * a.ld_tidx + t) * q;
    const size_t kstep = static_cast<size_t>(a.preds ? a.n_src : a.ld_tidx) * q;
    if constexpr (NANMODE) {
      for (int e = tid; e < K * q; e += SF_THREADS) {
        const int k = e / q, c = e - k * q;
        const double* Ck = Cs + static_cast<size_t>(k + 1) * k / 2 * q;
        double acc = 0.0;
        for (int i = 0; i <= k; ++i) acc = fma(s_part[i], Ck[i * q + c], acc);
        dst[k * kstep + c] = a.standardize ? acc * yscale[c] + ymean[c] : acc;
      }
    } else {
      for (int c = tid; c < q; c += SF_THREADS) {
        double acc = 0.0;
        for (int k = 0; k < K; ++k) {
          acc = fma(s_part[k], V[static_cast<size_t>(k) * q + c], acc);
          const double yh = a.standardize ? acc * yscale[c] + ymean[c] : acc;
          dst[k * kstep + c] = yh;
        }
      }
    }
    __syncthreads();
  }
}

// Both modes go through the one inlined copy of sf_fit, so a fit compiles to the same instructions in either.
template <bool NANMODE>
__global__ void __launch_bounds__(SF_THREADS, 1) smallfit_kernel(const mbpls_smallfit_args a) {
  while (true) {
    if (a.nslots > 0) {  // thread 0 claims the next fit for the whole CTA
      if (threadIdx.x == 0) s_fit = atomicAdd(a.ticket, 1);
      __syncthreads();
      if (s_fit >= a.nfits) return;
    }
    sf_fit<NANMODE>(a);
    if (a.nslots == 0) return;
    __syncthreads();  // the slot's workspace, s_fit and the shared arrays are reused by the next fit
  }
}

}  // namespace

extern "C" {

int mbpls_smallfit_scratch_doubles(int p, int B, long ldw) {
  const long v = 3 * ldw + static_cast<long>(B) * ldw + p;
  return v > 0x7fffffffL ? -1 : static_cast<int>(v);
}

int mbpls_smallfit_nan_scratch_doubles(int p, int q, int B, int K, long ldw) {
  const int dense = mbpls_smallfit_scratch_doubles(p, B, ldw);
  if (dense < 0 || p < 0 || q < 0 || B < 0 || K < 0 || K > SF_MAXK) return -1;
  const long Kl = K, v = dense + static_cast<long>(B) * ldw + p + q + 3 * Kl * Kl + Kl * (Kl + 1) / 2 * q;
  return v > 0x7fffffffL ? -1 : static_cast<int>(v);
}

int mbpls_smallfit_nipals_f64(const mbpls_smallfit_args* a, void* stream) {
  if (!a || !a->Xsrc || !a->Ysrc || !a->block_off || (a->train_idx && !a->train_cnt) || !a->Xw || !a->Yw || !a->stats || !a->Wt ||
      !a->W || !a->P || !a->Ts || !a->U || !a->Tb || !a->small || !a->R || (!a->beta && a->nslots == 0) || !a->scratch)
    return MBPLS_ERR_ARG;
  if (a->nslots < 0 || (a->nslots > 0 && (!a->ticket || a->preds))) return MBPLS_ERR_ARG;  // preds: test sets may overlap
  if ((a->ytrain_idx && !a->train_idx) || (a->fit_preds && (a->preds || !a->test_idx || !a->test_cnt))) return MBPLS_ERR_ARG;
  if (a->B < 1 || a->B > SF_MAXB || a->q < 1 || a->q > SF_MAXQ || a->K < 1 || a->K > SF_THREADS || a->p < 1 || a->nfits < 1 ||
      (a->nanmode && a->K > SF_MAXK))
    return MBPLS_ERR_SIZE;
  if (a->preds && (!a->test_idx || !a->test_cnt)) return MBPLS_ERR_ARG;
  if (!a->train_idx && (a->nfits != 1 || a->ldw < a->n_src)) return MBPLS_ERR_ARG;
  const int need = a->nanmode ? mbpls_smallfit_nan_scratch_doubles(a->p, a->q, a->B, a->K, a->ldw)
                              : mbpls_smallfit_scratch_doubles(a->p, a->B, a->ldw);
  if (need < 0 || a->scratch_stride < need) return MBPLS_ERR_ARG;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (a->perm_rows || a->fit_perm) {  // block permutation: every (r, b) pair must name a row of perm_rows and a block
    if (!a->perm_rows || !a->fit_perm || !a->train_idx || a->n_perm < 1) return MBPLS_ERR_ARG;
    std::vector<int> pairs(2 * static_cast<size_t>(a->nfits));
    cudaError_t e = cudaMemcpyAsync(pairs.data(), a->fit_perm, pairs.size() * sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return MBPLS_CUDA_ERR(e);
    for (int f = 0; f < a->nfits; ++f) {
      const int r = pairs[2 * f], b = pairs[2 * f + 1];
      if (r < -1 || r >= a->n_perm || (r >= 0 && (b < 0 || b >= a->B))) return MBPLS_ERR_ARG;
    }
  }
  if (a->nslots > 0) {
    const cudaError_t e = cudaMemsetAsync(a->ticket, 0, sizeof(int), st);
    if (e != cudaSuccess) return MBPLS_CUDA_ERR(e);
  }
  const int grid = a->nslots > 0 ? a->nslots : a->nfits;
  if (a->nanmode) smallfit_kernel<true><<<grid, SF_THREADS, 0, st>>>(*a);
  else smallfit_kernel<false><<<grid, SF_THREADS, 0, st>>>(*a);
  MBPLS_RETURN_LAST();
}

}  // extern "C"
