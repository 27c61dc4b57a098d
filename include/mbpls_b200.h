/*
 * mbpls_b200 -- C ABI of the B200 (sm_100a) kernels behind the MB-PLS latent-variable fitting path.
 *
 * The reference (DTUComputeStatisticsAndDataAnalysis/MBPLS v1.0.4) is pure Python and has NO plugin /
 * FFI / operator interface to mirror (SURVEY.md section 8b): its boundary is the sklearn-style class
 * `mbpls.mbpls.MBPLS` (mbpls/mbpls.py:22).  This header therefore *defines* the entry points a binding
 * for that class calls; every function cites the region of mbpls/mbpls.py whose numpy / scipy /
 * scikit-learn calls it replaces.  The Python host class `mbpls_b200.MBPLS` binds them with ctypes
 * (mbpls_b200/_cabi.py); INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless the name ends in `_host` or the doc says otherwise.
 *  - All matrices are float64 and FEATURE-MAJOR: a p x ld array with one feature (one column of the
 *    reference's n x p matrix) per row, ld >= n, ld % 16 == 0, padding [n, ld) zero.  Result matrices
 *    are COMPONENT-MAJOR (K x p or K x ld).  n-vectors have at least ld elements.
 *  - `stream` is a cudaStream_t passed as void*.  Functions never allocate, never synchronise and keep
 *    no global state; they return 0, a negative MBPLS_ERR_* code for bad arguments, or
 *    1000 + cudaError_t for a launch failure.
 *  - `done` arguments point at the int ctrl[MBPLS_CTRL_DONE] of a NIPALS component; when it is
 *    non-zero the kernel returns immediately (lets the host enqueue trips in batches).
 */
#ifndef MBPLS_B200_H
#define MBPLS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MBPLS_ABI_VERSION 16

/* indices into the per-fit scalar / control buffers */
#define MBPLS_SCAL_UU 0    /* u'u of the current Y-score vector (mbpls.py:847,856,879) */
#define MBPLS_SCAL_DIFF 1  /* last diff_t (mbpls.py:887) */
#define MBPLS_SCAL_TT 2    /* ts'ts */
#define MBPLS_SCAL_VV 3    /* v'v */
#define MBPLS_SCAL_COUNT 8
#define MBPLS_CTRL_DONE 0  /* 1 once diff_t <= max_tol (mbpls.py:841) */
#define MBPLS_CTRL_TRIPS 1 /* completed trips of the while loop for this component */
#define MBPLS_CTRL_ERROR 2 /* sticky: a peer GPU did not arrive at an in-kernel exchange (mbpls_nipals_xchg_epilogue_f64) */
#define MBPLS_CTRL_COUNT 4

/* nipals_convergence_norm: matrix-norm semantics of np.linalg.norm on an n x 1 array (mbpls.py:887) */
#define MBPLS_NORM_L2 0  /* ord = 2, -2, 'fro', 'nuc' */
#define MBPLS_NORM_L1 1  /* ord = 1, -1 */
#define MBPLS_NORM_MAX 2 /* ord = inf */
#define MBPLS_NORM_MIN 3 /* ord = -inf */

int mbpls_abi_version(void);

/* ---- ingest (mbpls.py:301-323 check_array copies, :379 hstack) ---------------------------------- */
/* row-major chunk (rows x cols, leading dim lds) -> feature-major dst[c*ld + row0 + r] */
int mbpls_transpose_in_f64(const double* src, long lds, int rows, int cols, double* dst, long ld, int row0, void* stream);
/* same from a single-precision row-major source: check_array(dtype=float64) (mbpls.py:310) widens float32 inputs on the
 * host; here they cross PCIe at half the size and are widened inside the transposition */
int mbpls_transpose_in_f32(const float* src, long lds, int rows, int cols, double* dst, long ld, int row0, void* stream);
/* feature-major -> row-major */
int mbpls_transpose_out_f64(const double* src, long ld, int rows, int cols, double* dst, long ldd, int row0, void* stream);

/* ---- NaN census: MBPLS.check_sparsity_level (mbpls.py:255-271) and check_array's finiteness test (:310,:336) ----
 * col_nan[j] = number of NaNs in feature j; row_flag[b*ldf + i] = 1 if sample i has a NaN in block b
 * (optional; must be zeroed by the caller); *inf_flag = 1 if any element is +-inf (optional).
 * block_off: B+1 ascending local feature offsets. */
int mbpls_nan_census_f64(const double* Xt, long ld, int n, int p, const int* block_off, int B, int* col_nan,
                         unsigned char* row_flag, long ldf, int* inf_flag, void* stream);

/* ---- StandardScaler.fit_transform on every feature, in place (mbpls.py:307,314,325-326) ----------
 * Outputs per feature: mean_, var_, scale_, n_samples_seen_ and nansum(z^2) (feeds varx, :826-829).
 * mode 0: feature-resident bulk-copy pipeline (1 read + 1 write) when a feature fits in shared
 * memory, otherwise the global-memory fallback; mode 1 forces the fallback. */
int mbpls_standardize_fit_f64(double* Xt, long ld, int n, int p, double* mean, double* var, double* scale,
                              long long* seen, double* zss, int mode, void* stream);
/* StandardScaler.transform on new data (mbpls.py:1097,1103,1125,1369,1372) */
int mbpls_standardize_apply_f64(double* Xt, long ld, int n, int p, const double* mean, const double* scale, void* stream);
/* y_scaler_.inverse_transform (mbpls.py:1384,1386) on a feature-major q x ld array */
int mbpls_scaler_inverse_f64(double* Zt, long ld, int n, int q, const double* mean, const double* scale, void* stream);
/* nansum(x_j^2) per feature: (X**2).sum() / np.nansum (mbpls.py:826-830, :943-945) */
int mbpls_feature_sumsq_f64(const double* Xt, long ld, int n, int p, double* out, void* stream);
/* row-sharded StandardScaler: var_/scale_ from the all-reduced centred sums sum(x-mean), sum((x-mean)^2) */
int mbpls_scaler_finish_f64(const double* corr, const double* ssq, const double* mean, double count, double* var, double* scale,
                            int p, void* stream);
/* deterministic segmented sum out[s] = sum v[off[s]:off[s+1]] */
int mbpls_segsum_f64(const double* v, const int* off, int nseg, double* out, void* stream);

/* ---- NIPALS inner loop (mbpls.py:841-914) -------------------------------------------------------- */
int mbpls_xtu_feats_per_cta(int p);
int mbpls_xtu_num_ctas(int p); /* rows of norm_part */
int mbpls_xw_ctas_per_sm(void); /* resident CTAs per SM of the sample-owning kernels: size grids to one wave */

/* w[j] = x_j . u / u'u (mbpls.py:847,856); NaN mode: masked ratio for features with NaN (:848-852).
 * uu == NULL: no division for fully observed features (the loadings of :920,:928).
 * norm_part[cta*B + b] = partial ||w_b||^2 (may be NULL). */
int mbpls_nipals_xtu_f64(const double* Xt, long ld, int n, int p, const double* u, const double* uu, const int* block_off,
                         int B, double* w, double* norm_part, int nanmode, const int* done, void* stream);
/* same partial norms for a w produced elsewhere (fused deflation) */
int mbpls_block_sumsq_parts_f64(const double* w, int p, const int* block_off, int B, double* norm_part, const int* done,
                                void* stream);
/* Tnum[s][i] = sum_{j in split s} w_j x_ij (mbpls.py:866,875); NaN mode also Tden[s][i] = masked sum of
 * w_j^2 (:867-872).  split s covers local features [split_f0[s], split_f1[s]) of a single block. */
int mbpls_nipals_xw_f64(const double* Xt, long ld, int n, const double* w, const int* split_f0, const int* split_f1,
                        int nsplit, double* Tnum, double* Tden, long ldt, int nanmode, const int* done, void* stream);
/* red = [B x ldt numerators | B x ldt denominators (NaN mode) | B squared block-weight norms]:
 * fixed-order sums over the splits of each block / over the xtu CTAs.  This is the buffer that is
 * all-reduced over NVLink when features are sharded across GPUs. */
int mbpls_nipals_reduce_partials_f64(const double* Tnum, const double* Tden, long ldt, int n, int B,
                                     const int* block_split_off, const double* norm_part, int n_norm_parts, double* red,
                                     int nanmode, const int* done, void* stream);
static inline long mbpls_red_elems(int B, long ldt, int nanmode) { return (long)(nanmode ? 2 : 1) * B * ldt + B; }

/* u <- u0, u'u, trips = 0, diff = 1, done = 0 (mbpls.py:832-840) */
int mbpls_nipals_begin_component_f64(const double* u0, int n, double* u, double* scal, int* ctrl, void* stream);

typedef struct mbpls_epilogue_args {
  int n, B, q, nanmode, norm_kind;
  long ldt, ldf;
  double max_tol;
  const double* red;             /* reduced partials, layout above */
  const double* Yt;              /* q x ldt */
  const unsigned char* row_flag; /* B x ldf, NaN mode */
  const unsigned char* ycol_flag;/* q, NaN mode: Y column has a NaN */
  double* T;                     /* B x ldt  block scores t_b of this trip (mbpls.py:863-875) */
  double* u;                     /* n  in: u of this trip, out: next u (:901-913) */
  double* ts;                    /* n  superscores (:882-883) */
  double* ts_old;                /* n  superscores_old (:888) */
  double* a;                     /* B  superweights (:879-880) */
  double* v;                     /* q  Y weights (:890-899) */
  double* scal;                  /* MBPLS_SCAL_COUNT */
  int* ctrl;                     /* MBPLS_CTRL_COUNT */
  double* diff_trace;            /* optional diff_t per trip */
  int diff_trace_len;
} mbpls_epilogue_args;
/* `args` is a HOST pointer; the struct is passed to the kernel by value. */
int mbpls_nipals_epilogue_f64(const mbpls_epilogue_args* args_host, void* stream);

/* reduce_partials + exchange between the GPUs + epilogue as ONE kernel (csrc/nipals.cu xchg_epilogue_kernel).
 * world == 1: the split partials are summed straight into epi.red and the last CTA runs the epilogue.
 * world > 1 (features sharded): peer_bufs is a DEVICE array of `world` addresses, entry r = rank r's symmetric buffer as
 * mapped into this process (peer memory over NVLink; torch.distributed._symmetric_memory hands out such arrays).  A buffer
 * holds 2 slots of slot_elems doubles followed, at flags_off doubles, by `world` 8-byte flag words (zero before the first
 * call).  seq > 0 must grow by one per call and be the same on every rank; every rank must make the same calls.  The sums
 * over the GPUs are formed in rank order on every GPU, i.e. bit-identical everywhere (replaces ncclAllReduce of epi.red,
 * SURVEY.md 8e).  counters: 2 zeroed unsigned ints in local memory.  On a peer timeout ctrl[MBPLS_CTRL_ERROR] is set. */
typedef struct mbpls_xchg_args {
  mbpls_epilogue_args epi;
  const double* Tnum;            /* [nsplit][ldp] split partials (as for mbpls_nipals_reduce_partials_f64) */
  const double* Tden;            /* NaN mode */
  long ldp;
  const int* block_split_off;    /* B + 1 */
  const double* norm_part;       /* [n_norm_parts][B] */
  int n_norm_parts;
  int world, rank;
  const unsigned long long* peer_bufs;
  long slot_elems, flags_off;
  unsigned long long seq;
  unsigned int* counters;
  double* work;                  /* optional: 32768 doubles of scratch, zero before the first call.  With it (and epoch > 0),
                                    dense fits with B <= 8, q <= 16 and n <= 1024 * CTAs spread the superlevel step over all
                                    CTAs of the launch (grid-wide sums through this buffer) */
  unsigned long long epoch;      /* with `work`: 1, 2, 3, ... growing by one per call on this buffer */
  int tpi, ch;                   /* set by the library (warps sharing one split sum, samples per CTA); callers leave them 0 */
} mbpls_xchg_args;
int mbpls_nipals_xchg_epilogue_f64(const mbpls_xchg_args* args_host, int ctas, void* stream);

typedef struct mbpls_record_args {
  int n, p, B, q, nanmode;
  long ldt, T_block_stride;
  const int* block_off;
  const double *w, *red, *T, *ts, *u, *v, *a;
  double *Wt_k, *W_k, *Ts_k, *U_k, *T_k, *V_k, *A_k;
  const int* only_if_done; /* may be NULL; else the launch is a no-op unless *only_if_done is set (see mbpls_fused_deflate_f64) */
} mbpls_record_args;
/* append the converged component (mbpls.py:975-983): W_non_normal_, W_, Ts_, U_, T_, V_, A_ */
int mbpls_nipals_record_component_f64(const mbpls_record_args* args_host, void* stream);

/* p_j = x_j . ts (masked ratio for features with NaN) and X <- X - ts p' in place (mbpls.py:917-930,
 * :968-969).  pss[j] = p_j^2.  If u0 != NULL also w_next[j] = x_j(deflated) . u0 / u0'u0, i.e. the first
 * weights of the next component (:847,856 with u = u0).  mode as in mbpls_standardize_fit_f64. */
int mbpls_loadings_deflate_f64(double* Xt, long ld, int n, int p, const double* ts, const double* u0, const double* u0u0,
                               double* P_k, double* w_next, double* pss, int nanmode, int mode, void* stream);

/* ---- one-pass NIPALS kernels (csrc/fused.cu) ---------------------------------------------------------
 * A trip of the reference's loop reads X twice (X_b'u at mbpls.py:847/:856, then X_b w_b at :866/:875).  Because
 * w~_j depends on feature j and u only, and t~_b is a sum over features, both are produced while a feature is
 * resident on the SM: ONE read of X per trip.  "Workers" (groups of threads inside a persistent CTA) own one
 * split each -- a contiguous local feature range inside one block, split_block[s] = its block -- and keep the
 * n-vector of partial block scores in registers; outputs have the layout of mbpls_nipals_xw_f64 /
 * mbpls_nipals_xtu_f64 (Tnum[s][.], w[j]) and norm_part[s*B + split_block[s]] = sum of w~_j^2
 * over the split (all other entries of norm_part must be zero), so mbpls_nipals_reduce_partials_f64 and the
 * epilogue apply unchanged.  Features of up to 10,240 samples are handled by one CTA; the deflation pass of features
 * longer than 5,120 samples, and both passes of features of up to 20,480 samples, split every feature by samples over
 * the two CTAs of a thread-block cluster (each keeps half of ts / u0 / u in shared memory; partial dot products meet
 * through distributed shared memory).  mbpls_fused_total_workers(ld) returns the number of splits to build on the
 * current device (0: the feature is too long for the register-resident accumulators, use the two-pass kernels);
 * mbpls_fused_workers_per_sm_pair(ld) is the device-independent density behind it; mbpls_fused_uses_clusters(ld)
 * reports which passes run on CTA pairs (bit 0: trip, bit 1: deflation). */
int mbpls_fused_workers_per_sm_pair(long ld);
int mbpls_fused_total_workers(long ld);
int mbpls_fused_uses_clusters(long ld);
/* rden == NULL: dense data.  NaN mode: rden[j] = reciprocal masked denominator of feature j for this u
 * (mbpls_masked_colden_f64); NaN entries count as zero; the masked score denominators come from
 * mbpls_masked_rowden_f64 afterwards. */
int mbpls_nipals_fused_trip_f64(const double* Xt, long ld, int n, const double* u, const double* uu, const double* rden,
                                const int* split_f0, const int* split_f1, const int* split_block, int nsplit, int B, double* w,
                                double* norm_part, double* Tnum, long ldt, const int* done, void* stream);
/* Loadings p_j = x_j . ts and X <- X - ts p' (mbpls.py:917-930, :968-969) in place, and -- if u0 != NULL -- the complete
 * first trip of the next component (u restarts from u0, :838): w_next[j] = x_j(deflated) . u0 / u0'u0, its squared norms
 * and its partial block scores Tnum.  1 read + 1 write of X.  NaN mode (rden_ts != NULL): masked loadings / weights through
 * the reciprocal denominators rden_ts (for ts, dense features: 1) and rden_u0 (for u0); NaN entries stay NaN.
 * only_if_done != NULL: the launch is a no-op unless *only_if_done (ctrl[MBPLS_CTRL_DONE]) is set -- the host enqueues the
 * closing pass of a component behind its trips before it knows whether they converged, so the GPU never idles while the
 * host reads the flag back; if they did not, it enqueues more trips and the closing pass again. */
int mbpls_fused_deflate_f64(double* Xt, long ld, int n, const double* ts, const double* rden_ts, const double* u0,
                            const double* u0u0, const double* rden_u0, const int* split_f0, const int* split_f1,
                            const int* split_block, int nsplit, int B, double* P_k, double* pss, double* w_next, double* norm_part,
                            double* Tnum, long ldt, const int* only_if_done, void* stream);

/* StandardScaler.fit_transform of X in place (mbpls.py:307,314) fused with the complete first trip of the first component
 * (u = u0 = the first standardised Y column, :838): per-feature statistics as mbpls_standardize_fit_f64, first weights w,
 * norm_part and Tnum as mbpls_nipals_fused_trip_f64 -- 1 read + 1 write of X instead of 2 reads + 1 write.  Dense data,
 * features of up to 10,240 samples (MBPLS_ERR_SIZE otherwise: standardise and trip separately). */
int mbpls_fused_standardize_f64(double* Xt, long ld, int n, const double* u0, const double* u0u0, const int* split_f0,
                                const int* split_f1, const int* split_block, int nsplit, int B, double* mean, double* var,
                                double* scale, long long* seen, double* zss, double* w, double* norm_part, double* Tnum, long ldt,
                                void* stream);

/* ---- whole dense NIPALS fits in one kernel (csrc/smallfit.cu): one persistent CTA per fit, device-side while loop -----
 * For problems that are launch-latency bound through the streaming kernels (README quickstart, the leave-one-out loops of
 * the reference's notebooks).  Fit f uses the samples train_idx[f*ld_idx .. + train_cnt[f]) of the shared feature-major
 * source (Xsrc p x ldx, Ysrc q x ldx, raw values): gather + StandardScaler (mbpls.py:303-326), the NIPALS loop :821-983,
 * results per fit (component-major, sample vectors with leading dimension ldw >= max train_cnt):
 *   stats  [4p + 4q]  x mean | x var | x scale | x sum z^2 | y mean | y var | y scale | y sum z^2
 *   Wt, W, P  [K][p]   un-normalised weights, block-normalised weights, loadings
 *   Ts, U  [K][ldw],  Tb [B][K][ldw]
 *   small  [K(q + 2B + 4) + B + 2]  V (K x q) | A (K x B) | sum p_j^2 per block (K x B) | ts'ts (K) | v'v (K) | diff_t (K) |
 *                                   trips (K) | varx per block (B) | vary | singular
 *   R [K][p], beta [q][p]   R = W (P'W)^-1 by substitution (P'W is upper triangular for NIPALS) and beta = R V' (:986-989);
 *                           singular = 1 flags a (near-)singular P'W: apply the pseudo-inverse on the host side instead
 * train_idx == NULL (nfits == 1): the fit uses every sample of the source, in order.
 * Xw [nfits][p*ldw] / Yw [nfits][q*ldw] receive the standardised (then deflated) copies; scratch holds
 * mbpls_smallfit_scratch_doubles(...) doubles per fit (scratch_stride).  With preds != NULL the CTA also predicts the
 * samples test_idx[f*ld_tidx .. + test_cnt[f]) for every prefix of its model: preds[k][sample][c], k+1 components
 * (the leading blocks of P'W, :1386).  Dense data only.
 * Resampling (permutation tests, bootstrap); every field below left zero / NULL keeps the behaviour above:
 *   ytrain_idx  per fit, ld_idx wide, counts of train_cnt: the rows of Ysrc gathered for the fit (NULL: those of train_idx);
 *               X row train_idx[t] is paired with Y row ytrain_idx[t] (a permuted y, a bootstrap resample)
 *   fit_preds   held-out predictions per fit by position in its test list: fit_preds[((f*K + k)*ld_tidx + t)*q + c], k+1
 *               components, computed like preds (one of preds and fit_preds, not both)
 *   nslots      0: a grid of nfits CTAs, everything indexed by fit.  > 0: a grid of nslots persistent CTAs; each claims the
 *               next fit with atomicAdd(ticket, 1) until the claims reach nfits.  Xw, Yw, scratch, stats, Wt, W, P, Ts, U, Tb
 *               and R are then indexed by slot (the CTA), small, beta and fit_preds by fit; beta may be NULL (not written);
 *               preds (indexed by sample) is rejected.  A fit's results do not depend on the mode or on the slot that ran it.
 *   ticket      one int, zeroed on the launch stream by the entry point (slot mode only). */
typedef struct mbpls_smallfit_args {
  int n_src, p, B, q, K, nfits;
  long ldx;
  const double* Xsrc;
  const double* Ysrc;
  const int* block_off;
  int standardize, norm_kind, max_iter;
  double max_tol;
  const int* train_idx;
  const int* train_cnt;
  long ld_idx;
  const int* test_idx;
  const int* test_cnt;
  long ld_tidx;
  long ldw;
  double* Xw;
  double* Yw;
  double* stats;
  double* Wt;
  double* W;
  double* P;
  double* Ts;
  double* U;
  double* Tb;
  double* small;
  double* R;
  double* beta;
  double* preds;
  double* scratch;
  long scratch_stride;
  const int* ytrain_idx;
  double* fit_preds;
  int nslots;
  int* ticket;
} mbpls_smallfit_args;
int mbpls_smallfit_scratch_doubles(int p, int B, long ldw);
int mbpls_smallfit_nipals_f64(const mbpls_smallfit_args* args_host, void* stream);

/* ---- NaN bit matrix and the masked denominators derived from it (csrc/nanmask.cu; mbpls.py:848-852, :867-872, :923-925)
 * bits[j*ldw + (i >> 5)] bit (i & 31) = 1 iff x_ij is NaN; ldw = mbpls_nan_bitmask_ldw(n) 32-bit words per feature. */
int mbpls_nan_bitmask_ldw(int n);
int mbpls_nan_bitmask_f64(const double* Xt, long ld, int n, int p, unsigned* bits, long ldw, void* stream);
/* Masked column sums from the bit matrix.  m_j = *vv - sum_{i: x_ij NaN} v_i v2_i  (v2 == NULL: v2 = v), *vv = v . v2 over all
 * samples; fully observed features (col_nan[j] == 0, from mbpls_nan_census_f64) have m_j = *vv.
 * mode 0: out[j] = 1 / m_j for features with NaN, 1 for fully observed ones (dense loadings are not divided, :920)
 * mode 1: out[j] = 1 / m_j (weights, :847-852)          mode 2: out[j] = m_j */
int mbpls_masked_colden_f64(const unsigned* bits, long ldw, int n, int p, const int* col_nan, const double* v, const double* v2,
                            const double* vv, int mode, double* out, const int* done, void* stream);
/* out[0] = a . b over n samples (single CTA, fixed order) */
int mbpls_vec_dot_f64(const double* a, const double* b, int n, double* out, void* stream);
/* Tden[s*ldt + i] = sum over the features j of split s observed in sample i of w_j^2 (:867-872) */
int mbpls_masked_rowden_f64(const unsigned* bits, long ldw, int n, const double* w, const int* split_f0, const int* split_f1,
                            int nsplit, double* Tden, long ldt, const int* done, void* stream);

/* ---- finalisation and new-data paths (mbpls.py:986-989, :1110-1117, :1379-1386) -------------------- */
/* Cpart[chunk][i*K2 + j] = sum_{f in chunk} A[i][f] * Bm[j][f]; A is K1 x p (lda), Bm is K2 x p (ldb).
 * Returns the number of chunks via mbpls_gram_num_chunks; reduce with mbpls_reduce_chunks_f64. */
int mbpls_gram_num_chunks(int p);
int mbpls_gram_partial_f64(const double* A, long lda, int K1, const double* Bm, long ldb, int K2, int p, double* Cpart,
                           void* stream);
int mbpls_reduce_chunks_f64(const double* Cpart, int nchunks, int len, double* C, void* stream);
/* out[c][j] = sum_k (in[k][j] * rowscale[k]) * M[k*C + c]   (R_ = W pinv(P'W), beta_ = R_ V_') */
int mbpls_right_multiply_f64(const double* in, long ldin, int K, int p, const double* rowscale, const double* M, int C,
                             double* out, long ldout, void* stream);
/* out_part[s][c][i] = sum_{j in split s} nan0(z_ij) * Bm[c][j]   (X.dot(beta_), X.dot(R_), X_b.dot(W_b));
 * z_ij = Xt[j][i], or (Xt[j][i] - mean[j]) / scale[j] when mean/scale are given (x_scalers_[b].transform fused
 * into the product, mbpls.py:1097,:1369, so predict reads new data exactly once); with mean given and scale == NULL
 * only the centring is applied -- the caller has folded 1 / scale[j] into Bm, which takes the fp64 division out of the
 * streaming loop.  nonfinite_flag (optional) is set to 1 if any raw element is NaN or inf (check_array's finiteness
 * test, :1368, without an extra pass). */
int mbpls_skinny_gemm_f64(const double* Xt, long ld, int n, const double* Bm, long ldb, int C, const int* split_f0,
                          const int* split_f1, int nsplit, double* out_part, long ldo, const double* mean,
                          const double* scale, int* nonfinite_flag, void* stream);
/* The same product for tall batches (m >> p, at most 4 outputs, all p features): out[c*ldo + i] written directly.
 * Persistent CTAs stream 16 KB chunks of every feature through a 192 KB ring of bulk (TMA) copies instead of issuing
 * per-thread loads 8 MB apart; the coefficients of a feature travel with its chunk.  coef: p x 8 doubles, row j =
 * {mean_j (0: no centring), b_0j, b_1j, b_2j, b_3j, 0, 0, 0} with 1 / scale_j already folded into the b's. */
int mbpls_skinny_gemm_tall_f64(const double* Xt, long ld, int n, int p, const double* coef, int C, double* out, long ldo,
                               int* nonfinite_flag, void* stream);
/* X_b <- X_b - ts p_b' for new data (transform, mbpls.py:1145,1204); NaNs stay NaN */
int mbpls_rank1_update_f64(double* Xt, long ld, int n, int p, const double* ts, const double* pvec, void* stream);
/* column norms / scaling of a C x ld feature-major array over n samples */
int mbpls_rows_sumsq_f64(const double* M, long ld, int rows, int n, double* out, void* stream);
int mbpls_rows_scale_f64(double* M, long ld, int rows, int n, const double* scale, int divide, void* stream);

/* ---- SIMPLS / UNIPALS / KERNEL building blocks (mbpls.py:384-807, :995-1048) ------------------------ */
/* out[c][j] = sum_i nan0(Xt[j][i]) * M[c][i]: X'Y (:396,:587,:998), X'U (:731), X'Ts (:734) */
int mbpls_xt_multi_f64(const double* Xt, long ld, int n, int p, const double* M, long ldm, int C, double* out, long ldo,
                       void* stream);
/* few, long features (n >= 2^16): the same product with every feature cut into mbpls_xt_multi_chunks(n, p) sample ranges so that
 * the whole GPU streams it; part[s][c][j] (C * ldo doubles per chunk s) receives the partial products, which are then added
 * in chunk order: mbpls_reduce_chunks_f64(part, chunks, C * ldo, out) */
int mbpls_xt_multi_chunks(int n, int p);
int mbpls_xt_multi_split_f64(const double* Xt, long ld, int n, int p, const double* M, long ldm, int C, double* part, long ldo,
                             int chunks, void* stream);
/* out[j] = base[j] - sum_k V[k][j]*coef[k]: SIMPLS orthogonalisation (:1016-1017) */
int mbpls_lincomb_sub_f64(double* out, const double* base, const double* V, long ldv, int K, const double* coef, int len,
                          void* stream);
/* t <- t - mean(t) (if center); *nrm_out = ||t||; t <- t/||t|| (if normalize)  (:1007-1009, :417, :424) */
int mbpls_center_normalize_f64(double* t, int n, int center, int normalize, double* nrm_out, void* stream);
/* out[b] = ||w_b||^2 and out[j] = w[j]/sqrt(a[block(j)]): block weights / importances (:405-408, :605-609, :746-750) */
int mbpls_block_sumsq_f64(const double* w, const int* off, int B, double* out, void* stream);
int mbpls_scale_by_block_f64(const double* w, const int* off, int B, const double* a, double* out, int p, void* stream);
/* FP64 tensor-core (DMMA m8n8k4) cross product with deterministic split-K:
 * kmajor=1: C = A B' (A: M x Kdim, B: N x Kdim)  -> X'X from the feature-major matrix (:586)
 * kmajor=0: C = A' B (A: Kdim x M, B: Kdim x N)  -> X X' from the feature-major matrix (:704)
 * Cpart: splits x M x ldc partials (splits = mbpls_crossprod_splits); sum them with mbpls_reduce_chunks_f64. */
int mbpls_crossprod_splits(int M, int N, long Kdim);
/* split count for symmetric=1 (X'X / XX'): balances the CTAs that do work (tiles on / above the diagonal) over whole rounds of
 * the SMs; a pure function of (M, Kdim, SM count) */
int mbpls_crossprod_splits_syrk(int M, long Kdim);
int mbpls_crossprod_f64(const double* A, long lda, const double* B, long ldb, int M, int N, long Kdim, int kmajor, int splits,
                        double* Cpart, long ldc, int symmetric, void* stream);
/* symmetric=1 (A == B, M == N): only the tiles on/above the diagonal are computed (SYRK); after the split-K
 * reduction call mbpls_symmetrize_f64 to mirror them below the diagonal. */
int mbpls_symmetrize_f64(double* C, long ldc, int M, void* stream);
/* y = A x for a dense m x ncols matrix (VAR w :595,:599; AS_Y ts :718) */
int mbpls_dense_gemv_f64(const double* A, long lda, int m, int ncols, const double* x, double* y, void* stream);
/* A += al*x y' + be*y x' + ga*x x' with al,be (ga) optionally multiplied by scal[alpha_from] (scal[gamma_from]):
 * the rank-1/2 forms of the sandwich deflations D'VAR D (:632) and D AS_X D (:723) */
int mbpls_dense_rank2_f64(double* A, long lda, int m, int ncols, const double* x, const double* y, const double* scal,
                          double alpha, double beta, double gamma, int alpha_from, int gamma_from, void* stream);

/* ---- small dense linear algebra of the per-component steps (single CTA, one-sided Jacobi SVD, m <= 64) ---- */
/* out[0..m) = unit top eigenvector of the symmetric PSD m x m matrix G: np.linalg.svd(S)[0][:, 0:1] for
 * S = C C' via the q x q matrix C'C (mbpls.py:398,:590,:1001) */
int mbpls_small_top_eigvec_f64(const double* G, long ld, int m, double* out, void* stream);
/* out = pinv(M) (m x m), singular values <= rcond * sigma_max dropped: np.linalg.pinv (:476,:569,:642,:734,:737,:988) */
int mbpls_small_pinv_f64(const double* M, long ld, int m, double rcond, double* out, long ldo, void* stream);
/* c with A c = top left singular vector of A B', given G = B'B and H = A'A: svd(XX'YY') (:491,:713) */
int mbpls_small_top_sv_product_f64(const double* G, long ldg, const double* H, long ldh, int m, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MBPLS_B200_H */
