/*
 * libevcplm -- C ABI of the B200-native pseudo-likelihood Potts-model engine.
 *
 * This is the drop-in boundary for the ONE numerically heavy step of the
 * EVcouplings pipeline: what evcouplings/couplings/tools.py:126-307 (run_plmc)
 * obtains today by fork/exec of the external `plmc` C/OpenMP binary
 * (argv built at tools.py:202-262, subprocess at tools.py:266, caller
 * evcouplings/couplings/protocol.py:203-218).  The entry points below are
 * what a ctypes binding of that call site needs (INTEGRATION.md shows the
 * binding); evcouplings_b200/ is the Python host that mirrors run_plmc on top
 * of them.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.
 *   - "d_" arguments are device pointers on the handle's device, "h_"/unprefixed
 *     host pointers.  `stream` is a cudaStream_t passed as void* (NULL = default).
 *   - every function returns 0 on success, non-zero on failure;
 *     evc_last_error() gives the message (thread-local).
 *   - the caller owns all buffers it passes; the library owns what it allocates
 *     inside a handle until evc_plm_destroy.
 *   - a handle is not re-entrant; independent handles may be used from
 *     different threads or processes (one process per GPU for multi-GPU runs).  The
 *     evc_vec_*, evc_lbfgs_*, evc_plm_add_regulariser and evc_hamming_* entry points keep
 *     their small reduction / candidate scratch per (device, stream) inside the library:
 *     concurrent callers must use different streams (or different devices).
 *
 * Parameter vector layout (identical to the plmc_v2 .model file read by
 * evcouplings/couplings/model.py:354-389):
 *     x = [ h : L*q floats | J : L(L-1)/2 blocks of q*q floats,
 *           pairs (i<j) in row-major (i,j) order, block[a][b], a = state at i ]
 * Sequence codes: uint8, 0..q-1 = model states; with gap_code >= 0 (plmc -g,
 * "ignore_gaps") the value gap_code (== q) marks a gap: the site is skipped as
 * a conditional and contributes nothing as a neighbour.
 */
#ifndef EVCPLM_H
#define EVCPLM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVCPLM_ABI_VERSION 2

typedef struct evc_plm evc_plm_t;

/* ---- library / device -------------------------------------------------- */
int evc_abi_version(void);
const char *evc_last_error(void);
int evc_device_count(void);                  /* <0 on error                */
int evc_device_info(int32_t device, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor,
                    int64_t *total_mem_bytes);

/* ---- (b) O(N^2 L) pairwise-Hamming sequence reweighting ------------------
 * Replaces plmc's reweighting pass (stderr "Effective number of samples",
 * parsed at tools.py:55) and the in-tree twin
 * evcouplings/align/alignment.py:1192-1233 (num_cluster_members).
 * counts[s] = #{ t : #(codes[s,k] == codes[t,k]) >= min_identical }, self
 * included, gap == gap counts as identical.  min_identical is the integer form
 * of "pair_id / L >= theta" (alignment.py:1229), computed by the host.
 */
int evc_hamming_counts(const uint8_t *codes, int64_t N, int32_t L, int32_t min_identical,
                       int32_t device, int32_t *counts_out);

/* device-resident building blocks (multi-GPU: each rank counts a tile range,
 * the host all-reduces the int32 counters) */
int64_t evc_hamming_plane_words(int64_t N, int32_t L);   /* uint32 words of the bit-plane buffer */
int64_t evc_hamming_num_tiles(int64_t N);                /* upper-triangular 128x128 pair tiles   */
int evc_hamming_pack(const uint8_t *d_codes, int64_t N, int32_t L, uint32_t *d_planes, void *stream);
int evc_hamming_count_tiles(const uint32_t *d_planes, int64_t N, int32_t L, int32_t min_identical,
                            int64_t tile_begin, int64_t tile_end, int32_t *d_counts /* += */,
                            void *stream);

/* f3 twin of identities_to_seq (evcouplings/align/alignment.py:1156-1189): d_out[n] = #{k : codes[n,k] == seq[k]} */
int evc_identities_to_seq(const uint8_t *d_codes /* N x L */, const uint8_t *d_seq /* L */, int64_t N, int32_t L,
                          int32_t *d_out, void *stream);

/* ---- f4: compiled A2M / FASTA ingest (host code) ---------------------------------------------------------
 * Replaces the reference's in-tree text readers (evcouplings/align/alignment.py:42-74 read_fasta, 410-443
 * sequences_to_matrix, 479-495 map_matrix) and plmc's own parser (8a row a4).  Return 0 ok, 1 I/O or argument
 * error, 2 malformed alignment (no sequences / zero length / ragged rows); message in evc_last_error().
 *   evc_a2m_scan:   number of records, common row width, bytes for the NUL-separated record ids
 *   evc_a2m_read:   raw characters (n_rows x width, as in the file: case and '.' preserved) and the ids
 *   evc_msa_encode: codes_out[v][k] = lut[raw[row_v][cols[k]]] for the VALID rows only (a row is valid iff no
 *                   character of the whole row maps to 255), valid_out[r] in {0,1}, *n_valid_out rows written */
int evc_a2m_scan(const char *path, int64_t *n_rows, int64_t *width, int64_t *ids_bytes);
int evc_a2m_read(const char *path, int64_t n_rows, int64_t width, uint8_t *raw, char *ids, int64_t ids_bytes);
int evc_msa_encode(const uint8_t *raw, int64_t n_rows, int64_t width, const uint8_t *lut, const int64_t *cols,
                   int64_t n_cols, uint8_t *valid_out, uint8_t *codes_out, int64_t *n_valid_out);

/* ---- (a) PLM objective + gradient -----------------------------------------
 * Replaces plmc's negative-log-posterior evaluation (the inner loop of its
 * L-BFGS; SURVEY.md 8a row a7).
 */
int evc_plm_create(evc_plm_t **out, const uint8_t *codes /* host, N x L */, int64_t N, int32_t L,
                   int32_t q, int32_t gap_code /* -1: gap is a model state */,
                   const float *weights /* host, N */, int32_t device);
void evc_plm_destroy(evc_plm_t *h);
int64_t evc_plm_num_params(const evc_plm_t *h);          /* L*q + L(L-1)/2*q*q */

/* data term on this handle's sequences:  d_g[0..n) = d/dx of
 * -sum_s w_s sum_i log P(s_i | s_-i),  d_fx[0] = that sum (double).
 * No regulariser (so shards can be summed with one all-reduce). */
int evc_plm_eval_data(evc_plm_t *h, const float *d_x, float *d_g, double *d_fx, void *stream);

/* Backward implementation of the data term: 0 = gather/bucket kernel (shared-memory bound, default),
 * 1 = dense one-hot contraction on the tcgen05 tensor cores (bf16 hi/lo split of the residuals, fp32
 * accumulation in TMEM).  Both produce the same gradient within fp32 tolerance; bench.py reports both. */
int evc_plm_set_backward(evc_plm_t *h, int32_t mode);
/* Forward implementation: 0 = gather kernel (fp32 couplings streamed through shared memory),
 * 1 = logits as a tcgen05 GEMM (couplings split in bf16 hi + lo, fp32 accumulation) followed by a
 * softmax/residual kernel; 2 = the same GEMM with softmax / residuals fused into its epilogue (no logits
 * matrix in HBM; protein alphabets, falls back to 1 otherwise).  Modes 1 and 2 imply the tensor-core backward. */
int evc_plm_set_forward(evc_plm_t *h, int32_t mode);

/* Arithmetic of the tensor-core products (SURVEY.md 8b `precision`; BASELINE configs[4] "bf16 tiles / fp32
 * parameters"): 0 (default) = fp32-equivalent: the real-valued operand (couplings forward, residuals backward)
 * enters as TWO bf16 terms hi + lo (16 mantissa bits), two tcgen05.mma per K slice; 1 = bf16 tiles: ONE bf16
 * term, one tcgen05.mma per K slice (half the tensor-core work).  Parameters, accumulation (TMEM, K chunks
 * promoted with fp32 round-to-nearest adds), softmax and the optimiser stay fp32 in both modes.  No effect on
 * the gather kernels.  May be changed between evaluations. */
int evc_plm_set_precision(evc_plm_t *h, int32_t mode);

/* Per-stage device timing of the LAST evc_plm_eval_data call (CUDA events recorded on the stream the
 * kernels were launched on): ms_out[5] = {expand (+ clear), forward (gather kernel or logits GEMM),
 * softmax kernel (0 on the gather forward), backward kernel, finalize}.
 * Used by bench.py to report the dominant kernel's roofline live. */
int evc_plm_set_profiling(evc_plm_t *h, int32_t enable);
int evc_plm_last_stage_ms(evc_plm_t *h, float *ms_out);

/* d_g += 2*lambda*x (lambda_h on the first L*q entries, lambda_J on the rest);
 * d_fx[1] = d_fx[0] + lambda_h*|h|^2 + lambda_J*|J|^2   (d_fx[0] = -loglk kept) */
int evc_plm_add_regulariser(evc_plm_t *h, const float *d_x, float *d_g, double *d_fx,
                            float lambda_h, float lambda_J, void *stream);

/* host-buffer convenience (H2D of x, evaluation, D2H of g inside the call):
 * fx_out[0] = -loglk, fx_out[1] = full objective. */
int evc_plm_eval_host(evc_plm_t *h, const float *x, float *g, double *fx_out,
                      float lambda_h, float lambda_J);

/* ---- a6: weighted single / pair counts for the .model file ---------------
 * d_fi_counts[L*q], d_fij_counts[L(L-1)/2*q*q] (tri blocks [a][b]) receive
 * sum_s w_s [s_i=a] and sum_s w_s [s_i=a][s_j=b]; the host normalises
 * (N_eff, or per-site / per-pair non-gap weight under ignore_gaps). */
int evc_plm_weighted_counts(evc_plm_t *h, float *d_fi_counts, float *d_fij_counts, void *stream);

/* ---- a8: the whole L-BFGS fit on the device (replaces plmc's libLBFGS loop; iteration cap = plmc `-m`,
 * evcouplings/couplings/tools.py:226-228) ---------------------------------------------------------------
 * Minimises  -sum_s w_s sum_i log P(s_i | s_-i) + lambda_h |h|^2 + lambda_J |J|^2  from the start point in d_x
 * (device, n floats; overwritten with the result).  All vectors live in the handle; the host sees six doubles
 * per objective evaluation.  Status codes carry libLBFGS's names (plmc prints them after
 * "Gradient optimization:", parsed at tools.py:57). */
enum {
    EVC_LBFGS_SUCCESS = 0,
    EVC_LBFGS_ALREADY_MINIMIZED = 2,
    EVC_LBFGSERR_CANCELED = -1021,
    EVC_LBFGSERR_INVALIDPARAMETERS = -1000,
    EVC_LBFGSERR_MINIMUMSTEP = -1001,
    EVC_LBFGSERR_MAXIMUMSTEP = -1002,
    EVC_LBFGSERR_MAXIMUMLINESEARCH = -1003,
    EVC_LBFGSERR_MAXIMUMITERATION = -1004,
    EVC_LBFGSERR_WIDTHTOOSMALL = -1005,
    EVC_LBFGSERR_ROUNDING_ERROR = -1006,
    EVC_LBFGSERR_INCREASEGRADIENT = -1007
};
typedef struct {
    int32_t max_iterations;      /* 0 = until convergence                                             */
    int32_t m;                   /* correction pairs kept (1..32)                                      */
    float epsilon;               /* stop when |g| / max(1, |x|) <= epsilon                             */
    float lambda_h, lambda_J;
    int32_t max_linesearch;
    double min_step, max_step, ftol, gtol, xtol;
    int32_t precision_schedule;  /* 0: keep the handle's precision; 1: bf16 tiles until
                                    |g|/max(1,|x|) <= switch_factor * epsilon (or the line search fails),
                                    then fp32-equivalent products to the end                            */
    float switch_factor;
} evc_fit_params_t;
typedef struct {
    int32_t status;              /* EVC_LBFGS*                                                          */
    int32_t iterations;
    int32_t evaluations;
    int32_t switched_at;         /* iteration at which precision_schedule 1 left the bf16 mode, or -1   */
    double fx, negloglk;
    double seconds;
} evc_fit_result_t;
/* Sum d_buf[0..count) over all ranks in place, asynchronously on `stream` (NCCL all-reduce in the Python host).
 * The buffer is the gradient followed by 4 floats that carry -loglk as exact fixed-point limbs: ONE collective
 * per evaluation.  NULL = single rank.  Return non-zero to abort. */
typedef int (*evc_allreduce_cb)(void *user, float *d_buf, int64_t count, void *stream);
/* Called once per iteration (the row of plmc's iteration table, tools.py:59-83); non-zero return cancels. */
typedef int (*evc_progress_cb)(void *user, int32_t iteration, double fx, double xnorm, double gnorm, double step,
                               int32_t linesearch_evals, double negloglk, double hnorm, double enorm);
void evc_fit_default_params(evc_fit_params_t *p);
int evc_plm_fit(evc_plm_t *h, float *d_x, const evc_fit_params_t *params, evc_allreduce_cb allreduce,
                void *allreduce_user, evc_progress_cb progress, void *progress_user, evc_fit_result_t *result,
                void *stream);

/* -loglk <-> 4 floats appended to the gradient (three exact fixed-point limbs, resolution 2^-16, |fx| < 1.3e11, up to 64 ranks):
 * a data-parallel evaluation then needs ONE all-reduce of n + 4 floats (SURVEY.md 8e `[fx, g]`). */
int evc_plm_pack_fx(const double *d_fx, float *d_limbs, void *stream);
int evc_plm_unpack_fx(const float *d_limbs, double *d_fx, void *stream);

/* ---- a8: on-device L-BFGS vector algebra ----------------------------------
 * All scalars stay on the device (double); the host reads back only what the
 * line search needs. */
int evc_vec_dot(const float *d_a, const float *d_b, int64_t n, double *d_out, void *stream);
int evc_vec_axpby(float *d_y, const float *d_x, float a, float b, int64_t n, void *stream); /* y = a*x + b*y */
int evc_vec_copy(float *d_dst, const float *d_src, int64_t n, void *stream);
int evc_vec_sub(float *d_out, const float *d_a, const float *d_b, int64_t n, void *stream);
/* two-loop recursion: d = -H g using `bound` stored pairs ending before slot
 * `end` (ring of m); d_S/d_Y are m x n row-major; d_ys[m] holds y.s per slot;
 * d_scratch needs m + 2 doubles. */
int evc_lbfgs_direction(float *d_d, const float *d_g, const float *d_S, const float *d_Y,
                        const double *d_ys, double *d_scratch, int64_t n, int32_t m,
                        int32_t bound, int32_t end, void *stream);
/* s = x - xp, y = g - gp into slot, d_ys[slot] = y.s, d_scratch[0] = y.y (fused) */
int evc_lbfgs_update_pair(float *d_S_slot, float *d_Y_slot, const float *d_x, const float *d_xp,
                          const float *d_g, const float *d_gp, double *d_ys_slot, double *d_yy,
                          int64_t n, void *stream);

/* ---- SURVEY 8(f) "next" rows ------------------------------------------------
 * f1: per-pair scores of CouplingsModel._calculate_ecs (evcouplings/couplings/model.py:777-827):
 *     Frobenius norm of each J_ij block in the raw gauge (plmc's _ECs.txt) and in the zero-sum gauge
 *     (model.py:179-233), and mutual information from f_ij / f_i (d_fij_tri / d_fi / d_mi may be NULL).
 *     The APC (model.py:744-775) is an L x L host operation.
 * f2: statistical energies of this handle's sequences under parameters x (model.py:25-60 _hamiltonians):
 *     d_out[n][3] = {H, H_J, H_h} (double). */
int evc_ec_scores(const float *d_J_tri, const float *d_fij_tri, const float *d_fi, int32_t L, int32_t q,
                  float *d_fn_raw, float *d_fn_zero_sum, float *d_mi, void *stream);
int evc_plm_energies(evc_plm_t *h, const float *d_x, double *d_out, void *stream);

/* ---- a10: EC scores (Frobenius norm of each J block, raw gauge) ---------- */
int evc_fn_scores(const float *d_J_tri, int32_t L, int32_t q, float *d_fn /* L(L-1)/2 */, void *stream);

/* ---- mean-field DCA (the couplings stage's `mean_field` protocol: evcouplings/couplings/mean_field.py) -------
 * Everything in fp64.  Sites L >= 2, states q in 2..21 (the gap is a state, alphabet order, last state = the
 * reference state of the model), n = L*(q-1).  All arrays are device arrays, row-major.
 *   evc_mf_weighted_counts_f64: d_F ((L*q) x (L*q), symmetric) at row i*q+a, column j*q+b =
 *       sum_s w_s [s_i = a][s_j = b] / n_eff  (so the (i,i) blocks hold f_i on their diagonal).
 *   evc_mf_covariance: from d_F and the pseudo-count pc, any output may be NULL:
 *       d_C (n x n): rf_ij[a][b] - rf_i[a] rf_j[b], a, b < q-1, with rf_i = (1-pc) f_i + pc/q,
 *           rf_ij = (1-pc) f_ij + pc/q^2 for i != j and (1-pc) f_i[a] d_ab + (pc/q) d_ab for i == j;
 *       d_fi, d_rfi (L x q): raw and regularised single-site frequencies;
 *       d_fij_tri (L(L-1)/2 blocks of q x q, pairs i<j row-major): raw pair frequencies.
 *   evc_spd_inverse_f64: d_A (n x n, symmetric positive definite, only the lower triangle is read) is replaced by
 *       its inverse (both triangles); d_work holds n*n doubles.  Blocked Cholesky, triangular inverse, X^T X.
 *       Synchronous.  Returns EVC_NOT_SPD, *info_out = 1-based column of the first non-positive pivot, when the
 *       matrix is not positive definite (d_A is then undefined); *info_out = 0 on success.
 *   evc_mf_couplings_fields: d_J_tri (tri blocks) = -Cinv[(i,a),(j,b)] for a, b < q-1, 0 on the last state;
 *       d_h (L x q) = log(rf_i[a] / rf_i[q-1]) - sum_{j != i} sum_b J_ij[a][b] rf_j[b].
 *   evc_mf_di_scores: direct information of every pair (tri order) from J and the regularised f_i: the two-site
 *       fixed point on exp(J_ij) from 1/q until the max-abs change is <= 1e-4; d_iters (may be NULL) receives
 *       the iteration count of each pair.
 *   evc_ec_scores_f64: evc_ec_scores in fp64 (the mean-field couplings are scored without a float32 rounding). */
#define EVC_NOT_SPD 2
int evc_mf_weighted_counts_f64(const uint8_t *d_codes /* N x L */, const double *d_weights, int64_t N, int32_t L,
                               int32_t q, double n_eff, double *d_F, void *stream);
int evc_mf_covariance(const double *d_F, int32_t L, int32_t q, double pseudo_count, double *d_C, double *d_fi,
                      double *d_rfi, double *d_fij_tri, void *stream);
int evc_spd_inverse_f64(double *d_A, int64_t n, double *d_work, int32_t *info_out, void *stream);
int evc_mf_couplings_fields(const double *d_Cinv, const double *d_rfi, int32_t L, int32_t q, double *d_J_tri,
                            double *d_h, void *stream);
int evc_mf_di_scores(const double *d_J_tri, const double *d_rfi, int32_t L, int32_t q, double *d_di,
                     int32_t *d_iters, void *stream);
int evc_ec_scores_f64(const double *d_J_tri, const double *d_fij_tri, const double *d_fi, int32_t L, int32_t q,
                      double *d_fn_raw, double *d_fn_zero_sum, double *d_mi, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* EVCPLM_H */
