// Internal C++ interfaces between the translation units of libevcplm.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace evc {

// hamming.cu
int64_t hamming_plane_words(int64_t N, int L);
int64_t hamming_num_tiles(int64_t N);
int hamming_pack(const uint8_t *d_codes, int64_t N, int L, uint32_t *d_planes, cudaStream_t st);
int hamming_count_tiles(const uint32_t *d_planes, int64_t N, int L, int min_identical,
                        int64_t tile_begin, int64_t tile_end, int *d_counts, cudaStream_t st);

int identities_to_seq(const uint8_t *d_codes, const uint8_t *d_seq, int64_t N, int L, int *d_out, cudaStream_t st);

// plm_gather.cu -- geometry of the expanded coupling tensor and the gather-path kernels
struct PlmGeom {
    int64_t N;        // sequences on this handle
    int L;            // sites
    int Lp;           // L rounded up to 4 (bulk-copy alignment of a site's row block)
    int q;            // model states (QA)
    int QB;           // neighbour states incl. the ignored-gap row (q or q+1)
    int S;            // row stride in floats (odd => conflict-free shared-memory gathers)
    int gap_code;     // -1 or q
    int64_t Nr;       // N rounded up to the backward tile (rows of the residual buffer)
    int64_t Nld;      // leading dimension of the packed column-major MSA
    int L4;           // ceil(L/4) packed site words
    int ntiles_f;     // forward sequence tiles
    int ntiles_b;     // backward sequence tiles
    int64_t n_params;
    __host__ __device__ int64_t blk() const { return (int64_t)QB * S; }                    // floats per (i,j) block
    __host__ __device__ int64_t row_block() const { return (int64_t)Lp * blk(); }          // floats per site i
    __host__ __device__ int64_t w_floats() const { return (int64_t)L * row_block(); }
};

constexpr int PLM_FWD_TS = 512;    // sequences per forward CTA (256 threads x 2)
constexpr int PLM_BWD_TS = 2048;   // sequences per backward tile (residual tile in shared memory)
constexpr int PLM_BWD_CAP = 2224;  // list entries per (tile, column): 2048 + up to 7 pads for each of <= 22 buckets
constexpr int PLM_BWD_BS = 24;     // bucket-boundary slots per list

bool plm_supported_q(int q);
int plm_pack_msa(const PlmGeom &g, const uint8_t *d_codes, uint32_t *d_msa4, cudaStream_t st);
int plm_build_buckets(const PlmGeom &g, const uint8_t *d_codes, uint32_t *d_perm, uint16_t *d_bstart,
                      cudaStream_t st);
int plm_expand(const PlmGeom &g, const float *d_x, float *d_W, cudaStream_t st);
int plm_forward(const PlmGeom &g, const float *d_W, const float *d_x, const uint32_t *d_msa4,
                const float *d_wts, float *d_R, void *d_rt_hi, void *d_rt_lo, int64_t Kp, float *d_gh_part,
                double *d_fx_part, cudaStream_t st);
int plm_onehot_residual(const PlmGeom &g, const uint32_t *d_msa4, const float *d_wts, float *d_R,
                        float *d_gh_part, cudaStream_t st);
int plm_backward(const PlmGeom &g, const float *d_R, const uint32_t *d_perm, const uint16_t *d_bstart,
                 float *d_G, cudaStream_t st);
int plm_finalize(const PlmGeom &g, const float *d_G, const float *d_gh_part, const double *d_fx_part,
                 float *d_gh, float *d_gJ, double *d_fx, float scale_pair, cudaStream_t st);
int plm_add_reg(const PlmGeom &g, const float *d_x, float *d_g, double *d_fx, float lambda_h,
                float lambda_J, cudaStream_t st);

// plm_tc.cu -- backward as a bf16 tcgen05 GEMM (dense one-hot contraction)
struct PlmTcGeom {
    int64_t Mp;   // L*q rounded up to the 128-row MMA tile  (rows of Xt, Gd)
    int64_t Np;   // L*q rounded up to the 192-column tile   (rows of Rt_hi / Rt_lo, columns of Gd)
    int64_t Kp;   // sequences rounded up to the 64-wide K block
};
void plm_tc_geometry(const PlmGeom &g, PlmTcGeom &t);
size_t plm_tc_map_bytes();
int plm_tc_build_xt(const PlmGeom &g, const PlmTcGeom &t, const uint32_t *d_msa4, void *d_xt, cudaStream_t st);
int plm_tc_make_maps(const PlmTcGeom &t, void *d_xt, void *d_rt_hi, void *d_rt_lo, void *maps_out_host);
int plm_tc_backward(const PlmGeom &g, const PlmTcGeom &t, const void *maps_host, float *d_Gd, int single,
                    cudaStream_t st);
int plm_tc_onehot_residual(const PlmGeom &g, int ntiles, const uint32_t *d_msa4, const float *d_wts, void *d_rt_hi,
                           void *d_rt_lo, int64_t Kp, float *d_gh_part, double *d_fx_part, cudaStream_t st);
int plm_tc_finalize_pairs(const PlmGeom &g, const PlmTcGeom &t, const float *d_Gd, float *d_gJ, float scale,
                          cudaStream_t st);
// tensor-core forward: Zt = (Wt_hi + Wt_lo) X^T on tcgen05, then softmax/residual kernel
struct PlmTcfGeom {
    int64_t Mp;      // L*q rounded to 128: rows of Wt_hi/Wt_lo and of Zt
    int64_t Kw;      // L*q rounded to 64: K extent
    int64_t Ns;      // sequences rounded to 192: leading dimension of Zt
    int64_t Xrows;   // allocated rows of the one-hot X (N rounded to 384)
    int ntiles_s;    // softmax-kernel sequence tiles (256 sequences)
};
void plm_tcf_geometry(const PlmGeom &g, PlmTcfGeom &t);
int plm_tcf_build_x(const PlmGeom &g, const PlmTcfGeom &t, const uint32_t *d_msa4, void *d_x1h, cudaStream_t st);
int plm_tcf_make_maps(const PlmTcfGeom &t, void *d_wt_hi, void *d_wt_lo, void *d_x1h, void *maps_out_host);
int plm_tcf_expand(const PlmGeom &g, const PlmTcfGeom &t, const float *d_x, void *d_wt_hi, void *d_wt_lo,
                   int single, cudaStream_t st);
int plm_tcf_logits(const PlmGeom &g, const PlmTcfGeom &t, const void *maps_host, float *d_zt, int single,
                   cudaStream_t st);
int plm_tcf_softmax(const PlmGeom &g, const PlmTcfGeom &t, const float *d_zt, const float *d_x,
                    const uint32_t *d_msa4, const float *d_wts, void *d_rt_hi, void *d_rt_lo, int64_t Kp,
                    float *d_gh_part, double *d_fx_part, cudaStream_t st);
// fused tensor-core forward (softmax / residual epilogue on the TMEM accumulator)
struct PlmTcffGeom {
    int n_tiles;       // site tiles (8 sites = 176 padded columns each)
    int m_tiles;       // sequence tiles (128 sequences)
    int64_t Np;        // rows of the padded coupling operand Wp_hi / Wp_lo
    int64_t Kw;        // K extent (L*q rounded to 64)
    int64_t Xrows;     // allocated rows of X
    int ntile_part;    // partial-sum slots per site (m_tiles * 4)
};
void plm_tcff_geometry(const PlmGeom &g, PlmTcffGeom &t);
bool plm_tcff_supported(const PlmGeom &g);
int plm_tcff_make_maps(const PlmTcffGeom &t, void *d_x1h, void *d_wp_hi, void *d_wp_lo, void *maps_out_host);
int plm_tcff_expand(const PlmGeom &g, const PlmTcffGeom &t, const float *d_x, void *d_wp_hi, void *d_wp_lo,
                    int single, cudaStream_t st);
int plm_tcff_forward(const PlmGeom &g, const PlmTcffGeom &t, const void *maps_host, const float *d_x,
                     const uint32_t *d_msa4, const float *d_wts, void *d_rt_hi, void *d_rt_lo, int64_t Kp,
                     float *d_gh_part, double *d_fx_part, int single, cudaStream_t st);
int plm_finalize_fields_n(const PlmGeom &g, const float *d_gh_part, const double *d_fx_part, float *d_gh,
                          double *d_fx, int ntiles, cudaStream_t st);
int plm_finalize_fields(const PlmGeom &g, const float *d_gh_part, const double *d_fx_part, float *d_gh,
                        double *d_fx, cudaStream_t st);

// model_ops.cu (SURVEY 8f rows f1 / f2)
int ec_scores(const float *d_J, const float *d_fij, const float *d_fi, int L, int q, float *d_fn_raw,
              float *d_fn_zs, float *d_mi, cudaStream_t st);
int plm_energies(const PlmGeom &g, const float *d_W, const float *d_x, const uint32_t *d_msa4, float *d_epart,
                 double *d_out, cudaStream_t st);
int ec_scores_f64(const double *d_J, const double *d_fij, const double *d_fi, int L, int q, double *d_fn_raw,
                  double *d_fn_zs, double *d_mi, cudaStream_t st);

// mean_field.cu (mean-field DCA, fp64)
int mf_weighted_counts(const uint8_t *d_codes, const double *d_w, int64_t N, int L, int q, double n_eff, double *d_F,
                       cudaStream_t st);
int mf_covariance(const double *d_F, int L, int q, double pc, double *d_C, double *d_fi, double *d_rfi,
                  double *d_fij_tri, cudaStream_t st);
int spd_inverse(double *d_A, int64_t n, double *d_X, int *d_info, cudaStream_t st);
int mf_couplings_fields(const double *d_Cinv, const double *d_rfi, int L, int q, double *d_J_tri, double *d_h,
                        cudaStream_t st);
int mf_di_scores(const double *d_J_tri, const double *d_rfi, int L, int q, double *d_di, int *d_iters,
                 cudaStream_t st);

// vecops.cu
int vec_dot(const float *a, const float *b, int64_t n, double *out, cudaStream_t st);
int vec_axpby(float *y, const float *x, float a, float b, int64_t n, cudaStream_t st);
int vec_sub(float *out, const float *a, const float *b, int64_t n, cudaStream_t st);
int lbfgs_direction(float *d, const float *g, const float *S, const float *Y, const double *ys,
                    double *scratch, int64_t n, int m, int bound, int end, cudaStream_t st);
int lbfgs_update_pair(float *s, float *y, const float *x, const float *xp, const float *g,
                      const float *gp, double *ys, double *yy, int64_t n, cudaStream_t st);
int fn_scores(const float *J, int L, int q, float *fn, cudaStream_t st);

// fit.cu
struct FitWork;
void fit_work_free(FitWork *w);

}  // namespace evc

// The handle behind evc_plm_t (include/evcplm.h).  Defined here because api.cu (objective) and fit.cu (L-BFGS
// driver) both work on it.
struct evc_plm {
    int device = 0;
    evc::PlmGeom g{};
    uint8_t *d_codes = nullptr;     // [N][L] (kept: the gather path's bucket lists are built lazily from it)
    uint32_t *d_msa4 = nullptr;
    float *d_wts = nullptr;
    // gather path (plm_gather.cu): allocated on first use (ensure_gather) -- the tensor-core path never needs it
    bool gather_ready = false;
    uint32_t *d_perm = nullptr;
    uint16_t *d_bstart = nullptr;
    float *d_W = nullptr;
    float *d_G = nullptr;
    float *d_R = nullptr;
    float *d_gh_part = nullptr;
    double *d_fx_part = nullptr;
    float *d_x_tmp = nullptr;       // host-buffer convenience path
    float *d_g_tmp = nullptr;
    double *d_fx_tmp = nullptr;
    int precision = 0;              // 0 = fp32-equivalent (bf16 hi + lo products), 1 = bf16 tiles (one product)
    // tensor-core backward (plm_tc.cu); allocated on first use
    int bwd_mode = 0;               // 0 = gather/bucket kernel, 1 = tcgen05 GEMM
    evc::PlmTcGeom tc{};
    void *d_xt = nullptr;
    void *d_rt_hi = nullptr;
    void *d_rt_lo = nullptr;
    float *d_Gd = nullptr;
    void *tc_maps = nullptr;        // host: 3 CUtensorMap
    // tensor-core forward (plm_tc.cu); allocated on first use
    int fwd_mode = 0;               // 0 = gather kernel, 1 = tcgen05 GEMM + softmax kernel, 2 = fused epilogue
    evc::PlmTcfGeom tcf{};
    void *d_x1h = nullptr;
    void *d_wt_hi = nullptr;
    void *d_wt_lo = nullptr;
    float *d_zt = nullptr;
    float *d_gh_part2 = nullptr;
    double *d_fx_part2 = nullptr;
    void *tcf_maps = nullptr;
    // fused tensor-core forward (softmax epilogue on the accumulator)
    evc::PlmTcffGeom tcff{};
    void *d_wp_hi = nullptr;
    void *d_wp_lo = nullptr;
    float *d_gh_part3 = nullptr;
    double *d_fx_part3 = nullptr;
    void *tcff_maps = nullptr;
    bool profiling = false;         // record CUDA events around the stages of evc_plm_eval_data
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool ev_valid = false;
    evc::FitWork *fit = nullptr;    // L-BFGS workspace (fit.cu), allocated by the first evc_plm_fit
};
