// C ABI of libevcplm (declared in include/evcplm.h).  This is the boundary a binding of the
// reference's plmc call site (evcouplings/couplings/tools.py:202-266) talks to.
#include "../../include/evcplm.h"

#include <stdlib.h>

#include <new>
#include <string>
#include <vector>

#include "common.cuh"
#include "internal.h"

namespace evc {
static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
}  // namespace evc

using namespace evc;

static cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

int evc_abi_version(void) { return EVCPLM_ABI_VERSION; }

const char *evc_last_error(void) { return g_err.c_str(); }

int evc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        set_error("cudaGetDeviceCount failed (no CUDA device / driver?)");
        return -1;
    }
    return n;
}

int evc_device_info(int32_t device, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor,
                    int64_t *total_mem_bytes)
{
    cudaDeviceProp p;
    EVC_CUDA(cudaGetDeviceProperties(&p, device));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem_bytes) *total_mem_bytes = (int64_t)p.totalGlobalMem;
    return 0;
}

// ---- (b) Hamming ---------------------------------------------------------------------------------
int64_t evc_hamming_plane_words(int64_t N, int32_t L) { return hamming_plane_words(N, L); }
int64_t evc_hamming_num_tiles(int64_t N) { return hamming_num_tiles(N); }

int evc_hamming_pack(const uint8_t *d_codes, int64_t N, int32_t L, uint32_t *d_planes, void *stream)
{
    return hamming_pack(d_codes, N, L, d_planes, as_stream(stream));
}

int evc_hamming_count_tiles(const uint32_t *d_planes, int64_t N, int32_t L, int32_t min_identical,
                            int64_t tile_begin, int64_t tile_end, int32_t *d_counts, void *stream)
{
    return hamming_count_tiles(d_planes, N, L, min_identical, tile_begin, tile_end, d_counts,
                               as_stream(stream));
}

int evc_hamming_counts(const uint8_t *codes, int64_t N, int32_t L, int32_t min_identical, int32_t device,
                       int32_t *counts_out)
{
    if (!codes || !counts_out || N <= 0 || L <= 0) {
        set_error("evc_hamming_counts: empty alignment or null pointer");
        return 1;
    }
    EVC_CUDA(cudaSetDevice(device));
    uint8_t *d_codes = nullptr;
    uint32_t *d_planes = nullptr;
    int32_t *d_counts = nullptr;
    int rc = 1;
    do {
        if (cudaMalloc(&d_codes, (size_t)N * L) != cudaSuccess ||
            cudaMalloc(&d_planes, (size_t)hamming_plane_words(N, L) * sizeof(uint32_t)) != cudaSuccess ||
            cudaMalloc(&d_counts, (size_t)N * sizeof(int32_t)) != cudaSuccess) {
            set_error("evc_hamming_counts: device allocation failed");
            break;
        }
        if (cudaMemcpy(d_codes, codes, (size_t)N * L, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemset(d_counts, 0, (size_t)N * sizeof(int32_t)) != cudaSuccess) {
            set_error("evc_hamming_counts: H2D failed");
            break;
        }
        if (hamming_pack(d_codes, N, L, d_planes, 0)) break;
        if (hamming_count_tiles(d_planes, N, L, min_identical, 0, hamming_num_tiles(N), d_counts, 0)) break;
        if (cudaMemcpy(counts_out, d_counts, (size_t)N * sizeof(int32_t), cudaMemcpyDeviceToHost) !=
            cudaSuccess) {
            set_error(std::string("evc_hamming_counts: kernel/D2H failed: ") +
                      cudaGetErrorString(cudaGetLastError()));
            break;
        }
        rc = 0;
    } while (0);
    cudaFree(d_codes);
    cudaFree(d_planes);
    cudaFree(d_counts);
    return rc;
}

int evc_identities_to_seq(const uint8_t *d_codes, const uint8_t *d_seq, int64_t N, int32_t L, int32_t *d_out,
                          void *stream)
{
    if (!d_codes || !d_seq || !d_out) { set_error("evc_identities_to_seq: null pointer"); return 1; }
    return identities_to_seq(d_codes, d_seq, N, L, d_out, as_stream(stream));
}

// ---- (a) PLM ---------------------------------------------------------------------------------------
void evc_plm_destroy(evc_plm_t *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaFree(h->d_codes);
    cudaFree(h->d_msa4);
    cudaFree(h->d_perm);
    cudaFree(h->d_bstart);
    cudaFree(h->d_wts);
    cudaFree(h->d_W);
    cudaFree(h->d_G);
    cudaFree(h->d_R);
    cudaFree(h->d_gh_part);
    cudaFree(h->d_fx_part);
    cudaFree(h->d_x_tmp);
    cudaFree(h->d_g_tmp);
    cudaFree(h->d_fx_tmp);
    cudaFree(h->d_xt);
    cudaFree(h->d_rt_hi);
    cudaFree(h->d_rt_lo);
    cudaFree(h->d_Gd);
    free(h->tc_maps);
    cudaFree(h->d_x1h);
    cudaFree(h->d_wt_hi);
    cudaFree(h->d_wt_lo);
    cudaFree(h->d_zt);
    cudaFree(h->d_gh_part2);
    cudaFree(h->d_fx_part2);
    free(h->tcf_maps);
    cudaFree(h->d_wp_hi);
    cudaFree(h->d_wp_lo);
    cudaFree(h->d_gh_part3);
    cudaFree(h->d_fx_part3);
    free(h->tcff_maps);
    for (int k = 0; k < 6; k++)
        if (h->ev[k]) cudaEventDestroy(h->ev[k]);
    fit_work_free(h->fit);
    delete h;
}

int evc_plm_create(evc_plm_t **out, const uint8_t *codes, int64_t N, int32_t L, int32_t q, int32_t gap_code,
                   const float *weights, int32_t device)
{
    if (!out || !codes || !weights) { set_error("evc_plm_create: null pointer"); return 1; }
    *out = nullptr;
    if (N <= 0 || L < 2) { set_error("evc_plm_create: need N >= 1 sequences and L >= 2 sites"); return 1; }
    if (!plm_supported_q(q)) {
        set_error("evc_plm_create: unsupported number of states q=" + std::to_string(q) +
                  " (supported: 4, 5, 20, 21)");
        return 1;
    }
    if (gap_code >= 0 && gap_code != q) {
        set_error("evc_plm_create: gap_code must be -1 or q");
        return 1;
    }
    if (L > 65535) { set_error("evc_plm_create: L too large"); return 1; }
    // every code must address a row of a coupling block: 0..q-1, or q for the ignored gap (the kernels index
    // shared-memory rows with the raw byte, so an out-of-range code would silently read another site's block)
    {
        unsigned mx = 0;
        const size_t total = (size_t)N * L;
        for (size_t e = 0; e < total; e++) mx = codes[e] > mx ? codes[e] : mx;
        if ((int)mx >= (gap_code >= 0 ? q + 1 : q)) {
            set_error("evc_plm_create: sequence code " + std::to_string(mx) + " out of range (valid: 0.." +
                      std::to_string((gap_code >= 0 ? q + 1 : q) - 1) + (gap_code >= 0 ? ", the last one being the ignored gap)" : ")"));
            return 1;
        }
    }
    EVC_CUDA(cudaSetDevice(device));
    evc_plm *h = new (std::nothrow) evc_plm();
    if (!h) { set_error("evc_plm_create: out of host memory"); return 1; }
    h->device = device;
    PlmGeom &g = h->g;
    g.N = N;
    g.L = L;
    g.Lp = (int)round_up(L, 4);
    g.q = q;
    g.gap_code = gap_code;
    g.QB = gap_code >= 0 ? q + 1 : q;
    g.S = (q % 2) ? q : q + 1;
    g.Nr = round_up(N, PLM_BWD_TS);
    g.Nld = round_up(N, 32);
    g.L4 = g.Lp / 4;
    g.ntiles_f = (int)ceil_div(N, PLM_FWD_TS);
    g.ntiles_b = (int)ceil_div(N, PLM_BWD_TS);
    g.n_params = (int64_t)L * q + (int64_t)L * (L - 1) / 2 * q * q;

    bool ok = cudaMalloc(&h->d_codes, (size_t)N * L) == cudaSuccess &&
              cudaMalloc(&h->d_msa4, (size_t)g.L4 * g.Nld * sizeof(uint32_t)) == cudaSuccess &&
              cudaMalloc(&h->d_wts, (size_t)N * sizeof(float)) == cudaSuccess;
    if (!ok) {
        set_error(std::string("evc_plm_create: device allocation failed: ") +
                  cudaGetErrorString(cudaGetLastError()));
        evc_plm_destroy(h);
        return 1;
    }
    ok = cudaMemcpy(h->d_codes, codes, (size_t)N * L, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(h->d_wts, weights, (size_t)N * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok || plm_pack_msa(g, h->d_codes, h->d_msa4, 0) || cudaDeviceSynchronize() != cudaSuccess) {
        if (ok) set_error(std::string("evc_plm_create: packing failed: ") + cudaGetErrorString(cudaGetLastError()));
        else set_error("evc_plm_create: H2D failed");
        evc_plm_destroy(h);
        return 1;
    }
    *out = h;
    return 0;
}

// Buffers of the gather path (expanded couplings W, their gradient G, residuals R, state-sorted bucket lists):
// 6.7 GB of R alone at N = 100k, L = 800 -- allocated only when a gather kernel is actually selected.
static int ensure_gather(evc_plm *h)
{
    if (h->gather_ready) return 0;
    EVC_CUDA(cudaSetDevice(h->device));
    const PlmGeom &g = h->g;
    const size_t w_bytes = (size_t)g.w_floats() * sizeof(float);
    const size_t r_bytes = (size_t)g.L * g.Nr * g.S * sizeof(float);
    const bool ok = cudaMalloc(&h->d_perm, (size_t)g.ntiles_b * g.L * PLM_BWD_CAP * sizeof(uint32_t)) == cudaSuccess &&
                    cudaMalloc(&h->d_bstart, (size_t)g.ntiles_b * g.L * PLM_BWD_BS * sizeof(uint16_t)) == cudaSuccess &&
                    cudaMalloc(&h->d_W, w_bytes) == cudaSuccess && cudaMalloc(&h->d_G, w_bytes) == cudaSuccess &&
                    cudaMalloc(&h->d_R, r_bytes) == cudaSuccess &&
                    cudaMalloc(&h->d_gh_part, (size_t)g.L * g.ntiles_f * g.S * sizeof(float)) == cudaSuccess &&
                    cudaMalloc(&h->d_fx_part, (size_t)g.L * g.ntiles_f * sizeof(double)) == cudaSuccess;
    if (!ok) {
        set_error(std::string("libevcplm: device allocation of the gather-path buffers failed: ") +
                  cudaGetErrorString(cudaGetLastError()));
        return 1;
    }
    EVC_CUDA(cudaMemset(h->d_W, 0, w_bytes));
    EVC_CUDA(cudaMemset(h->d_R, 0, r_bytes));
    if (plm_build_buckets(g, h->d_codes, h->d_perm, h->d_bstart, 0)) return 1;
    EVC_CUDA(cudaDeviceSynchronize());
    h->gather_ready = true;
    return 0;
}

int64_t evc_plm_num_params(const evc_plm_t *h) { return h ? h->g.n_params : -1; }

int evc_plm_set_precision(evc_plm_t *h, int32_t mode)
{
    if (!h) { set_error("evc_plm_set_precision: null handle"); return 1; }
    if (mode != 0 && mode != 1) {
        set_error("evc_plm_set_precision: mode must be 0 (fp32-equivalent, bf16 hi+lo products) or 1 (bf16 tiles)");
        return 1;
    }
    h->precision = mode;
    return 0;
}

int evc_plm_eval_data(evc_plm_t *h, const float *d_x, float *d_g, double *d_fx, void *stream)
{
    if (!h || !d_x || !d_g || !d_fx) { set_error("evc_plm_eval_data: null pointer"); return 1; }
    cudaStream_t st = as_stream(stream);
    const PlmGeom &g = h->g;
    const bool prof = h->profiling;
    const bool tc = h->bwd_mode == 1;
    const bool tcf = h->fwd_mode == 1;
    const bool tcff = h->fwd_mode == 2;
    const int single = h->precision == 1 ? 1 : 0;      // only the tensor-core products have a reduced mode
    void *rt_lo = single ? nullptr : h->d_rt_lo;
    float *gJ = d_g + (int64_t)g.L * g.q;
    if ((!tc || (!tcf && !tcff)) && ensure_gather(h)) return 1;
    if (prof) EVC_CUDA(cudaEventRecord(h->ev[0], st));
    if (tcff) {
        // expand -> fused tcgen05 forward (logits + softmax + residuals) -> tcgen05 backward GEMM
        if (plm_tcff_expand(g, h->tcff, d_x, h->d_wp_hi, h->d_wp_lo, single, st)) return 1;
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[1], st));
        if (plm_tcff_forward(g, h->tcff, h->tcff_maps, d_x, h->d_msa4, h->d_wts, h->d_rt_hi, h->d_rt_lo, h->tc.Kp,
                             h->d_gh_part3, h->d_fx_part3, single, st))
            return 1;
        if (prof) {
            EVC_CUDA(cudaEventRecord(h->ev[2], st));
            EVC_CUDA(cudaEventRecord(h->ev[3], st));
        }
        if (plm_tc_backward(g, h->tc, h->tc_maps, h->d_Gd, single, st)) return 1;
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[4], st));
        if (plm_tc_finalize_pairs(g, h->tc, h->d_Gd, gJ, 1.0f, st)) return 1;
        if (plm_finalize_fields_n(g, h->d_gh_part3, h->d_fx_part3, d_g, d_fx, h->tcff.ntile_part, st)) return 1;
    } else if (tcf) {
        // expand -> tcgen05 logits GEMM -> softmax/residuals -> tcgen05 backward GEMM
        if (plm_tcf_expand(g, h->tcf, d_x, h->d_wt_hi, h->d_wt_lo, single, st)) return 1;
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[1], st));
        if (plm_tcf_logits(g, h->tcf, h->tcf_maps, h->d_zt, single, st)) return 1;
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[2], st));
        if (plm_tcf_softmax(g, h->tcf, h->d_zt, d_x, h->d_msa4, h->d_wts, h->d_rt_hi, rt_lo, h->tc.Kp,
                            h->d_gh_part2, h->d_fx_part2, st))
            return 1;
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[3], st));
        if (plm_tc_backward(g, h->tc, h->tc_maps, h->d_Gd, single, st)) return 1;
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[4], st));
        if (plm_tc_finalize_pairs(g, h->tc, h->d_Gd, gJ, 1.0f, st)) return 1;
        if (plm_finalize_fields_n(g, h->d_gh_part2, h->d_fx_part2, d_g, d_fx, h->tcf.ntiles_s, st)) return 1;
    } else {
        if (plm_expand(g, d_x, h->d_W, st)) return 1;
        if (!tc) EVC_CUDA(cudaMemsetAsync(h->d_G, 0, (size_t)g.w_floats() * sizeof(float), st));
        if (prof) EVC_CUDA(cudaEventRecord(h->ev[1], st));
        if (plm_forward(g, h->d_W, d_x, h->d_msa4, h->d_wts, h->d_R, tc ? h->d_rt_hi : nullptr,
                        tc ? h->d_rt_lo : nullptr, h->tc.Kp, h->d_gh_part, h->d_fx_part, st))
            return 1;
        if (prof) {
            EVC_CUDA(cudaEventRecord(h->ev[2], st));
            EVC_CUDA(cudaEventRecord(h->ev[3], st));
        }
        if (tc) {
            if (plm_tc_backward(g, h->tc, h->tc_maps, h->d_Gd, single, st)) return 1;
            if (prof) EVC_CUDA(cudaEventRecord(h->ev[4], st));
            if (plm_tc_finalize_pairs(g, h->tc, h->d_Gd, gJ, 1.0f, st)) return 1;
            if (plm_finalize_fields(g, h->d_gh_part, h->d_fx_part, d_g, d_fx, st)) return 1;
        } else {
            if (plm_backward(g, h->d_R, h->d_perm, h->d_bstart, h->d_G, st)) return 1;
            if (prof) EVC_CUDA(cudaEventRecord(h->ev[4], st));
            if (plm_finalize(g, h->d_G, h->d_gh_part, h->d_fx_part, d_g, gJ, d_fx, 1.0f, st)) return 1;
        }
    }
    if (prof) {
        EVC_CUDA(cudaEventRecord(h->ev[5], st));
        h->ev_valid = true;
    }
    return 0;
}

int evc_plm_set_backward(evc_plm_t *h, int32_t mode)
{
    if (!h) { set_error("evc_plm_set_backward: null handle"); return 1; }
    if (mode != 0 && mode != 1) { set_error("evc_plm_set_backward: mode must be 0 (gather) or 1 (tensor core)"); return 1; }
    EVC_CUDA(cudaSetDevice(h->device));
    if (mode == 1 && !h->d_xt) {
        plm_tc_geometry(h->g, h->tc);
        const PlmTcGeom &t = h->tc;
        const size_t xb = (size_t)t.Mp * t.Kp * 2, rb = (size_t)t.Np * t.Kp * 2;
        if (cudaMalloc(&h->d_xt, xb) != cudaSuccess || cudaMalloc(&h->d_rt_hi, rb) != cudaSuccess ||
            cudaMalloc(&h->d_rt_lo, rb) != cudaSuccess ||
            cudaMalloc(&h->d_Gd, (size_t)t.Mp * t.Np * sizeof(float)) != cudaSuccess) {
            set_error(std::string("evc_plm_set_backward: device allocation failed: ") +
                      cudaGetErrorString(cudaGetLastError()));
            return 1;
        }
        EVC_CUDA(cudaMemset(h->d_rt_hi, 0, rb));
        EVC_CUDA(cudaMemset(h->d_rt_lo, 0, rb));
        EVC_CUDA(cudaMemset(h->d_Gd, 0, (size_t)t.Mp * t.Np * sizeof(float)));
        if (plm_tc_build_xt(h->g, t, h->d_msa4, h->d_xt, 0)) return 1;
        EVC_CUDA(cudaDeviceSynchronize());
        h->tc_maps = aligned_alloc(64, round_up((int64_t)plm_tc_map_bytes(), 64));
        if (!h->tc_maps) { set_error("evc_plm_set_backward: out of host memory"); return 1; }
        if (plm_tc_make_maps(t, h->d_xt, h->d_rt_hi, h->d_rt_lo, h->tc_maps)) return 1;
    }
    h->bwd_mode = mode;
    return 0;
}

int evc_plm_set_forward(evc_plm_t *h, int32_t mode)
{
    if (!h) { set_error("evc_plm_set_forward: null handle"); return 1; }
    if (mode < 0 || mode > 2) {
        set_error("evc_plm_set_forward: mode must be 0 (gather), 1 (tensor core) or 2 (tensor core, fused softmax)");
        return 1;
    }
    EVC_CUDA(cudaSetDevice(h->device));
    // the fused variant needs the 21-wide site layout and keeps the whole K extent in one TMEM accumulation
    // chain (no K-chunk promotion): nucleotide alphabets and L*q > 8192 use the unfused tensor-core forward
    if (mode == 2 && (!plm_tcff_supported(h->g) || (int64_t)h->g.L * h->g.q > 8192)) mode = 1;
    if (mode >= 1) {
        if (evc_plm_set_backward(h, 1)) return 1;     // the tensor-core forward feeds the tensor-core backward
        if (!h->d_x1h) {
            plm_tcf_geometry(h->g, h->tcf);
            const PlmTcfGeom &t = h->tcf;
            const size_t xb = (size_t)t.Xrows * t.Kw * 2;
            if (cudaMalloc(&h->d_x1h, xb) != cudaSuccess) {
                set_error("evc_plm_set_forward: device allocation failed (one-hot operand)");
                return 1;
            }
            if (plm_tcf_build_x(h->g, t, h->d_msa4, h->d_x1h, 0)) return 1;
            EVC_CUDA(cudaDeviceSynchronize());
        }
    }
    if (mode == 1 && !h->d_zt) {
        const PlmTcfGeom &t = h->tcf;
        const size_t wb = (size_t)t.Mp * t.Kw * 2;
        const size_t zb = (size_t)t.Mp * t.Ns * sizeof(float);
        if (cudaMalloc(&h->d_wt_hi, wb) != cudaSuccess || cudaMalloc(&h->d_wt_lo, wb) != cudaSuccess ||
            cudaMalloc(&h->d_zt, zb) != cudaSuccess ||
            cudaMalloc(&h->d_gh_part2, (size_t)h->g.L * t.ntiles_s * h->g.S * sizeof(float)) != cudaSuccess ||
            cudaMalloc(&h->d_fx_part2, (size_t)h->g.L * t.ntiles_s * sizeof(double)) != cudaSuccess) {
            set_error(std::string("evc_plm_set_forward: device allocation failed: ") +
                      cudaGetErrorString(cudaGetLastError()));
            return 1;
        }
        EVC_CUDA(cudaMemset(h->d_wt_hi, 0, wb));
        EVC_CUDA(cudaMemset(h->d_wt_lo, 0, wb));
        h->tcf_maps = aligned_alloc(64, round_up((int64_t)plm_tc_map_bytes(), 64));
        if (!h->tcf_maps) { set_error("evc_plm_set_forward: out of host memory"); return 1; }
        if (plm_tcf_make_maps(t, h->d_wt_hi, h->d_wt_lo, h->d_x1h, h->tcf_maps)) return 1;
    }
    if (mode == 2 && !h->d_wp_hi) {
        plm_tcff_geometry(h->g, h->tcff);
        const PlmTcffGeom &t = h->tcff;
        const size_t wb = (size_t)t.Np * t.Kw * 2;
        if (cudaMalloc(&h->d_wp_hi, wb) != cudaSuccess || cudaMalloc(&h->d_wp_lo, wb) != cudaSuccess ||
            cudaMalloc(&h->d_gh_part3, (size_t)h->g.L * t.ntile_part * h->g.S * sizeof(float)) != cudaSuccess ||
            cudaMalloc(&h->d_fx_part3, (size_t)h->g.L * t.ntile_part * sizeof(double)) != cudaSuccess) {
            set_error(std::string("evc_plm_set_forward: device allocation failed: ") +
                      cudaGetErrorString(cudaGetLastError()));
            return 1;
        }
        EVC_CUDA(cudaMemset(h->d_wp_hi, 0, wb));
        EVC_CUDA(cudaMemset(h->d_wp_lo, 0, wb));
        h->tcff_maps = aligned_alloc(64, round_up((int64_t)plm_tc_map_bytes(), 64));
        if (!h->tcff_maps) { set_error("evc_plm_set_forward: out of host memory"); return 1; }
        if (plm_tcff_make_maps(t, h->d_x1h, h->d_wp_hi, h->d_wp_lo, h->tcff_maps)) return 1;
    }
    h->fwd_mode = mode;
    return 0;
}

int evc_plm_set_profiling(evc_plm_t *h, int32_t enable)
{
    if (!h) { set_error("evc_plm_set_profiling: null handle"); return 1; }
    EVC_CUDA(cudaSetDevice(h->device));
    if (enable && !h->ev[0])
        for (int k = 0; k < 6; k++) EVC_CUDA(cudaEventCreate(&h->ev[k]));
    h->profiling = enable != 0;
    h->ev_valid = false;
    return 0;
}

int evc_plm_last_stage_ms(evc_plm_t *h, float *ms_out)
{
    if (!h || !ms_out) { set_error("evc_plm_last_stage_ms: null pointer"); return 1; }
    if (!h->ev_valid) { set_error("evc_plm_last_stage_ms: no profiled evaluation recorded"); return 1; }
    EVC_CUDA(cudaEventSynchronize(h->ev[5]));
    for (int k = 0; k < 5; k++) EVC_CUDA(cudaEventElapsedTime(&ms_out[k], h->ev[k], h->ev[k + 1]));
    return 0;
}

int evc_plm_add_regulariser(evc_plm_t *h, const float *d_x, float *d_g, double *d_fx, float lambda_h,
                            float lambda_J, void *stream)
{
    if (!h || !d_x || !d_g || !d_fx) { set_error("evc_plm_add_regulariser: null pointer"); return 1; }
    return plm_add_reg(h->g, d_x, d_g, d_fx, lambda_h, lambda_J, as_stream(stream));
}

int evc_plm_eval_host(evc_plm_t *h, const float *x, float *gout, double *fx_out, float lambda_h,
                      float lambda_J)
{
    if (!h || !x || !gout || !fx_out) { set_error("evc_plm_eval_host: null pointer"); return 1; }
    EVC_CUDA(cudaSetDevice(h->device));
    const size_t nb = (size_t)h->g.n_params * sizeof(float);
    if (!h->d_x_tmp) {
        EVC_CUDA(cudaMalloc(&h->d_x_tmp, nb));
        EVC_CUDA(cudaMalloc(&h->d_g_tmp, nb));
        EVC_CUDA(cudaMalloc(&h->d_fx_tmp, 2 * sizeof(double)));
    }
    EVC_CUDA(cudaMemcpyAsync(h->d_x_tmp, x, nb, cudaMemcpyHostToDevice, 0));
    if (evc_plm_eval_data(h, h->d_x_tmp, h->d_g_tmp, h->d_fx_tmp, nullptr)) return 1;
    if (evc_plm_add_regulariser(h, h->d_x_tmp, h->d_g_tmp, h->d_fx_tmp, lambda_h, lambda_J, nullptr)) return 1;
    EVC_CUDA(cudaMemcpyAsync(gout, h->d_g_tmp, nb, cudaMemcpyDeviceToHost, 0));
    EVC_CUDA(cudaMemcpyAsync(fx_out, h->d_fx_tmp, 2 * sizeof(double), cudaMemcpyDeviceToHost, 0));
    EVC_CUDA(cudaStreamSynchronize(0));
    return 0;
}

int evc_plm_weighted_counts(evc_plm_t *h, float *d_fi_counts, float *d_fij_counts, void *stream)
{
    if (!h || !d_fi_counts || !d_fij_counts) { set_error("evc_plm_weighted_counts: null pointer"); return 1; }
    cudaStream_t st = as_stream(stream);
    const PlmGeom &g = h->g;
    if (h->bwd_mode == 1 && h->d_gh_part2) {
        // tensor-core path: f_ij = Xt (w X)^T through the same backward product (weights as bf16 hi + lo)
        const int ntiles = h->tcf.ntiles_s;
        if (plm_tc_onehot_residual(g, ntiles, h->d_msa4, h->d_wts, h->d_rt_hi, h->d_rt_lo, h->tc.Kp, h->d_gh_part2,
                                   h->d_fx_part2, st))
            return 1;
        if (plm_tc_backward(g, h->tc, h->tc_maps, h->d_Gd, 0, st)) return 1;
        if (plm_tc_finalize_pairs(g, h->tc, h->d_Gd, d_fij_counts, 0.5f, st)) return 1;
        return plm_finalize_fields_n(g, h->d_gh_part2, nullptr, d_fi_counts, nullptr, ntiles, st);
    }
    if (ensure_gather(h)) return 1;
    EVC_CUDA(cudaMemsetAsync(h->d_G, 0, (size_t)g.w_floats() * sizeof(float), st));
    if (plm_onehot_residual(g, h->d_msa4, h->d_wts, h->d_R, h->d_gh_part, st)) return 1;
    if (plm_backward(g, h->d_R, h->d_perm, h->d_bstart, h->d_G, st)) return 1;
    return plm_finalize(g, h->d_G, h->d_gh_part, nullptr, d_fi_counts, d_fij_counts, nullptr, 0.5f, st);
}

// ---- 8(f) rows f1 / f2 ------------------------------------------------------------------------------
int evc_ec_scores(const float *d_J_tri, const float *d_fij_tri, const float *d_fi, int32_t L, int32_t q,
                  float *d_fn_raw, float *d_fn_zero_sum, float *d_mi, void *stream)
{
    if (!d_J_tri) { set_error("evc_ec_scores: null pointer"); return 1; }
    return ec_scores(d_J_tri, d_fij_tri, d_fi, L, q, d_fn_raw, d_fn_zero_sum, d_mi, as_stream(stream));
}

int evc_plm_energies(evc_plm_t *h, const float *d_x, double *d_out, void *stream)
{
    if (!h || !d_x || !d_out) { set_error("evc_plm_energies: null pointer"); return 1; }
    cudaStream_t st = as_stream(stream);
    const PlmGeom &g = h->g;
    if (ensure_gather(h)) return 1;
    if (plm_expand(g, d_x, h->d_W, st)) return 1;
    // the residual buffer (L * Nr * S floats) is free outside an evaluation: reuse it for the per-site partials
    return plm_energies(g, h->d_W, d_x, h->d_msa4, h->d_R, d_out, st);
}

// ---- a8 vector algebra --------------------------------------------------------------------------
int evc_vec_dot(const float *d_a, const float *d_b, int64_t n, double *d_out, void *stream)
{
    return vec_dot(d_a, d_b, n, d_out, as_stream(stream));
}
int evc_vec_axpby(float *d_y, const float *d_x, float a, float b, int64_t n, void *stream)
{
    return vec_axpby(d_y, d_x, a, b, n, as_stream(stream));
}
int evc_vec_copy(float *d_dst, const float *d_src, int64_t n, void *stream)
{
    EVC_CUDA(cudaMemcpyAsync(d_dst, d_src, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice,
                             as_stream(stream)));
    return 0;
}
int evc_vec_sub(float *d_out, const float *d_a, const float *d_b, int64_t n, void *stream)
{
    return vec_sub(d_out, d_a, d_b, n, as_stream(stream));
}
int evc_lbfgs_direction(float *d_d, const float *d_g, const float *d_S, const float *d_Y, const double *d_ys,
                        double *d_scratch, int64_t n, int32_t m, int32_t bound, int32_t end, void *stream)
{
    return lbfgs_direction(d_d, d_g, d_S, d_Y, d_ys, d_scratch, n, m, bound, end, as_stream(stream));
}
int evc_lbfgs_update_pair(float *d_S_slot, float *d_Y_slot, const float *d_x, const float *d_xp,
                          const float *d_g, const float *d_gp, double *d_ys_slot, double *d_yy, int64_t n,
                          void *stream)
{
    return lbfgs_update_pair(d_S_slot, d_Y_slot, d_x, d_xp, d_g, d_gp, d_ys_slot, d_yy, n, as_stream(stream));
}
int evc_fn_scores(const float *d_J_tri, int32_t L, int32_t q, float *d_fn, void *stream)
{
    return fn_scores(d_J_tri, L, q, d_fn, as_stream(stream));
}

// ---- mean-field DCA (mean_field.cu) ----------------------------------------------------------------------
static int mf_check_dims(const char *what, int32_t L, int32_t q)
{
    if (L < 2 || q < 2 || q > 21) {
        set_error(std::string(what) + ": need L >= 2 and 2 <= q <= 21");
        return 1;
    }
    return 0;
}

int evc_mf_weighted_counts_f64(const uint8_t *d_codes, const double *d_weights, int64_t N, int32_t L, int32_t q,
                               double n_eff, double *d_F, void *stream)
{
    if (!d_codes || !d_weights || !d_F || N < 1) { set_error("evc_mf_weighted_counts_f64: bad argument"); return 1; }
    if (mf_check_dims("evc_mf_weighted_counts_f64", L, q)) return 1;
    if (!(n_eff > 0.0)) { set_error("evc_mf_weighted_counts_f64: n_eff must be > 0"); return 1; }
    return mf_weighted_counts(d_codes, d_weights, N, L, q, n_eff, d_F, as_stream(stream));
}

int evc_mf_covariance(const double *d_F, int32_t L, int32_t q, double pseudo_count, double *d_C, double *d_fi,
                      double *d_rfi, double *d_fij_tri, void *stream)
{
    if (!d_F) { set_error("evc_mf_covariance: null pointer"); return 1; }
    if (mf_check_dims("evc_mf_covariance", L, q)) return 1;
    return mf_covariance(d_F, L, q, pseudo_count, d_C, d_fi, d_rfi, d_fij_tri, as_stream(stream));
}

int evc_spd_inverse_f64(double *d_A, int64_t n, double *d_work, int32_t *info_out, void *stream)
{
    if (!d_A || !d_work || !info_out || n < 1) { set_error("evc_spd_inverse_f64: bad argument"); return 1; }
    *info_out = 0;
    cudaStream_t st = as_stream(stream);
    int *d_info = nullptr;
    EVC_CUDA(cudaMallocAsync(&d_info, sizeof(int), st));
    const int rc = spd_inverse(d_A, n, d_work, d_info, st);
    int info = 0;
    if (rc == 0) {
        EVC_CUDA(cudaMemcpyAsync(&info, d_info, sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    EVC_CUDA(cudaFreeAsync(d_info, st));
    EVC_CUDA(cudaStreamSynchronize(st));
    if (rc) return rc;
    *info_out = info;
    if (info) {
        set_error("evc_spd_inverse_f64: matrix is not positive definite (non-positive pivot at column " +
                  std::to_string(info) + ")");
        return EVC_NOT_SPD;
    }
    return 0;
}

int evc_mf_couplings_fields(const double *d_Cinv, const double *d_rfi, int32_t L, int32_t q, double *d_J_tri,
                            double *d_h, void *stream)
{
    if (!d_Cinv || !d_rfi) { set_error("evc_mf_couplings_fields: null pointer"); return 1; }
    if (mf_check_dims("evc_mf_couplings_fields", L, q)) return 1;
    return mf_couplings_fields(d_Cinv, d_rfi, L, q, d_J_tri, d_h, as_stream(stream));
}

int evc_mf_di_scores(const double *d_J_tri, const double *d_rfi, int32_t L, int32_t q, double *d_di,
                     int32_t *d_iters, void *stream)
{
    if (!d_J_tri || !d_rfi || !d_di) { set_error("evc_mf_di_scores: null pointer"); return 1; }
    if (mf_check_dims("evc_mf_di_scores", L, q)) return 1;
    return mf_di_scores(d_J_tri, d_rfi, L, q, d_di, d_iters, as_stream(stream));
}

int evc_ec_scores_f64(const double *d_J_tri, const double *d_fij_tri, const double *d_fi, int32_t L, int32_t q,
                      double *d_fn_raw, double *d_fn_zero_sum, double *d_mi, void *stream)
{
    if (!d_J_tri) { set_error("evc_ec_scores_f64: null pointer"); return 1; }
    return ec_scores_f64(d_J_tri, d_fij_tri, d_fi, L, q, d_fn_raw, d_fn_zero_sum, d_mi, as_stream(stream));
}

}  // extern "C"
