// SURVEY.md 8(f) rows f1 / f2 -- consumers of the fitted model, on the device.
//
// f1  EC scoring as done by the reference's CouplingsModel._calculate_ecs
//     (evcouplings/couplings/model.py:777-827): zero-sum gauge (model.py:179-233) Frobenius norm of
//     every J_ij block, raw-gauge Frobenius norm (what plmc writes to _ECs.txt) and mutual information
//     from f_ij / f_i.  The APC (model.py:744-775) is an L x L operation done by the host.
//     ||J0||_F^2 = sum J^2 - (1/q) sum_a r_a^2 - (1/q) sum_b c_b^2 + T^2/q^2   (r, c row/column sums, T total).
// f2  statistical energies of many sequences (model.py:25-60 _hamiltonians): for each sequence
//     H_J = sum_{i<j} J_ij(s_i, s_j),  H_h = sum_i h_i(s_i).  Same streaming of the expanded coupling rows
//     through shared memory as plm_fwd_kernel, but ONE gathered element per (sequence, i, j).
#include "common.cuh"
#include "internal.h"

namespace evc {

// Real = float for the PLM models; Real = double for the mean-field scores (accumulation is fp64 in both)
template <typename Real>
__global__ void ec_block_scores_kernel(const Real *__restrict__ J, const Real *__restrict__ fij,
                                       const Real *__restrict__ fi, int L, int q, int64_t npairs,
                                       Real *__restrict__ fn_raw, Real *__restrict__ fn_zs,
                                       Real *__restrict__ mi)
{
    const int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= npairs) return;
    const int qq = q * q;
    const Real *B = J + p * qq;
    // lane a (< q) owns row a: row sum, sum of squares; column sums via a second pass
    double rs = 0.0, ss = 0.0, cs = 0.0;
    if (lane < q) {
        for (int b = 0; b < q; b++) {
            const double v = B[lane * q + b];
            rs += v;
            ss += v * v;
            cs += (double)B[b * q + lane];
        }
    }
    const double T = warp_sum(rs);
    const double SS = warp_sum(ss);
    const double R2 = warp_sum(rs * rs);
    const double C2 = warp_sum(cs * cs);
    if (lane == 0) {
        if (fn_raw) fn_raw[p] = (Real)sqrt(SS);
        double z = SS - R2 / q - C2 / q + T * T / ((double)q * q);
        if (fn_zs) fn_zs[p] = (Real)sqrt(z > 0.0 ? z : 0.0);
    }
    if (mi != nullptr && fij != nullptr) {
        // pair index -> (i, j)
        int i = 0;
        int64_t rem = p;
        while (rem >= L - 1 - i) { rem -= L - 1 - i; i++; }
        const int j = i + 1 + (int)rem;
        const Real *F = fij + p * qq;
        double acc = 0.0;
        for (int e = lane; e < qq; e += 32) {
            const int a = e / q, b = e - a * q;
            const double pv = F[e];
            const double m = (double)fi[i * q + a] * (double)fi[j * q + b];
            if (pv > 0.0 && m > 0.0) acc += pv * log(pv / m);
        }
        acc = warp_sum(acc);
        if (lane == 0) mi[p] = (Real)acc;
    }
}

template <typename Real>
static int ec_scores_t(const Real *d_J, const Real *d_fij, const Real *d_fi, int L, int q, Real *d_fn_raw,
                       Real *d_fn_zs, Real *d_mi, cudaStream_t st)
{
    const int64_t npairs = (int64_t)L * (L - 1) / 2;
    if (npairs == 0) return 0;
    if (q > 32) { set_error("ec_scores: q > 32 not supported"); return 1; }
    ec_block_scores_kernel<Real><<<(unsigned)ceil_div(npairs, 8), 256, 0, st>>>(d_J, d_fij, d_fi, L, q, npairs,
                                                                              d_fn_raw, d_fn_zs, d_mi);
    EVC_KERNEL_CHECK();
    return 0;
}

int ec_scores(const float *d_J, const float *d_fij, const float *d_fi, int L, int q, float *d_fn_raw,
              float *d_fn_zs, float *d_mi, cudaStream_t st)
{
    return ec_scores_t(d_J, d_fij, d_fi, L, q, d_fn_raw, d_fn_zs, d_mi, st);
}

int ec_scores_f64(const double *d_J, const double *d_fij, const double *d_fi, int L, int q, double *d_fn_raw,
                  double *d_fn_zs, double *d_mi, cudaStream_t st)
{
    return ec_scores_t(d_J, d_fij, d_fi, L, q, d_fn_raw, d_fn_zs, d_mi, st);
}

// ---- f2: energies --------------------------------------------------------------------------------
constexpr int EN_JC = 24;
constexpr int EN_THREADS = 256;

template <int S>
__global__ void __launch_bounds__(EN_THREADS, 2)
plm_energy_kernel(const float *__restrict__ W, const uint32_t *__restrict__ msa4, float *__restrict__ Epart,
                  PlmGeom g)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int BLK = g.QB * S;
    const int chunk_floats = EN_JC * BLK;
    float *buf0 = reinterpret_cast<float *>(smem_raw);
    float *buf1 = buf0 + chunk_floats;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)2 * chunk_floats * sizeof(float));
    const int tile = blockIdx.x, i = blockIdx.y, tid = threadIdx.x;
    const int64_t N = g.N;
    const int64_t n0 = (int64_t)tile * (2 * EN_THREADS) + tid, n1 = n0 + EN_THREADS;
    const int64_t m0 = n0 < N ? n0 : N - 1, m1 = n1 < N ? n1 : N - 1;
    const int Lp = g.Lp;
    const int nchunks = (Lp + EN_JC - 1) / EN_JC;
    const float *Wi = W + (int64_t)i * g.row_block();
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)(min(EN_JC, Lp) * BLK * sizeof(float));
        mbar_expect_tx(&bars[0], bytes);
        bulk_g2s(buf0, Wi, bytes, &bars[0]);
    }
    const uint32_t wi0 = msa4[(int64_t)(i >> 2) * g.Nld + m0], wi1 = msa4[(int64_t)(i >> 2) * g.Nld + m1];
    int s0 = (int)((wi0 >> (8 * (i & 3))) & 0xffu), s1 = (int)((wi1 >> (8 * (i & 3))) & 0xffu);
    const bool ok0 = s0 < g.q, ok1 = s1 < g.q;      // ignored gap at site i: contributes nothing
    if (!ok0) s0 = 0;
    if (!ok1) s1 = 0;
    float e0 = 0.f, e1 = 0.f;
    for (int c = 0; c < nchunks; c++) {
        const int j0 = c * EN_JC;
        const int jc = min(EN_JC, Lp - j0);
        if (tid == 0 && c + 1 < nchunks) {
            const int jn = min(EN_JC, Lp - (j0 + EN_JC));
            const uint32_t bytes = (uint32_t)(jn * BLK * sizeof(float));
            uint64_t *bar = &bars[(c + 1) & 1];
            mbar_expect_tx(bar, bytes);
            bulk_g2s(((c + 1) & 1) ? buf1 : buf0, Wi + (int64_t)(j0 + EN_JC) * BLK, bytes, bar);
        }
        uint32_t pk0[EN_JC / 4], pk1[EN_JC / 4];
#pragma unroll
        for (int u = 0; u < EN_JC / 4; u++) {
            pk0[u] = 0; pk1[u] = 0;
            if (u * 4 < jc) {
                const int64_t off = (int64_t)(j0 / 4 + u) * g.Nld;
                pk0[u] = msa4[off + m0];
                pk1[u] = msa4[off + m1];
            }
        }
        mbar_wait(&bars[c & 1], (uint32_t)((c >> 1) & 1));
        const float *B = (c & 1) ? buf1 : buf0;
#pragma unroll
        for (int u = 0; u < EN_JC / 4; u++) {
            if (u * 4 < jc) {
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    const int jj = u * 4 + v;
                    const uint32_t b0 = (pk0[u] >> (8 * v)) & 0xffu, b1 = (pk1[u] >> (8 * v)) & 0xffu;
                    e0 += B[jj * BLK + b0 * S + s0];      // W[i][j][b][a]: zero for j == i, padded j, gap b
                    e1 += B[jj * BLK + b1 * S + s1];
                }
            }
        }
        __syncthreads();
    }
    if (n0 < N) Epart[(int64_t)i * g.Nld + n0] = ok0 ? e0 : 0.f;
    if (n1 < N) Epart[(int64_t)i * g.Nld + n1] = ok1 ? e1 : 0.f;
}

__global__ void energy_reduce_kernel(const float *__restrict__ Epart, const float *__restrict__ h,
                                     const uint32_t *__restrict__ msa4, double *__restrict__ out, PlmGeom g)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= g.N) return;
    double hj = 0.0, hh = 0.0;
    for (int i = 0; i < g.L; i++) {
        hj += (double)Epart[(int64_t)i * g.Nld + n];
        const int s = (int)((msa4[(int64_t)(i >> 2) * g.Nld + n] >> (8 * (i & 3))) & 0xffu);
        if (s < g.q) hh += (double)h[i * g.q + s];
    }
    hj *= 0.5;                      // every pair was visited from both of its sites
    out[n * 3 + 0] = hj + hh;
    out[n * 3 + 1] = hj;
    out[n * 3 + 2] = hh;
}

int plm_energies(const PlmGeom &g, const float *d_W, const float *d_x, const uint32_t *d_msa4, float *d_epart,
                 double *d_out, cudaStream_t st)
{
    dim3 grid((unsigned)ceil_div(g.N, 2 * EN_THREADS), (unsigned)g.L);
    const size_t smem = (size_t)2 * EN_JC * g.QB * g.S * sizeof(float) + 2 * sizeof(uint64_t);
    if (g.S == 21) {
        EVC_CUDA(cudaFuncSetAttribute(plm_energy_kernel<21>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        plm_energy_kernel<21><<<grid, EN_THREADS, smem, st>>>(d_W, d_msa4, d_epart, g);
    } else if (g.S == 5) {
        plm_energy_kernel<5><<<grid, EN_THREADS, smem, st>>>(d_W, d_msa4, d_epart, g);
    } else {
        set_error("plm_energies: unsupported row stride");
        return 1;
    }
    EVC_KERNEL_CHECK();
    energy_reduce_kernel<<<(unsigned)ceil_div(g.N, 256), 256, 0, st>>>(d_epart, d_x, d_msa4, d_out, g);
    EVC_KERNEL_CHECK();
    return 0;
}

}  // namespace evc
