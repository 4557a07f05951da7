// Mean-field DCA (the reference's evcouplings/couplings/mean_field.py, MeanFieldDCA.fit and
// MeanFieldCouplingsModel's DI), in fp64 throughout.
//
// One tile-GEMM engine (fp64 FFMA, 64x64 tiles, 4x4 outputs per thread) serves
//   - the weighted one-hot counts  F = X^T diag(w) X / N_eff  (X: N x L*q one-hot, generated from the codes
//     while loading the tile; lower tiles only, mirrored on store), and
//   - the O(n^3) products of the SPD inverse: the trailing update of a blocked right-looking Cholesky, the
//     block update of the triangular inverse X = L^-1, and C^-1 = X^T X (lower tiles, K range clipped to the
//     non-zero part of the triangular operand, mirrored on store).
// Pseudo-counts need the counts accurate to about 1e-7 relative (the couplings amplify an error in f_ij by the
// condition number of the covariance, ~1e3-1e4), which rules out the bf16/fp32 tensor-core counts of the PLM path.
#include "common.cuh"
#include "internal.h"

#include <math.h>

namespace evc {

namespace {

constexpr int GT = 64;          // GEMM tile edge (M and N)
constexpr int GK = 16;          // K slice
constexpr int GTHREADS = 256;   // 16 x 16 threads, 4 x 4 outputs each
constexpr int NB = 64;          // Cholesky / triangular-inverse block size
constexpr int TS_VEC = 128;     // vectors per CTA of the triangular solve
constexpr int MF_MAX_Q = 21;    // largest alphabet (protein with gap)

// Operand of the tile GEMM: element (r, k) of a dense matrix at base[r * sr + k * sk], or of the one-hot
// alignment matrix: r = site * q + state, k = sequence, value = [codes[k][site] == state] * (w ? w[k] : 1).
struct Operand {
    const double *base;
    int64_t sr, sk;
    const uint8_t *codes;
    const double *w;
    int L, q;
};

__device__ __forceinline__ double load_op(const Operand &o, int64_t r, int64_t k)
{
    if (o.codes) {
        const int site = (int)(r / o.q), state = (int)(r - (int64_t)site * o.q);
        if (o.codes[k * o.L + site] != state) return 0.0;
        return o.w ? o.w[k] : 1.0;
    }
    return o.base[r * o.sr + k * o.sk];
}

struct GemmArgs {
    Operand a, b;
    double *c;
    int64_t ldc;
    int64_t M, N, K;
    double alpha, beta;   // C = beta * C + alpha * A B^T (beta == 0: C is not read)
    int lower;            // compute only tiles with n0 <= m0 (on the tile diagonal: all of it)
    int mirror;           // also store C(n, m) = C(m, n) for n < m
    int tri_k;            // A(r, k) = B(r, k) = 0 for k < r: start K at max(m0, n0)
    const int *info;      // non-zero: a previous factorisation step failed, do nothing
};

__global__ void __launch_bounds__(GTHREADS) mf_gemm_f64_kernel(GemmArgs g)
{
    const int64_t m0 = (int64_t)blockIdx.y * GT, n0 = (int64_t)blockIdx.x * GT;
    if (g.lower && n0 > m0) return;
    if (g.info && *g.info) return;
    __shared__ double As[GK][GT + 1];
    __shared__ double Bs[GK][GT + 1];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    double acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; u++)
#pragma unroll
        for (int v = 0; v < 4; v++) acc[u][v] = 0.0;
    int64_t k0 = 0;
    if (g.tri_k) k0 = (m0 > n0 ? m0 : n0) / GK * GK;
    // loader thread mapping: consecutive threads walk the unit-stride index of the operand
    for (; k0 < g.K; k0 += GK) {
#pragma unroll
        for (int e = tid; e < GK * GT; e += GTHREADS) {
            int kk, rr;
            if (g.a.codes || g.a.sr == 1) { rr = e % GT; kk = e / GT; } else { kk = e % GK; rr = e / GK; }
            const int64_t r = m0 + rr, k = k0 + kk;
            As[kk][rr] = (r < g.M && k < g.K) ? load_op(g.a, r, k) : 0.0;
            if (g.b.codes || g.b.sr == 1) { rr = e % GT; kk = e / GT; } else { kk = e % GK; rr = e / GK; }
            const int64_t rn = n0 + rr, kn = k0 + kk;
            Bs[kk][rr] = (rn < g.N && kn < g.K) ? load_op(g.b, rn, kn) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; kk++) {
            double a[4], b[4];
#pragma unroll
            for (int u = 0; u < 4; u++) a[u] = As[kk][ty + 16 * u];
#pragma unroll
            for (int v = 0; v < 4; v++) b[v] = Bs[kk][tx + 16 * v];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int v = 0; v < 4; v++) acc[u][v] = fma(a[u], b[v], acc[u][v]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const int64_t m = m0 + ty + 16 * u;
        if (m >= g.M) continue;
#pragma unroll
        for (int v = 0; v < 4; v++) {
            const int64_t n = n0 + tx + 16 * v;
            if (n >= g.N) continue;
            if (g.lower && n > m && !g.mirror) continue;
            double val = g.alpha * acc[u][v];
            if (g.beta != 0.0) val += g.beta * g.c[m * g.ldc + n];
            g.c[m * g.ldc + n] = val;
            if (g.mirror && n < m) g.c[n * g.ldc + m] = val;
        }
    }
}

int gemm(const GemmArgs &g, cudaStream_t st)
{
    if (g.M <= 0 || g.N <= 0) return 0;
    dim3 grid((unsigned)ceil_div(g.N, GT), (unsigned)ceil_div(g.M, GT));
    mf_gemm_f64_kernel<<<grid, GTHREADS, 0, st>>>(g);
    EVC_KERNEL_CHECK();
    return 0;
}

Operand dense(const double *p, int64_t sr, int64_t sk) { return Operand{p, sr, sk, nullptr, nullptr, 0, 0}; }

// Unblocked Cholesky of one kb x kb diagonal block (row-major, lda) in shared memory; lower triangle written back.
// A pivot <= 0 (or NaN) stores its 1-based global column in *info and stops.
__global__ void __launch_bounds__(256) mf_potrf_block_kernel(double *A, int64_t lda, int kb, int64_t col0, int *info)
{
    if (*info) return;
    __shared__ double S[NB][NB + 1];
    __shared__ int bad;
    const int tid = threadIdx.x;
    for (int e = tid; e < kb * kb; e += blockDim.x) S[e / kb][e % kb] = A[(int64_t)(e / kb) * lda + e % kb];
    if (tid == 0) bad = 0;
    __syncthreads();
    for (int j = 0; j < kb; j++) {
        const double d = S[j][j];
        if (!(d > 0.0)) {
            if (tid == 0) { bad = 1; *info = (int)(col0 + j + 1); }
            break;                                      // uniform: every thread read the same S[j][j]
        }
        const double r = sqrt(d);
        __syncthreads();
        if (tid == 0) S[j][j] = r;
        for (int i = j + 1 + tid; i < kb; i += blockDim.x) S[i][j] /= r;
        __syncthreads();
        const int m = kb - j - 1;
        for (int e = tid; e < m * m; e += blockDim.x) {
            const int i = j + 1 + e / m, c = j + 1 + e % m;
            if (c <= i) S[i][c] -= S[i][j] * S[c][j];
        }
        __syncthreads();
    }
    __syncthreads();
    if (bad) return;
    for (int e = tid; e < kb * kb; e += blockDim.x) {
        const int i = e / kb, c = e % kb;
        if (c <= i) A[(int64_t)i * lda + c] = S[i][c];
    }
}

// Solve T y = b in place for nvec vectors b (element e of vector v at B[v * vs + e * es]); T is the kb x kb lower
// triangle at Tm (row-major, ldt).  One thread per vector, the vector lives in a shared-memory column.
__global__ void __launch_bounds__(TS_VEC) mf_trsm_lower_kernel(const double *Tm, int64_t ldt, int kb, double *B,
                                                               int64_t vs, int64_t es, int64_t nvec, const int *info)
{
    if (*info) return;
    extern __shared__ double sm[];
    double *T = sm;                       // kb x kb
    double *Y = sm + NB * NB;             // kb x TS_VEC
    const int tid = threadIdx.x;
    const int64_t v0 = (int64_t)blockIdx.x * TS_VEC;
    for (int e = tid; e < kb * kb; e += TS_VEC) T[e] = Tm[(int64_t)(e / kb) * ldt + e % kb];
    for (int e = tid; e < kb * TS_VEC; e += TS_VEC) {
        int vv, ee;
        if (es == 1) { ee = e % kb; vv = e / kb; } else { vv = e % TS_VEC; ee = e / TS_VEC; }
        const int64_t v = v0 + vv;
        Y[ee * TS_VEC + vv] = v < nvec ? B[v * vs + ee * es] : 0.0;
    }
    __syncthreads();
    for (int r = 0; r < kb; r++) {
        double s = Y[r * TS_VEC + tid];
        for (int c = 0; c < r; c++) s -= T[r * kb + c] * Y[c * TS_VEC + tid];
        Y[r * TS_VEC + tid] = s / T[r * kb + r];
    }
    __syncthreads();
    for (int e = tid; e < kb * TS_VEC; e += TS_VEC) {
        int vv, ee;
        if (es == 1) { ee = e % kb; vv = e / kb; } else { vv = e % TS_VEC; ee = e / TS_VEC; }
        const int64_t v = v0 + vv;
        if (v < nvec) B[v * vs + ee * es] = Y[ee * TS_VEC + vv];
    }
}

int trsm(const double *T, int64_t ldt, int kb, double *B, int64_t vs, int64_t es, int64_t nvec, const int *info,
         cudaStream_t st)
{
    if (nvec <= 0) return 0;
    const size_t smem = (size_t)(NB * NB + NB * TS_VEC) * sizeof(double);
    mf_trsm_lower_kernel<<<(unsigned)ceil_div(nvec, TS_VEC), TS_VEC, smem, st>>>(T, ldt, kb, B, vs, es, nvec, info);
    EVC_KERNEL_CHECK();
    return 0;
}

__global__ void mf_identity_kernel(double *X, int64_t n)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n * n) X[e] = (e / n == e % n) ? 1.0 : 0.0;
}

// ---- covariance ---------------------------------------------------------------------------------------------
// F: (L*q)^2 normalised counts (symmetric).  C[(i,a),(j,b)] = rf_ij[a][b] - rf_i[a] rf_j[b], a, b < q-1, with
// rf_ij = (1-pc) f_ij + pc/q^2 off the diagonal blocks and (1-pc) f_i[a] d_ab + (pc/q) d_ab on them.
__global__ void mf_covariance_kernel(const double *F, int L, int q, double pc, double *C)
{
    const int Q = q - 1;
    const int64_t n = (int64_t)L * Q, ldf = (int64_t)L * q;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * n) return;
    const int64_t r = e / n, c = e % n;
    const int i = (int)(r / Q), a = (int)(r % Q), j = (int)(c / Q), b = (int)(c % Q);
    const double fia = F[((int64_t)i * q + a) * ldf + (int64_t)i * q + a];
    const double fjb = F[((int64_t)j * q + b) * ldf + (int64_t)j * q + b];
    const double rfi = (1.0 - pc) * fia + pc / q, rfj = (1.0 - pc) * fjb + pc / q;
    double rfij;
    if (i == j) rfij = a == b ? (1.0 - pc) * fia + pc / q : 0.0;
    else rfij = (1.0 - pc) * F[((int64_t)i * q + a) * ldf + (int64_t)j * q + b] + pc / ((double)q * q);
    C[e] = rfij - rfi * rfj;
}

__global__ void mf_site_freqs_kernel(const double *F, int L, int q, double pc, double *fi, double *rfi)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= L * q) return;
    const int64_t ldf = (int64_t)L * q;
    const double f = F[(int64_t)e * ldf + e];
    if (fi) fi[e] = f;
    if (rfi) rfi[e] = (1.0 - pc) * f + pc / q;
}

// pair p = (i, j), i < j, in row-major order; one CTA per site i
__device__ __forceinline__ int64_t pair_base(int i, int L) { return (int64_t)i * (2 * L - i - 1) / 2; }

__global__ void mf_pair_freqs_kernel(const double *F, int L, int q, double *fij_tri)
{
    const int i = blockIdx.x, qq = q * q;
    const int64_t ldf = (int64_t)L * q, base = pair_base(i, L) * qq;
    const int64_t cnt = (int64_t)(L - 1 - i) * qq;
    for (int64_t e = threadIdx.x; e < cnt; e += blockDim.x) {
        const int j = i + 1 + (int)(e / qq), ab = (int)(e % qq), a = ab / q, b = ab % q;
        fij_tri[base + e] = F[((int64_t)i * q + a) * ldf + (int64_t)j * q + b];
    }
}

// J_ij[a][b] = -Cinv[(i,a),(j,b)] for a, b < q-1, 0 on the last symbol; tri blocks
__global__ void mf_couplings_kernel(const double *Ci, int L, int q, double *J_tri)
{
    const int i = blockIdx.x, qq = q * q, Q = q - 1;
    const int64_t n = (int64_t)L * Q, base = pair_base(i, L) * qq;
    const int64_t cnt = (int64_t)(L - 1 - i) * qq;
    for (int64_t e = threadIdx.x; e < cnt; e += blockDim.x) {
        const int j = i + 1 + (int)(e / qq), ab = (int)(e % qq), a = ab / q, b = ab % q;
        J_tri[base + e] = (a < Q && b < Q) ? -Ci[((int64_t)i * Q + a) * n + (int64_t)j * Q + b] : 0.0;
    }
}

// h_i[a] = log(rf_i[a] / rf_i[q-1]) - sum_{j != i} sum_b J_ij[a][b] rf_j[b]; one CTA per (i, a)
__global__ void __launch_bounds__(256) mf_fields_kernel(const double *Ci, const double *rfi, int L, int q, double *h)
{
    const int i = blockIdx.x / q, a = blockIdx.x % q, Q = q - 1;
    if (a == Q) {
        if (threadIdx.x == 0) h[i * q + a] = 0.0;
        return;
    }
    const int64_t n = (int64_t)L * Q;
    const double *row = Ci + ((int64_t)i * Q + a) * n;
    double s = 0.0;
    for (int64_t c = threadIdx.x; c < n; c += blockDim.x) {
        const int j = (int)(c / Q), b = (int)(c % Q);
        if (j != i) s += row[c] * rfi[j * q + b];      // -J = Cinv
    }
    __shared__ double red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += red[w];
        h[i * q + a] = log(rfi[i * q + a] / rfi[i * q + Q]) + t;
    }
}

// ---- direct information: one warp per pair ------------------------------------------------------------------
constexpr int DI_WARPS = 8;
constexpr int DI_MAX_ITER = 1000000;    // the reference iterates without a cap; this only bounds a runaway pair

__global__ void __launch_bounds__(DI_WARPS * 32) mf_di_kernel(const double *J_tri, const double *rf, int L, int q,
                                                              int64_t npairs, double *di, int *iters)
{
    __shared__ double Es[DI_WARPS][MF_MAX_Q * MF_MAX_Q];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t p = (int64_t)blockIdx.x * DI_WARPS + w;
    if (p >= npairs) return;
    int i = 0;
    int64_t rem = p;
    while (rem >= L - 1 - i) { rem -= L - 1 - i; i++; }
    const int j = i + 1 + (int)rem;
    const int qq = q * q;
    double *E = Es[w];
    for (int e = lane; e < qq; e += 32) E[e] = exp(J_tri[p * qq + e]);
    __syncwarp();
    const bool on = lane < q;
    const double fi = on ? rf[i * q + lane] : 0.0, fj = on ? rf[j * q + lane] : 0.0;
    double hi = on ? 1.0 / q : 0.0, hj = hi;
    double diff = 1.0;
    int it = 0;
    while (diff > 1e-4 && it < DI_MAX_ITER) {
        // t1[a] = sum_b E[a][b] hj[b],  t2[b] = sum_a hi[a] E[a][b]  (both from the previous iterate)
        double t1 = 0.0, t2 = 0.0;
        for (int k = 0; k < q; k++) {
            const double hjk = __shfl_sync(0xffffffffu, hj, k), hik = __shfl_sync(0xffffffffu, hi, k);
            if (on) {
                t1 += E[lane * q + k] * hjk;
                t2 += hik * E[k * q + lane];
            }
        }
        double ni = on ? fi / t1 : 0.0, nj = on ? fj / t2 : 0.0;
        ni /= warp_sum(ni);
        nj /= warp_sum(nj);
        double d = on ? fmax(fabs(ni - hi), fabs(nj - hj)) : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d = fmax(d, __shfl_xor_sync(0xffffffffu, d, o));
        diff = d;
        hi = ni;
        hj = nj;
        it++;
    }
    // P = E * (hi hj^T), normalised; DI = sum P log((P + 1e-100) / (rf_i rf_j^T + 1e-100))
    // gather hi, hj into shared memory so every lane can read any entry
    __shared__ double Hs[DI_WARPS][2][32];
    Hs[w][0][lane] = hi;
    Hs[w][1][lane] = hj;
    __syncwarp();
    double sum = 0.0;
    for (int e = lane; e < qq; e += 32) sum += E[e] * (Hs[w][0][e / q] * Hs[w][1][e % q]);
    sum = warp_sum(sum);
    double acc = 0.0;
    for (int e = lane; e < qq; e += 32) {
        const int a = e / q, b = e % q;
        const double P = E[e] * (Hs[w][0][a] * Hs[w][1][b]) / sum;
        acc += P * log((P + 1e-100) / (rf[i * q + a] * rf[j * q + b] + 1e-100));
    }
    acc = warp_sum(acc);
    if (lane == 0) {
        di[p] = acc;
        if (iters) iters[p] = it;
    }
}

}  // namespace

// ---- entry points (api.cu) ----------------------------------------------------------------------------------
int mf_weighted_counts(const uint8_t *d_codes, const double *d_w, int64_t N, int L, int q, double n_eff, double *d_F,
                       cudaStream_t st)
{
    GemmArgs g{};
    g.a = Operand{nullptr, 0, 0, d_codes, d_w, L, q};
    g.b = Operand{nullptr, 0, 0, d_codes, nullptr, L, q};
    g.c = d_F;
    g.ldc = (int64_t)L * q;
    g.M = g.N = (int64_t)L * q;
    g.K = N;
    g.alpha = 1.0 / n_eff;
    g.beta = 0.0;
    g.lower = 1;
    g.mirror = 1;
    return gemm(g, st);
}

int mf_covariance(const double *d_F, int L, int q, double pc, double *d_C, double *d_fi, double *d_rfi,
                  double *d_fij_tri, cudaStream_t st)
{
    const int64_t n = (int64_t)L * (q - 1);
    if (d_C) {
        mf_covariance_kernel<<<(unsigned)ceil_div(n * n, 256), 256, 0, st>>>(d_F, L, q, pc, d_C);
        EVC_KERNEL_CHECK();
    }
    if (d_fi || d_rfi) {
        mf_site_freqs_kernel<<<(unsigned)ceil_div((int64_t)L * q, 256), 256, 0, st>>>(d_F, L, q, pc, d_fi, d_rfi);
        EVC_KERNEL_CHECK();
    }
    if (d_fij_tri && L > 1) {
        mf_pair_freqs_kernel<<<L - 1, 256, 0, st>>>(d_F, L, q, d_fij_tri);
        EVC_KERNEL_CHECK();
    }
    return 0;
}

int spd_inverse(double *d_A, int64_t n, double *d_X, int *d_info, cudaStream_t st)
{
    const size_t ts_smem = (size_t)(NB * NB + NB * TS_VEC) * sizeof(double);
    EVC_CUDA(cudaFuncSetAttribute(mf_trsm_lower_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ts_smem));
    EVC_CUDA(cudaMemsetAsync(d_info, 0, sizeof(int), st));
    const int64_t lda = n;
    // 1) A = L L^T (lower triangle of d_A overwritten by L)
    for (int64_t k0 = 0; k0 < n; k0 += NB) {
        const int kb = (int)(n - k0 < NB ? n - k0 : NB);
        double *Akk = d_A + k0 * lda + k0;
        mf_potrf_block_kernel<<<1, 256, 0, st>>>(Akk, lda, kb, k0, d_info);
        EVC_KERNEL_CHECK();
        const int64_t r0 = k0 + kb, rest = n - r0;
        if (rest <= 0) break;
        double *P = d_A + r0 * lda + k0;                 // panel rows r0.., columns k0..k0+kb
        if (trsm(Akk, lda, kb, P, lda, 1, rest, d_info, st)) return 1;   // L11 P^T = A21^T
        GemmArgs g{};
        g.a = dense(P, lda, 1);
        g.b = dense(P, lda, 1);
        g.c = d_A + r0 * lda + r0;
        g.ldc = lda;
        g.M = g.N = rest;
        g.K = kb;
        g.alpha = -1.0;
        g.beta = 1.0;
        g.lower = 1;
        g.info = d_info;
        if (gemm(g, st)) return 1;
    }
    // 2) X = L^-1: solve L X = I block row by block row, updating the rows below (right-looking)
    mf_identity_kernel<<<(unsigned)ceil_div(n * n, 256), 256, 0, st>>>(d_X, n);
    EVC_KERNEL_CHECK();
    for (int64_t k0 = 0; k0 < n; k0 += NB) {
        const int kb = (int)(n - k0 < NB ? n - k0 : NB);
        const int64_t ncols = k0 + kb;
        double *Xk = d_X + k0 * n;                       // block row k, columns 0..ncols
        if (trsm(d_A + k0 * lda + k0, lda, kb, Xk, 1, n, ncols, d_info, st)) return 1;
        const int64_t r0 = k0 + kb;
        if (r0 >= n) break;
        GemmArgs g{};
        g.a = dense(d_A + r0 * lda + k0, lda, 1);        // L[r0.., k0..k0+kb]
        g.b = dense(Xk, 1, n);                           // B(c, kk) = X[k0 + kk][c]
        g.c = d_X + r0 * n;
        g.ldc = n;
        g.M = n - r0;
        g.N = ncols;
        g.K = kb;
        g.alpha = -1.0;
        g.beta = 1.0;
        g.info = d_info;
        if (gemm(g, st)) return 1;
    }
    // 3) A^-1 = X^T X (symmetric: lower tiles, mirrored), X[k][m] = 0 for k < m
    GemmArgs g{};
    g.a = dense(d_X, 1, n);
    g.b = dense(d_X, 1, n);
    g.c = d_A;
    g.ldc = lda;
    g.M = g.N = g.K = n;
    g.alpha = 1.0;
    g.beta = 0.0;
    g.lower = 1;
    g.mirror = 1;
    g.tri_k = 1;
    g.info = d_info;
    return gemm(g, st);
}

int mf_couplings_fields(const double *d_Cinv, const double *d_rfi, int L, int q, double *d_J_tri, double *d_h,
                        cudaStream_t st)
{
    if (d_J_tri && L > 1) {
        mf_couplings_kernel<<<L - 1, 256, 0, st>>>(d_Cinv, L, q, d_J_tri);
        EVC_KERNEL_CHECK();
    }
    if (d_h) {
        mf_fields_kernel<<<L * q, 256, 0, st>>>(d_Cinv, d_rfi, L, q, d_h);
        EVC_KERNEL_CHECK();
    }
    return 0;
}

int mf_di_scores(const double *d_J_tri, const double *d_rfi, int L, int q, double *d_di, int *d_iters,
                 cudaStream_t st)
{
    const int64_t npairs = (int64_t)L * (L - 1) / 2;
    if (npairs == 0) return 0;
    mf_di_kernel<<<(unsigned)ceil_div(npairs, DI_WARPS), DI_WARPS * 32, 0, st>>>(d_J_tri, d_rfi, L, q, npairs, d_di,
                                                                               d_iters);
    EVC_KERNEL_CHECK();
    return 0;
}

}  // namespace evc
