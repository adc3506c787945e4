// Closed-form variance-based sensitivity of the emulator's mean (gladsgp_b200.sensitivity.gp_sensitivity_indices).
//
// A function f(x) = sum_n a_n prod_k exp(-beta_nk (x_k - z_nk)^2) of independent uniform inputs on [0,1]^q has every Sobol'
// integral in closed form:
//   I1(b, z)         = int_0^1 e^{-b(x-z)^2} dx            = 1/2 sqrt(pi/b) [erf(sqrt(b)(1-z)) + erf(sqrt(b) z)]
//   I2(b, z; b', z') = int_0^1 e^{-b(x-z)^2-b'(x-z')^2} dx = exp(-b b'(z-z')^2/B) 1/2 sqrt(pi/B) [erf(sqrt(B)(1-c)) + erf(sqrt(B) c)]
//                      with B = b + b', c = (b z + b' z') / B;  both are exactly 1 at beta = 0
//   M(u) = sum_{n,n'} a_n a_n' prod_{k in u} I2_k(n,n') prod_{k not in u} I1_k(n) I1_k(n'),   E0 = sum_n a_n prod_k I1_k(n).
// gp_pair_kernel forms M({k}), M(all\k) and M(all) for every input k in one pass over the pairs n <= n' (a pair n < n'
// counts twice).  Products over all inputs but one come from prefix / suffix products, never from a division (an I1 can
// underflow).  The per-term factors I1_k(n), prod_{r != k} I1_r(n) and prod_k I1_k(n) are tabulated first
// (gp_table_kernel).  Everything is libdevice erf / exp / sqrt in FP64 (no fast-math, -fmad=false for the whole library);
// every sum runs in a fixed order, so two identical calls give identical bits.
//
// Functions and terms.  Blocks b = s * pu + j (posterior sample s, PC j) carry beta[b][q] and the weights a[b][m] of the
// m training rows Z[m][q].  mode 0: one function per block, terms n = i.  mode 1: one function per PC j, terms
// n = (s, i) over all samples (the caller scales the weights, e.g. by 1 / S for the posterior-mean function).
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int GS_TILE = 32;          // terms per tile side: a lane per column term
constexpr int GS_NT = 128;           // threads of the pair kernel: 4 warps x 8 row terms each
constexpr int GS_RNT = 256;          // threads of the term-sum kernels
constexpr long long GS_CTAS = 8192;  // pair-kernel CTAs aimed for: slices per function = ceil(GS_CTAS / functions)
constexpr double GS_PI = 3.14159265358979323846;

__device__ __forceinline__ double gs_i1(double b, double z)
{
    if (b == 0.0) return 1.0;
    const double sb = sqrt(b);
    return 0.5 * sqrt(GS_PI / b) * (erf(sb * (1.0 - z)) + erf(sb * z));
}

__device__ __forceinline__ double gs_i2(double b, double z, double b2, double z2)
{
    const double B = b + b2;
    if (B == 0.0) return 1.0;
    const double c = (b * z + b2 * z2) / B;
    const double sB = sqrt(B);
    const double d = z - z2;
    return exp(-b * b2 * d * d / B) * 0.5 * sqrt(GS_PI / B) * (erf(sB * (1.0 - c)) + erf(sB * c));
}

// I2 of two terms with the same beta (mode 0): B = 2b, c = (z + z') / 2, exp(-b (z-z')^2 / 2); sB = sqrt(2b),
// h = 1/2 sqrt(pi / 2b) precomputed per input
__device__ __forceinline__ double gs_i2_same(double b, double sB, double h, double z, double z2)
{
    const double c = 0.5 * (z + z2);
    const double d = z - z2;
    return exp(-0.5 * b * d * d) * h * (erf(sB * (1.0 - c)) + erf(sB * c));
}

__device__ __forceinline__ void gs_term(int mode, int f, long long n, int m, int pu, int& b, int& i)
{
    if (mode == 0) { b = f; i = (int)n; }
    else { const int s = (int)(n / m); i = (int)(n - (long long)s * m); b = s * pu + f; }
}

// per (block b, row i): I1[b][i][k], the exclusive products E[b][i][k] = prod_{r != k} I1_r and P[b][i] = prod_k I1_k
__global__ void gp_table_kernel(const double* __restrict__ Z, int m, int q, const double* __restrict__ beta, int nblk,
                                double* __restrict__ I1t, double* __restrict__ Et, double* __restrict__ Pt)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)nblk * m) return;
    const int b = (int)(t / m), i = (int)(t - (long long)b * m);
    double* __restrict__ I = I1t + t * q;
    double* __restrict__ E = Et + t * q;
    double pre = 1.0;
    for (int k = 0; k < q; ++k) {
        const double v = gs_i1(beta[(size_t)b * q + k], Z[(size_t)i * q + k]);
        I[k] = v;
        E[k] = pre;
        pre *= v;
    }
    Pt[t] = pre;
    double suf = 1.0;
    for (int k = q - 1; k >= 0; --k) {
        E[k] *= suf;
        suf *= I[k];
    }
}

// Shared tile of GS_TILE terms: [k][term] arrays (a lane reads consecutive words), beta only where it varies per term
template <int QP, bool SAME>
struct GsTile {
    double z[QP][GS_TILE], i1[QP][GS_TILE], ex[QP][GS_TILE], b[SAME ? 1 : QP][GS_TILE], a[GS_TILE];
};

template <int QP, bool SAME>
__device__ __forceinline__ void gs_load_tile(GsTile<QP, SAME>& T, long long n0, long long N, int mode, int f, int m,
                                             int q, int pu, const double* __restrict__ Z, const double* __restrict__ beta,
                                             const double* __restrict__ a, const double* __restrict__ I1t,
                                             const double* __restrict__ Et)
{
    for (int e = threadIdx.x; e < GS_TILE * QP; e += GS_NT) {
        const int t = e % GS_TILE, k = e / GS_TILE;
        const long long n = n0 + t;
        double z = 0.0, i1 = 1.0, ex = 1.0, bb = 0.0;
        if (n < N && k < q) {
            int b, i;
            gs_term(mode, f, n, m, pu, b, i);
            const size_t r = ((size_t)b * m + i) * q + k;
            z = Z[(size_t)i * q + k];
            i1 = I1t[r];
            ex = Et[r];
            bb = beta[(size_t)b * q + k];
        }
        T.z[k][t] = z; T.i1[k][t] = i1; T.ex[k][t] = ex;
        if (!SAME) T.b[k][t] = bb;
        if (k == 0) {
            double av = 0.0;
            if (n < N) {
                int b, i;
                gs_term(mode, f, n, m, pu, b, i);
                av = a[(size_t)b * m + i];
            }
            T.a[t] = av;
        }
    }
}

// One CTA = (function f, slice p): the upper-triangle tile pairs tp = p, p + P, p + 2P, ... of the function, in that order.
// Thread (warp w, lane c) takes column term c and row terms w + 4u of each tile; its 2q + 1 sums stay in registers, then
// a fixed warp tree and a fixed sum over the 4 warps give the slice's partial [f][p][2q+1].
template <int QP, bool SAME>
__global__ void __launch_bounds__(GS_NT)
gp_pair_kernel(const double* __restrict__ Z, int m, int q, const double* __restrict__ beta, const double* __restrict__ a,
               int pu, int mode, long long N, int P, const double* __restrict__ I1t, const double* __restrict__ Et,
               double* __restrict__ partial)
{
    extern __shared__ __align__(16) unsigned char gs_smem[];
    GsTile<QP, SAME>& R = *reinterpret_cast<GsTile<QP, SAME>*>(gs_smem);
    GsTile<QP, SAME>& Cm = *reinterpret_cast<GsTile<QP, SAME>*>(gs_smem + sizeof(GsTile<QP, SAME>));
    __shared__ double sb[QP], ssB[QP], sh[QP];
    __shared__ double red[GS_NT / 32][2 * QP + 1];
    const int f = (int)(blockIdx.x / P), p = (int)(blockIdx.x - (long long)f * P);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (SAME && threadIdx.x < QP) {
        const int k = threadIdx.x;
        const double bk = (k < q) ? beta[(size_t)f * q + k] : 0.0;
        sb[k] = bk;
        ssB[k] = sqrt(2.0 * bk);
        sh[k] = (bk == 0.0) ? 0.0 : 0.5 * sqrt(GS_PI / (2.0 * bk));
    }
    double M1[QP], Mt[QP], Mall = 0.0;
#pragma unroll
    for (int k = 0; k < QP; ++k) { M1[k] = 0.0; Mt[k] = 0.0; }

    const long long nt = (N + GS_TILE - 1) / GS_TILE;
    const long long ntp = nt * (nt + 1) / 2;
    for (long long tp = p; tp < ntp; tp += P) {
        // row ti of the upper triangle starts at st(ti) = ti nt - ti (ti - 1) / 2
        long long ti = (long long)((2.0 * nt + 1.0 - sqrt((2.0 * nt + 1.0) * (2.0 * nt + 1.0) - 8.0 * (double)tp)) * 0.5);
        if (ti < 0) ti = 0;
        if (ti > nt - 1) ti = nt - 1;
        while (ti > 0 && ti * nt - ti * (ti - 1) / 2 > tp) --ti;
        while (ti + 1 < nt && (ti + 1) * nt - (ti + 1) * ti / 2 <= tp) ++ti;
        const long long tj = ti + (tp - (ti * nt - ti * (ti - 1) / 2));
        __syncthreads();                                 // previous tiles consumed (and sb / ssB / sh written)
        gs_load_tile<QP, SAME>(R, ti * GS_TILE, N, mode, f, m, q, pu, Z, beta, a, I1t, Et);
        gs_load_tile<QP, SAME>(Cm, tj * GS_TILE, N, mode, f, m, q, pu, Z, beta, a, I1t, Et);
        __syncthreads();
        const bool diag = (ti == tj);
        const long long cn = tj * GS_TILE + lane;
        if (cn >= N) continue;
#pragma unroll 1
        for (int u = 0; u < GS_TILE / (GS_NT / 32); ++u) {
            const int r = warp + (GS_NT / 32) * u;
            if (ti * GS_TILE + r >= N || (diag && lane < r)) continue;
            const double wgt = R.a[r] * Cm.a[lane] * ((diag && lane == r) ? 1.0 : 2.0);
            double Bv[QP], suf[QP];
#pragma unroll
            for (int k = 0; k < QP; ++k) {
                double v = 1.0;
                if (k < q) {
                    if (SAME) {
                        if (sb[k] != 0.0) v = gs_i2_same(sb[k], ssB[k], sh[k], R.z[k][r], Cm.z[k][lane]);
                    } else {
                        v = gs_i2(R.b[SAME ? 0 : k][r], R.z[k][r], Cm.b[SAME ? 0 : k][lane], Cm.z[k][lane]);
                    }
                }
                Bv[k] = v;
            }
            suf[QP - 1] = 1.0;
#pragma unroll
            for (int k = QP - 2; k >= 0; --k) suf[k] = suf[k + 1] * Bv[k + 1];
            double pre = 1.0;
#pragma unroll
            for (int k = 0; k < QP; ++k) {
                if (k < q) {
                    M1[k] += wgt * (R.ex[k][r] * Cm.ex[k][lane]) * Bv[k];
                    Mt[k] += wgt * (pre * suf[k]) * (R.i1[k][r] * Cm.i1[k][lane]);
                }
                pre *= Bv[k];
            }
            Mall += wgt * pre;
        }
    }
#pragma unroll
    for (int k = 0; k < QP; ++k) {
        const double s1 = warp_sum(M1[k]), st = warp_sum(Mt[k]);
        if (lane == 0) { red[warp][k] = s1; red[warp][QP + k] = st; }
    }
    const double sa = warp_sum(Mall);
    if (lane == 0) red[warp][2 * QP] = sa;
    __syncthreads();
    const int nout = 2 * q + 1;
    if (threadIdx.x < nout) {
        const int j = threadIdx.x;
        const int src = (j < q) ? j : (j < 2 * q) ? QP + (j - q) : 2 * QP;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < GS_NT / 32; ++w) s += red[w][src];
        partial[((size_t)f * P + p) * nout + j] = s;
    }
}

// fixed-order sum of the slices: M[f][j] = sum_p partial[f][p][j]
__global__ void gp_reduce_kernel(const double* __restrict__ partial, int F, int P, int nout, double* __restrict__ M)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)F * nout) return;
    const int f = (int)(t / nout), j = (int)(t - (long long)f * nout);
    double s = 0.0;
    for (int p = 0; p < P; ++p) s += partial[((size_t)f * P + p) * nout + j];
    M[t] = s;
}

// fixed tree over a CTA of GS_RNT threads; the result is valid in thread 0
__device__ __forceinline__ double gs_block_sum(double v, double* sred)
{
    v = warp_sum(v);
    __syncthreads();                                      // sred free from the previous use
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < GS_RNT / 32; ++w) s += sred[w];
    return s;
}

// E0[f] = sum_n a_n P_n, one CTA per function, terms strided over the threads
__global__ void __launch_bounds__(GS_RNT)
gp_mean_kernel(const double* __restrict__ a, int m, int pu, int mode, long long N, const double* __restrict__ Pt,
               double* __restrict__ E0)
{
    __shared__ double sred[GS_RNT / 32];
    const int f = blockIdx.x;
    double s = 0.0;
    for (long long n = threadIdx.x; n < N; n += GS_RNT) {
        int b, i;
        gs_term(mode, f, n, m, pu, b, i);
        const size_t r = (size_t)b * m + i;
        s += a[r] * Pt[r];
    }
    s = gs_block_sum(s, sred);
    if (threadIdx.x == 0) E0[f] = s;
}

// main-effect curves: out[f][k][g] = sum_n a_n exp(-beta_nk (grid_g - z_nk)^2) prod_{r != k} I1_r(n); one CTA per (f, k)
__global__ void __launch_bounds__(GS_RNT)
gp_main_effects_kernel(const double* __restrict__ Z, int m, int q, const double* __restrict__ beta,
                       const double* __restrict__ a, int pu, int mode, long long N, const double* __restrict__ Et,
                       const double* __restrict__ grid, int ngrid, double* __restrict__ out)
{
    __shared__ double sred[GS_RNT / 32];
    const int f = blockIdx.x / q, k = blockIdx.x - f * q;
    for (int g = 0; g < ngrid; ++g) {
        const double x = grid[g];
        double s = 0.0;
        for (long long n = threadIdx.x; n < N; n += GS_RNT) {
            int b, i;
            gs_term(mode, f, n, m, pu, b, i);
            const size_t r = (size_t)b * m + i;
            const double d = x - Z[(size_t)i * q + k];
            s += a[r] * Et[r * q + k] * exp(-beta[(size_t)b * q + k] * d * d);
        }
        s = gs_block_sum(s, sred);
        if (threadIdx.x == 0) out[((size_t)f * q + k) * ngrid + g] = s;
    }
}

struct GsShape {
    int F;            // functions
    long long N;      // terms per function
    int P;            // slices per function
    long long table;  // doubles of the I1 and E tables (each) -- B m q
};

static GsShape gs_shape(int m, int q, int S, int pu, int mode)
{
    GsShape s;
    s.F = mode == 0 ? S * pu : pu;
    s.N = mode == 0 ? (long long)m : (long long)S * m;
    const long long nt = (s.N + GS_TILE - 1) / GS_TILE;
    const long long ntp = nt * (nt + 1) / 2;
    long long P = (GS_CTAS + s.F - 1) / s.F;
    if (P > ntp) P = ntp;
    if (P < 1) P = 1;
    s.P = (int)P;
    s.table = (long long)S * pu * m * q;
    return s;
}

static long long gs_workspace(const GsShape& s, int q, int S, int pu, int m)
{
    return 8LL * (2 * s.table + (long long)S * pu * m + (long long)s.F * s.P * (2 * q + 1));
}

static const char* gs_check(int m, int q, int S, int pu, int mode)
{
    if (m <= 0 || S <= 0 || pu <= 0) return "m, S, pu must be positive";
    if (q < 1 || q > 32) return "q must be in [1, 32]";
    if (mode != 0 && mode != 1) return "mode must be 0 (per block) or 1 (sum over samples)";
    if ((long long)S * pu >= (1LL << 31) || (long long)S * m >= (1LL << 31)) return "S * pu and S * m must be below 2^31";
    return nullptr;
}

static int gs_tables(const double* Z, int m, int q, const double* beta, int nblk, double* ws, cudaStream_t st)
{
    const long long rows = (long long)nblk * m;
    const long long tab = rows * q;
    gp_table_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(Z, m, q, beta, nblk, ws, ws + tab, ws + 2 * tab);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

template <int QP, bool SAME>
static int gs_launch_pairs(const double* Z, int m, int q, const double* beta, const double* a, int pu, int mode,
                           const GsShape& s, const double* I1t, const double* Et, double* partial, cudaStream_t st)
{
    const size_t smem = 2 * sizeof(GsTile<QP, SAME>);
    GGP_CUDA(cudaFuncSetAttribute(gp_pair_kernel<QP, SAME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gp_pair_kernel<QP, SAME><<<(unsigned)((long long)s.F * s.P), GS_NT, smem, st>>>(Z, m, q, beta, a, pu, mode, s.N, s.P,
                                                                                   I1t, Et, partial);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

template <bool SAME>
static int gs_dispatch(int QP, const double* Z, int m, int q, const double* beta, const double* a, int pu, int mode,
                       const GsShape& s, const double* I1t, const double* Et, double* partial, cudaStream_t st)
{
    switch (QP) {
        case 4: return gs_launch_pairs<4, SAME>(Z, m, q, beta, a, pu, mode, s, I1t, Et, partial, st);
        case 8: return gs_launch_pairs<8, SAME>(Z, m, q, beta, a, pu, mode, s, I1t, Et, partial, st);
        case 16: return gs_launch_pairs<16, SAME>(Z, m, q, beta, a, pu, mode, s, I1t, Et, partial, st);
        default: return gs_launch_pairs<32, SAME>(Z, m, q, beta, a, pu, mode, s, I1t, Et, partial, st);
    }
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_gp_sens_workspace_bytes(int m, int q, int S, int pu, int mode)
{
    if (gs_check(m, q, S, pu, mode)) return -1;
    return gs_workspace(gs_shape(m, q, S, pu, mode), q, S, pu, m);
}

int ggp_gp_sens_f64(const double* Z, int m, int q, const double* beta, const double* a, int S, int pu, int mode,
                    double* M_out, double* E0_out, void* workspace, long long workspace_bytes, void* stream)
{
    GGP_ARG(Z && beta && a && M_out && E0_out && workspace, "null pointer");
    const char* bad = gs_check(m, q, S, pu, mode);
    GGP_ARG(!bad, bad);
    const GsShape s = gs_shape(m, q, S, pu, mode);
    GGP_ARG((long long)s.F * s.P < (1LL << 31), "too many functions");
    const long long need = gs_workspace(s, q, S, pu, m);
    if (workspace_bytes < need) {
        set_error("ggp_gp_sens_f64: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* ws = reinterpret_cast<double*>(workspace);
    const int nblk = S * pu;
    int rc = gs_tables(Z, m, q, beta, nblk, ws, st);
    if (rc != GGP_OK) return rc;
    const double* I1t = ws;
    const double* Et = ws + s.table;
    const double* Pt = ws + 2 * s.table;
    double* partial = ws + 2 * s.table + (long long)nblk * m;
    const int QP = q <= 4 ? 4 : q <= 8 ? 8 : q <= 16 ? 16 : 32;
    rc = mode == 0 ? gs_dispatch<true>(QP, Z, m, q, beta, a, pu, mode, s, I1t, Et, partial, st)
                   : gs_dispatch<false>(QP, Z, m, q, beta, a, pu, mode, s, I1t, Et, partial, st);
    if (rc != GGP_OK) return rc;
    const long long nred = (long long)s.F * (2 * q + 1);
    gp_reduce_kernel<<<(unsigned)((nred + 255) / 256), 256, 0, st>>>(partial, s.F, s.P, 2 * q + 1, M_out);
    GGP_CUDA(cudaGetLastError());
    gp_mean_kernel<<<s.F, GS_RNT, 0, st>>>(a, m, pu, mode, s.N, Pt, E0_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_main_effects_f64(const double* Z, int m, int q, const double* beta, const double* a, int S, int pu, int mode,
                         const double* grid, int ngrid, double* out, void* workspace, long long workspace_bytes,
                         void* stream)
{
    GGP_ARG(Z && beta && a && grid && out && workspace, "null pointer");
    const char* bad = gs_check(m, q, S, pu, mode);
    GGP_ARG(!bad, bad);
    GGP_ARG(ngrid > 0, "ngrid must be positive");
    const GsShape s = gs_shape(m, q, S, pu, mode);
    GGP_ARG((long long)s.F * q < (1LL << 31), "too many functions");
    const long long need = gs_workspace(s, q, S, pu, m);
    if (workspace_bytes < need) {
        set_error("ggp_main_effects_f64: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* ws = reinterpret_cast<double*>(workspace);
    const int rc = gs_tables(Z, m, q, beta, S * pu, ws, st);
    if (rc != GGP_OK) return rc;
    gp_main_effects_kernel<<<(unsigned)((long long)s.F * q), GS_RNT, 0, st>>>(Z, m, q, beta, a, pu, mode, s.N,
                                                                             ws + s.table, grid, ngrid, out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
