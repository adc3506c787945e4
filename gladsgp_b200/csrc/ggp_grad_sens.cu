// Closed-form gradient outer-product matrix of the emulator's mean (gladsgp_b200.sensitivity.gp_active_subspace).
//
// For f(x) = sum_n a_n phi_n(x), phi_n(x) = prod_k exp(-b_nk (x_k - z_nk)^2), with independent inputs uniform on [0,1]^q,
//   C = E[grad f grad f^T] = sum_{n,n'} a_n a_n' Omega_{j(n) j(n')} int grad phi_n grad phi_n'^T dx.
// Its eigenvectors span the active subspace; its diagonal is the derivative-based sensitivity nu_k = E[(d_k f)^2].
// Per input, with B = b + b', c = (b z + b' z') / B, e = exp(-b b' (z - z')^2 / B):
//   It = int_0^1 e^{-B(x-c)^2} dx = 1/2 sqrt(pi/B) [erf(sqrt(B)(1-c)) + erf(sqrt(B) c)],  E0 = e^{-B c^2}, E1 = e^{-B(1-c)^2}
//   m1 = (E0 - E1) / 2B,  m2 = It / 2B - ((1-c) E1 + c E0) / 2B
//   I2 = e It,  G(n,n') = int d phi_n phi_n' = -2 b e (m1 + (c-z) It),  H = int d phi_n d phi_n' = 4 b b' e (m2 + m1 (2c-z-z') + (c-z)(c-z') It)
// Every integral of a pair carries the factor e of its input, so a pair's entries all carry eps J with
// eps = exp(-sum_r b_r b'_r d_r^2 / B_r) and J = prod_r It_r: one exp per pair, no products over all inputs but one.
// With u_r = G_r(n,n') / (e_r It_r), v_r = G_r(n',n) / (e_r It_r), h_r = H_r / (e_r It_r) and W = a a' Omega eps J
// (doubled for n != n'), the pair adds W/2 (u v^T + v u^T) off the diagonal and W h on it.  E0 - E1 is formed as the
// larger exponential times expm1 of the exponent difference (no cancellation at small B, no overflow at large B).
// An input with b = 0 on both sides has u = v = h = 0 exactly; on one side, that side's u (or v) and h are 0.
//
// gg_pair_kernel walks the upper-triangle 32x32 tile pairs of one function in a fixed slice per CTA (gp_pair_kernel's
// scheme).  Each lane forms u, v, h and W of one pair at a time and stages them in its warp's shared rows; the warp then
// adds X += sum_p (W_p u_p) v_p^T on the FP64 tensor cores (DMMA m8n8k4, the accumulator in fragments, (QP/8)^2 of them)
// and the diagonal D += sum_p W_p h_p as a fixed-order column sum.  The four warps' X and D are added in a fixed order
// into the slice's partial; gg_reduce_kernel sums the slices in order and writes C_kl = (X_kl + X_lk)/2, C_kk = D_k, so C
// is exactly symmetric and two identical calls give identical bits.  FP64 libdevice erf / exp / expm1 / sqrt, no fast-math.
//
// Functions and terms (blocks b = s * pu + j carry beta[b][q] and a[b][m]; training rows Z[m][q]):
//   mode 0: one function per block, terms n = i, Omega = 1 (same beta on both sides of every pair);
//   mode 1: one per PC j, terms n = (s, i), Omega = 1;   mode 2: one per sample s, terms n = (j, i), Omega = omega[pu][pu];
//   mode 3: one function, terms n = (s, j, i), Omega = omega.
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int GG_TILE = 32;          // terms per tile side: a lane per column term
constexpr int GG_NT = 128;           // threads of the pair kernel: 4 warps x 8 row terms each
constexpr long long GG_CTAS = 8192;  // pair-kernel CTAs aimed for: slices per function = ceil(GG_CTAS / functions)
constexpr double GG_PI = 3.14159265358979323846;

__device__ __forceinline__ void gg_term(int mode, int f, long long n, int m, int pu, int& b, int& i)
{
    if (mode == 0) { b = f; i = (int)n; return; }
    const long long r = n / m;                           // mode 1: s; mode 2: j; mode 3: s * pu + j
    i = (int)(n - r * m);
    b = mode == 1 ? (int)r * pu + f : mode == 2 ? f * pu + (int)r : (int)r;
}

template <int QP>
struct GgTile {
    double z[QP][GG_TILE], b[QP][GG_TILE], a[GG_TILE];
    int pc[GG_TILE];
};

template <int QP>
__device__ __forceinline__ void gg_load_tile(GgTile<QP>& T, long long n0, long long N, int mode, int f, int m, int q,
                                             int pu, const double* __restrict__ Z, const double* __restrict__ beta,
                                             const double* __restrict__ a)
{
    for (int e = threadIdx.x; e < GG_TILE * QP; e += GG_NT) {
        const int t = e % GG_TILE, k = e / GG_TILE;
        const long long n = n0 + t;
        int b = 0, i = 0;
        if (n < N) gg_term(mode, f, n, m, pu, b, i);
        const bool ok = n < N && k < q;
        T.z[k][t] = ok ? Z[(size_t)i * q + k] : 0.0;
        T.b[k][t] = ok ? beta[(size_t)b * q + k] : 0.0;
        if (k == 0) {
            T.a[t] = n < N ? a[(size_t)b * m + i] : 0.0;
            T.pc[t] = b % pu;
        }
    }
}

// per-warp staging of 32 pairs: rows [pair][k] of u, v, h (stride QP + 1 against bank conflicts) and W
template <int QP>
struct GgStage {
    double u[GG_TILE][QP + 1], v[GG_TILE][QP + 1], h[GG_TILE][QP + 1], w[GG_TILE];
};

// u, v, h of input k for one pair; returns It (1 at B = 0) and adds b b' d^2 / B to lnE
template <bool SAME>
__device__ __forceinline__ double gg_input(double b, double b2, double z, double z2, double sB, double hB, double i2B,
                                           double& lnE, double& u, double& v, double& h)
{
    u = 0.0; v = 0.0; h = 0.0;
    const double B = b + b2;
    if (B == 0.0) return 1.0;
    const double d = z - z2;
    double c;
    if (SAME) {
        c = 0.5 * (z + z2);
        lnE += 0.5 * b * d * d;
    } else {
        const double iB = 1.0 / B;
        c = (b * z + b2 * z2) * iB;
        sB = sqrt(B);
        hB = 0.5 * sqrt(GG_PI * iB);
        i2B = 0.5 * iB;
        lnE += b * b2 * d * d * iB;
    }
    const double It = hB * (erf(sB * (1.0 - c)) + erf(sB * c));
    const double t = B * (1.0 - 2.0 * c);                // B (1-c)^2 - B c^2
    const bool lo = t >= 0.0;                            // c <= 1/2: E0 is the larger exponential
    const double Ebig = exp(-B * (lo ? c * c : (1.0 - c) * (1.0 - c)));
    const double em = expm1(-fabs(t));
    const double Esmall = Ebig + Ebig * em;
    const double E0 = lo ? Ebig : Esmall, E1 = lo ? Esmall : Ebig;
    const double m1 = (lo ? -Ebig : Ebig) * em * i2B;
    const double m2 = (It - (1.0 - c) * E1 - c * E0) * i2B;
    const double rI = It > 0.0 ? 1.0 / It : 0.0;         // It = 0 only for c far outside [0,1]: then J = 0 and W = 0
    const double cz = c - z, cz2 = c - z2, r1 = m1 * rI;
    u = -2.0 * b * (r1 + cz);
    v = -2.0 * b2 * (r1 + cz2);
    h = 4.0 * b * b2 * ((m2 + m1 * (2.0 * c - z - z2)) * rI + cz * cz2);
    return It;
}

// One CTA = (function f, slice p): the upper-triangle tile pairs tp = p, p + P, ... of the function, in that order.
// Thread (warp w, lane c) takes column term c and row terms w + 4s of each tile.  partial[f][p][k][l] holds X_kl
// (k != l) and D_k (k == l) of the slice.
template <int QP, bool SAME>
__global__ void __launch_bounds__(GG_NT)
gg_pair_kernel(const double* __restrict__ Z, int m, int q, const double* __restrict__ beta, const double* __restrict__ a,
               int pu, int mode, const double* __restrict__ omega, long long N, int P, double* __restrict__ partial)
{
    constexpr int NB = QP < 8 ? 1 : QP / 8;              // 8x8 fragments per side
    extern __shared__ __align__(16) unsigned char gg_smem[];
    GgTile<QP>& R = *reinterpret_cast<GgTile<QP>*>(gg_smem);
    GgTile<QP>& Cm = *reinterpret_cast<GgTile<QP>*>(gg_smem + sizeof(GgTile<QP>));
    GgStage<QP>* stages = reinterpret_cast<GgStage<QP>*>(gg_smem + 2 * sizeof(GgTile<QP>));
    __shared__ double sb[QP], ssB[QP], sh[QP], si2B[QP];
    const int f = (int)(blockIdx.x / P), p = (int)(blockIdx.x - (long long)f * P);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    GgStage<QP>& st = stages[warp];
    if (SAME && threadIdx.x < QP) {
        const int k = threadIdx.x;
        const double bk = (k < q) ? beta[(size_t)f * q + k] : 0.0;
        sb[k] = bk;
        ssB[k] = sqrt(2.0 * bk);
        sh[k] = (bk == 0.0) ? 0.0 : 0.5 * sqrt(GG_PI / (2.0 * bk));
        si2B[k] = (bk == 0.0) ? 0.0 : 0.25 / bk;
    }
    double acc[NB][NB][2];
#pragma unroll
    for (int i = 0; i < NB; ++i)
#pragma unroll
        for (int j = 0; j < NB; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
    double dsum = 0.0;                                   // D of input k = lane

    const long long nt = (N + GG_TILE - 1) / GG_TILE;
    const long long ntp = nt * (nt + 1) / 2;
    for (long long tp = p; tp < ntp; tp += P) {
        // row ti of the upper triangle starts at st(ti) = ti nt - ti (ti - 1) / 2
        long long ti = (long long)((2.0 * nt + 1.0 - sqrt((2.0 * nt + 1.0) * (2.0 * nt + 1.0) - 8.0 * (double)tp)) * 0.5);
        if (ti < 0) ti = 0;
        if (ti > nt - 1) ti = nt - 1;
        while (ti > 0 && ti * nt - ti * (ti - 1) / 2 > tp) --ti;
        while (ti + 1 < nt && (ti + 1) * nt - (ti + 1) * ti / 2 <= tp) ++ti;
        const long long tj = ti + (tp - (ti * nt - ti * (ti - 1) / 2));
        __syncthreads();                                 // previous tiles consumed (and sb / ssB / sh / si2B written)
        gg_load_tile<QP>(R, ti * GG_TILE, N, mode, f, m, q, pu, Z, beta, a);
        gg_load_tile<QP>(Cm, tj * GG_TILE, N, mode, f, m, q, pu, Z, beta, a);
        __syncthreads();
        const bool diag = (ti == tj);
        const bool cok = tj * GG_TILE + lane < N;
#pragma unroll 1
        for (int s = 0; s < GG_TILE / (GG_NT / 32); ++s) {
            const int r = warp + (GG_NT / 32) * s;
            const bool ok = cok && ti * GG_TILE + r < N && !(diag && lane < r);
            double lnE = 0.0, J = 1.0;
#pragma unroll
            for (int k = 0; k < QP; ++k) {
                double uk = 0.0, vk = 0.0, hk = 0.0;
                if (ok && k < q) {
                    if (SAME) {
                        if (sb[k] != 0.0)
                            J *= gg_input<true>(sb[k], sb[k], R.z[k][r], Cm.z[k][lane], ssB[k], sh[k], si2B[k], lnE,
                                                uk, vk, hk);
                    } else {
                        J *= gg_input<false>(R.b[k][r], Cm.b[k][lane], R.z[k][r], Cm.z[k][lane], 0.0, 0.0, 0.0, lnE,
                                             uk, vk, hk);
                    }
                }
                st.u[lane][k] = uk; st.v[lane][k] = vk; st.h[lane][k] = hk;
            }
            double W = 0.0;
            if (ok) {
                const double om = mode >= 2 ? __ldg(omega + (size_t)R.pc[r] * pu + Cm.pc[lane]) : 1.0;
                W = R.a[r] * Cm.a[lane] * om * ((diag && lane == r) ? 1.0 : 2.0) * exp(-lnE) * J;
            }
            st.w[lane] = W;
            __syncwarp();
            // X += sum_p (W_p u_p) v_p^T: A[row k][col p] = W_p u_p[k], B[row p][col l] = v_p[l]
#pragma unroll
            for (int k4 = 0; k4 < GG_TILE; k4 += 4) {
                const int pp = k4 + t4;
                const double wp = st.w[pp];
                double af[NB], bf[NB];
#pragma unroll
                for (int i = 0; i < NB; ++i) {
                    const int k = 8 * i + g;
                    af[i] = k < QP ? wp * st.u[pp][k] : 0.0;
                    bf[i] = k < QP ? st.v[pp][k] : 0.0;
                }
#pragma unroll
                for (int i = 0; i < NB; ++i)
#pragma unroll
                    for (int j = 0; j < NB; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
            }
            if (lane < QP) {
#pragma unroll 4
                for (int pp = 0; pp < GG_TILE; ++pp) dsum += st.w[pp] * st.h[pp][lane];
            }
            __syncwarp();                                // stage consumed before the next pairs overwrite it
        }
    }
    // fixed-order sum of the four warps' X and D into the slice's partial (the stages are free now)
    __syncthreads();
    constexpr int QQ = (QP < 8 ? 8 : QP);
    double* red = reinterpret_cast<double*>(gg_smem + 2 * sizeof(GgTile<QP>));     // [warp][QQ][QQ]
    double* mine = red + (size_t)warp * QQ * QQ;
#pragma unroll
    for (int i = 0; i < NB; ++i)
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            const int row = 8 * i + g, col = 8 * j + 2 * t4;
            mine[row * QQ + col] = acc[i][j][0];
            mine[row * QQ + col + 1] = acc[i][j][1];
        }
    __syncwarp();
    if (lane < QP) mine[lane * QQ + lane] = dsum;
    __syncthreads();
    double* out = partial + ((size_t)f * P + p) * q * q;
    for (int e = threadIdx.x; e < q * q; e += GG_NT) {
        const int k = e / q, l = e - k * q;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < GG_NT / 32; ++w) s += red[(size_t)w * QQ * QQ + k * QQ + l];
        out[e] = s;
    }
}

// fixed-order sum of the slices; C_kl = (X_kl + X_lk) / 2 off the diagonal (exactly symmetric), C_kk = D_k
__global__ void gg_reduce_kernel(const double* __restrict__ partial, int F, int P, int q, double* __restrict__ C)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long qq = (long long)q * q;
    if (t >= (long long)F * qq) return;
    const int f = (int)(t / qq), e = (int)(t - (long long)f * qq);
    const int k = e / q, l = e - k * q;
    const double* src = partial + (size_t)f * P * qq;
    double s = 0.0, s2 = 0.0;
    for (int p = 0; p < P; ++p) {
        s += src[(size_t)p * qq + (size_t)k * q + l];
        s2 += src[(size_t)p * qq + (size_t)l * q + k];
    }
    C[t] = k == l ? s : 0.5 * (s + s2);
}

struct GgShape {
    int F;            // functions
    long long N;      // terms per function
    int P;            // slices per function
};

static GgShape gg_shape(int m, int S, int pu, int mode)
{
    GgShape s;
    s.F = mode == 0 ? S * pu : mode == 1 ? pu : mode == 2 ? S : 1;
    s.N = (long long)m * (mode == 0 ? 1 : mode == 1 ? S : mode == 2 ? pu : (long long)S * pu);
    const long long nt = (s.N + GG_TILE - 1) / GG_TILE;
    const long long ntp = nt * (nt + 1) / 2;
    long long P = (GG_CTAS + s.F - 1) / s.F;
    if (P > ntp) P = ntp;
    if (P < 1) P = 1;
    s.P = (int)P;
    return s;
}

static long long gg_workspace(const GgShape& s, int q)
{
    return 8LL * s.F * s.P * q * q;
}

static const char* gg_check(int m, int q, int S, int pu, int mode)
{
    if (m <= 0 || S <= 0 || pu <= 0) return "m, S, pu must be positive";
    if (q < 1 || q > 32) return "q must be in [1, 32]";
    if (mode < 0 || mode > 3) return "mode must be 0 (per block), 1 (per PC), 2 (per sample) or 3 (one function)";
    if ((long long)S * pu >= (1LL << 31)) return "S * pu must be below 2^31";
    const long long N = (long long)m * (mode == 0 ? 1 : mode == 1 ? S : mode == 2 ? pu : (long long)S * pu);
    if (N >= (1LL << 31)) return "the terms of a function must number below 2^31";
    return nullptr;
}

template <int QP, bool SAME>
static int gg_launch(const double* Z, int m, int q, const double* beta, const double* a, int pu, int mode,
                     const double* omega, const GgShape& s, double* partial, cudaStream_t st)
{
    const size_t smem = 2 * sizeof(GgTile<QP>) + (GG_NT / 32) * sizeof(GgStage<QP>);
    GGP_CUDA(cudaFuncSetAttribute(gg_pair_kernel<QP, SAME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gg_pair_kernel<QP, SAME><<<(unsigned)((long long)s.F * s.P), GG_NT, smem, st>>>(Z, m, q, beta, a, pu, mode, omega,
                                                                                   s.N, s.P, partial);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

template <bool SAME>
static int gg_dispatch(int QP, const double* Z, int m, int q, const double* beta, const double* a, int pu, int mode,
                       const double* omega, const GgShape& s, double* partial, cudaStream_t st)
{
    switch (QP) {
        case 4: return gg_launch<4, SAME>(Z, m, q, beta, a, pu, mode, omega, s, partial, st);
        case 8: return gg_launch<8, SAME>(Z, m, q, beta, a, pu, mode, omega, s, partial, st);
        case 16: return gg_launch<16, SAME>(Z, m, q, beta, a, pu, mode, omega, s, partial, st);
        default: return gg_launch<32, SAME>(Z, m, q, beta, a, pu, mode, omega, s, partial, st);
    }
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_grad_sens_workspace_bytes(int m, int q, int S, int pu, int mode)
{
    if (gg_check(m, q, S, pu, mode)) return -1;
    return gg_workspace(gg_shape(m, S, pu, mode), q);
}

int ggp_grad_sens_f64(const double* Z, int m, int q, const double* beta, const double* a, int S, int pu, int mode,
                      const double* omega, double* C_out, void* workspace, long long workspace_bytes, void* stream)
{
    GGP_ARG(Z && beta && a && C_out && workspace, "null pointer");
    const char* bad = gg_check(m, q, S, pu, mode);
    GGP_ARG(!bad, bad);
    GGP_ARG(mode < 2 || omega, "null pointer (omega, modes 2 and 3)");
    const GgShape s = gg_shape(m, S, pu, mode);
    GGP_ARG((long long)s.F * s.P < (1LL << 31), "too many functions");
    const long long need = gg_workspace(s, q);
    if (workspace_bytes < need) {
        set_error("ggp_grad_sens_f64: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* partial = reinterpret_cast<double*>(workspace);
    const int QP = q <= 4 ? 4 : q <= 8 ? 8 : q <= 16 ? 16 : 32;
    const int rc = mode == 0 ? gg_dispatch<true>(QP, Z, m, q, beta, a, pu, mode, omega, s, partial, st)
                             : gg_dispatch<false>(QP, Z, m, q, beta, a, pu, mode, omega, s, partial, st);
    if (rc != GGP_OK) return rc;
    const long long nred = (long long)s.F * q * q;
    gg_reduce_kernel<<<(unsigned)((nred + 255) / 256), 256, 0, st>>>(partial, s.F, s.P, q, C_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
