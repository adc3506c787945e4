// Emulator Jacobians: the gradient of the predictive mean with respect to the inputs, the joint posterior covariance
// of the value and the gradient, and from it the gradient of the predictive variance (DESIGN.md section 2 item 13).
//
// For a (sample, PC) block b with k(x, z_i) = exp(-sum_k beta_k (x_k - z_ik)^2) / lamz, the cached packed factor L of
// S22 and u = L^-1 w, ggp_predict_f64 forms V = L^-1 k(x, Z), mu = V.u and v = s11 - |V|^2.  Here every design gets one
// more row per differentiated input k:
//   g_k(x)_i = d k(x, z_i) / d x_k = -2 beta_k (x_k - z_ik) k(x, z_i),     D_k = L^-1 g_k,
// and with R = [V; D_1; ...; D_q] the mean vector is [mu, grad mu] = R u and the joint covariance of [f, grad f] is
// P - R R^T, P = diag(s11, 2 beta_1 / lamz, ..., 2 beta_q / lamz) (d k(x, x') / d x' vanishes at x' = x).
//
// The q + 1 rows of a design are consecutive rows of one warp, 32 / (q + 1) designs per warp, and go through
// predict_kernel's left-looking DMMA panel loop.  The rows never reach HBM: since the accumulator and A-fragment layouts
// coincide under the k permutation, a lane's fragment of X_b is both the A operand of X_b and the B operand of X_b^T, and
// acc_ab += X_a X_b^T over a panel's 32 columns is eight DMMA.8x8x4.  A unit's diagonal block is formed from its solved
// fragments while they are in registers; the blocks of two units holding rows of a common design stream both fragments
// back from the CTA's V workspace, where the same lane has just written them (fewer live registers than keeping them).
// The Gram blocks of a warp live in a per-warp shared-memory area (each lane touches only its own entries).
// Every row's panel product, covariance step and unit solve are those of predict_kernel and do not depend on the other
// rows, and the value row's mean and |V|^2 are summed in predict_kernel's order: mu and v equal ggp_predict_f64's bit
// for bit.  The diagonal of P - R R^T comes from those per-row sums, the off-diagonal entries from the DMMA Gram,
// written once for both triangles (exactly symmetric).
#include "ggp_chol.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int JNT = 256;          // threads of the Jacobian kernel
constexpr int JNW = JNT / 32;
constexpr int JPB = 256;          // rows per task: 8 warps x 4 units x 8 rows (the V workspace pitch, as predict's PB)
constexpr int JGRAM = 10 * 64;    // per-warp Gram area: unit pairs (a, b), b <= a < 4, 2 accumulator doubles per lane
constexpr int JWS = JGRAM + 8 * 32;   // per-warp area: the Gram, then the running mean and |R_k|^2 sums of the 4 units

struct JacSmem {
    double* Minv;   // [32][MI_LD] inverted diagonal block of the current panel
    double* uj;     // [32]
    double* etab;   // [ETAB]
    double* SC;     // [sc_doubles(d)] B fragments of the distance product for the current panel's columns
    double* sb;     // [d] sqrt(beta)
    double* ZS;     // [32][d] raw coordinates of the current panel's training points (the derivative factors)
    double* scr;    // [JNW][512] per-warp scratch of the covariance step
    double* gram;   // [JNW][JWS] per-warp Gram accumulators and row sums
};

__host__ __device__ inline size_t jac_smem_bytes(int d) {
    return (size_t)(32 * MI_LD + 32 + ETAB + sc_doubles(d) + ((d + 1) & ~1) + 32 * ((d + 1) & ~1) + JNW * 512 +
                    JNW * JWS) * sizeof(double);
}

// designs per warp for q differentiated inputs: q + 1 consecutive rows each, packed into the warp's 32 (q <= 31)
__host__ __device__ inline int jac_designs_per_warp(int q) { return 32 / (q + 1); }

// pair_cov for rows that are either a design's value row (kcol < 0: the cross-covariance k(x, z_c), as pair_cov with
// self = false computes it) or its derivative row for input kcol: k(x, z_c) times -2 beta (x_kcol - z_c,kcol)
// (nb2 = -2 beta, xk = x_kcol).  xr: each unit's row coordinates.  p = C - p.
template <int NU>
static __device__ __forceinline__ void pair_cov_grad(double (&p)[2][4][2], const double* const (&xr)[2],
                                                     const bool (&row_ok)[2], const int (&kcol)[2],
                                                     const double (&nb2)[2], const double (&xk)[2],
                                                     const double* __restrict__ ZS, const double* __restrict__ SCB,
                                                     const double* __restrict__ sb, int d, int m, int row0, int q,
                                                     double inv_lamz, const double* __restrict__ etab,
                                                     double* __restrict__ scr, int lane)
{
    double dn[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) { dn[i][cb][0] = 0.0; dn[i][cb][1] = 0.0; }
    switch (cov_ksteps(d)) {
        case 1: cov_dist<NU, 1>(dn, xr, SCB, sb, d, q, lane); break;
        case 2: cov_dist<NU, 2>(dn, xr, SCB, sb, d, q, lane); break;
        case 3: cov_dist<NU, 3>(dn, xr, SCB, sb, d, q, lane); break;
        case 4: cov_dist<NU, 4>(dn, xr, SCB, sb, d, q, lane); break;
        case 5: cov_dist<NU, 5>(dn, xr, SCB, sb, d, q, lane); break;
        default: cov_dist<NU, 0>(dn, xr, SCB, sb, d, q, lane); break;
    }
#pragma unroll
    for (int i = 0; i < NU; ++i)
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            scr[(8 * i + 2 * cb) * 32 + lane] = dn[i][cb][0];
            scr[(8 * i + 2 * cb + 1) * 32 + lane] = dn[i][cb][1];
        }
#pragma unroll 8
    for (int e = 0; e < 8 * NU; ++e) scr[e * 32 + lane] = exp_neg(scr[e * 32 + lane], etab);
#pragma unroll
    for (int i = 0; i < NU; ++i)
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int cc = 8 * cb + 2 * q + e;
                const int c = row0 + cc;
                double v = (row_ok[i] && c < m) ? scr[(8 * i + 2 * cb + e) * 32 + lane] * inv_lamz : 0.0;
                if (kcol[i] >= 0) v *= nb2[i] * (xk[i] - ZS[cc * d + kcol[i]]);
                p[i][cb][e] = v - p[i][cb][e];
            }
        }
}

// acc_ab += X_a X_b^T over one panel's 32 columns: a lane's accumulator fragment of X_a is the A operand and its
// fragment of X_b the B operand (both under the k permutation of the factorisation).  gp: this lane's entries.
static __device__ __forceinline__ void gram_add(double* __restrict__ gp, const double (&xa)[4][2], const double (&xb)[4][2])
{
    double c0 = gp[0], c1 = gp[32];
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) {
        dmma884(c0, c1, xa[cb][0], xb[cb][0]);
        dmma884(c0, c1, xa[cb][1], xb[cb][1]);
    }
    gp[0] = c0;
    gp[32] = c1;
}

__device__ __forceinline__ int gram_idx(int a, int b) { return a * (a + 1) / 2 + b; }

// One CTA pushes blocks of JNW * dpw designs (q + 1 rows each) through the cached factor of block b.  Warp w owns
// local rows 32 w .. 32 w + 31 (units u = 0..3 at rows 32 w + 8 u); row k of the warp's design slot s (k = 0: value,
// k >= 1: input col0 + k - 1) is within-warp row s (q + 1) + k, so a design may straddle units.  Units a > b share a
// design when the first slot of a is at most the last slot of b; the Gram of such a pair is accumulated.
__global__ void __launch_bounds__(JNT, 2)
jacobian_kernel(const double* __restrict__ X, int m, int Mp, int d, int col0, const double* __restrict__ factor,
                long long l_stride, const double* __restrict__ U, const double* __restrict__ beta,
                const double* __restrict__ lamz, const double* __restrict__ s11, const double* __restrict__ Xp, int n,
                int B, int full, double* __restrict__ mean_out, double* __restrict__ cov_out, double* __restrict__ Vws)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    JacSmem sm;
    const int dpad = (d + 1) & ~1;
    {
        double* p = reinterpret_cast<double*>(smem_raw);
        sm.Minv = p;  p += 32 * MI_LD;
        sm.uj = p;    p += 32;
        sm.etab = p;  p += ETAB;
        sm.SC = p;    p += sc_doubles(d);
        sm.sb = p;    p += dpad;
        sm.ZS = p;    p += 32 * dpad;
        sm.scr = p;   p += JNW * 512;
        sm.gram = p;
    }
    __shared__ int soff[1024];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int nP = Mp >> 5;
    const int nq = d - col0;                       // differentiated inputs
    const int nr = nq + 1;                         // rows per design
    const int dpw = jac_designs_per_warp(nq);
    const int dpt = JNW * dpw;                     // designs per task
    fill_slab_offsets(soff, Mp);
    fill_exp_table(sm.etab);
    const int nblk = (n + dpt - 1) / dpt;
    const long long ntask = (long long)B * nblk;
    double* __restrict__ Vw = Vws + (size_t)blockIdx.x * Mp * JPB;   // [nP*4][JPB][8]
    double* __restrict__ gw = sm.gram + warp * JWS + lane;
    double* __restrict__ msum = gw + JGRAM;        // [u][lane] running R u, then [4 + u][lane] running |R_k|^2
    const int units_used = (dpw * nr + 7) >> 3;    // units holding rows of a design
    auto share = [&](int a, int bu) { return (8 * a) / nr <= (8 * bu + 7) / nr; };   // units a >= bu: a common design

    for (long long task = blockIdx.x; task < ntask; task += gridDim.x) {
        const int b = (int)(task / nblk);
        const int t0 = (int)(task - (long long)b * nblk) * dpt;
        const int nt = min(dpt, n - t0);
        const double inv_lamz = 1.0 / lamz[b];
        const double* __restrict__ Lp = factor + (size_t)b * l_stride;
        const double* __restrict__ ub = U + (size_t)b * Mp;
        const double* __restrict__ be = beta + (size_t)b * d;
        const double* __restrict__ Xt = Xp + (size_t)t0 * d;
        __syncthreads();
        if (tid < d) sm.sb[tid] = sqrt(be[tid]);
        for (int e = 0; e < JWS; e += 32) gw[e] = 0.0;

        for (int j = 0; j < nP; ++j) {
            const int row0 = j << 5;
            __syncthreads();                       // previous panel done with Minv / uj / SC / ZS (and sb visible)
            for (int idx = tid; idx < 32 * d; idx += JNT)
                sm.ZS[idx] = (row0 + idx / d < m) ? __ldg(X + (size_t)row0 * d + idx) : 0.0;
            fill_panel_coords(sm.SC, X, sm.sb, d, m, row0);
            for (int idx = tid; idx < 1024; idx += JNT)
                sm.Minv[(idx >> 5) * MI_LD + (idx & 31)] = Lp[minv_off(Mp) + 1024LL * j + idx];
            if (tid < 32) sm.uj[tid] = ub[row0 + tid];
            __syncthreads();
#pragma unroll 1                           // one copy of the pair body: unrolled, it spills at 128 registers
            for (int h = 0; h < 2; ++h) {
                // a pair whose first unit holds no design of this task does nothing (warp-uniform)
                if (2 * h >= units_used || warp * dpw + (16 * h) / nr >= nt) continue;
                double acc[2][4][2];
                int rb[2];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    rb[i] = 8 * (4 * warp + 2 * h + i);
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
                }
                if (j > 0) panel_gemm<2>(acc, Vw, Lp, soff, j, row0, rb, g, q, JPB);
                // the rows' roles, formed after the product (fewer registers live across it)
                const double* xr[2];
                bool ok[2];
                int kcol[2];
                double nb2[2], xk[2];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int wr = 8 * (2 * h + i) + g, slot = wr / nr, k = wr - slot * nr;
                    const int ld = warp * dpw + slot;
                    ok[i] = slot < dpw && ld < nt;
                    xr[i] = Xt + (size_t)(ok[i] ? ld : 0) * d;
                    kcol[i] = (ok[i] && k > 0) ? col0 + k - 1 : -1;
                    nb2[i] = (kcol[i] >= 0) ? -2.0 * be[kcol[i]] : 0.0;
                    xk[i] = (kcol[i] >= 0) ? __ldg(xr[i] + kcol[i]) : 0.0;
                }
                pair_cov_grad<2>(acc, xr, ok, kcol, nb2, xk, sm.ZS, sm.SC, sm.sb, d, m, row0, q, inv_lamz, sm.etab,
                                 sm.scr + warp * 512, lane);
                const int a0 = 2 * h, a1 = 2 * h + 1;
                const bool has1 = a1 < units_used;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int r = rb[i] + g;                       // local row
                    double xt[4][2];
                    unit_trsm(acc[i], xt, sm.Minv, g, q);
                    double s0 = 0.0, q0 = 0.0;
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) {
                        const double2 u2 = *reinterpret_cast<const double2*>(sm.uj + 8 * cb + 2 * q);
                        s0 = fma(xt[cb][0], u2.x, s0);
                        s0 = fma(xt[cb][1], u2.y, s0);
                        q0 = fma(xt[cb][0], xt[cb][0], q0);
                        q0 = fma(xt[cb][1], xt[cb][1], q0);
                        *reinterpret_cast<double2*>(Vw + ((size_t)(4 * j + cb) * JPB + r) * 8 + 2 * q) =
                            make_double2(xt[cb][0], xt[cb][1]);
                    }
                    msum[32 * (2 * h + i)] += s0;
                    msum[32 * (4 + 2 * h + i)] += q0;
                    // the unit's diagonal Gram block, from its fragments while they are in registers
                    if (i == 0 || has1) gram_add(gw + gram_idx(2 * h + i, 2 * h + i) * 64, xt, xt);
                }
                // blocks of units sharing a design (a > bu, bu in an earlier unit of the warp): both operands streamed
                // back from the V workspace (this lane wrote them above) two doubles at a time
                if (has1 || h == 1) {
#pragma unroll 1
                    for (int a = a0; a <= a1; ++a) {
                        if (a >= units_used) break;
#pragma unroll 1
                        for (int bu = 0; bu < a; ++bu) {
                            if (!share(a, bu)) continue;
                            double* gp = gw + gram_idx(a, bu) * 64;
                            double c0 = gp[0], c1 = gp[32];
                            const double* pa = Vw + ((size_t)(4 * j) * JPB + 8 * (4 * warp + a) + g) * 8 + 2 * q;
                            const double* pb = Vw + ((size_t)(4 * j) * JPB + 8 * (4 * warp + bu) + g) * 8 + 2 * q;
#pragma unroll
                            for (int cb = 0; cb < 4; ++cb) {
                                const double2 xa = *reinterpret_cast<const double2*>(pa + (size_t)cb * JPB * 8);
                                const double2 xb = *reinterpret_cast<const double2*>(pb + (size_t)cb * JPB * 8);
                                dmma884(c0, c1, xa.x, xb.x);
                                dmma884(c0, c1, xa.y, xb.y);
                            }
                            gp[0] = c0;
                            gp[32] = c1;
                        }
                    }
                }
            }
        }
        // ---- outputs: [mu, grad mu] from the per-row sums, the covariance diagonal from |R_k|^2, the rest from the Gram
        const size_t cstride = full ? (size_t)nr * nr : (size_t)(2 * nq + 1);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            double s = msum[32 * u], v = msum[32 * (4 + u)];
            s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 1); v += __shfl_xor_sync(0xffffffffu, v, 2);
            const int wr = 8 * u + g, slot = wr / nr, k = wr - slot * nr;
            const int ld = warp * dpw + slot;
            if (q == 0 && slot < dpw && ld < nt) {
                const size_t t = (size_t)b * n + t0 + ld;
                mean_out[t * nr + k] = s;
                const double prior = (k == 0) ? s11[b] : (2.0 * be[col0 + k - 1]) * inv_lamz;
                const double c = prior - v;
                if (full) cov_out[t * cstride + (size_t)k * nr + k] = c;
                else cov_out[t * cstride + (k == 0 ? 0 : nq + k)] = c;
            }
        }
        __syncwarp();
        for (int a = 0; a < units_used; ++a)
            for (int bu = 0; bu <= a; ++bu) {
                if (bu < a && !share(a, bu)) continue;
                const double* gp = gw + gram_idx(a, bu) * 64;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int wr = 8 * a + g, wc = 8 * bu + 2 * q + e, slot = wr / nr;
                    const int ld = warp * dpw + slot;
                    if (slot != wc / nr || slot >= dpw || ld >= nt) continue;
                    const int ki = wr - slot * nr, kj = wc - slot * nr;
                    if (kj >= ki) continue;
                    const size_t t = (size_t)b * n + t0 + ld;
                    const double c = -gp[32 * e];
                    if (full) {
                        cov_out[t * cstride + (size_t)ki * nr + kj] = c;
                        cov_out[t * cstride + (size_t)kj * nr + ki] = c;
                    } else if (kj == 0) {
                        cov_out[t * cstride + ki] = c;
                    }
                }
            }
    }
}

static int jacobian_grid(int B, int n, int q)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int dpt = JNW * jac_designs_per_warp(q);
    const long long ntask = (long long)B * ((n + dpt - 1) / dpt);
    return (int)(ntask < 2LL * sms ? ntask : 2LL * sms);       // two CTAs per SM
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_jacobian_workspace_bytes(int m, int d, int col0, int n, int B)
{
    if (m <= 0 || m > 8192 || d <= 0 || n <= 0 || B <= 0 || col0 < 0 || d - col0 < 1 || d - col0 > 31) return -1;
    return (long long)jacobian_grid(B, n, d - col0) * round_up32(m) * JPB * (long long)sizeof(double);
}

int ggp_jacobian_f64(const double* X, int m, int d, const double* factor, const double* u, const double* beta,
                     const double* lamz, const double* s11_diag, const double* Xp, int n, int B, int col0, int full,
                     double* mean_out, double* cov_out, void* workspace, long long workspace_bytes, void* stream)
{
    GGP_ARG(X && factor && u && beta && lamz && s11_diag && Xp && mean_out && cov_out && workspace, "null pointer");
    GGP_ARG(m > 0 && d > 0 && n > 0 && B > 0, "m, d, n, B must be positive");
    GGP_ARG(m <= 8192, "m must be <= 8192");
    GGP_ARG(col0 >= 0 && d - col0 >= 1 && d - col0 <= 31, "the differentiated inputs q = d - col0 must be in [1, 31]");
    GGP_ARG(full == 0 || full == 1, "full must be 0 or 1");
    const int Mp = round_up32(m);
    const size_t smem = jac_smem_bytes(d);
    const long long need = ggp_jacobian_workspace_bytes(m, d, col0, n, B);
    if (workspace_bytes < need) {
        set_error("ggp_jacobian_f64: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    GGP_CUDA(cudaFuncSetAttribute(jacobian_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    jacobian_kernel<<<jacobian_grid(B, n, d - col0), JNT, smem, (cudaStream_t)stream>>>(
        X, m, Mp, d, col0, factor, packed_doubles(Mp), u, beta, lamz, s11_diag, Xp, n, B, full, mean_out, cov_out,
        reinterpret_cast<double*>(workspace));
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
