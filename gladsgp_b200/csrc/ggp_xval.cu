// Cross-validated emulator predictions from the cached factor of the FULL training covariance (SepiaXvalEmulatorPrediction).
//
// SEPIA refits a sub-model per fold F of held-out training rows and predicts them from the rest.  With P = S22^-1 the
// held-out moments are closed forms in P (Schur complement):  mu_F = w_F - (P_FF)^-1 (P w)_F,  Sig_F = (P_FF)^-1 - c I.
// P_FF = Z_F Z_F^T with rows z_i = L^-1 e_i (S22 = L L^T), and (P w)_i = z_i . u with u = L^-1 w (kept with the factor).
// This kernel solves L z_i = e_i for a list of training rows i and returns alpha_i = z_i . u, p_i = |z_i|^2 and optionally
// the rows z_i themselves; for a leave-one-out fold those two numbers are the whole answer (mu_i = w_i - alpha_i / p_i,
// var_i = 1 / p_i - c).
//
// It is predict_kernel with the cross-covariance right-hand side replaced by the unit matrix of the held-out indices.
// z_i is zero above row i, so an 8-row unit pair starts both its panel loop and the k-range of its update at the panel of
// its smallest index: for ascending indices that is m^3/3 flop per (sample, PC) block instead of m^3.  Panels and k-blocks
// that a pair skips would only contribute exact zeros, so the results do not depend on the order of the indices.
#include "ggp_chol.cuh"
#include "../../include/gladsgp_b200.h"

#include <climits>

namespace ggp {

constexpr int XNT = 256;          // threads of the kernel
constexpr int XNW = XNT / 32;
constexpr int XB = 256;           // held-out rows per task: 8 warps x 4 units x 8 rows

// Tasks are (row block tb, block b) pairs handed out in the order tb-major through a counter in global memory: with
// ascending indices the first row blocks are the expensive ones (their rows start in early panels), so they go first and
// the cheap ones fill in behind them.  Which CTA runs a task does not change its result.
__global__ void __launch_bounds__(XNT, 2)
xval_kernel(int m, int Mp, const double* __restrict__ factor, long long l_stride, const double* __restrict__ U,
            const int* __restrict__ idx, int nidx, int B, double* __restrict__ alpha_out, double* __restrict__ p_out,
            double* __restrict__ Z_out, double* __restrict__ Vws, int* __restrict__ task_ctr)
{
    __shared__ __align__(16) double Minv[32 * MI_LD];
    __shared__ __align__(16) double uj[32];
    __shared__ int soff[1024];
    __shared__ int s_task, s_j0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int nP = Mp >> 5;
    fill_slab_offsets(soff, Mp);
    const int nblk = (nidx + XB - 1) / XB;
    const int ntask = B * nblk;
    double* __restrict__ Vw = Vws + (size_t)blockIdx.x * Mp * XB;   // [nP*4][XB][8]

    while (true) {
        __syncthreads();                                  // previous task done with s_task / s_j0 / Minv / uj
        if (tid == 0) { s_task = atomicAdd(task_ctr, 1); s_j0 = nP; }
        __syncthreads();
        const int task = s_task;
        if (task >= ntask) break;
        const int tb = task / B;
        const int b = task - tb * B;
        const int t0 = tb * XB;
        const int nt = min(XB, nidx - t0);
        const double* __restrict__ Lp = factor + (size_t)b * l_stride;
        const double* __restrict__ ub = U + (size_t)b * Mp;

        // held-out index of each of this lane's rows (-1: past the end of the list, or outside [0, m): a zero row) and
        // the first panel of each of the warp's two unit pairs
        int ir[2][2], jp[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int lo = INT_MAX;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int r = 8 * (warp + XNW * (2 * h + i)) + g;
                int v = (r < nt) ? idx[t0 + r] : -1;
                if (v < 0 || v >= m) v = -1;
                ir[h][i] = v;
                if (v >= 0) lo = min(lo, v);
            }
            lo = __reduce_min_sync(0xffffffffu, lo);
            jp[h] = (lo == INT_MAX) ? nP : (lo >> 5);
        }
        if (lane == 0) atomicMin(&s_j0, min(jp[0], jp[1]));
        if (Z_out) {                                      // the skipped leading panels of z are zero
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int r = 8 * (warp + XNW * (2 * h + i)) + g;
                    if (r < nt)
                        for (int c = 2 * q; c < 32 * jp[h]; c += 8)
                            *reinterpret_cast<double2*>(Z_out + ((size_t)b * nidx + t0 + r) * Mp + c) = make_double2(0.0, 0.0);
                }
        }
        double asum[4], psum[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { asum[i] = 0.0; psum[i] = 0.0; }
        __syncthreads();
        const int j0 = s_j0;

        for (int j = j0; j < nP; ++j) {
            const int row0 = j << 5;
            __syncthreads();                              // previous panel done with Minv / uj
            for (int e = tid; e < 1024; e += XNT)
                Minv[(e >> 5) * MI_LD + (e & 31)] = Lp[minv_off(Mp) + 1024LL * j + e];
            if (tid < 32) uj[tid] = ub[row0 + tid];
            __syncthreads();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (j < jp[h]) continue;                  // the pair's rows are still zero here (or it has none)
                const int kb0 = jp[h];
                double acc[2][4][2];
                int rb[2];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    rb[i] = 8 * (warp + XNW * (2 * h + i));
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
                }
                // S = Z[:, kb0-th k-block .. j) L[panel, same]^T: the k-range starts at the pair's first non-zero column
                if (j > kb0) panel_gemm<2>(acc, Vw + (size_t)(4 * kb0) * XB * 8, Lp, soff + 4 * kb0, j - kb0, row0, rb, g, q, XB);
#pragma unroll
                for (int i = 0; i < 2; ++i)
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                        for (int e = 0; e < 2; ++e)
                            acc[i][cb][e] = ((ir[h][i] == row0 + 8 * cb + 2 * q + e) ? 1.0 : 0.0) - acc[i][cb][e];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int r = rb[i] + g;
                    double xt[4][2];
                    unit_trsm(acc[i], xt, Minv, g, q);
                    double s0 = 0.0, q0 = 0.0;
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) {
                        const double2 u2 = *reinterpret_cast<const double2*>(uj + 8 * cb + 2 * q);
                        s0 = fma(xt[cb][0], u2.x, s0);
                        s0 = fma(xt[cb][1], u2.y, s0);
                        q0 = fma(xt[cb][0], xt[cb][0], q0);
                        q0 = fma(xt[cb][1], xt[cb][1], q0);
                        *reinterpret_cast<double2*>(Vw + ((size_t)(4 * j + cb) * XB + r) * 8 + 2 * q) =
                            make_double2(xt[cb][0], xt[cb][1]);
                        if (Z_out && r < nt)
                            *reinterpret_cast<double2*>(Z_out + ((size_t)b * nidx + t0 + r) * Mp + row0 + 8 * cb + 2 * q) =
                                make_double2(xt[cb][0], xt[cb][1]);
                    }
                    asum[2 * h + i] += s0;
                    psum[2 * h + i] += q0;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double s = asum[i], v = psum[i];
            s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 1); v += __shfl_xor_sync(0xffffffffu, v, 2);
            const int r = 8 * (warp + XNW * i) + g;
            if (q == 0 && r < nt) {
                alpha_out[(size_t)b * nidx + t0 + r] = s;
                p_out[(size_t)b * nidx + t0 + r] = v;
            }
        }
    }
}

}  // namespace ggp

using namespace ggp;

static int xval_grid(int B, int nidx)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long ntask = (long long)B * ((nidx + XB - 1) / XB);
    return (int)(ntask < 2LL * sms ? ntask : 2LL * sms);       // two CTAs per SM
}

// per-CTA unit-pair rows [Mp / 8][XB][8], then the task counter
static long long xval_rows_bytes(int m, int grid) { return (long long)grid * round_up32(m) * XB * (long long)sizeof(double); }

extern "C" {

long long ggp_xval_workspace_bytes(int m, int nidx, int B)
{
    if (m <= 0 || nidx <= 0 || B <= 0) return -1;
    return xval_rows_bytes(m, xval_grid(B, nidx)) + 16;
}

int ggp_xval_solve_f64(const double* factor, const double* u, int m, int B, const int* idx, int nidx,
                       double* alpha_out, double* pdiag_out, double* Z_out, void* workspace, long long workspace_bytes,
                       void* stream)
{
    GGP_ARG(factor && u && idx && alpha_out && pdiag_out && workspace, "null pointer");
    GGP_ARG(m > 0 && nidx > 0 && B > 0, "m, nidx, B must be positive");
    GGP_ARG(m <= 8192, "m must be <= 8192");
    GGP_ARG((long long)B * ((nidx + XB - 1) / XB) < (1LL << 31), "B * ceil(nidx / 256) must be below 2^31");
    const int grid = xval_grid(B, nidx);
    const long long need = xval_rows_bytes(m, grid) + 16;
    if (workspace_bytes < need) {
        set_error("ggp_xval_solve_f64: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int* ctr = reinterpret_cast<int*>(reinterpret_cast<char*>(workspace) + xval_rows_bytes(m, grid));
    GGP_CUDA(cudaMemsetAsync(ctr, 0, sizeof(int), st));
    const int Mp = round_up32(m);
    xval_kernel<<<grid, XNT, 0, st>>>(m, Mp, factor, packed_doubles(Mp), u, idx, nidx, B, alpha_out, pdiag_out, Z_out,
                                      reinterpret_cast<double*>(workspace), ctr);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
