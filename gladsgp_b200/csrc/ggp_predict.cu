// Posterior prediction kernels: predictive mean / variance through the cached factor, predictive
// covariance for joint draws, and the PC-basis reconstruction.
//
// Replaces SepiaPredict.wPred and SepiaEmulatorPrediction.get_y (SURVEY.md 8a rows a7, a8;
// Appendix A.7, A.10 w_pred / get_y; callers e.g.
// /root/reference/experiments/synthetic/analysis/assess_all_models.py:489-492).
//
// The reference solves S22 W = S21 from scratch for every (sample, PC, call).  Here the packed
// Cholesky factor L and u = L^-1 w of every (sample, PC) are computed once
// (ggp_loglik_batched_f64) and a block of test designs is pushed through
//   V = S21^T L^-T  (rows = designs; same left-looking DMMA panel loop as the factorisation),
//   mean = V u,  var = s11 - rowsum(V^2),  Sigma = S11 - V V^T.
#include "ggp_chol.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int PNT = 256;          // threads of the prediction kernel
constexpr int PNW = PNT / 32;
constexpr int PB = 256;           // designs per task: 8 warps x 4 units x 8 rows

struct PredSmem {
    double* Minv;   // [32][MI_LD] inverted diagonal block of the current panel (from the packed factor)
    double* uj;     // [32]
    double* etab;   // [ETAB]
    double* sb;     // [d]
    double* SC;     // [d][32] scaled training coordinates of the current panel
    double* scr;    // [PNW][16][32] per-warp scratch of the covariance step
};

__host__ __device__ inline size_t pred_smem_bytes(int d) {
    return (size_t)(32 * MI_LD + 32 + ETAB + sc_doubles(d) + 2 * ((d + 1) & ~1) + PNW * 512) * sizeof(double);
}

// One CTA pushes blocks of PB test designs through the cached factor of block b.  Rows = designs: each
// warp owns four 8-row units; per panel  S = V[:,0:32j] L[panel,0:32j]^T (DMMA),  P = cross-cov - S,
// X = P Minv^T (DMMA), V[:,panel] = X.  A lane reads back exactly the V entries it wrote (accumulator and
// A-fragment layouts coincide under the k permutation), so V needs no block-level synchronisation.
__global__ void __launch_bounds__(PNT, 2)
predict_kernel(const double* __restrict__ X, int m, int Mp, int d, const double* __restrict__ factor,
               long long l_stride, const double* __restrict__ U, const double* __restrict__ beta,
               const double* __restrict__ lamz, const double* __restrict__ s11,
               const double* __restrict__ Xp, int n, int B, double* __restrict__ mean_out,
               double* __restrict__ var_out, double* __restrict__ V_out, double* __restrict__ Vws)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PredSmem sm;
    {
        double* p = reinterpret_cast<double*>(smem_raw);
        sm.Minv = p;  p += 32 * MI_LD;
        sm.uj = p;    p += 32;
        sm.etab = p;  p += ETAB;
        sm.SC = p;    p += sc_doubles(d);
        sm.sb = p;    p += ((d + 1) & ~1);
        sm.scr = p;
    }
    __shared__ int soff[1024];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int nP = Mp >> 5;
    fill_slab_offsets(soff, Mp);
    fill_exp_table(sm.etab);
    const int nblk = (n + PB - 1) / PB;
    const long long ntask = (long long)B * nblk;
    double* __restrict__ Vw = Vws + (size_t)blockIdx.x * Mp * PB;   // [nP*4][PB][8]

    for (long long task = blockIdx.x; task < ntask; task += gridDim.x) {
        const int b = (int)(task / nblk);
        const int t0 = (int)(task - (long long)b * nblk) * PB;
        const int nt = min(PB, n - t0);
        const double inv_lamz = 1.0 / lamz[b];
        const double* __restrict__ Lp = factor + (size_t)b * l_stride;
        const double* __restrict__ ub = U + (size_t)b * Mp;
        __syncthreads();
        if (tid < d) sm.sb[tid] = sqrt(beta[(size_t)b * d + tid]);
        double mean[4], vsum[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { mean[i] = 0.0; vsum[i] = 0.0; }

        for (int j = 0; j < nP; ++j) {
            const int row0 = j << 5;
            __syncthreads();                       // previous panel done with Minv / uj / SC (and sb visible)
            fill_panel_coords(sm.SC, X, sm.sb, d, m, row0);
            for (int idx = tid; idx < 1024; idx += PNT)
                sm.Minv[(idx >> 5) * MI_LD + (idx & 31)] = Lp[minv_off(Mp) + 1024LL * j + idx];
            if (tid < 32) sm.uj[tid] = ub[row0 + tid];
            __syncthreads();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                double acc[2][4][2];
                int rb[2];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    rb[i] = 8 * (warp + PNW * (2 * h + i));
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
                }
                // a pair without a real design (the reference predicts 1-4 designs per call, assess_all_models.py:481: 4 of the
                // task's 256 rows) does nothing: small calls cost the latency of the warps that hold designs, not the full tile
                if (rb[0] >= nt) continue;
                if (j > 0) panel_gemm<2>(acc, Vw, Lp, soff, j, row0, rb, g, q, PB);
                {
                    const int rr[2] = {rb[0] + g, rb[1] + g};
                    const bool ok[2] = {rr[0] < nt, rr[1] < nt};
                    pair_cov<2>(acc, Xp + (size_t)t0 * d, rr, ok, sm.SC, sm.sb, d, m, row0, q, inv_lamz, 0.0, false, sm.etab,
                                sm.scr + warp * 512, lane);
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int r = rb[i] + g;                       // local design index
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
                        *reinterpret_cast<double2*>(Vw + ((size_t)(4 * j + cb) * PB + r) * 8 + 2 * q) =
                            make_double2(xt[cb][0], xt[cb][1]);
                        if (V_out && r < nt)
                            *reinterpret_cast<double2*>(V_out + ((size_t)b * n + t0 + r) * Mp + row0 + 8 * cb + 2 * q) =
                                make_double2(xt[cb][0], xt[cb][1]);
                    }
                    mean[2 * h + i] += s0;
                    vsum[2 * h + i] += q0;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double s = mean[i], v = vsum[i];
            s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 1); v += __shfl_xor_sync(0xffffffffu, v, 2);
            const int r = 8 * (warp + PNW * i) + g;
            if (q == 0 && r < nt) {
                mean_out[(size_t)b * n + t0 + r] = s;
                var_out[(size_t)b * n + t0 + r] = s11[b] - v;
            }
        }
    }
}

// Sigma[b][t1][t2] = S11 - V V^T ; S11 diagonal = s11[b], off-diagonal = cov(xp_t1, xp_t2)   (the per-PC block of SEPIA's
// predictive covariance, SepiaPredict.wPred).  The V V^T contraction (2 n^2 Mp flop per block: at the reference's
// largest call size, n = 256 designs, as much work as the moments themselves) runs on the FP64 tensor cores: one CTA
// (4 warps) per 64 x 32 tile of the lower triangle, a warp owns two 8-row units x 32 columns (DMMA.8x8x4, accumulators in
// registers, fragments are 16-byte loads from the row-major V with the same k permutation as the factorisation); tiles
// above the diagonal are not computed, every entry is written together with its mirror image.
__global__ void __launch_bounds__(128)
pred_cov_kernel(const double* __restrict__ Xp, int n, int d, const double* __restrict__ beta,
                const double* __restrict__ lamz, const double* __restrict__ s11,
                const double* __restrict__ V, int Mp, double* __restrict__ Sigma, int n_ct, int n_tiles)
{
    const int b = blockIdx.x / n_tiles;
    const int tile = blockIdx.x - b * n_tiles;
    // tiles of the lower triangle in row-tile-major order: row tile rt has min(n_ct, 2 rt + 2) column tiles
    int rt = 0, ct = tile;
    while (true) {
        const int w = min(n_ct, 2 * rt + 2);
        if (ct < w) break;
        ct -= w; ++rt;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int row0 = 64 * rt + 16 * warp, col0 = 32 * ct;
    if (col0 > row0 + 15) return;                      // this warp's rows lie entirely above the tile's columns
    const double* Vb = V + (size_t)b * n * Mp;
    const double* ap[2];
    const double* bp[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) ap[i] = Vb + (size_t)min(row0 + 8 * i + g, n - 1) * Mp + 2 * q;
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) bp[cb] = Vb + (size_t)min(col0 + 8 * cb + g, n - 1) * Mp + 2 * q;
    double acc[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
    double2 a[2], bb[4], an[2], bn[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) a[i] = *reinterpret_cast<const double2*>(ap[i]);
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) bb[cb] = *reinterpret_cast<const double2*>(bp[cb]);
    for (int k = 0; k < Mp; k += 8) {
        if (k + 8 < Mp) {
#pragma unroll
            for (int i = 0; i < 2; ++i) an[i] = *reinterpret_cast<const double2*>(ap[i] + k + 8);
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) bn[cb] = *reinterpret_cast<const double2*>(bp[cb] + k + 8);
        }
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int i = 0; i < 2; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].x, bb[cb].x);
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int i = 0; i < 2; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].y, bb[cb].y);
#pragma unroll
        for (int i = 0; i < 2; ++i) a[i] = an[i];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) bb[cb] = bn[cb];
    }
    const double* be = beta + (size_t)b * d;
    const double il = 1.0 / lamz[b];
    double* Sb = Sigma + (size_t)b * n * n;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int t1 = row0 + 8 * i + g;
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int t2 = col0 + 8 * cb + 2 * q + e;
                if (t1 >= n || t2 > t1) continue;
                double c11;
                if (t1 == t2) {
                    c11 = s11[b];
                } else {
                    double dist = 0.0;
                    for (int kk = 0; kk < d; ++kk) {
                        const double df = Xp[(size_t)t1 * d + kk] - Xp[(size_t)t2 * d + kk];
                        dist = fma(be[kk] * df, df, dist);
                    }
                    c11 = exp(-dist) * il;
                }
                const double v = c11 - acc[i][cb][e];
                Sb[(size_t)t1 * n + t2] = v;
                if (t1 != t2) Sb[(size_t)t2 * n + t1] = v;
            }
    }
}

// ---------------------------------------------------------------------------------------------
// PC-basis reconstruction  y[r][c] = (sum_p w[r][p] K[p][c]) * sd[c] + mean[c]   (get_y), float32.
// HBM-write bound: 4*R*n_y bytes.  Each thread owns 4 columns and keeps their K entries for all PCs in
// registers (PUMAX x 4), the w rows of the CTA's row range sit in shared memory and are read as
// broadcast LDS.128 (16 FMAs per load); stores are 16-byte streaming stores (512 B contiguous per warp).
// ---------------------------------------------------------------------------------------------
constexpr int RC_COLS = 1024;
constexpr int RC_RT = 128;       // rows of w staged per shared-memory tile

template <int PUMAX, bool VEC>
__global__ void __launch_bounds__(256)
reconstruct_kernel(const float* __restrict__ w, const float* __restrict__ K, const float* __restrict__ sd,
                   int sd_len, const float* __restrict__ mu, int mu_len, int R, int pu, long long n_y,
                   int rows_per_cta, float* __restrict__ y)
{
    __shared__ __align__(16) float ws[RC_RT * PUMAX];
    const long long c0 = (long long)blockIdx.x * RC_COLS;
    const int tid = threadIdx.x;
    long long col[4];
    float sdv[4], muv[4], kreg[PUMAX][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        col[i] = VEC ? c0 + 4 * tid + i : c0 + tid + 256 * i;
        const bool in = col[i] < n_y;
        sdv[i] = in ? (sd_len == 1 ? sd[0] : sd[col[i]]) : 0.f;
        muv[i] = in ? (mu_len == 1 ? mu[0] : mu[col[i]]) : 0.f;
#pragma unroll
        for (int p = 0; p < PUMAX; ++p) kreg[p][i] = (in && p < pu) ? __ldg(K + (size_t)p * n_y + col[i]) : 0.f;
    }
    const int r_begin = blockIdx.y * rows_per_cta;
    const int r_end = min(R, r_begin + rows_per_cta);
    for (int r0 = r_begin; r0 < r_end; r0 += RC_RT) {
        const int nr = min(RC_RT, r_end - r0);
        __syncthreads();
        for (int idx = tid; idx < nr * PUMAX; idx += 256) {
            const int rr = idx / PUMAX, p = idx - rr * PUMAX;
            ws[idx] = (p < pu) ? w[(size_t)(r0 + rr) * pu + p] : 0.f;
        }
        __syncthreads();
#pragma unroll 2
        for (int rr = 0; rr < nr; ++rr) {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int p4 = 0; p4 < PUMAX; p4 += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(ws + rr * PUMAX + p4);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    acc[c] = fmaf(w4.x, kreg[p4 + 0][c], acc[c]);
                    acc[c] = fmaf(w4.y, kreg[p4 + 1][c], acc[c]);
                    acc[c] = fmaf(w4.z, kreg[p4 + 2][c], acc[c]);
                    acc[c] = fmaf(w4.w, kreg[p4 + 3][c], acc[c]);
                }
            }
            float* yr = y + (size_t)(r0 + rr) * n_y;
            if (VEC && col[3] < n_y) {
                __stcs(reinterpret_cast<float4*>(yr + col[0]),
                       make_float4(acc[0] * sdv[0] + muv[0], acc[1] * sdv[1] + muv[1], acc[2] * sdv[2] + muv[2],
                                   acc[3] * sdv[3] + muv[3]));
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (col[c] < n_y) __stcs(yr + col[c], acc[c] * sdv[c] + muv[c]);
            }
        }
    }
}

// error statistics of one output against its test value (assess_all_models.py:523-538), accumulated in FP64 per thread:
// e = { resid^2, |resid / y_test| and its count over y_test >= mape_floor, covered count, lower limit, upper limit }
__device__ __forceinline__ void errstats_add(double (&e)[6], float vm, float vl, float vh, float yt, float mape_floor)
{
    const float res = vm - yt;
    e[0] += (double)(res * res);
    if (!(yt < mape_floor)) { e[1] += (double)fabsf(res / yt); e[2] += 1.0; }
    if (yt >= vl && yt <= vh) e[3] += 1.0;
    e[4] += (double)vl;
    e[5] += (double)vh;
}

// fixed-order reduction of e over a 256-thread block -> row[0..5] (summed over the tiles in order by errstats_reduce_kernel)
__device__ __forceinline__ void errstats_block_store(double (&e)[6], double* __restrict__ row)
{
    __shared__ double red[8][6];
    const int tid = threadIdx.x;
#pragma unroll
    for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) e[k] += __shfl_xor_sync(0xffffffffu, e[k], o);
    if ((tid & 31) == 0)
#pragma unroll
        for (int k = 0; k < 6; ++k) red[tid >> 5][k] = e[k];
    __syncthreads();
    if (tid < 6) {
        double sacc = 0.0;
        for (int wv = 0; wv < 8; ++wv) sacc += red[wv][tid];
        row[tid] = sacc;
    }
}

// ---------------------------------------------------------------------------------------------
// Fused predictive-distribution statistics (SURVEY 8f rank 1; the post-processing every caller does right
// after get_y: assess_all_models.py:493-500, plot_test_error.py:81-87).  For design t and output c, over the
// posterior samples s:   y_s = (w[s][t] . K[:,c]) * sd[c] + mu[c],   z_s = y_s + sd[c] * noise[s][t]
//   ymean = mean_s y_s ,  ylo / yhi = q and 1-q quantiles of z_s (np.quantile, linear interpolation).
// The per-sample fields never touch HBM: each thread streams the samples for 4 columns and keeps only the
// KQ smallest and KQ largest values (the quantiles the reference uses, 2.5 % / 97.5 % of 64-128 samples,
// need 3-5 of them).
// ---------------------------------------------------------------------------------------------
template <int PUMAX, int KQ>
__global__ void __launch_bounds__(256)
reconstruct_stats_kernel(const float* __restrict__ w, const float* __restrict__ K, const float* __restrict__ sd,
                         int sd_len, const float* __restrict__ mu, int mu_len, const float* __restrict__ noise,
                         int nsamp, int npred, int pu, long long n_y, int i0, float frac,
                         float* __restrict__ ymean, float* __restrict__ ylo, float* __restrict__ yhi,
                         const float* __restrict__ ytest, float mape_floor, double* __restrict__ err_part)
{
    extern __shared__ __align__(16) float ws[];          // [nsamp][PUMAX] then noise [nsamp]
    float* ns = ws + (size_t)nsamp * PUMAX;
    const int t = blockIdx.y;
    const long long c0 = (long long)blockIdx.x * RC_COLS;
    const int tid = threadIdx.x;
    for (int idx = tid; idx < nsamp * PUMAX; idx += 256) {
        const int s_ = idx / PUMAX, p = idx - s_ * PUMAX;
        ws[idx] = (p < pu) ? w[((size_t)s_ * npred + t) * pu + p] : 0.f;
    }
    for (int s_ = tid; s_ < nsamp; s_ += 256) ns[s_] = noise ? noise[(size_t)s_ * npred + t] : 0.f;
    long long col[4];
    float sdv[4], muv[4], kreg[PUMAX][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        col[i] = c0 + tid + 256 * i;                       // coalesced scalar access (n_y may be odd)
        const bool in = col[i] < n_y;
        sdv[i] = in ? (sd_len == 1 ? sd[0] : sd[col[i]]) : 0.f;
        muv[i] = in ? (mu_len == 1 ? mu[0] : mu[col[i]]) : 0.f;
#pragma unroll
        for (int p = 0; p < PUMAX; ++p) kreg[p][i] = (in && p < pu) ? __ldg(K + (size_t)p * n_y + col[i]) : 0.f;
    }
    __syncthreads();
    float lo[4][KQ], hi[4][KQ], sum[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        sum[c] = 0.f;
#pragma unroll
        for (int k = 0; k < KQ; ++k) { lo[c][k] = INFINITY; hi[c][k] = -INFINITY; }
    }
    for (int s_ = 0; s_ < nsamp; ++s_) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int p4 = 0; p4 < PUMAX; p4 += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(ws + s_ * PUMAX + p4);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                acc[c] = fmaf(w4.x, kreg[p4 + 0][c], acc[c]);
                acc[c] = fmaf(w4.y, kreg[p4 + 1][c], acc[c]);
                acc[c] = fmaf(w4.z, kreg[p4 + 2][c], acc[c]);
                acc[c] = fmaf(w4.w, kreg[p4 + 3][c], acc[c]);
            }
        }
        const float e = ns[s_];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float yv = acc[c] * sdv[c] + muv[c];
            sum[c] += yv;
            const float z = yv + sdv[c] * e;
            float v = z;
#pragma unroll
            for (int k = 0; k < KQ; ++k) { const float a = lo[c][k]; lo[c][k] = fminf(a, v); v = fmaxf(a, v); }
            v = z;
#pragma unroll
            for (int k = 0; k < KQ; ++k) { const float a = hi[c][k]; hi[c][k] = fmaxf(a, v); v = fminf(a, v); }
        }
    }
    const float inv_n = 1.f / (float)nsamp;
    double e[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        if (col[c] < n_y) {
            float a = 0.f, b = 0.f, ha = 0.f, hb = 0.f;
#pragma unroll
            for (int k = 0; k < KQ - 1; ++k)
                if (k == i0) { a = lo[c][k]; b = lo[c][k + 1]; ha = hi[c][k + 1]; hb = hi[c][k]; }
            const size_t o = (size_t)t * n_y + col[c];
            const float vm = sum[c] * inv_n, vl = a + (b - a) * frac, vh = ha + (hb - ha) * (1.f - frac);
            if (ymean) {
                __stcs(ymean + o, vm);
                __stcs(ylo + o, vl);
                __stcs(yhi + o, vh);
            }
            if (ytest) errstats_add(e, vm, vl, vh, __ldcs(ytest + o), mape_floor);
        }
    }
    if (ytest) errstats_block_store(e, err_part + ((size_t)t * gridDim.x + blockIdx.x) * 6);
}

// The same error sums from stored mean / limit fields (of ggp_reconstruct_quantiles_f32): the tiles, the per-thread
// columns and the reduction order are those of reconstruct_stats_kernel.  Block b = (design t, tile b % ntile).
__global__ void __launch_bounds__(256)
fields_errstats_kernel(const float* __restrict__ ymean, const float* __restrict__ ylo, const float* __restrict__ yhi,
                       const float* __restrict__ ytest, long long n_y, int ntile, float mape_floor,
                       double* __restrict__ err_part)
{
    const int t = blockIdx.x / ntile;
    const long long c0 = (long long)(blockIdx.x - t * ntile) * RC_COLS;
    double e[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const long long col = c0 + threadIdx.x + 256 * c;
        if (col < n_y) {
            const size_t o = (size_t)t * n_y + col;
            errstats_add(e, __ldcs(ymean + o), __ldcs(ylo + o), __ldcs(yhi + o), __ldcs(ytest + o), mape_floor);
        }
    }
    errstats_block_store(e, err_part + (size_t)blockIdx.x * 6);
}

// err[t][k] = sum over the column tiles of err_part[t][tile][k], in tile order
__global__ void errstats_reduce_kernel(const double* __restrict__ part, int ntile, int npred, double* __restrict__ err)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npred * 6) return;
    const int t = idx / 6, k = idx - 6 * t;
    double sacc = 0.0;
    for (int b = 0; b < ntile; ++b) sacc += part[((size_t)t * ntile + b) * 6 + k];
    err[idx] = sacc;
}

template <int PUMAX>
static int launch_stats(const float* w, const float* K, const float* sd, int sd_len, const float* mean, int mean_len,
                        const float* noise, int nsamp, int npred, int pu, long long n_y, int i0, float frac,
                        float* ymean, float* ylo, float* yhi, cudaStream_t st,
                        const float* ytest = nullptr, float mape_floor = 0.f, double* err_part = nullptr)
{
    const dim3 grid((unsigned)((n_y + RC_COLS - 1) / RC_COLS), (unsigned)npred);
    const size_t smem = ((size_t)nsamp * PUMAX + nsamp) * sizeof(float);
    // the staged samples exceed the default 48 KB of dynamic shared memory from about 700 samples at pu = 16
    if (i0 + 2 <= 4) {
        GGP_CUDA(cudaFuncSetAttribute(reconstruct_stats_kernel<PUMAX, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        reconstruct_stats_kernel<PUMAX, 4><<<grid, 256, smem, st>>>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu,
                                                                   n_y, i0, frac, ymean, ylo, yhi, ytest, mape_floor, err_part);
    } else {
        GGP_CUDA(cudaFuncSetAttribute(reconstruct_stats_kernel<PUMAX, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        reconstruct_stats_kernel<PUMAX, 8><<<grid, 256, smem, st>>>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu,
                                                                   n_y, i0, frac, ymean, ylo, yhi, ytest, mape_floor, err_part);
    }
    return GGP_OK;
}

template <int PUMAX>
static int launch_reconstruct(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                              int mean_len, int R, int pu, long long n_y, float* y_out, cudaStream_t st)
{
    const unsigned gx = (unsigned)((n_y + RC_COLS - 1) / RC_COLS);
    // enough CTAs to fill the machine a few times over, but long row ranges per CTA (K is loaded once per CTA)
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    unsigned gy = (unsigned)((8u * sms + gx - 1) / gx);
    const unsigned gymax = (unsigned)((R + 31) / 32);
    if (gy > gymax) gy = gymax;
    if (gy < 1) gy = 1;
    const int rows_per_cta = (R + gy - 1) / gy;
    gy = (unsigned)((R + rows_per_cta - 1) / rows_per_cta);
    const bool vec = (n_y % 4 == 0) && ((reinterpret_cast<uintptr_t>(y_out) & 15) == 0);
    if (vec)
        reconstruct_kernel<PUMAX, true><<<dim3(gx, gy), 256, 0, st>>>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, rows_per_cta, y_out);
    else
        reconstruct_kernel<PUMAX, false><<<dim3(gx, gy), 256, 0, st>>>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, rows_per_cta, y_out);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Multivariate-normal deviate of a (sample, PC) block from its joint predictive covariance: dev = L z, Sigma = L L^T.
// One CTA per block; the factorisation is eval_block_loglik's (DMMA left-looking panels, packed factor as scratch) with
// the matrix entries read from memory instead of generated, and a product in place of the forward solve.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, CTAS_PER_SM)
chol_draw_kernel(const double* __restrict__ Sigma, int n, int Mp, const double* __restrict__ z, double* __restrict__ Lws,
                 long long l_stride, double* __restrict__ dev, int* __restrict__ info, int b0)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const size_t b = (size_t)b0 + blockIdx.x;
    EvalSmem sm = carve_eval_smem(smem_raw, Mp, 0);
    eval_block_loglik<false, 1>(sm, Sigma + b * n * n, n, Mp, 0, nullptr, 1.0, 0.0, z + b * n,
                                        Lws + (size_t)blockIdx.x * l_stride, dev + b * n, info + b);
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_chol_draw_workspace_bytes(int n, int B)
{
    if (n <= 0 || B <= 0) return -1;
    return (long long)B * packed_doubles(round_up32(n)) * (long long)sizeof(double);
}

int ggp_chol_draw_f64(const double* Sigma, int n, int B, const double* z, double* dev_out, int* info_out,
                      void* workspace, long long workspace_bytes, void* stream)
{
    GGP_ARG(Sigma && z && dev_out && info_out && workspace, "null pointer");
    GGP_ARG(n > 0 && B > 0, "n, B must be positive");
    const int Mp = round_up32(n);
    const size_t smem = eval_smem_bytes(Mp, 0);
    if (smem > 227 * 1024) {
        set_error("ggp_chol_draw_f64: n=%d needs %zu B of shared memory (> 227 KB)", n, smem);
        return GGP_ERR_UNSUPPORTED;
    }
    const long long per = ggp_chol_draw_workspace_bytes(n, 1);
    const long long chunk = workspace_bytes / per;            // blocks whose scratch factor fits the workspace
    if (chunk < 1) {
        set_error("ggp_chol_draw_f64: workspace too small (%lld < %lld for one block)", workspace_bytes, per);
        return GGP_ERR_WORKSPACE;
    }
    GGP_CUDA(cudaFuncSetAttribute(chol_draw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GGP_CUDA(cudaFuncSetAttribute(chol_draw_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, eval_carveout_pct(smem)));
    for (long long b0 = 0; b0 < B; b0 += chunk) {
        const int nb = (int)((B - b0 < chunk) ? B - b0 : chunk);
        chol_draw_kernel<<<nb, NT, smem, (cudaStream_t)stream>>>(Sigma, n, Mp, z, reinterpret_cast<double*>(workspace),
                                                                 packed_doubles(Mp), dev_out, info_out, (int)b0);
        GGP_CUDA(cudaGetLastError());
    }
    return GGP_OK;
}

static int predict_grid(int B, int n)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long ntask = (long long)B * ((n + PB - 1) / PB);
    return (int)(ntask < 2LL * sms ? ntask : 2LL * sms);       // two CTAs per SM
}

long long ggp_predict_workspace_bytes(int m, int n, int B)
{
    if (m <= 0 || n <= 0 || B <= 0) return -1;
    const int Mp = round_up32(m);
    return (long long)predict_grid(B, n) * Mp * PB * (long long)sizeof(double);
}

int ggp_predict_f64(const double* X, int m, int d, const double* factor, const double* u, const double* beta,
                    const double* lamz, const double* s11_diag, const double* Xp, int n, int B,
                    double* mean_out, double* var_out, double* V_out, void* workspace, long long workspace_bytes,
                    void* stream)
{
    GGP_ARG(X && factor && u && beta && lamz && s11_diag && Xp && mean_out && var_out && workspace, "null pointer");
    GGP_ARG(m > 0 && d > 0 && n > 0 && B > 0, "m, d, n, B must be positive");
    GGP_ARG(m <= 8192, "m must be <= 8192");
    const int Mp = round_up32(m);
    const size_t smem = pred_smem_bytes(d);
    if (smem > 100 * 1024) {
        set_error("ggp_predict_f64: m=%d d=%d needs %zu B of shared memory (> 100 KB)", m, d, smem);
        return GGP_ERR_UNSUPPORTED;
    }
    const long long need = ggp_predict_workspace_bytes(m, n, B);
    if (workspace_bytes < need) {
        set_error("ggp_predict_f64: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    GGP_CUDA(cudaFuncSetAttribute(predict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    predict_kernel<<<predict_grid(B, n), PNT, smem, (cudaStream_t)stream>>>(
        X, m, Mp, d, factor, packed_doubles(Mp), u, beta, lamz, s11_diag, Xp, n, B, mean_out, var_out, V_out,
        reinterpret_cast<double*>(workspace));
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_pred_cov_f64(const double* Xp, int n, int d, const double* beta, const double* lamz,
                     const double* s11_diag, const double* V, int m, int B, double* Sigma_out, void* stream)
{
    GGP_ARG(Xp && beta && lamz && s11_diag && V && Sigma_out, "null pointer");
    GGP_ARG(n > 0 && d > 0 && m > 0 && B > 0, "n, d, m, B must be positive");
    const int n_rt = (n + 63) / 64, n_ct = (n + 31) / 32;
    long long n_tiles = 0;
    for (int rt = 0; rt < n_rt; ++rt) n_tiles += (n_ct < 2 * rt + 2) ? n_ct : 2 * rt + 2;
    GGP_ARG(n_tiles * (long long)B < (1LL << 31), "B * tiles(n) must be below 2^31 CTAs");
    pred_cov_kernel<<<(unsigned)(n_tiles * B), 128, 0, (cudaStream_t)stream>>>(Xp, n, d, beta, lamz, s11_diag, V, round_up32(m),
                                                                              Sigma_out, n_ct, (int)n_tiles);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_reconstruct_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                        int mean_len, int R, int pu, long long n_y, float* y_out, void* stream)
{
    GGP_ARG(w && K && sd && mean && y_out, "null pointer");
    GGP_ARG(R > 0 && pu > 0 && n_y > 0, "R, pu, n_y must be positive");
    GGP_ARG((sd_len == 1 || sd_len == n_y) && (mean_len == 1 || mean_len == n_y), "sd/mean length must be 1 or n_y");
    GGP_ARG(pu <= 32, "pu must be <= 32");
    cudaStream_t st = (cudaStream_t)stream;
    if (pu <= 4) launch_reconstruct<4>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, y_out, st);
    else if (pu <= 8) launch_reconstruct<8>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, y_out, st);
    else if (pu <= 12) launch_reconstruct<12>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, y_out, st);
    else if (pu <= 16) launch_reconstruct<16>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, y_out, st);
    else if (pu <= 24) launch_reconstruct<24>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, y_out, st);
    else launch_reconstruct<32>(w, K, sd, sd_len, mean, mean_len, R, pu, n_y, y_out, st);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_reconstruct_stats_supported(int nsamp, int pu, double q)
{
    const int i0 = (int)floor(q * (nsamp - 1));
    return !(pu > 16 || i0 + 2 > 8 || i0 + 2 > nsamp || (size_t)nsamp * 17 * sizeof(float) > 200 * 1024);
}

int ggp_reconstruct_stats_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                              int mean_len, const float* noise, int nsamp, int npred, int pu, long long n_y, double q,
                              float* ymean_out, float* ylo_out, float* yhi_out, void* stream)
{
    GGP_ARG(w && K && sd && mean && ymean_out && ylo_out && yhi_out, "null pointer");
    GGP_ARG(nsamp > 1 && npred > 0 && pu > 0 && n_y > 0, "nsamp, npred, pu, n_y must be positive");
    GGP_ARG((sd_len == 1 || sd_len == n_y) && (mean_len == 1 || mean_len == n_y), "sd/mean length must be 1 or n_y");
    GGP_ARG(q > 0.0 && q < 0.5, "q must be in (0, 0.5)");
    GGP_ARG(npred <= 65535, "npred must be <= 65535 per call");
    const double pos = q * (nsamp - 1);
    const int i0 = (int)floor(pos);
    const float frac = (float)(pos - i0);
    if (!ggp_reconstruct_stats_supported(nsamp, pu, q)) {
        set_error("ggp_reconstruct_stats_f32: unsupported (pu=%d > 16 or quantile needs %d > 8 order statistics)", pu, i0 + 2);
        return GGP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (pu <= 4) rc = launch_stats<4>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st);
    else if (pu <= 8) rc = launch_stats<8>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st);
    else if (pu <= 12) rc = launch_stats<12>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st);
    else rc = launch_stats<16>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st);
    if (rc != GGP_OK) return rc;
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

long long ggp_errstats_workspace_bytes(int npred, long long n_y)
{
    if (npred <= 0 || n_y <= 0) return -1;
    return (long long)npred * ((n_y + RC_COLS - 1) / RC_COLS) * 6 * (long long)sizeof(double);
}

int ggp_reconstruct_errstats_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                                 int mean_len, const float* noise, int nsamp, int npred, int pu, long long n_y, double q,
                                 const float* y_test, float mape_floor, float* ymean_out, float* ylo_out, float* yhi_out,
                                 double* err_out, void* workspace, long long workspace_bytes, void* stream)
{
    GGP_ARG(w && K && sd && mean && y_test && err_out && workspace, "null pointer");
    GGP_ARG((ymean_out && ylo_out && yhi_out) || (!ymean_out && !ylo_out && !yhi_out), "field outputs: all three or none");
    GGP_ARG(nsamp > 1 && npred > 0 && pu > 0 && n_y > 0, "nsamp, npred, pu, n_y must be positive");
    GGP_ARG((sd_len == 1 || sd_len == n_y) && (mean_len == 1 || mean_len == n_y), "sd/mean length must be 1 or n_y");
    GGP_ARG(q > 0.0 && q < 0.5, "q must be in (0, 0.5)");
    GGP_ARG(npred <= 65535, "npred must be <= 65535 per call");
    const double pos = q * (nsamp - 1);
    const int i0 = (int)floor(pos);
    const float frac = (float)(pos - i0);
    if (!ggp_reconstruct_stats_supported(nsamp, pu, q)) {
        set_error("ggp_reconstruct_errstats_f32: unsupported (pu=%d > 16 or quantile needs %d > 8 order statistics)", pu, i0 + 2);
        return GGP_ERR_UNSUPPORTED;
    }
    const long long need = ggp_errstats_workspace_bytes(npred, n_y);
    if (workspace_bytes < need) {
        set_error("ggp_reconstruct_errstats_f32: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* part = reinterpret_cast<double*>(workspace);
    int rc;
    if (pu <= 4) rc = launch_stats<4>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st, y_test, mape_floor, part);
    else if (pu <= 8) rc = launch_stats<8>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st, y_test, mape_floor, part);
    else if (pu <= 12) rc = launch_stats<12>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st, y_test, mape_floor, part);
    else rc = launch_stats<16>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, i0, frac, ymean_out, ylo_out, yhi_out, st, y_test, mape_floor, part);
    if (rc != GGP_OK) return rc;
    GGP_CUDA(cudaGetLastError());
    const int ntile = (int)((n_y + RC_COLS - 1) / RC_COLS);
    errstats_reduce_kernel<<<(npred * 6 + 127) / 128, 128, 0, st>>>(part, ntile, npred, err_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_fields_errstats_f32(const float* ymean, const float* ylo, const float* yhi, const float* y_test, int npred,
                            long long n_y, float mape_floor, double* err_out, void* workspace, long long workspace_bytes,
                            void* stream)
{
    GGP_ARG(ymean && ylo && yhi && y_test && err_out && workspace, "null pointer");
    GGP_ARG(npred > 0 && n_y > 0, "npred, n_y must be positive");
    const long long ntile = (n_y + RC_COLS - 1) / RC_COLS;
    GGP_ARG(6 * ntile * npred < (1LL << 31), "6 npred ceil(n_y / 1024) must be below 2^31");
    const long long need = ggp_errstats_workspace_bytes(npred, n_y);
    if (workspace_bytes < need) {
        set_error("ggp_fields_errstats_f32: workspace too small (%lld < %lld)", workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* part = reinterpret_cast<double*>(workspace);
    fields_errstats_kernel<<<(unsigned)(ntile * npred), 256, 0, st>>>(ymean, ylo, yhi, y_test, n_y, (int)ntile, mape_floor, part);
    GGP_CUDA(cudaGetLastError());
    errstats_reduce_kernel<<<(npred * 6 + 127) / 128, 128, 0, st>>>(part, (int)ntile, npred, err_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
