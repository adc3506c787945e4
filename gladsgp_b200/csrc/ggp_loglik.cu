// Covariance build, cross-covariance and batched fused log-likelihood entry points.
// C-ABI declared in include/gladsgp_b200.h.
#include "ggp_chol.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

// ---------------------------------------------------------------------------------------------
// (1) product squared-exponential covariance, materialised (SepiaDistCov type 1).
// 8*m*m bytes written per matrix.  One CTA per (64x64 tile pair, matrix): the tile (bi >= bj) is
// computed once (half the exps) and written twice -- directly and transposed -- as 16-byte streaming stores.
// Distances are the rank-(d+2) DMMA product of pair_cov (ggp_chol.cuh): warp w owns the 8 rows 8w..8w+7 of the tile,
// 3 DMMA steps per 8x8 block at d = 9; the 16 exponentials of a lane are inlined; the tile goes through shared memory
// so that both copies leave as full 128-byte lines.
// ---------------------------------------------------------------------------------------------
constexpr int CT = 64;
constexpr int CT_LD = CT + 1;

// KSC: compile-time number of DMMA steps of the distance product (0 = runtime), so that the fragment addresses are constants
template <int KSC>
__global__ void __launch_bounds__(256, 4)
cov_build_kernel(const double* __restrict__ X, int m, int d, const double* __restrict__ beta,
                 const double* __restrict__ lamz, const double* __restrict__ diag_add,
                 double* __restrict__ C, int ntile)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int KS = KSC > 0 ? KSC : cov_ksteps(d), K4 = 4 * KS;
    double* XA = reinterpret_cast<double*>(smem_raw);      // [CT][K4] row side:    [x~, |x~|^2, 1, 0..]
    double* XB = XA + CT * K4;                             // [CT][K4] column side: [2 x~, -1, -|x~|^2, 0..]
    double* T = XB + CT * K4;                              // [CT][CT_LD] the tile
    double* etab = T + CT * CT_LD;                         // [ETAB]
    double* sbs = etab + ETAB;                               // [d] sqrt(beta)
    const int b = blockIdx.y;
    // decode lower-triangular tile index
    int t = blockIdx.x;
    int bi = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
    while (bi * (bi + 1) / 2 > t) --bi;
    const int bj = t - bi * (bi + 1) / 2;
    const double* be = beta + (size_t)b * d;
    const double il = 1.0 / lamz[b];
    const double dg = il + diag_add[b];
    const int r0 = bi * CT, c0 = bj * CT;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    fill_exp_table(etab);
    if (tid >= 128 && tid < 128 + d) sbs[tid - 128] = sqrt(be[tid - 128]);
    __syncthreads();
    if (tid < 2 * CT) {
        // thread per point: rows of the tile (tid < CT) and columns (tid >= CT)
        const bool colside = tid >= CT;
        const int lr = colside ? tid - CT : tid;
        const int pt = (colside ? c0 : r0) + lr;
        double* dst = (colside ? XB : XA) + lr * K4;
        double rr = 0.0;
        for (int k = 0; k < d; ++k) {
            const double x = (pt < m) ? __ldg(X + (size_t)pt * d + k) * sbs[k] : 0.0;
            rr = fma(x, x, rr);
            dst[k] = colside ? 2.0 * x : x;
        }
        for (int k = d; k < K4; ++k) dst[k] = 0.0;
        if (pt < m) {
            dst[d] = colside ? -1.0 : rr;
            dst[d + 1] = colside ? -rr : 1.0;
        }
    }
    __syncthreads();
    // -dist for the warp's 8 rows x 64 columns
    double dn[8][2];
#pragma unroll
    for (int cb = 0; cb < 8; ++cb) { dn[cb][0] = 0.0; dn[cb][1] = 0.0; }
#pragma unroll
    for (int s = 0; s < KS; ++s) {
        const double a = XA[(8 * warp + g) * K4 + 4 * s + q];
#pragma unroll
        for (int cb = 0; cb < 8; ++cb) dmma884(dn[cb][0], dn[cb][1], a, XB[(8 * cb + g) * K4 + 4 * s + q]);
    }
    {
        const int lr = 8 * warp + g;
        double* trow = T + lr * CT_LD + 2 * q;
        const int dcol = r0 + lr - c0 - 2 * q;               // tile-local column (minus 2q) of the diagonal entry, if any
#pragma unroll
        for (int cb = 0; cb < 8; ++cb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double v = exp_neg(dn[cb][e], etab) * il;
                trow[8 * cb + e] = (dcol == 8 * cb + e) ? dg : v;
            }
    }
    __syncthreads();
    double* Cb = C + (size_t)b * m * m;
    const bool vec2 = (m % 2 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
    const int cc = 2 * lane;
    if (vec2 && r0 + CT <= m && c0 + CT <= m) {
        // interior tile: no bounds checks.  8 rows x 64 columns per pass, a warp writes one 512-byte row segment
        double* dst = Cb + (size_t)(r0 + warp) * m + c0 + cc;
        const double* src = T + warp * CT_LD + cc;
#pragma unroll
        for (int it = 0; it < 8; ++it)
            __stcs(reinterpret_cast<double2*>(dst + (size_t)it * 8 * m), make_double2(src[it * 8 * CT_LD], src[it * 8 * CT_LD + 1]));
        if (bi != bj) {
            double* dt = Cb + (size_t)(c0 + warp) * m + r0 + cc;           // transposed copy: output row = column of the tile
            const double* st = T + cc * CT_LD + warp;
#pragma unroll
            for (int it = 0; it < 8; ++it)
                __stcs(reinterpret_cast<double2*>(dt + (size_t)it * 8 * m), make_double2(st[it * 8], st[it * 8 + CT_LD]));
        }
        return;
    }
    for (int it = 0; it < 8; ++it) {
        const int lr = it * 8 + warp;
        const int r = r0 + lr, c = c0 + cc;
        if (r < m) {
            const double v0 = T[lr * CT_LD + cc], v1 = T[lr * CT_LD + cc + 1];
            if (vec2 && c + 1 < m) __stcs(reinterpret_cast<double2*>(Cb + (size_t)r * m + c), make_double2(v0, v1));
            else {
                if (c < m) Cb[(size_t)r * m + c] = v0;
                if (c + 1 < m) Cb[(size_t)r * m + c + 1] = v1;
            }
        }
    }
    if (bi != bj) {
        for (int it = 0; it < 8; ++it) {
            const int lc = it * 8 + warp;                  // tile column -> output row
            const int r = c0 + lc, c = r0 + cc;
            if (r < m) {
                const double v0 = T[cc * CT_LD + lc], v1 = T[(cc + 1) * CT_LD + lc];
                if (vec2 && c + 1 < m) __stcs(reinterpret_cast<double2*>(Cb + (size_t)r * m + c), make_double2(v0, v1));
                else {
                    if (c < m) Cb[(size_t)r * m + c] = v0;
                    if (c + 1 < m) Cb[(size_t)r * m + c + 1] = v1;
                }
            }
        }
    }
}

// Row-block version (round 2) for m a multiple of 64 and a 16-byte aligned output: one CTA per (64-row block bi, matrix)
// walks the tiles bj = 0 .. bi of its block.  Per CTA, not per tile: the exponential table, sqrt(beta) and the row side of the
// distance product; the column side of the next tile is staged (two warps) while the current tile is computed.  The tile's own
// copy AND its mirror image leave straight from the accumulator fragments (streaming stores: 64 contiguous bytes per row and
// instruction either way; no tile in shared memory, one barrier per tile); the diagonal rule is applied in the diagonal tile alone.  Same arithmetic
// per entry as cov_build_kernel: identical bits.  (A two-level-table exponential with the scale folded into the exponent, 9 instead
// of 14 FP64 operations per entry, made this kernel slower: 0.356 vs 0.333 ms -- the second table lookup costs more than the operations.)
template <int KSC>
__global__ void __launch_bounds__(256, 4)
cov_build_rows_kernel(const double* __restrict__ X, int m, int d, const double* __restrict__ beta,
                      const double* __restrict__ lamz, const double* __restrict__ diag_add, double* __restrict__ C)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int KS = KSC > 0 ? KSC : cov_ksteps(d), K4 = 4 * KS;
    double* XA = reinterpret_cast<double*>(smem_raw);      // [CT][K4] row side:    [x~, |x~|^2, 1, 0..]
    double* XB = XA + CT * K4;                             // [2][CT][K4] column side: [2 x~, -1, -|x~|^2, 0..] (double-buffered)
    double* etab = XB + 2 * CT * K4;                       // [ETAB]
    double* sbs = etab + ETAB;                             // [d] sqrt(beta)
    const int b = blockIdx.y;
    const int bi = (int)gridDim.x - 1 - (int)blockIdx.x;   // long row blocks first
    const double* be = beta + (size_t)b * d;
    const double il = 1.0 / lamz[b];
    const double dg = il + diag_add[b];
    const int r0 = bi * CT;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    fill_exp_table(etab);
    if (tid >= 128 && tid < 128 + d) sbs[tid - 128] = sqrt(be[tid - 128]);
    __syncthreads();
    // coordinates of 64 points -> one side of the distance product (thread lr of a 64-thread group)
    auto stage = [&](double* dst0, int p0, bool colside, int lr) {
        double* dst = dst0 + lr * K4;
        double rr = 0.0;
        for (int k = 0; k < d; ++k) {
            const double x = __ldg(X + (size_t)(p0 + lr) * d + k) * sbs[k];
            rr = fma(x, x, rr);
            dst[k] = colside ? 2.0 * x : x;
        }
        for (int k = d + 2; k < K4; ++k) dst[k] = 0.0;
        dst[d] = colside ? -1.0 : rr;
        dst[d + 1] = colside ? -rr : 1.0;
    };
    if (tid < CT) stage(XA, r0, false, tid);
    else if (tid < 2 * CT) stage(XB, 0, true, tid - CT);
    __syncthreads();
    double* Cb = C + (size_t)b * m * m;
    const int lr = 8 * warp + g;
    for (int bj = 0; bj <= bi; ++bj) {
        const int c0 = bj * CT;
        const double* XBc = XB + (bj & 1) * CT * K4;
        // column side of the next tile (warps 4 and 5; visible after the barrier at the end of this iteration)
        if (bj < bi && tid >= 2 * CT && tid < 3 * CT) stage(XB + ((bj + 1) & 1) * CT * K4, c0 + CT, true, tid - 2 * CT);
        double dn[8][2];
#pragma unroll
        for (int cb = 0; cb < 8; ++cb) { dn[cb][0] = 0.0; dn[cb][1] = 0.0; }
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const double a = XA[lr * K4 + 4 * s + q];
#pragma unroll
            for (int cb = 0; cb < 8; ++cb) dmma884(dn[cb][0], dn[cb][1], a, XBc[(8 * cb + g) * K4 + 4 * s + q]);
        }
#pragma unroll
        for (int cb = 0; cb < 8; ++cb)
#pragma unroll
            for (int e = 0; e < 2; ++e) dn[cb][e] = exp_neg(dn[cb][e], etab) * il;
        if (bj == bi) {                                      // diagonal tile: complete (both triangles), no mirror image
            const int dcol = lr - 2 * q;
#pragma unroll
            for (int cb = 0; cb < 8; ++cb)
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    if (dcol == 8 * cb + e) dn[cb][e] = dg;
        }
        double* drow = Cb + (size_t)(r0 + lr) * m + c0 + 2 * q;
#pragma unroll
        for (int cb = 0; cb < 8; ++cb) __stcs(reinterpret_cast<double2*>(drow + 8 * cb), make_double2(dn[cb][0], dn[cb][1]));
        if (bj != bi) {
            // mirror image, also straight from the fragments: entry (row g, column 2q + e) of an 8 x 8 block goes to output row
            // c0 + 8 cb + 2q + e, column r0 + 8 warp + g -- per store instruction the eight lanes with the same q write 64
            // contiguous bytes, the same segment size as the tile's own copy; no transposition through shared memory
            double* dt = Cb + (size_t)(c0 + 2 * q) * m + r0 + lr;
#pragma unroll
            for (int cb = 0; cb < 8; ++cb) {
                __stcs(dt + (size_t)(8 * cb) * m, dn[cb][0]);
                __stcs(dt + (size_t)(8 * cb + 1) * m, dn[cb][1]);
            }
        }
        __syncthreads();                                     // the next tile's column side is in place
    }
}

// SepiaDistCov type 2: S21[b][i][t] = exp(-sum_k beta_k (x_ik - xp_tk)^2) / lamz, (m x n) row-major.
// Round 2: same scheme as the row-block covariance build -- 64 x 64 tile per CTA, squared distances as the rank-(d+2) DMMA
// product (row side from X, column side from Xp), exp_neg fused, the tile stored straight from the accumulator fragments
// (64 contiguous bytes per row and store instruction) -- instead of scalar difference sums and libm exp per entry.
template <int KSC>
__global__ void __launch_bounds__(256, 4)
cross_cov_kernel(const double* __restrict__ X, int m, const double* __restrict__ Xp, int n, int d,
                 const double* __restrict__ beta, const double* __restrict__ lamz,
                 double* __restrict__ S21, int n_ct, int n_rt, int ct_per_cta)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int KS = KSC > 0 ? KSC : cov_ksteps(d), K4 = 4 * KS;
    double* XA = reinterpret_cast<double*>(smem_raw);      // [CT][K4] row side:    [x~, |x~|^2, 1, 0..]
    double* XB = XA + CT * K4;                             // [2][CT][K4] column side: [2 x~, -1, -|x~|^2, 0..] (double-buffered)
    double* etab = XB + 2 * CT * K4;                       // [ETAB]
    double* sbs = etab + ETAB;                             // [d]
    // CTA = (matrix b, 64-row block, run of ct_per_cta column tiles): prologue and row side once per CTA
    const int runs = (n_ct + ct_per_cta - 1) / ct_per_cta;
    const int per_b = n_rt * runs;
    const int b = blockIdx.x / per_b;
    const int tix = blockIdx.x - b * per_b;
    const int r0 = (tix / runs) * CT;
    const int ct0 = (tix % runs) * ct_per_cta, ct1 = min(n_ct, ct0 + ct_per_cta);
    const double* be = beta + (size_t)b * d;
    const double il = 1.0 / lamz[b];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    fill_exp_table(etab);
    if (tid >= 128 && tid < 128 + d) sbs[tid - 128] = sqrt(be[tid - 128]);
    __syncthreads();
    auto stage = [&](double* dst0, const double* P, int p0, int np, bool colside, int lr) {
        const bool in = p0 + lr < np;
        const double* src = P + (size_t)(in ? p0 + lr : 0) * d;
        double* dst = dst0 + lr * K4;
        double rr = 0.0;
        for (int k = 0; k < d; ++k) {
            const double x = in ? __ldg(src + k) * sbs[k] : 0.0;
            rr = fma(x, x, rr);
            dst[k] = colside ? 2.0 * x : x;
        }
        for (int k = d; k < K4; ++k) dst[k] = 0.0;
        if (in) {
            dst[d] = colside ? -1.0 : rr;
            dst[d + 1] = colside ? -rr : 1.0;
        }
    };
    if (tid < CT) stage(XA, X, r0, m, false, tid);
    else if (tid < 2 * CT) stage(XB + (ct0 & 1) * CT * K4, Xp, ct0 * CT, n, true, tid - CT);
    __syncthreads();
    const int lr = 8 * warp + g;
    const int r = r0 + lr;
    double* Sb = S21 + (size_t)b * m * n;
    const bool vec2 = (n % 2 == 0) && ((reinterpret_cast<uintptr_t>(S21) & 15) == 0);
    for (int ct = ct0; ct < ct1; ++ct) {
        const int c0 = ct * CT;
        const double* XBc = XB + (ct & 1) * CT * K4;
        if (ct + 1 < ct1 && tid >= 2 * CT && tid < 3 * CT) stage(XB + ((ct + 1) & 1) * CT * K4, Xp, c0 + CT, n, true, tid - 2 * CT);
        double dn[8][2];
#pragma unroll
        for (int cb = 0; cb < 8; ++cb) { dn[cb][0] = 0.0; dn[cb][1] = 0.0; }
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const double a = XA[lr * K4 + 4 * s + q];
#pragma unroll
            for (int cb = 0; cb < 8; ++cb) dmma884(dn[cb][0], dn[cb][1], a, XBc[(8 * cb + g) * K4 + 4 * s + q]);
        }
#pragma unroll
        for (int cb = 0; cb < 8; ++cb) {
            const double v0 = exp_neg(dn[cb][0], etab) * il, v1 = exp_neg(dn[cb][1], etab) * il;
            const int c = c0 + 8 * cb + 2 * q;
            if (r < m) {
                if (vec2 && c + 1 < n) __stcs(reinterpret_cast<double2*>(Sb + (size_t)r * n + c), make_double2(v0, v1));
                else {
                    if (c < n) Sb[(size_t)r * n + c] = v0;
                    if (c + 1 < n) Sb[(size_t)r * n + c + 1] = v1;
                }
            }
        }
        __syncthreads();                                     // the next tile's column side is in place
    }
}

// ---------------------------------------------------------------------------------------------
// (2) batched fused log-likelihood: one CTA (look-ahead schedule) or one thread-block cluster (CL) per matrix.
// ---------------------------------------------------------------------------------------------
template <bool CL>
__global__ void __launch_bounds__(NT, CL ? CL_CTAS_PER_SM : CTAS_PER_SM)
loglik_batched_kernel(const double* __restrict__ X, int m, int Mp, int d, const double* __restrict__ W,
                      long long w_stride, const double* __restrict__ beta, const double* __restrict__ lamz,
                      const double* __restrict__ diag_add, double* __restrict__ Lws, long long l_stride,
                      double* __restrict__ u_out, double* __restrict__ loglik, int* __restrict__ info)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = CL ? blockIdx.x / cluster_nctarank() : blockIdx.x;
    double ll;
    if constexpr (CL) {
        EvalSmem sm = carve_eval_smem(smem_raw, Mp, d);
        ll = eval_block_loglik<true>(sm, X, m, Mp, d, beta + (size_t)b * d, lamz[b], diag_add[b],
                                     W + (size_t)b * w_stride, Lws + (size_t)b * l_stride,
                                     u_out ? u_out + (size_t)b * Mp : nullptr, info ? info + b : nullptr);
    } else {
        LaSmem sm = carve_la_smem(smem_raw, Mp, d);
        const int rot = cta_role_rotation();
        ll = eval_block_loglik_la(sm, X, m, Mp, d, beta + (size_t)b * d, lamz[b], diag_add[b],
                                  W + (size_t)b * w_stride, Lws + (size_t)b * l_stride,
                                  u_out ? u_out + (size_t)b * Mp : nullptr, info ? info + b : nullptr, rot);
    }
    if (threadIdx.x == 0 && (!CL || cluster_ctarank() == 0)) loglik[b] = ll;
}

// packed factor -> dense lower-triangular (m x m row-major), for tests / inspection
__global__ void unpack_factor_kernel(const double* __restrict__ Lws, long long l_stride, int m, int Mp,
                                     double* __restrict__ Ld)
{
    const int b = blockIdx.y;
    const double* Lp = Lws + (size_t)b * l_stride;
    double* out = Ld + (size_t)b * m * m;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < (long long)m * m;
         idx += (long long)gridDim.x * blockDim.x) {
        int r = (int)(idx / m), c = (int)(idx - (long long)r * m);
        double v = 0.0;
        if (c <= r) {
            int kb = c >> 5, ks = (c >> 3) & 3, cc = c & 7;
            v = Lp[panel_off(kb, Mp) + (long long)ks * (Mp - 32 * kb) * 8 + (long long)(r - 32 * kb) * 8 + cc];
        }
        out[idx] = v;
    }
}

// test hook for the in-kernel exponential
__global__ void exp_neg_kernel(const double* __restrict__ y, double* __restrict__ out, int n)
{
    __shared__ double etab[ETAB];
    fill_exp_table(etab);
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = exp_neg(y[i], etab);
}

}  // namespace ggp

using namespace ggp;

extern "C" {

int ggp_cov_build_f64(const double* X, int m, int d, const double* beta, const double* lamz,
                      const double* diag_add, int B, double* C_out, void* stream)
{
    GGP_ARG(X && beta && lamz && diag_add && C_out, "null pointer");
    GGP_ARG(m > 0 && d > 0 && B > 0, "m, d, B must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    int nt = (m + CT - 1) / CT;
    int ntile = nt * (nt + 1) / 2;
    size_t smem = (size_t)(2 * CT * 4 * cov_ksteps(d) + CT * CT_LD + ETAB + d) * sizeof(double);
    GGP_ARG(smem <= 200 * 1024, "d too large for cov_build");
    auto run = [&](auto kern) -> int {
        GGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<dim3(ntile, B), 256, smem, st>>>(X, m, d, beta, lamz, diag_add, C_out, ntile);
        GGP_CUDA(cudaGetLastError());
        return GGP_OK;
    };
    // whole 64-row blocks and a 16-byte aligned output: the row-block kernel
    if (m % CT == 0 && (reinterpret_cast<uintptr_t>(C_out) & 15) == 0) {
        const size_t smem_r = (size_t)(3 * CT * 4 * cov_ksteps(d) + ETAB + d) * sizeof(double);
        auto run_rows = [&](auto kern) -> int {
            GGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_r));
            kern<<<dim3(nt, B), 256, smem_r, st>>>(X, m, d, beta, lamz, diag_add, C_out);
            GGP_CUDA(cudaGetLastError());
            return GGP_OK;
        };
        if (smem_r <= 200 * 1024) {
            switch (cov_ksteps(d)) {
                case 1: return run_rows(cov_build_rows_kernel<1>);
                case 2: return run_rows(cov_build_rows_kernel<2>);
                case 3: return run_rows(cov_build_rows_kernel<3>);
                case 4: return run_rows(cov_build_rows_kernel<4>);
                case 5: return run_rows(cov_build_rows_kernel<5>);
                default: return run_rows(cov_build_rows_kernel<0>);
            }
        }
    }
    switch (cov_ksteps(d)) {
        case 1: return run(cov_build_kernel<1>);
        case 2: return run(cov_build_kernel<2>);
        case 3: return run(cov_build_kernel<3>);
        case 4: return run(cov_build_kernel<4>);
        case 5: return run(cov_build_kernel<5>);
        default: return run(cov_build_kernel<0>);
    }
}

int ggp_cross_cov_f64(const double* X, int m, const double* Xp, int n, int d, const double* beta,
                      const double* lamz, int B, double* S21_out, void* stream)
{
    GGP_ARG(X && Xp && beta && lamz && S21_out, "null pointer");
    GGP_ARG(m > 0 && n > 0 && d > 0 && B > 0, "m, n, d, B must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)(3 * CT * 4 * cov_ksteps(d) + ETAB + d) * sizeof(double);
    GGP_ARG(smem <= 200 * 1024, "d too large for cross_cov");
    const int n_ct = (n + CT - 1) / CT, n_rt = (m + CT - 1) / CT;
    // runs of up to 8 column tiles per CTA (prologue and row side amortised), but at least ~4 CTAs per SM slot in total
    int ct_per_cta = 8;
    while (ct_per_cta > 1 && (long long)n_rt * B * ((n_ct + ct_per_cta - 1) / ct_per_cta) < 4LL * 592) ct_per_cta >>= 1;
    const long long nblk = (long long)n_rt * B * ((n_ct + ct_per_cta - 1) / ct_per_cta);
    GGP_ARG(nblk < (1LL << 31), "B * tiles(m, n) must be below 2^31 CTAs");
    auto run = [&](auto kern) -> int {
        GGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)nblk, 256, smem, st>>>(X, m, Xp, n, d, beta, lamz, S21_out, n_ct, n_rt, ct_per_cta);
        GGP_CUDA(cudaGetLastError());
        return GGP_OK;
    };
    switch (cov_ksteps(d)) {
        case 1: return run(cross_cov_kernel<1>);
        case 2: return run(cross_cov_kernel<2>);
        case 3: return run(cross_cov_kernel<3>);
        case 4: return run(cross_cov_kernel<4>);
        case 5: return run(cross_cov_kernel<5>);
        default: return run(cross_cov_kernel<0>);
    }
}

int ggp_debug_exp_neg_f64(const double* y, double* out, int n, void* stream)
{
    GGP_ARG(y && out && n > 0, "bad argument");
    exp_neg_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(y, out, n);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

long long ggp_factor_doubles(int m) { return packed_doubles(round_up32(m)); }

int ggp_padded_m(int m) { return round_up32(m); }

int ggp_loglik_batched_f64(const double* X, int m, int d, const double* W, long long w_stride,
                           const double* beta, const double* lamz, const double* diag_add, int B,
                           double* factor_ws, double* u_out, double* loglik_out, int* info_out, void* stream)
{
    GGP_ARG(X && W && beta && lamz && diag_add && factor_ws && loglik_out, "null pointer");
    GGP_ARG(m > 0 && d > 0 && B > 0, "m, d, B must be positive");
    const int Mp = round_up32(m);
    const size_t smem = eval_smem_bytes(Mp, d);
    if (smem > 227 * 1024) {
        set_error("ggp_loglik_batched_f64: m=%d d=%d needs %zu B of shared memory (> 227 KB)", m, d, smem);
        return GGP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int G = choose_cluster(B, round_up32(m));
    const long long ls = packed_doubles(Mp);
    if (G > 1) {
        GGP_CUDA(cudaFuncSetAttribute(loglik_batched_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int Gc = checked_cluster(loglik_batched_kernel<true>, G, smem);
        GGP_CUDA(cudaFuncSetAttribute(loglik_batched_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, eval_carveout_pct(smem)));
        GGP_CUDA(launch_maybe_cluster(loglik_batched_kernel<true>, dim3(B * Gc), dim3(NT), smem, st, Gc, X, m, Mp, d, W, w_stride,
                                      beta, lamz, diag_add, factor_ws, ls, u_out, loglik_out, info_out));
    } else {
        const size_t sla = la_smem_bytes(Mp, d);
        if (sla > 227 * 1024) {
            set_error("ggp_loglik_batched_f64: m=%d d=%d needs %zu B of shared memory (> 227 KB)", m, d, sla);
            return GGP_ERR_UNSUPPORTED;
        }
        GGP_CUDA(cudaFuncSetAttribute(loglik_batched_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sla));
        GGP_CUDA(cudaFuncSetAttribute(loglik_batched_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, eval_carveout_pct(sla)));
        loglik_batched_kernel<false><<<B, NT, sla, st>>>(X, m, Mp, d, W, w_stride, beta, lamz, diag_add, factor_ws, ls, u_out,
                                                         loglik_out, info_out);
    }
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_factor_unpack_f64(const double* factor_ws, int m, int B, double* L_dense, void* stream)
{
    GGP_ARG(factor_ws && L_dense && m > 0 && B > 0, "bad argument");
    const int Mp = round_up32(m);
    unpack_factor_kernel<<<dim3(64, B), 256, 0, (cudaStream_t)stream>>>(factor_ws, packed_doubles(Mp), m, Mp, L_dense);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
