// Sequential design (gladsgp_b200.design; DESIGN.md section 2 item 10): greedy ALC scores of candidate simulator runs
// and the rank-one update that conditions the emulator on a chosen run.
//
// For a (sample, PC) block b, V_x = L^-1 k(X, x) is the row ggp_predict_f64 writes for a design x (Mp columns, zero
// beyond m), and A_x (pitch Kp) holds one column per run chosen so far.  After t picks the posterior covariance between
// a reference point r and a candidate c is
//   Sigma_t(r, c) = k_b(r, c) - V_r . V_c - A_r . A_c,    k_b(x, x') = exp(-sum_k beta_bk (x_k - x'_k)^2) / lamUz_b,
// and adding c as a training row (nugget dadd_b) lowers the variance at r by Sigma_t(r, c)^2 / den_t(c), with
//   den_t(c) = 1/lamUz_b + dadd_b - |V_c|^2 - |A_c|^2   (the Schur complement of the enlarged S22, >= dadd_b > 0).
// design_score_kernel forms Sigma_t on the FP64 tensor cores, tile by tile (never written to memory), squares it and
// sums over r inside the CTA; design_reduce_kernel weights each block and sums the blocks in block order.
// design_condition_kernel appends column t of A:  a(x) = Sigma_t(x, c*) / sqrt(den_t(c*)).
// Every sum runs in a fixed order: identical calls give identical bits, and so does any split of the blocks over calls.
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int DS_NT = 128;       // 4 warps: a 2 x 2 grid of 32 x 32 warp tiles over a 64 x 64 (reference x candidate) tile
constexpr int DS_T = 64;
constexpr int DC_NT = 256;       // condition kernel: one warp per point
constexpr int DC_PTS = 64;       // points per CTA
constexpr int DR_NT = 256;       // row-variance kernel: one CTA per block

__host__ __device__ inline size_t ds_smem_bytes(int d) {
    return (size_t)(2 * DS_T * d + d + DS_T + 2 * DS_T) * sizeof(double);
}

// acc[i][cb] += sum_k P[row 8i+g][k] Q[col 8cb+g][k] over k < K (a multiple of 8) on DMMA.8x8x4.  ap / bp point at the
// lane's rows + 2q; the fragment scheme is pred_cov_kernel's (16-byte loads, k permuted identically on both sides).
__device__ __forceinline__ void ds_mma(double (&acc)[4][4][2], const double* const (&ap)[4], const double* const (&bp)[4],
                                       int K)
{
    double2 a[4], bb[4], an[4], bn[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const double2*>(ap[i]);
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) bb[cb] = *reinterpret_cast<const double2*>(bp[cb]);
    for (int k = 0; k < K; k += 8) {
        if (k + 8 < K) {
#pragma unroll
            for (int i = 0; i < 4; ++i) an[i] = *reinterpret_cast<const double2*>(ap[i] + k + 8);
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) bn[cb] = *reinterpret_cast<const double2*>(bp[cb] + k + 8);
        }
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int i = 0; i < 4; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].x, bb[cb].x);
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int i = 0; i < 4; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].y, bb[cb].y);
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = an[i];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) bb[cb] = bn[cb];
    }
}

// |V_x|^2 + |A_x|^2 over the first Mp and Kt columns, valid in every lane (lanes stride, then a butterfly)
__device__ __forceinline__ double ds_norm2(const double* __restrict__ v, int Mp, const double* __restrict__ a, int Kt)
{
    const int lane = threadIdx.x & 31;
    double s = 0.0;
    for (int k = lane; k < Mp; k += 32) s = fma(v[k], v[k], s);
    for (int k = lane; k < Kt; k += 32) s = fma(a[k], a[k], s);
    return warp_sum(s);
}

__device__ __forceinline__ double ds_kern(const double* __restrict__ x, const double* __restrict__ y,
                                          const double* __restrict__ be, int d, double inv_lamz)
{
    double dist = 0.0;
    for (int k = 0; k < d; ++k) {
        const double df = x[k] - y[k];
        dist = fma(be[k] * df, df, dist);
    }
    return exp(-dist) * inv_lamz;
}

// CTA (block b, candidate tile): part[b][c] = sum_r Sigma_t(r, c)^2 / den_t(c) for the tile's 64 candidates, over every
// reference point in tiles of 64.  Kt: the columns of A in use, rounded up to 8 (the rest of the pitch is not read).
__global__ void __launch_bounds__(DS_NT)
design_score_kernel(const double* __restrict__ XR, int n_ref, const double* __restrict__ XC, int n_cand, int d,
                    const double* __restrict__ beta, const double* __restrict__ lamz, const double* __restrict__ dadd,
                    const double* __restrict__ V_R, const double* __restrict__ V_C, int Mp,
                    const double* __restrict__ A_R, const double* __restrict__ A_C, int Kp, int Kt, int ntile,
                    double* __restrict__ part)
{
    extern __shared__ __align__(16) double ds_sm[];
    double* sc = ds_sm;                      // [64][d] candidate designs of the tile
    double* sr = sc + DS_T * d;              // [64][d] reference designs of the current row tile
    double* be = sr + DS_T * d;              // [d]
    double* den = be + d;                    // [64]
    double* red = den + DS_T;                // [2][64] column sums of the two row warps
    const int b = blockIdx.x / ntile;
    const int c0 = (blockIdx.x - b * ntile) * DS_T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int wr = warp >> 1, wc = warp & 1;
    const double il = 1.0 / lamz[b];
    const double* __restrict__ VRb = V_R + (size_t)b * n_ref * Mp;
    const double* __restrict__ VCb = V_C + (size_t)b * n_cand * Mp;
    const double* __restrict__ ARb = A_R + (size_t)b * n_ref * Kp;
    const double* __restrict__ ACb = A_C + (size_t)b * n_cand * Kp;
    for (int idx = tid; idx < DS_T * d; idx += DS_NT) {
        const int c = c0 + idx / d;
        sc[idx] = c < n_cand ? XC[(size_t)c0 * d + idx] : 0.0;
    }
    for (int k = tid; k < d; k += DS_NT) be[k] = beta[(size_t)b * d + k];
    for (int j = warp; j < DS_T; j += DS_NT / 32) {
        const int c = min(c0 + j, n_cand - 1);
        const double s = ds_norm2(VCb + (size_t)c * Mp, Mp, ACb + (size_t)c * Kp, Kt);
        if (lane == 0) den[j] = (il + dadd[b]) - s;
    }
    const double* bp[4];
    const double* bpa[4];
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) {
        const int c = min(c0 + 32 * wc + 8 * cb + g, n_cand - 1);
        bp[cb] = VCb + (size_t)c * Mp + 2 * q;
        bpa[cb] = ACb + (size_t)c * Kp + 2 * q;
    }
    double csum[4][2];
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) { csum[cb][0] = 0.0; csum[cb][1] = 0.0; }

    for (int r0 = 0; r0 < n_ref; r0 += DS_T) {
        __syncthreads();                                   // sr of the previous tile consumed (and sc, be, den visible)
        for (int idx = tid; idx < DS_T * d; idx += DS_NT) {
            const int r = r0 + idx / d;
            sr[idx] = r < n_ref ? XR[(size_t)r0 * d + idx] : 0.0;
        }
        __syncthreads();
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
        {
            const double* ap[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) ap[i] = VRb + (size_t)min(r0 + 32 * wr + 8 * i + g, n_ref - 1) * Mp + 2 * q;
            ds_mma(acc, ap, bp, Mp);
        }
        if (Kt > 0) {
            const double* ap[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) ap[i] = ARb + (size_t)min(r0 + 32 * wr + 8 * i + g, n_ref - 1) * Kp + 2 * q;
            ds_mma(acc, ap, bpa, Kt);
        }
        // epilogue: Sigma = k - acc, squared and summed over the lane's rows (i ascending, tiles ascending)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = 32 * wr + 8 * i + g;
            if (r0 + rl >= n_ref) continue;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int cl = 32 * wc + 8 * cb + 2 * q + e;
                    const double sg = ds_kern(sr + rl * d, sc + cl * d, be, d, il) - acc[i][cb][e];
                    csum[cb][e] = fma(sg, sg, csum[cb][e]);
                }
        }
    }
    // sum over the 8 row groups of the warp (butterfly), then the two row warps in order
#pragma unroll
    for (int cb = 0; cb < 4; ++cb)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double v = csum[cb][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            if (g == 0) red[wr * DS_T + 32 * wc + 8 * cb + 2 * q + e] = v;
        }
    __syncthreads();
    if (tid < DS_T && c0 + tid < n_cand)
        part[(size_t)b * n_cand + c0 + tid] = (red[tid] + red[DS_T + tid]) / den[tid];
}

// vsum[b] = sum_r max(s11_b - |V_r|^2 - |A_r|^2, 0): warp w takes rows w, w + 8, ... in order, the warps are summed in order
__global__ void __launch_bounds__(DR_NT)
design_rowvar_kernel(int n_ref, const double* __restrict__ s11, const double* __restrict__ V_R, int Mp,
                     const double* __restrict__ A_R, int Kp, int t, double* __restrict__ vsum)
{
    __shared__ double ws[DR_NT / 32];
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double sb = s11[b];
    double acc = 0.0;
    for (int r = warp; r < n_ref; r += DR_NT / 32) {
        const size_t row = (size_t)b * n_ref + r;
        const double s = ds_norm2(V_R + row * Mp, Mp, A_R + row * Kp, t);
        acc += fmax(sb - s, 0.0);
    }
    if (lane == 0) ws[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0.0;
        for (int w = 0; w < DR_NT / 32; ++w) v += ws[w];
        vsum[b] = v;
    }
}

// score[c] (c < n_cand) and imse (index n_cand): start value (0, or the output when accumulate) + sum_b wgt[b] * x_b, b
// ascending.  A null score skips the candidates.
__global__ void design_reduce_kernel(const double* __restrict__ part, const double* __restrict__ vsum,
                                     const double* __restrict__ wgt, int B, int n_cand, int accumulate,
                                     double* __restrict__ score, double* __restrict__ imse)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cand && score) {
        double acc = accumulate ? score[c] : 0.0;
        for (int b = 0; b < B; ++b) acc += wgt[b] * part[(size_t)b * n_cand + c];
        score[c] = acc;
    } else if (c == n_cand) {
        double acc = accumulate ? imse[0] : 0.0;
        for (int b = 0; b < B; ++b) acc += wgt[b] * vsum[b];
        imse[0] = acc;
    }
}

// Column t of A for every point of block b: a(x) = (k_b(x, c*) - V_x . V_c* - A_x . A_c*) / sqrt(den_t(c*)), the dot
// products over the Mp columns of V and the t columns of A already written.  Points p < n_r are reference points, the
// rest candidates (n_r = 0 when the reference set is the candidate set).
__global__ void __launch_bounds__(DC_NT)
design_condition_kernel(const double* __restrict__ XR, int n_ref, int n_r, const double* __restrict__ XC, int n_cand, int d,
                        const double* __restrict__ beta, const double* __restrict__ lamz, const double* __restrict__ dadd,
                        const double* __restrict__ V_R, const double* __restrict__ V_C, int Mp,
                        double* A_R, double* A_C, int Kp, int t, int cstar, int ntile)
{
    __shared__ double s_isd;
    const int b = blockIdx.x / ntile;
    const int p0 = (blockIdx.x - b * ntile) * DC_PTS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int npts = n_r + n_cand;
    const double il = 1.0 / lamz[b];
    const double* __restrict__ vs = V_C + ((size_t)b * n_cand + cstar) * Mp;
    const double* as = A_C + ((size_t)b * n_cand + cstar) * Kp;      // A is read and written: no __restrict__
    const double* __restrict__ xs = XC + (size_t)cstar * d;
    const double* __restrict__ be = beta + (size_t)b * d;
    if (warp == 0) {
        const double s = ds_norm2(vs, Mp, as, t);
        if (lane == 0) s_isd = 1.0 / sqrt((il + dadd[b]) - s);
    }
    __syncthreads();
    const double isd = s_isd;
    for (int p = p0 + warp; p < min(p0 + DC_PTS, npts); p += DC_NT / 32) {
        const bool ref = p < n_r;
        const size_t row = ref ? (size_t)b * n_ref + p : (size_t)b * n_cand + (p - n_r);
        const double* __restrict__ v = (ref ? V_R : V_C) + row * Mp;
        double* a = (ref ? A_R : A_C) + row * Kp;
        const double* __restrict__ x = ref ? XR + (size_t)p * d : XC + (size_t)(p - n_r) * d;
        double s = 0.0;
        for (int k = lane; k < Mp; k += 32) s = fma(v[k], vs[k], s);
        for (int k = lane; k < t; k += 32) s = fma(a[k], as[k], s);
        s = warp_sum(s);
        if (lane == 0) a[t] = (ds_kern(x, xs, be, d, il) - s) * isd;
    }
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_design_workspace_bytes(int n_cand, int B)
{
    if (n_cand <= 0 || B <= 0) return -1;
    return ((long long)B * n_cand + B) * (long long)sizeof(double);
}

static const char* ds_check(int n_ref, int n_cand, int d, int m, int Kp, int B)
{
    if (n_ref <= 0 || n_cand <= 0 || d <= 0 || m <= 0 || Kp <= 0 || B <= 0)
        return "n_ref, n_cand, d, m, Kp and B must be positive";
    if (Kp % 8 != 0) return "Kp must be a multiple of 8";
    if (m > 8192) return "m must be <= 8192";
    return nullptr;
}

int ggp_design_score_f64(const double* XR, int n_ref, const double* XC, int n_cand, int d, const double* beta,
                         const double* lamz, const double* dadd, const double* s11, const double* wgt, const double* V_R,
                         const double* V_C, int m, const double* A_R, const double* A_C, int Kp, int t, int B,
                         int accumulate, double* score_out, double* imse_out, void* workspace, long long workspace_bytes,
                         void* stream)
{
    GGP_ARG(XR && XC && beta && lamz && dadd && s11 && wgt && V_R && V_C && A_R && A_C && imse_out && workspace,
            "null pointer");
    const char* bad = ds_check(n_ref, n_cand, d, m, Kp, B);
    GGP_ARG(!bad, bad);
    GGP_ARG(t >= 0 && t <= Kp, "t must be in [0, Kp]");
    const long long ntile = (n_cand + DS_T - 1) / DS_T;
    GGP_ARG(ntile * B < (1LL << 31), "B * ceil(n_cand / 64) must be below 2^31");
    const long long need = ggp_design_workspace_bytes(n_cand, B);
    GGP_ARG(workspace_bytes >= need, "workspace too small");
    const size_t smem = ds_smem_bytes(d);
    if (smem > 200 * 1024) {
        set_error("ggp_design_score_f64: d=%d needs %zu B of shared memory (> 200 KB)", d, smem);
        return GGP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int Mp = round_up32(m);
    double* part = reinterpret_cast<double*>(workspace);
    double* vsum = part + (size_t)B * n_cand;
    if (score_out) {
        GGP_CUDA(cudaFuncSetAttribute(design_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        design_score_kernel<<<(unsigned)(ntile * B), DS_NT, smem, st>>>(XR, n_ref, XC, n_cand, d, beta, lamz, dadd, V_R, V_C,
                                                                          Mp, A_R, A_C, Kp, (t + 7) & ~7, (int)ntile, part);
        GGP_CUDA(cudaGetLastError());
    }
    design_rowvar_kernel<<<B, DR_NT, 0, st>>>(n_ref, s11, V_R, Mp, A_R, Kp, t, vsum);
    GGP_CUDA(cudaGetLastError());
    design_reduce_kernel<<<(n_cand + 1 + 127) / 128, 128, 0, st>>>(part, vsum, wgt, B, n_cand, accumulate, score_out,
                                                                   imse_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_design_condition_f64(const double* XR, int n_ref, const double* XC, int n_cand, int d, const double* beta,
                             const double* lamz, const double* dadd, const double* V_R, const double* V_C, int m,
                             double* A_R, double* A_C, int Kp, int t, int B, int index, void* stream)
{
    GGP_ARG(XR && XC && beta && lamz && dadd && V_R && V_C && A_R && A_C, "null pointer");
    const char* bad = ds_check(n_ref, n_cand, d, m, Kp, B);
    GGP_ARG(!bad, bad);
    GGP_ARG(t >= 0 && t < Kp, "t must be in [0, Kp)");
    GGP_ARG(index >= 0 && index < n_cand, "index out of range [0, n_cand)");
    const bool same = XR == XC && V_R == V_C && A_R == A_C;
    GGP_ARG(!same || n_ref == n_cand, "a shared reference / candidate set needs n_ref == n_cand");
    const int n_r = same ? 0 : n_ref;
    const long long ntile = ((long long)n_r + n_cand + DC_PTS - 1) / DC_PTS;
    GGP_ARG(ntile * B < (1LL << 31), "B * ceil((n_ref + n_cand) / 64) must be below 2^31");
    design_condition_kernel<<<(unsigned)(ntile * B), DC_NT, 0, (cudaStream_t)stream>>>(
        XR, n_ref, n_r, XC, n_cand, d, beta, lamz, dadd, V_R, V_C, round_up32(m), A_R, A_C, Kp, t, index, (int)ntile);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
