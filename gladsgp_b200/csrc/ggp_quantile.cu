// Exact posterior quantile fields over any number of samples (up to 16 384), any list of quantiles and up to 32 PCs.
//
// The post-processing every caller does after get_y (assess_all_models.py:493-500, plot_test_error.py:81-87; SURVEY 8f
// rank 1) without writing the nsamp x npred x n_y per-sample fields: for design t and output c, over the samples s,
//   y_s = (w[s][t] . K[:,c]) * sd[c] + mu[c],   z_s = y_s + sd[c] * noise[s][t]   (z_s = y_s without noise)
//   ymean = mean_s y_s  (FP64 sum in a fixed order, rounded once),   yq[k] = np.quantile(z, q[k]) on the float32 z_s.
// y_s and z_s are formed exactly as reconstruct_kernel and `y + sd * noise` form them (an fmaf chain over the PCs from
// 0, then an unfused multiply-add; the library is compiled with -fmad=false), so the results can be checked bit for bit.
//
// One CTA per (design, tile of C columns); C is chosen so that the tile's nsamp x C keys fit QT_SMEM_TARGET.
//   Phase 1: every thread holds the PC weights of one sample in registers and runs over the tile's columns, whose K
//            entries, sd and mu are read from shared memory as broadcasts; z_s is stored as an order-preserving
//            uint32 key (sign bit set for positives, all bits inverted for negatives, every NaN as 0xffffffff).
//   Phase 2: one warp per column.  The mean and a NaN check take one pass over the column; the order statistic of
//            rank i is found by a 32-step bitwise search on the keys (count of keys below a candidate, one warp
//            reduction per step), rank i + 1 by one more pass (count <= x_i and the smallest key above x_i).
//   Phase 3: NumPy's float32 linear interpolation between the two, as in numpy.lib._function_base_impl._lerp.
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int QT_NT = 256;
constexpr int QT_NW = QT_NT / 32;
constexpr int QT_MAXQ = 32;
constexpr int QT_MAXSAMP = 16384;
constexpr int QT_CMAX = 256;                       // columns per tile
constexpr size_t QT_SMEM_TARGET = 96 * 1024;       // two CTAs per SM while a tile's keys fit

// Ranks and weights of every quantile, computed on the host as NumPy does for a float32 array:
//   pos = float32(n - 1) * float32(q),  i = floor(pos),  j = min(i + 1, n - 1),  t = pos - i  (all float32)
struct QuantileRanks {
    int nq;
    int i[QT_MAXQ];
    int j[QT_MAXQ];
    float t[QT_MAXQ];
};

__device__ __forceinline__ unsigned order_key(float z)
{
    const unsigned b = __float_as_uint(z);
    return (z != z) ? 0xffffffffu : ((b & 0x80000000u) ? ~b : (b | 0x80000000u));
}

__device__ __forceinline__ float key_value(unsigned k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// the key of rank r (0-based) among kc[0, n): the largest x with count(key < x) <= r, built bit by bit
__device__ unsigned select_rank(const unsigned* __restrict__ kc, int n, int r, int lane)
{
    unsigned x = 0u;
    for (int b = 31; b >= 0; --b) {
        const unsigned cand = x | (1u << b);
        int cnt = 0;
#pragma unroll 4
        for (int s = lane; s < n; s += 32) cnt += (kc[s] < cand) ? 1 : 0;
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (cnt <= r) x = cand;
    }
    return x;
}

// the key of rank r + 1 given the key x of rank r
__device__ unsigned next_rank(const unsigned* __restrict__ kc, int n, int r, unsigned x, int lane)
{
    int le = 0;
    unsigned above = 0xffffffffu;
#pragma unroll 4
    for (int s = lane; s < n; s += 32) {
        const unsigned k = kc[s];
        le += (k <= x) ? 1 : 0;
        if (k > x) above = min(above, k);
    }
    le = __reduce_add_sync(0xffffffffu, le);
    above = __reduce_min_sync(0xffffffffu, above);
    return le > r + 1 ? x : above;
}

template <int PUMAX>
__global__ void __launch_bounds__(QT_NT, 2)
reconstruct_quantiles_kernel(const float* __restrict__ w, const float* __restrict__ K, const float* __restrict__ sd,
                             int sd_len, const float* __restrict__ mu, int mu_len, const float* __restrict__ noise,
                             int nsamp, int npred, int pu, long long n_y, int C, int SL, long long ntiles,
                             const QuantileRanks qr, float* __restrict__ ymean, float* __restrict__ yq)
{
    constexpr int KLD = PUMAX + 4;                                    // K[:, c] (PUMAX), sd[c], mu[c], padding
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* kt = reinterpret_cast<float*>(smem_raw);                   // [C][KLD]
    unsigned* keys = reinterpret_cast<unsigned*>(kt + (size_t)C * KLD);  // [C][nsamp]
    float* yb = reinterpret_cast<float*>(keys + (size_t)C * nsamp);   // [C][nsamp] y_s, only with noise
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sl = tid % SL, cg = tid / SL, CG = QT_NT / SL;          // phase 1: sample lane, column group
    const long long ntask = (long long)npred * ntiles;
    const size_t field = (size_t)npred * n_y;

    for (long long task = blockIdx.x; task < ntask; task += gridDim.x) {
        const int t = (int)(task / ntiles);
        const long long c0 = (task - (long long)t * ntiles) * C;
        const int nc = (int)min((long long)C, n_y - c0);
        __syncthreads();                                              // the previous tile is done with kt / keys
        for (int idx = tid; idx < KLD * C; idx += QT_NT) {
            const int p = idx / C, c = idx - p * C;                   // consecutive threads read consecutive columns
            const long long col = c0 + c;
            float v = 0.f;
            if (c < nc) {
                if (p < pu) v = __ldg(K + (size_t)p * n_y + col);
                else if (p == PUMAX) v = sd_len == 1 ? sd[0] : sd[col];
                else if (p == PUMAX + 1) v = mu_len == 1 ? mu[0] : mu[col];
            }
            kt[c * KLD + p] = v;
        }
        __syncthreads();

        // ---- phase 1: keys (and y_s when z_s differs from it)
        for (int s0 = 0; s0 < nsamp; s0 += SL) {
            const int s = s0 + sl;
            if (s >= nsamp) break;
            float wr[PUMAX];
            const float* ws = w + ((size_t)s * npred + t) * pu;
#pragma unroll
            for (int p = 0; p < PUMAX; ++p) wr[p] = (p < pu) ? __ldg(ws + p) : 0.f;
            const float e = noise ? __ldg(noise + (size_t)s * npred + t) : 0.f;
#pragma unroll 2
            for (int c = cg; c < nc; c += CG) {
                const float* kc = kt + c * KLD;
                float acc = 0.f;
#pragma unroll
                for (int p4 = 0; p4 < PUMAX; p4 += 4) {
                    const float4 k4 = *reinterpret_cast<const float4*>(kc + p4);
                    acc = fmaf(wr[p4 + 0], k4.x, acc);
                    acc = fmaf(wr[p4 + 1], k4.y, acc);
                    acc = fmaf(wr[p4 + 2], k4.z, acc);
                    acc = fmaf(wr[p4 + 3], k4.w, acc);
                }
                const float2 sm = *reinterpret_cast<const float2*>(kc + PUMAX);
                const float y = acc * sm.x + sm.y;
                if (noise) {
                    keys[(size_t)c * nsamp + s] = order_key(y + sm.x * e);
                    yb[(size_t)c * nsamp + s] = y;
                } else {
                    keys[(size_t)c * nsamp + s] = order_key(y);
                }
            }
        }
        __syncthreads();

        // ---- phases 2 and 3: one warp per column
        for (int c = warp; c < nc; c += QT_NW) {
            const unsigned* kc = keys + (size_t)c * nsamp;
            const float* yc = yb + (size_t)c * nsamp;
            const size_t o = (size_t)t * n_y + c0 + c;
            double sum = 0.0;
            bool nan = false;
            for (int s = lane; s < nsamp; s += 32) {
                const unsigned k = kc[s];
                nan |= (k == 0xffffffffu);
                sum += (double)(noise ? yc[s] : key_value(k));
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
            nan = __any_sync(0xffffffffu, nan);
            if (ymean && lane == 0) ymean[o] = (float)(sum / (double)nsamp);
            int ri_prev = -1, rj_prev = -1;
            unsigned xi = 0u, xj = 0u;
            for (int k = 0; k < qr.nq; ++k) {
                float r = __uint_as_float(0x7fffffffu);               // NumPy: a NaN sample makes every quantile NaN
                if (!nan) {
                    const int ri = qr.i[k], rj = qr.j[k];
                    if (ri != ri_prev) {
                        xi = (ri == rj_prev) ? xj : select_rank(kc, nsamp, ri, lane);
                        xj = (rj == ri) ? xi : next_rank(kc, nsamp, ri, xi, lane);
                    }
                    ri_prev = ri;
                    rj_prev = rj;
                    const float a = key_value(xi), b = key_value(xj), tt = qr.t[k];
                    const float d = b - a;
                    r = (tt >= 0.5f) ? b - d * (1.f - tt) : a + d * tt;
                }
                if (lane == 0) yq[(size_t)k * field + o] = r;
            }
        }
    }
}

template <int PUMAX>
static int launch_quantiles(const float* w, const float* K, const float* sd, int sd_len, const float* mean, int mean_len,
                            const float* noise, int nsamp, int npred, int pu, long long n_y, const QuantileRanks& qr,
                            float* ymean, float* yq, cudaStream_t st)
{
    const size_t per_col = (size_t)nsamp * sizeof(unsigned) * (noise ? 2 : 1) + (PUMAX + 4) * sizeof(float);
    long long C = (long long)(QT_SMEM_TARGET / per_col);
    if (C < 1) C = 1;
    if (C > QT_CMAX) C = QT_CMAX;
    if (C > n_y) C = n_y;
    if (C > QT_NW) C -= C % QT_NW;                                    // whole warps in phase 2
    const size_t smem = (size_t)C * per_col;
    int SL = 32;                                                      // sample lanes: a power of two >= nsamp, <= QT_NT
    while (SL < QT_NT && SL < nsamp) SL <<= 1;
    const long long ntiles = (n_y + C - 1) / C;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long ntask = ntiles * npred;
    const long long gmax = 64LL * sms;
    const unsigned grid = (unsigned)(ntask < gmax ? ntask : gmax);
    GGP_CUDA(cudaFuncSetAttribute(reconstruct_quantiles_kernel<PUMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    reconstruct_quantiles_kernel<PUMAX><<<grid, QT_NT, smem, st>>>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu,
                                                                   n_y, (int)C, SL, ntiles, qr, ymean, yq);
    return GGP_OK;
}

}  // namespace ggp

using namespace ggp;

extern "C" {

int ggp_reconstruct_quantiles_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                                  int mean_len, const float* noise, int nsamp, int npred, int pu, long long n_y,
                                  const double* q_host, int nq, float* ymean_out, float* yq_out, void* stream)
{
    GGP_ARG(w && K && sd && mean && q_host && yq_out, "null pointer");
    GGP_ARG(nsamp > 0 && npred > 0 && pu > 0 && n_y > 0, "nsamp, npred, pu, n_y must be positive");
    GGP_ARG((sd_len == 1 || sd_len == n_y) && (mean_len == 1 || mean_len == n_y), "sd/mean length must be 1 or n_y");
    GGP_ARG(nq >= 1 && nq <= QT_MAXQ, "nq must be in [1, 32]");
    for (int k = 0; k < nq; ++k) GGP_ARG(q_host[k] >= 0.0 && q_host[k] <= 1.0, "quantiles must be in [0, 1]");
    if (nsamp > QT_MAXSAMP || pu > 32) {
        set_error("ggp_reconstruct_quantiles_f32: unsupported (nsamp=%d > %d or pu=%d > 32)", nsamp, QT_MAXSAMP, pu);
        return GGP_ERR_UNSUPPORTED;
    }
    QuantileRanks qr;
    qr.nq = nq;
    for (int k = 0; k < nq; ++k) {
        const float pos = (float)(nsamp - 1) * (float)q_host[k];
        const int i = (int)floorf(pos);
        qr.i[k] = i;
        qr.j[k] = i + 1 < nsamp ? i + 1 : nsamp - 1;
        qr.t[k] = pos - (float)i;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (pu <= 4) rc = launch_quantiles<4>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, qr, ymean_out, yq_out, st);
    else if (pu <= 8) rc = launch_quantiles<8>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, qr, ymean_out, yq_out, st);
    else if (pu <= 12) rc = launch_quantiles<12>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, qr, ymean_out, yq_out, st);
    else if (pu <= 16) rc = launch_quantiles<16>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, qr, ymean_out, yq_out, st);
    else if (pu <= 24) rc = launch_quantiles<24>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, qr, ymean_out, yq_out, st);
    else rc = launch_quantiles<32>(w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, qr, ymean_out, yq_out, st);
    if (rc != GGP_OK) return rc;
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
