// History matching (gladsgp_b200.history; DESIGN.md section 2 item 11): the implausibility of every input point against
// every observed output, reduced to the `order` largest values and a count over the cutoff per point.
//
// For posterior sample s the predictive means mu (pu) and variances v (pu) of the PC weights at a point come from
// ggp_predict_f64 (block s * pu + j).  hm_mix_kernel forms the mixture over the samples,
//   m_j = (1/S) sum_s mu_sj,   M_jk = (1/S) sum_s [delta_jk max(v_sj, 0) + (mu_sj - m_j)(mu_sk - m_k)],
// and writes two feature rows per point: a_e = [1, m_1 .. m_pu] and a_v = [M_jj and 2 M_jk (j < k), packed; 1].  With the
// output-side rows b_e = [r_i, -K_1i .. -K_pu,i] and b_v = [K_ji K_ki, packed the same way; c_i] (c_i = rho + tau_i^2 +
// delta_i^2), e_i = a_e . b_e and V_i = a_v . b_v, and I_i = |e_i| / sqrt(V_i).  hm_pair_kernel forms both products on
// the FP64 tensor cores (DMMA.8x8x4, the fragment scheme of design_score_kernel) for a 64-point tile against 64-output
// tiles of one slab of the outputs, building b_e and b_v in shared memory from K_O; e and V are never written.  Its
// epilogue counts I_i > cutoff and keeps, per point, the `order` largest I_i (NaN counted as +inf); hm_merge_kernel
// merges the slabs.  A top list of a multiset and an integer count do not depend on how the outputs are split, and every
// e_i, V_i is the same sum in the same order wherever its tile runs: identical calls give identical bits, and so does
// any split of the points over calls.
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int HM_NT = 128;         // 4 warps: a 2 x 2 grid of 32 x 32 warp tiles over a 64 x 64 (point x output) tile
constexpr int HM_T = 64;
constexpr int HM_FVC = 64;         // columns of b_v built in shared memory at a time
constexpr int HM_MAXPU = 32;
constexpr int HM_MAXORD = 8;
constexpr int HM_HOLD = 8;         // threads that hold columns of one row: 2 column warps x 4 lanes
constexpr int HM_MIX_NT = 256;     // mixture kernel: one warp per point
constexpr int HM_TARGET_CTAS = 592;   // 148 SMs x 4: the output slabs are chosen to give at least this many CTAs

__host__ __device__ inline int hm_fe(int pu) { return (pu + 1 + 7) & ~7; }
__host__ __device__ inline int hm_npair(int pu) { return pu * (pu + 1) / 2; }
__host__ __device__ inline int hm_fv(int pu) { return (hm_npair(pu) + 1 + 7) & ~7; }
// shared row pitch (doubles) of a 16-byte fragment load: = 8 mod 16, so the 8 lanes of a phase hit distinct banks
__host__ __device__ inline int hm_pitch(int f) { return (f & 15) ? f : f + 8; }

__host__ inline int hm_nslab(int n, int n_o)
{
    const long long tp = ((long long)n + HM_T - 1) / HM_T, to = ((long long)n_o + HM_T - 1) / HM_T;
    const long long want = (HM_TARGET_CTAS + tp - 1) / tp;
    return (int)(want < to ? want : to);
}

__host__ inline size_t hm_smem_bytes(int pu, int order)
{
    return (size_t)(HM_T * hm_pitch(hm_fe(pu)) + HM_T * hm_pitch(HM_FVC) + pu * HM_T + 2 * HM_T +
                    HM_T * HM_HOLD * order) * sizeof(double) + (size_t)2 * HM_T * sizeof(int) +
           (size_t)2 * hm_npair(pu);
}

// I = |e| / sqrt(V): +inf for V = 0 and e != 0, 0 for V = 0 and e = 0, a NaN counted as +inf
__device__ __forceinline__ double hm_impl(double e, double V)
{
    if (V == 0.0) return e == 0.0 ? 0.0 : INFINITY;
    const double I = fabs(e) / sqrt(V);
    return I != I ? INFINITY : I;
}

// I > t decided from e^2 against tv = t^2 V where the gap exceeds every rounding: 1 (above), -1 (not above), 0 (compute
// I).  Only normal-range operands are decided.
__device__ __forceinline__ int hm_cmp(double e2, double tv)
{
    if (e2 >= 1e-250 && e2 <= 1e250 && tv >= 1e-250 && tv <= 1e250) {
        if (e2 > tv * (1.0 + 1e-9)) return 1;
        if (e2 < tv * (1.0 - 1e-9)) return -1;
    }
    return 0;
}

// insert v (> L[ord-1]) into the descending list L; equal values keep their order.  Returns the new L[ord-1].
__device__ __forceinline__ double hm_insert(double* L, int ord, double v)
{
    int k = ord - 1;
    while (k > 0 && L[k - 1] < v) { L[k] = L[k - 1]; --k; }
    L[k] = v;
    return L[ord - 1];
}

// acc[i][cb] += sum_k P[row 8i+g][k] Q[col 8cb+g][k] over k < K (a multiple of 8): ds_mma of ggp_design.cu without the
// register double buffer (two accumulators are live here).
__device__ __forceinline__ void hm_mma(double (&acc)[4][4][2], const double* const (&ap)[4], const double* const (&bp)[4],
                                       int K)
{
#pragma unroll 1
    for (int k = 0; k < K; k += 8) {
        double2 a[4], bb[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const double2*>(ap[i] + k);
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) bb[cb] = *reinterpret_cast<const double2*>(bp[cb] + k);
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int i = 0; i < 4; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].x, bb[cb].x);
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
            for (int i = 0; i < 4; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].y, bb[cb].y);
    }
}

// One warp per point: lane j owns PC j.  ae (n, Fe), av (n, Fv) with zero padding.
__global__ void __launch_bounds__(HM_MIX_NT)
hm_mix_kernel(const double* __restrict__ mean, const double* __restrict__ var, int S, int pu, int n,
              double* __restrict__ ae, int Fe, double* __restrict__ av, int Fv)
{
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * (HM_MIX_NT / 32) + (threadIdx.x >> 5);
    if (p >= n) return;
    const bool own = lane < pu;
    double m = 0.0;
    if (own)
        for (int s = 0; s < S; ++s) m += mean[((size_t)s * pu + lane) * n + p];
    m /= S;
    double acc[HM_MAXPU];
#pragma unroll
    for (int k = 0; k < HM_MAXPU; ++k) acc[k] = 0.0;
    double vs = 0.0;
    for (int s = 0; s < S; ++s) {
        const size_t at = ((size_t)s * pu + (own ? lane : 0)) * n + p;
        const double d = own ? mean[at] - m : 0.0;
        if (own) vs += fmax(var[at], 0.0);
#pragma unroll
        for (int k = 0; k < HM_MAXPU; ++k) {
            if (k >= pu) break;
            acc[k] = fma(d, __shfl_sync(0xffffffffu, d, k), acc[k]);
        }
    }
    double* __restrict__ e = ae + (size_t)p * Fe;
    double* __restrict__ v = av + (size_t)p * Fv;
    const int P = hm_npair(pu);
    if (own) {
        e[1 + lane] = m;
        const int row = lane * pu - lane * (lane - 1) / 2 - lane;      // packed index of (j, k) is row + k, k >= j
#pragma unroll
        for (int k = 0; k < HM_MAXPU; ++k) {
            if (k >= pu) break;
            if (k == lane) v[row + k] = (acc[k] + vs) / S;
            else if (k > lane) v[row + k] = (2.0 * acc[k]) / S;
        }
    }
    if (lane == 0) { e[0] = 1.0; v[P] = 1.0; }
    for (int f = pu + 1 + lane; f < Fe; f += 32) e[f] = 0.0;
    for (int f = P + 1 + lane; f < Fv; f += 32) v[f] = 0.0;
}

// CTA (point tile, output slab): the top `order` I and the count over the cutoff of each of the tile's 64 points over the
// slab's outputs, to top (nslab, n, order) and cnt (nslab, n).
__global__ void __launch_bounds__(HM_NT)
hm_pair_kernel(const double* __restrict__ ae, int Fe, const double* __restrict__ av, int Fv, int n, int pu,
               const double* __restrict__ K_O, const double* __restrict__ r, const double* __restrict__ c, int n_o,
               int order, double cutoff, int ntp, int nslab, double* __restrict__ top, int* __restrict__ cnt)
{
    extern __shared__ __align__(16) double hm_sm[];
    const int pe = hm_pitch(Fe), pv = hm_pitch(HM_FVC);
    double* se = hm_sm;                        // [64][pe] b_e of the output tile
    double* sv = se + HM_T * pe;               // [64][pv] one chunk of b_v
    double* sk = sv + HM_T * pv;               // [pu][64] K_O of the tile
    double* sr = sk + pu * HM_T;               // [64] r
    double* sc = sr + HM_T;                    // [64] c
    double* tl = sc + HM_T;                    // [64 rows][8 holders][order] top lists
    int* red = reinterpret_cast<int*>(tl + HM_T * HM_HOLD * order);   // [2][64] counts of the two column warps
    unsigned char* pj = reinterpret_cast<unsigned char*>(red + 2 * HM_T);
    const int P = hm_npair(pu);
    unsigned char* pk = pj + P;

    const int slab = blockIdx.x / ntp;
    const int x0 = (blockIdx.x - slab * ntp) * HM_T;
    const int nto = (n_o + HM_T - 1) / HM_T;
    const int t_beg = (int)((long long)slab * nto / nslab), t_end = (int)((long long)(slab + 1) * nto / nslab);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int wr = warp >> 1, wc = warp & 1;
    const int hold = wc * 4 + q;
    const double cut2 = cutoff * cutoff;

    for (int j = tid; j < pu; j += HM_NT) {
        const int row = j * pu - j * (j - 1) / 2 - j;
        for (int k = j; k < pu; ++k) { pj[row + k] = (unsigned char)j; pk[row + k] = (unsigned char)k; }
    }
    for (int idx = tid; idx < HM_T * HM_HOLD * order; idx += HM_NT) tl[idx] = -1.0;   // below every I (I >= 0)
    const double* ape[4];
    const double* apv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int x = min(x0 + 32 * wr + 8 * i + g, n - 1);
        ape[i] = ae + (size_t)x * Fe + 2 * q;
        apv[i] = av + (size_t)x * Fv + 2 * q;
    }
    const double* bpe[4];
    const double* bpv[4];
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) {
        const int o = 32 * wc + 8 * cb + g;
        bpe[cb] = se + o * pe + 2 * q;
        bpv[cb] = sv + o * pv + 2 * q;
    }
    double th[4];                              // the lane's current order-th largest I of each of its rows
    int nover[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { th[i] = -1.0; nover[i] = 0; }

    for (int t = t_beg; t < t_end; ++t) {
        const int o0 = t * HM_T;
        __syncthreads();                                     // the previous tile's se / sv / sk consumed
        for (int idx = tid; idx < pu * HM_T; idx += HM_NT) {
            const int j = idx / HM_T, o = o0 + idx - j * HM_T;
            sk[idx] = o < n_o ? K_O[(size_t)j * n_o + o] : 0.0;
        }
        for (int o = tid; o < HM_T; o += HM_NT) {
            sr[o] = o0 + o < n_o ? r[o0 + o] : 0.0;
            sc[o] = o0 + o < n_o ? c[o0 + o] : 0.0;
        }
        __syncthreads();
        for (int idx = tid; idx < HM_T * Fe; idx += HM_NT) {
            const int o = idx / Fe, f = idx - o * Fe;
            se[o * pe + f] = f == 0 ? sr[o] : (f <= pu ? -sk[(f - 1) * HM_T + o] : 0.0);
        }
        double acc_e[4][4][2], acc_v[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                acc_e[i][cb][0] = 0.0; acc_e[i][cb][1] = 0.0;
                acc_v[i][cb][0] = 0.0; acc_v[i][cb][1] = 0.0;
            }
        for (int f0 = 0; f0 < Fv; f0 += HM_FVC) {
            const int w = min(HM_FVC, Fv - f0);
            if (f0 > 0) __syncthreads();                     // the previous chunk of sv consumed
            for (int idx = tid; idx < HM_T * w; idx += HM_NT) {
                const int o = idx / w, f = f0 + idx - o * w;
                double x = 0.0;
                if (f < P) x = sk[pj[f] * HM_T + o] * sk[pk[f] * HM_T + o];
                else if (f == P) x = sc[o];
                sv[o * pv + (f - f0)] = x;
            }
            __syncthreads();
            if (f0 == 0) hm_mma(acc_e, ape, bpe, Fe);
            {
                const double* ap[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) ap[i] = apv[i] + f0;
                hm_mma(acc_v, ap, bpv, w);
            }
        }
        // epilogue: count and top list of each of the lane's rows, columns in ascending order
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = 32 * wr + 8 * i + g;
            if (x0 + rl >= n) continue;
            double* L = tl + (rl * HM_HOLD + hold) * order;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    if (o0 + 32 * wc + 8 * cb + 2 * q + e >= n_o) continue;
                    const double E = acc_e[i][cb][e], V = acc_v[i][cb][e];
                    const double e2 = E * E;
                    int over = hm_cmp(e2, cut2 * V);
                    int in = th[i] < 0.0 ? 1 : hm_cmp(e2, th[i] * th[i] * V);
                    if (over == 0 || in >= 0) {
                        const double I = hm_impl(E, V);
                        if (over == 0) over = I > cutoff ? 1 : -1;
                        if (I > th[i]) th[i] = hm_insert(L, order, I);
                    }
                    nover[i] += over > 0;
                }
        }
    }
    // counts: the 4 lanes of a row (butterfly), then the two column warps in order
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int v = nover[i];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if (q == 0) red[wc * HM_T + 32 * wr + 8 * i + g] = v;
    }
    __syncthreads();
    if (tid < HM_T && x0 + tid < n) {
        double* L = tl + tid * HM_HOLD * order;
        double lo = L[order - 1];
        for (int h = 1; h < HM_HOLD; ++h)
            for (int k = 0; k < order; ++k) {
                const double v = L[h * order + k];
                if (v > lo) lo = hm_insert(L, order, v);
            }
        const size_t x = (size_t)slab * n + x0 + tid;
        for (int k = 0; k < order; ++k) top[x * order + k] = L[k];
        cnt[x] = red[tid] + red[HM_T + tid];
    }
}

// impl_out (n, order), nover_out (n): the slabs' lists merged in slab order and their counts summed
__global__ void hm_merge_kernel(const double* __restrict__ top, const int* __restrict__ cnt, int n, int order, int nslab,
                                double* __restrict__ impl_out, int* __restrict__ nover_out)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    double L[HM_MAXORD];
    for (int k = 0; k < order; ++k) L[k] = top[(size_t)x * order + k];
    int total = cnt[x];
    double lo = L[order - 1];
    for (int s = 1; s < nslab; ++s) {
        const size_t row = (size_t)s * n + x;
        for (int k = 0; k < order; ++k) {
            const double v = top[row * order + k];
            if (v > lo) lo = hm_insert(L, order, v);
        }
        total += cnt[row];
    }
    for (int k = 0; k < order; ++k) impl_out[(size_t)x * order + k] = L[k];
    nover_out[x] = total;
}

struct HmLayout {
    int Fe, Fv, nslab;
    size_t ae, av, top, cnt, total;       // byte offsets and size
};

static bool hm_layout(int n, int n_o, int pu, int S, HmLayout& l)
{
    if (S < 1 || n < 1 || n_o < 1 || pu < 1 || pu > HM_MAXPU || (long long)S * pu >= (1LL << 31)) return false;
    l.Fe = hm_fe(pu);
    l.Fv = hm_fv(pu);
    l.nslab = hm_nslab(n, n_o);
    l.ae = 0;
    l.av = l.ae + (size_t)n * l.Fe * sizeof(double);
    l.top = l.av + (size_t)n * l.Fv * sizeof(double);
    l.cnt = l.top + (size_t)l.nslab * n * HM_MAXORD * sizeof(double);
    l.total = l.cnt + (size_t)l.nslab * n * sizeof(int);
    return true;
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_hm_workspace_bytes(int n, int n_o, int pu, int S)
{
    HmLayout l;
    if (!hm_layout(n, n_o, pu, S, l)) return -1;
    return (long long)l.total;
}

int ggp_hm_impl_f64(const double* mean, const double* var, int S, int pu, int n, const double* K_O, const double* r,
                    const double* c, int n_o, int order, double cutoff, double* impl_out, int* nover_out,
                    void* workspace, long long workspace_bytes, void* stream)
{
    GGP_ARG(mean && var && K_O && r && c && impl_out && nover_out && workspace, "null pointer");
    GGP_ARG(S >= 1 && n >= 1 && n_o >= 1, "S, n and n_o must be positive");
    GGP_ARG(pu >= 1 && pu <= HM_MAXPU, "pu must be in [1, 32]");
    GGP_ARG(order >= 1 && order <= HM_MAXORD && order <= n_o, "order must be in [1, min(8, n_o)]");
    GGP_ARG(cutoff > 0.0 && cutoff <= 1.7976931348623157e308, "cutoff must be finite and positive");
    GGP_ARG((long long)S * pu < (1LL << 31), "S * pu must be below 2^31");
    HmLayout l;
    hm_layout(n, n_o, pu, S, l);
    GGP_ARG(workspace_bytes >= (long long)l.total, "workspace too small");
    const long long ntp = ((long long)n + HM_T - 1) / HM_T;
    GGP_ARG(ntp * l.nslab < (1LL << 31), "too many point tiles");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(workspace);
    double* ae = reinterpret_cast<double*>(ws + l.ae);
    double* av = reinterpret_cast<double*>(ws + l.av);
    double* top = reinterpret_cast<double*>(ws + l.top);
    int* cnt = reinterpret_cast<int*>(ws + l.cnt);
    hm_mix_kernel<<<(unsigned)((n + HM_MIX_NT / 32 - 1) / (HM_MIX_NT / 32)), HM_MIX_NT, 0, st>>>(mean, var, S, pu, n, ae,
                                                                                                 l.Fe, av, l.Fv);
    GGP_CUDA(cudaGetLastError());
    const size_t smem = hm_smem_bytes(pu, order);
    GGP_CUDA(cudaFuncSetAttribute(hm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    hm_pair_kernel<<<(unsigned)(ntp * l.nslab), HM_NT, smem, st>>>(ae, l.Fe, av, l.Fv, n, pu, K_O, r, c, n_o, order,
                                                                   cutoff, (int)ntp, l.nslab, top, cnt);
    GGP_CUDA(cudaGetLastError());
    hm_merge_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(top, cnt, n, order, l.nslab, impl_out, nover_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
