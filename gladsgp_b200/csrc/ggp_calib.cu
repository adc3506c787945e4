// Emulator-based calibration (gladsgp_b200.calibration; DESIGN.md section 2 item 9): the log-likelihood of observed
// outputs at candidate inputs theta, and one Metropolis step of many chains.
//
// For posterior sample s the predictive means mu (pu) and variances v (pu) of the PC weights at a design come from
// ggp_predict_f64 (block s * pu + j).  With the per-sample observation terms precomputed by the caller,
//   G = K_O D^-1 K_O^T,  b = K_O D^-1 r,  c0 = r^T D^-1 r + sum log D_ii + n_o log 2 pi,
// Woodbury gives, with A = I + V^1/2 G V^1/2 (eigenvalues >= 1) and h = b - G mu,
//   l_s = -1/2 (c0 - 2 mu^T b + mu^T G mu - h^T V^1/2 A^-1 V^1/2 h + log det A),
// so the number of observed outputs never enters a step.  l = log mean_s exp l_s, accumulated over s in ascending order
// with a running maximum.  One warp per (point, sample): lane i owns row i of A in shared memory, a right-looking
// Cholesky broadcasts the multipliers of column k by shuffles and runs the forward solve L z = V^1/2 h alongside.
// Every sum runs in a fixed order: identical calls give identical bits.
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int CA_NW = 4;                 // warps per CTA; one CTA per point
constexpr int CA_NT = CA_NW * 32;
constexpr int CA_LD = 33;                // row stride of a warp's A (conflict-free row-per-lane access)
constexpr int CA_CHUNK = 128;            // l_s staged per round of the sample loop
constexpr int CA_MAXPU = 32;
constexpr int CA_MAXQ = 32;

struct CalibSmem {
    double A[CA_NW][CA_MAXPU * CA_LD];
    double ls[CA_CHUNK];
};

// l_s of point p under sample s, valid in every lane.  mean / var: (S pu, n); G: (S, pu, pu) symmetric; b: (S, pu).
__device__ double calib_sample_ll(const double* __restrict__ mean, const double* __restrict__ var, int pu, int n, int p,
                                  int s, const double* __restrict__ G, const double* __restrict__ b,
                                  const double* __restrict__ c0, double* __restrict__ A)
{
    const int lane = threadIdx.x & 31;
    const bool own = lane < pu;
    const size_t blk = (size_t)s * pu + lane;
    const double mu = own ? mean[blk * n + p] : 0.0;
    const double sv = own ? sqrt(fmax(var[blk * n + p], 0.0)) : 0.0;
    const double bj = own ? b[blk] : 0.0;
    const double* __restrict__ Gs = G + (size_t)s * pu * pu;
    // row `lane` of A (lower triangle) and (G mu)_lane, in ascending column order
    double gmu = 0.0;
    for (int k = 0; k < pu; ++k) {
        const double muk = __shfl_sync(0xffffffffu, mu, k);
        const double svk = __shfl_sync(0xffffffffu, sv, k);
        if (own) {
            const double g = Gs[(size_t)lane * pu + k];
            gmu += g * muk;
            if (k <= lane) A[lane * CA_LD + k] = (sv * svk) * g + (k == lane ? 1.0 : 0.0);
        }
    }
    const double quad = warp_sum(mu * (gmu - 2.0 * bj));          // mu^T G mu - 2 mu^T b
    double y = sv * (bj - gmu);                                    // V^1/2 h, reduced in place to the forward residual
    double zz = 0.0, logd = 0.0;
    for (int k = 0; k < pu; ++k) {
        const double akk = __shfl_sync(0xffffffffu, own ? A[lane * CA_LD + min(lane, k)] : 0.0, k);
        const double dk = sqrt(akk);
        const double lik = (own && lane > k) ? A[lane * CA_LD + k] / dk : 0.0;
        const double zk = __shfl_sync(0xffffffffu, y, k) / dk;
        y -= lik * zk;
        zz += zk * zk;
        logd += log(dk);
        for (int j = k + 1; j < pu; ++j) {
            const double ljk = __shfl_sync(0xffffffffu, lik, j);
            if (own && lane >= j) A[lane * CA_LD + j] -= lik * ljk;
        }
    }
    return -0.5 * (c0[s] + quad - zz + 2.0 * logd);
}

// l of point p over all S samples by the CTA's warps; l_s also to ll_s (S, n) when it is not null.  Valid in thread 0.
__device__ double calib_point_ll(const double* __restrict__ mean, const double* __restrict__ var, int S, int pu, int n,
                                 int p, const double* __restrict__ G, const double* __restrict__ b,
                                 const double* __restrict__ c0, double* __restrict__ ll_s, CalibSmem& sm)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double mx = -INFINITY, acc = 0.0;
    for (int s0 = 0; s0 < S; s0 += CA_CHUNK) {
        const int ns = min(CA_CHUNK, S - s0);
        for (int t = warp; t < ns; t += CA_NW) {
            const double l = calib_sample_ll(mean, var, pu, n, p, s0 + t, G, b, c0, sm.A[warp]);
            if (lane == 0) {
                sm.ls[t] = l;
                if (ll_s) ll_s[(size_t)(s0 + t) * n + p] = l;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int t = 0; t < ns; ++t) {
                const double l = sm.ls[t];
                if (l > mx) { acc = acc * exp(mx - l) + 1.0; mx = l; }
                else if (l != -INFINITY) acc += exp(l - mx);             // a NaN l_s makes l NaN
            }
        }
        __syncthreads();                                           // ls is refilled by the next chunk
    }
    return mx + log(acc) - log((double)S);
}

__global__ void __launch_bounds__(CA_NT)
calib_loglik_kernel(const double* __restrict__ mean, const double* __restrict__ var, int S, int pu, int n,
                    const double* __restrict__ G, const double* __restrict__ b, const double* __restrict__ c0,
                    double* __restrict__ ll, double* __restrict__ ll_s)
{
    __shared__ CalibSmem sm;
    const int p = blockIdx.x;
    const double l = calib_point_ll(mean, var, S, pu, n, p, G, b, c0, ll_s, sm);
    if (threadIdx.x == 0) ll[p] = l;
}

// One Metropolis step of chain c = blockIdx.x: the candidate is row c of Xp (its last q columns), its mean / var come
// from the ggp_predict_f64 call on Xp that precedes this launch.
__global__ void __launch_bounds__(CA_NT)
calib_step_kernel(const double* __restrict__ mean, const double* __restrict__ var, int S, int pu, int C,
                  const double* __restrict__ G, const double* __restrict__ b, const double* __restrict__ c0,
                  double* __restrict__ Xp, int d, int q, const double* __restrict__ lo, const double* __restrict__ hi,
                  const double* __restrict__ Lprop, const double* __restrict__ z_next, const double* __restrict__ logu,
                  double* __restrict__ theta, double* __restrict__ ll, double* __restrict__ rec_theta,
                  double* __restrict__ rec_ll, unsigned char* __restrict__ rec_acc)
{
    __shared__ CalibSmem sm;
    __shared__ double th[CA_MAXQ];
    __shared__ int s_valid, s_acc;
    const int c = blockIdx.x, tid = threadIdx.x;
    double* __restrict__ xc = Xp + (size_t)c * d + (d - q);
    if (tid == 0) s_valid = 1;
    __syncthreads();
    if (tid < q) {
        const double x = xc[tid];
        if (!(x >= lo[tid] && x <= hi[tid])) s_valid = 0;          // a NaN coordinate is outside too
    }
    __syncthreads();
    const bool valid = s_valid != 0;
    double lnew = NAN;
    if (valid) lnew = calib_point_ll(mean, var, S, pu, C, c, G, b, c0, nullptr, sm);
    if (tid == 0) {
        const double lold = ll[c];
        const int acc = valid && logu[c] < lnew - lold;            // false for a NaN l'
        if (acc) ll[c] = lnew;
        rec_ll[c] = acc ? lnew : lold;
        rec_acc[c] = (unsigned char)acc;
        s_acc = acc;
    }
    __syncthreads();
    if (tid < q) {
        double t = theta[(size_t)c * q + tid];
        if (s_acc) t = xc[tid];
        theta[(size_t)c * q + tid] = t;
        rec_theta[(size_t)c * q + tid] = t;
        th[tid] = t;
    }
    __syncthreads();
    if (z_next && tid < q) {
        // next candidate theta + L z, L lower triangular, summed over k ascending
        const double* __restrict__ z = z_next + (size_t)c * q;
        double x = th[tid];
        for (int k = 0; k <= tid; ++k) x += Lprop[tid * q + k] * z[k];
        xc[tid] = x;
    }
}

static const char* ca_check(int S, int pu, int n)
{
    if (S <= 0 || n <= 0) return "S and the number of points must be positive";
    if (pu < 1 || pu > CA_MAXPU) return "pu must be in [1, 32]";
    if ((long long)S * pu >= (1LL << 31)) return "S * pu must be below 2^31";
    return nullptr;
}

}  // namespace ggp

using namespace ggp;

extern "C" {

int ggp_calib_loglik_f64(const double* mean, const double* var, int S, int pu, int n, const double* G, const double* b,
                         const double* c0, double* ll_out, double* ll_s_out, void* stream)
{
    GGP_ARG(mean && var && G && b && c0 && ll_out, "null pointer");
    const char* bad = ca_check(S, pu, n);
    GGP_ARG(!bad, bad);
    calib_loglik_kernel<<<n, CA_NT, 0, (cudaStream_t)stream>>>(mean, var, S, pu, n, G, b, c0, ll_out, ll_s_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_calib_step_f64(const double* mean, const double* var, int S, int pu, int C, const double* G, const double* b,
                       const double* c0, double* Xp, int d, int q, const double* lo, const double* hi,
                       const double* L_prop, const double* z_next, const double* logu, double* theta, double* ll,
                       double* rec_theta, double* rec_ll, unsigned char* rec_acc, void* stream)
{
    GGP_ARG(mean && var && G && b && c0 && Xp && lo && hi && L_prop && logu && theta && ll && rec_theta && rec_ll &&
            rec_acc, "null pointer");
    const char* bad = ca_check(S, pu, C);
    GGP_ARG(!bad, bad);
    GGP_ARG(q >= 1 && q <= CA_MAXQ, "q must be in [1, 32]");
    GGP_ARG(d >= q, "d must be at least q");
    calib_step_kernel<<<C, CA_NT, 0, (cudaStream_t)stream>>>(mean, var, S, pu, C, G, b, c0, Xp, d, q, lo, hi, L_prop,
                                                             z_next, logu, theta, ll, rec_theta, rec_ll, rec_acc);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
