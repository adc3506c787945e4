// Ensemble ingest and initialisation passes (SURVEY 8f rank 2): the streaming work of the reference's
// init_model / fit_models around the PCA, each as one pass over the (m x n) float32 ensemble.
//
//   /root/reference/src/model.py:60-64    mu_y = mean(y, 0); sd_y = std(y, ddof=1, 0); sd_y[sd_y < thr] = thr
//   /root/reference/src/model.py:71-72    y_std = (y - mu_y) / sd_y                       (SepiaData.standardize_y)
//   /root/reference/src/model.py:219-223  w = (pinv(K)^T y_std^T)^T ; pc_prec = 1 / var(y_std - w K)
//   SepiaModel.__init__ (SURVEY A.2/A.3)  w, LamSim = diag(K K^T), ||y_std - w K||^2 for the lamWOs prior
//   /root/reference/src/aggregate_outputs.py:61-68  ensemble file layout (n_y, m): `transposed` inputs
//
// All three are HBM-bound streaming kernels (bytes per element: colstats 4 read; standardise 4 read + 4 written;
// projection 4 read) except the projection, which also does m*n*pu FP64 FMAs (accumulation in double so that the
// PC weights w keep FP64 accuracy: they are the data vector of every log-likelihood evaluation).
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

// ---------------------------------------------------------------------------------------------------------
// column statistics, Y[m][n]: thread (x, y) owns 4 consecutive columns and the rows y, y+8, ...; sums are taken
// about the first row of the column (pivot) in FP64, so the variance has no cancellation problem.
template <bool VEC>
__global__ void __launch_bounds__(256)
colstats_kernel(const float* __restrict__ Y, long long ld, int m, long long n, int ddof, float sd_floor,
                float* __restrict__ mean, float* __restrict__ sd)
{
    __shared__ double red[2][8][128 + 1];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const long long c0 = ((long long)blockIdx.x * 32 + tx) * 4;
    float piv[4];
    bool in[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        in[c] = c0 + c < n;
        piv[c] = in[c] ? __ldg(Y + c0 + c) : 0.f;
    }
    double s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
#pragma unroll 4
    for (int i = ty; i < m; i += 8) {
        float v[4];
        const float* row = Y + (size_t)i * ld + c0;
        if (VEC && in[3]) {
            const float4 q = __ldcs(reinterpret_cast<const float4*>(row));
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) v[c] = in[c] ? __ldcs(row + c) : 0.f;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const double dv = (double)v[c] - (double)piv[c];
            s1[c] += dv;
            s2[c] = fma(dv, dv, s2[c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        red[0][ty][4 * tx + c] = s1[c];
        red[1][ty][4 * tx + c] = s2[c];
    }
    __syncthreads();
    const int t = ty * 32 + tx;
    if (t < 128) {
        const long long col = (long long)blockIdx.x * 128 + t;
        if (col < n) {
            double a = 0.0, b = 0.0;
#pragma unroll
            for (int k = 0; k < 8; ++k) { a += red[0][k][t]; b += red[1][k][t]; }
            const double mu = (double)__ldg(Y + col) + a / m;
            double var = (b - a * a / m) / (double)(m - ddof);
            if (var < 0.0) var = 0.0;
            float s = (float)sqrt(var);
            if (s < sd_floor) s = sd_floor;
            mean[col] = (float)mu;
            sd[col] = s;
        }
    }
}

// column statistics of the transposed layout Yt[n][m]: one warp per output column (its m samples are contiguous)
__global__ void __launch_bounds__(256)
colstats_t_kernel(const float* __restrict__ Yt, long long ld, int m, long long n, int ddof, float sd_floor,
                  float* __restrict__ mean, float* __restrict__ sd)
{
    const int lane = threadIdx.x & 31;
    const long long col = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (col >= n) return;
    const float* row = Yt + (size_t)col * ld;
    const double piv = (double)__ldg(row);
    double s1 = 0.0, s2 = 0.0;
#pragma unroll 4
    for (int i = lane; i < m; i += 32) {
        const double dv = (double)__ldcs(row + i) - piv;
        s1 += dv;
        s2 = fma(dv, dv, s2);
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) {
        double var = (s2 - s1 * s1 / m) / (double)(m - ddof);
        if (var < 0.0) var = 0.0;
        float s = (float)sqrt(var);
        if (s < sd_floor) s = sd_floor;
        mean[col] = (float)(piv + s1 / m);
        sd[col] = s;
    }
}

// ---------------------------------------------------------------------------------------------------------
// y_std = (y - mean) / sd in float32 (IEEE subtract and divide: bit-identical to NumPy on the same mean / sd)
template <bool VEC>
__global__ void __launch_bounds__(256)
standardize_kernel(const float* __restrict__ Y, long long ld, int m, long long n, const float* __restrict__ mean, long long mean_len,
                   const float* __restrict__ sd, long long sd_len, int rows_per_cta, float* __restrict__ out)
{
    const long long c0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
    if (c0 >= n) return;
    float mu[4], s[4];
    bool in[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        in[c] = c0 + c < n;
        mu[c] = in[c] ? (mean_len == 1 ? mean[0] : mean[c0 + c]) : 0.f;
        s[c] = in[c] ? (sd_len == 1 ? sd[0] : sd[c0 + c]) : 1.f;
    }
    const int r0 = blockIdx.y * rows_per_cta, r1 = min(m, r0 + rows_per_cta);
#pragma unroll 4
    for (int i = r0; i < r1; ++i) {
        const float* row = Y + (size_t)i * ld + c0;
        float* orow = out + (size_t)i * n + c0;
        if (VEC && in[3]) {
            const float4 q = __ldcs(reinterpret_cast<const float4*>(row));
            __stcs(reinterpret_cast<float4*>(orow),
                   make_float4((q.x - mu[0]) / s[0], (q.y - mu[1]) / s[1], (q.z - mu[2]) / s[2], (q.w - mu[3]) / s[3]));
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (in[c]) __stcs(orow + c, (__ldcs(row + c) - mu[c]) / s[c]);
        }
    }
}

// transposed input Yt[n][m] -> out[m][n]: 32 x 32 tiles through shared memory, both sides in 128-byte segments
__global__ void __launch_bounds__(256)
standardize_t_kernel(const float* __restrict__ Yt, long long ld, int m, long long n, const float* __restrict__ mean,
                     long long mean_len, const float* __restrict__ sd, long long sd_len, float* __restrict__ out)
{
    __shared__ float tile[32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;             // (32, 8)
    const long long c0 = (long long)blockIdx.x * 32;           // output columns (rows of Yt)
    const int s0 = blockIdx.y * 32;                            // samples (columns of Yt)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long c = c0 + ty + 8 * k;
        const int sidx = s0 + tx;
        tile[ty + 8 * k][tx] = (c < n && sidx < m) ? __ldcs(Yt + (size_t)c * ld + sidx) : 0.f;
    }
    __syncthreads();
    const long long c = c0 + tx;
    if (c >= n) return;
    const float mu = mean_len == 1 ? mean[0] : mean[c];
    const float s = sd_len == 1 ? sd[0] : sd[c];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int sidx = s0 + ty + 8 * k;
        if (sidx < m) __stcs(out + (size_t)sidx * n + c, (tile[tx][ty + 8 * k] - mu) / s);
    }
}

// ---------------------------------------------------------------------------------------------------------
// projection on the basis, FP64 accumulation:  P[i][k] = sum_c X[i][c] * Kt[k][c]  (k < pu),
// P[i][pu] = sum_c X[i][c],  P[i][pu+1] = sum_c X[i][c]^2.
// Same streaming structure as the FP32-FMA rSVD sketch of commit 667fe96 (csrc/ggp_rsvd.cu): the CTA pulls 32-column chunks of its 256*RPT rows
// through a padded shared-memory tile, each thread owns RPT rows and keeps their pu + 2 sums in registers.
constexpr int PJ_THREADS = 256;

template <int PU, int RPT>
__global__ void __launch_bounds__(PJ_THREADS, 2)
project_kernel(const float* __restrict__ X, int m, long long n, const float* __restrict__ Kt, int pu,
               double* __restrict__ partial)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* Xs = reinterpret_cast<float*>(smem_raw);                 // [RPT*256][33]
    float* Ks = Xs + (size_t)RPT * PJ_THREADS * 33;                 // [32][PU]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row_base = blockIdx.y * RPT * PJ_THREADS;
    double acc[RPT][PU], rs[RPT], rq[RPT];
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        rs[i] = 0.0; rq[i] = 0.0;
#pragma unroll
        for (int k = 0; k < PU; ++k) acc[i][k] = 0.0;
    }
    constexpr int mrows = RPT * PJ_THREADS;
    const long long nchunk = (n + 31) / 32;
    for (long long ch = blockIdx.x; ch < nchunk; ch += gridDim.x) {
        const long long c0 = ch * 32;
        const bool cin = c0 + lane < n;
        __syncthreads();
        for (int rb = warp; rb < mrows; rb += 8 * 16) {
            float v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int row = row_base + rb + 8 * u;
                v[u] = (rb + 8 * u < mrows && row < m && cin) ? __ldcs(X + (size_t)row * n + c0 + lane) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 16; ++u)
                if (rb + 8 * u < mrows) Xs[(rb + 8 * u) * 33 + lane] = v[u];
        }
        for (int idx = tid; idx < PU * 32; idx += PJ_THREADS) {
            const int k = idx >> 5, c = idx & 31;
            Ks[c * PU + k] = (k < pu && c0 + c < n) ? Kt[(size_t)k * n + c0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll 2
        for (int c = 0; c < 32; ++c) {
            double x[RPT];
#pragma unroll
            for (int i = 0; i < RPT; ++i) {
                x[i] = (double)Xs[(tid + PJ_THREADS * i) * 33 + c];
                rs[i] += x[i];
                rq[i] = fma(x[i], x[i], rq[i]);
            }
#pragma unroll
            for (int k4 = 0; k4 < PU; k4 += 4) {
                const float4 o4 = *reinterpret_cast<const float4*>(Ks + c * PU + k4);
#pragma unroll
                for (int i = 0; i < RPT; ++i) {
                    acc[i][k4 + 0] = fma(x[i], (double)o4.x, acc[i][k4 + 0]);
                    acc[i][k4 + 1] = fma(x[i], (double)o4.y, acc[i][k4 + 1]);
                    acc[i][k4 + 2] = fma(x[i], (double)o4.z, acc[i][k4 + 2]);
                    acc[i][k4 + 3] = fma(x[i], (double)o4.w, acc[i][k4 + 3]);
                }
            }
        }
    }
    // partial[blockIdx.x][m][PU + 2]
    double* out = partial + (size_t)blockIdx.x * m * (PU + 2);
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const int row = row_base + tid + PJ_THREADS * i;
        if (row < m) {
#pragma unroll
            for (int k = 0; k < PU; ++k) out[(size_t)row * (PU + 2) + k] = acc[i][k];
            out[(size_t)row * (PU + 2) + PU] = rs[i];
            out[(size_t)row * (PU + 2) + PU + 1] = rq[i];
        }
    }
}

// fixed-order (deterministic) sum of the per-CTA partials
__global__ void project_reduce_kernel(const double* __restrict__ partial, int nparts, int m, int PU, int pu,
                                      double* __restrict__ P)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= m * (PU + 2)) return;
    const int row = idx / (PU + 2), k = idx - row * (PU + 2);
    double s = 0.0;
    for (int p = 0; p < nparts; ++p) s += partial[(size_t)p * m * (PU + 2) + idx];
    if (k < pu) P[(size_t)row * (pu + 2) + k] = s;
    else if (k >= PU) P[(size_t)row * (pu + 2) + pu + (k - PU)] = s;
}

static int ingest_sm_count()
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

static int project_pu_pad(int pu) { return pu <= 4 ? 4 : pu <= 12 ? 12 : pu <= 20 ? 20 : 32; }

template <int PU, int RPT>
static int launch_project(const float* X, int m, long long n, const float* Kt, int pu, double* partial, int gx,
                          cudaStream_t st)
{
    const size_t smem = ((size_t)RPT * PJ_THREADS * 33 + 32 * PU) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(project_kernel<PU, RPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(project_kernel)");
    const int gy = (m + RPT * PJ_THREADS - 1) / (RPT * PJ_THREADS);
    project_kernel<PU, RPT><<<dim3(gx, gy), PJ_THREADS, smem, st>>>(X, m, n, Kt, pu, partial);
    return GGP_OK;
}

}  // namespace ggp

using namespace ggp;

extern "C" {

int ggp_colstats_f32(const float* Y, long long ld, int m, long long n, int transposed, int ddof, float sd_floor,
                     float* mean_out, float* sd_out, void* stream)
{
    if (ld <= 0) ld = transposed ? m : n;
    GGP_ARG(ld >= (transposed ? (long long)m : n), "ld smaller than the row length");
    GGP_ARG(Y && mean_out && sd_out, "null pointer");
    GGP_ARG(m > 0 && n > 0, "m, n must be positive");
    GGP_ARG(ddof >= 0 && ddof < m, "ddof must be in [0, m)");
    cudaStream_t st = (cudaStream_t)stream;
    if (transposed) {
        colstats_t_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(Y, ld, m, n, ddof, sd_floor, mean_out, sd_out);
    } else {
        const unsigned gx = (unsigned)((n + 127) / 128);
        const bool vec = (n % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(Y) & 15) == 0);
        if (vec) colstats_kernel<true><<<gx, dim3(32, 8), 0, st>>>(Y, ld, m, n, ddof, sd_floor, mean_out, sd_out);
        else colstats_kernel<false><<<gx, dim3(32, 8), 0, st>>>(Y, ld, m, n, ddof, sd_floor, mean_out, sd_out);
    }
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_standardize_f32(const float* Y, long long ld, int m, long long n, int transposed, const float* mean,
                        long long mean_len, const float* sd, long long sd_len, float* Ystd_out, void* stream)
{
    if (ld <= 0) ld = transposed ? m : n;
    GGP_ARG(ld >= (transposed ? (long long)m : n), "ld smaller than the row length");
    GGP_ARG(Y && mean && sd && Ystd_out, "null pointer");
    GGP_ARG(m > 0 && n > 0, "m, n must be positive");
    GGP_ARG((mean_len == 1 || mean_len == n) && (sd_len == 1 || sd_len == n), "mean / sd must have 1 or n entries");
    cudaStream_t st = (cudaStream_t)stream;
    if (transposed) {
        GGP_ARG(Y != Ystd_out, "the transposing pass cannot run in place");
        const dim3 grid((unsigned)((n + 31) / 32), (unsigned)((m + 31) / 32));
        GGP_ARG(grid.y <= 65535, "m too large");
        standardize_t_kernel<<<grid, dim3(32, 8), 0, st>>>(Y, ld, m, n, mean, mean_len, sd, sd_len, Ystd_out);
    } else {
        const unsigned gx = (unsigned)((n + 1023) / 1024);
        // enough CTAs to fill the machine, at least 16 rows each
        long long gy = (8LL * ingest_sm_count() + gx - 1) / gx;
        if (gy > (m + 15) / 16) gy = (m + 15) / 16;
        if (gy < 1) gy = 1;
        const int rows_per_cta = (int)((m + gy - 1) / gy);
        gy = (m + rows_per_cta - 1) / rows_per_cta;
        const bool vec = (n % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(Y) & 15) == 0) &&
                         ((reinterpret_cast<uintptr_t>(Ystd_out) & 15) == 0);
        if (vec) standardize_kernel<true><<<dim3(gx, (unsigned)gy), 256, 0, st>>>(Y, ld, m, n, mean, mean_len, sd, sd_len, rows_per_cta, Ystd_out);
        else standardize_kernel<false><<<dim3(gx, (unsigned)gy), 256, 0, st>>>(Y, ld, m, n, mean, mean_len, sd, sd_len, rows_per_cta, Ystd_out);
    }
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

long long ggp_project_workspace_bytes(int m, int pu)
{
    if (m <= 0 || pu <= 0 || pu > 32) return -1;
    return 2LL * ingest_sm_count() * m * (project_pu_pad(pu) + 2) * (long long)sizeof(double);
}

int ggp_project_f32(const float* X, int m, long long n, const float* Kt, int pu, double* P_out, void* workspace,
                    long long workspace_bytes, void* stream)
{
    GGP_ARG(X && Kt && P_out && workspace, "null pointer");
    GGP_ARG(m > 0 && n > 0, "m, n must be positive");
    GGP_ARG(pu > 0 && pu <= 32, "pu must be in [1, 32]");
    if (workspace_bytes < ggp_project_workspace_bytes(m, pu)) {
        set_error("ggp_project_f32: workspace too small");
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* partial = reinterpret_cast<double*>(workspace);
    const int PU = project_pu_pad(pu);
    const long long nchunk = (n + 31) / 32;
    const long long cap = 2LL * ingest_sm_count();
    const int gx = (int)(nchunk < cap ? nchunk : cap);
    int rc;
    const bool one = m <= PJ_THREADS;
    switch (PU) {
        case 4: rc = one ? launch_project<4, 1>(X, m, n, Kt, pu, partial, gx, st) : launch_project<4, 2>(X, m, n, Kt, pu, partial, gx, st); break;
        case 12: rc = one ? launch_project<12, 1>(X, m, n, Kt, pu, partial, gx, st) : launch_project<12, 2>(X, m, n, Kt, pu, partial, gx, st); break;
        case 20: rc = one ? launch_project<20, 1>(X, m, n, Kt, pu, partial, gx, st) : launch_project<20, 2>(X, m, n, Kt, pu, partial, gx, st); break;
        default: rc = launch_project<32, 1>(X, m, n, Kt, pu, partial, gx, st); break;
    }
    if (rc != GGP_OK) return rc;
    project_reduce_kernel<<<(m * (PU + 2) + 255) / 256, 256, 0, st>>>(partial, gx, m, PU, pu, P_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
