// gladsgp_b200 -- shared device/host helpers (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cmath>

#define GGP_OK 0
#define GGP_ERR_ARG (-1)
#define GGP_ERR_CUDA (-2)
#define GGP_ERR_UNSUPPORTED (-3)
#define GGP_ERR_WORKSPACE (-4)

namespace ggp {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define GGP_CUDA(call)                                             \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return ::ggp::cuda_fail(e__, #call); \
    } while (0)

#define GGP_ARG(cond, msg)                                         \
    do {                                                           \
        if (!(cond)) { ::ggp::set_error("bad argument: %s", msg); return GGP_ERR_ARG; } \
    } while (0)

constexpr int NB = 32;          // panel width of the blocked factorisation
constexpr int NT = 128;         // threads per CTA of the fused kernels
constexpr int NWARP = NT / 32;
constexpr int CTAS_PER_SM = 4;     // 4 warps x 4 CTAs per SM, 128 registers per thread (tools/quick_bench.py sweep)
constexpr int CL_CTAS_PER_SM = 3;  // cluster variant (few matrices in flight): 168 registers per thread, no spills
constexpr int D_LD = 33;        // staging of the 32x32 diagonal block
constexpr int MI_LD = 40;       // leading dimension of the inverted diagonal block (conflict-free LDS.128)
constexpr int LT_LD = 34;       // leading dimension of the transposed diagonal factor (even: 16 B pairs)

__host__ __device__ inline int round_up32(int m) { return (m + 31) & ~31; }

// Packed factor layout (doubles).  Panel kb holds rows [32kb, Mp) of columns [32kb, 32kb+32) as
// four sub-slabs of 8 columns, each stored row-major with 8 doubles per row:
//   L[r][32kb + 8ks + c]  ->  poff(kb) + ks*(Mp-32kb)*8 + (r-32kb)*8 + c
__host__ __device__ inline long long panel_off(int kb, int Mp) {
    return 32LL * ((long long)kb * Mp - 16LL * kb * (kb - 1));
}
// after the panels: nP inverted diagonal blocks, [nP][32][32] row-major (Minv[c][k] = (Ljj^-1)[c][k])
__host__ __device__ inline long long minv_off(int Mp) { return panel_off(Mp / 32, Mp); }
// after those: auxiliary area of the cluster (multi-CTA) variant: running forward solve wres[Mp], the current
// u block [32], a failure flag [32]
__host__ __device__ inline long long aux_off(int Mp) { return panel_off(Mp / 32, Mp) + 1024LL * (Mp / 32); }
__host__ __device__ inline long long packed_doubles(int Mp) { return aux_off(Mp) + Mp + 64; }

__device__ __forceinline__ unsigned cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cluster_nctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// FP64 tensor-core MMA: D(8x8) += A(8x4) * B(4x8).  SASS: DMMA.8x8x4
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

__device__ __forceinline__ double2 ldcg2(const double* p) {
    return __ldcg(reinterpret_cast<const double2*>(p));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ggp
