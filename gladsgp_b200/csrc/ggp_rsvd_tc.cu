// Randomized-SVD passes on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM).
//
// The products of the reference's src/svd.py:52-60 -- Y = X Omega and Bt = Y^T X over the (m x n) float32 ensemble --
// with the multiply-adds as 3xTF32 split products on the tensor pipe, so that the pass is bound by the HBM read of X
// instead of the FP32 FMA rate:
//     x = x_hi + x_lo (x_hi = tf32(x), x_lo = tf32(x - x_hi)),   x*o ~= x_hi*o_hi + x_hi*o_lo + x_lo*o_hi
// (error ~2^-21 relative per product, i.e. FP32-level; the dropped x_lo*o_lo term is 2^-22 smaller than the product).
// The tensor core adds into its FP32 accumulator with truncation, so a K-chunk (32 columns, 12 accumulator updates)
// is summed in TMEM and then added to round-to-nearest FP32 register accumulators by the CUDA cores -- the long sum
// over n never runs inside the tensor core.
//
// Operands reach shared memory in the UMMA canonical K-major 128-byte-swizzle layout.  Y = X Omega has one kernel per
// pitch class: when the row pitch is a multiple of 16 bytes and both bases are 16-byte aligned, TMA writes the tiles
// (sketch_tma_kernel); otherwise -- e.g. the reference's ensembles, 4*n_y bytes with n_y = 3693*365 -- the producer
// warps stage them through registers (sketch_tc_kernel).  Bt = Y^T X writes its X operand straight into tensor memory
// (xty_ts_kernel).  One elected thread issues tcgen05.mma and signals completion with tcgen05.commit on an mbarrier.
#include <cuda.h>                 // CUtensorMap and the cuTensorMapEncodeTiled prototype (resolved at run time, no -lcuda)
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

constexpr int TC_ROWS = 256;                 // rows of X per CTA (two M = 128 tiles)
constexpr int TC_K = 32;                     // columns of X per chunk (four K = 8 steps)
constexpr int TC_STAGES = 3;
constexpr int TC_PRODUCERS = 256;            // 8 producer warps
constexpr int TC_THREADS = TC_PRODUCERS + 128;  // + 4 epilogue warps (the first one also issues the MMAs)
constexpr int TC_A_BYTES = TC_ROWS * TC_K * 4;  // 32 KB (one of hi / lo)
constexpr int TC_B_BYTES = 32 * TC_K * 4;       // 4 KB
constexpr int TC_STAGE_BYTES = 2 * TC_A_BYTES + 2 * TC_B_BYTES;    // 72 KB
constexpr int TC_TMEM_COLS = 128;            // 2 buffers x 2 tiles x 32 columns

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded spin: a protocol error traps instead of hanging the device
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t addr = smem_u32(bar);
    for (int spin = 0; spin < 4000; ++spin) {               // each try_wait may suspend the thread for up to 1 ms
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(addr), "r"(parity), "r"(1000000u)
            : "memory");
        if (ok) return;
    }
    __trap();
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (the tensor core reads operands through it)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// K-major, 128-byte swizzle: a row is 128 contiguous bytes (32 tf32 = one K chunk), rows 128 B apart, 8-row groups
// 1024 B apart, and the 16-byte piece kc of row r sits at position kc ^ (r % 8) (Swizzle<3,4,3>; tile 1024-B aligned).
// A K = 8 step advances the start address by 32 bytes.
// The same descriptor as two words, so that the issuing thread only adds a byte offset to the low word per MMA
// (it is a single thread: every instruction it spends on descriptors is on the critical path of the chunk).
constexpr uint32_t UMMA_SW128_HI = 64u | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t umma_sw128_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | (1u << 16); }
__device__ __forceinline__ uint64_t umma_join(uint32_t lo, uint32_t hi)
{
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
template <bool ACC>
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "n"(ACC ? 1 : 0)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
// issue all tcgen05.ld of an epilogue first, then wait once
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// x = hi + lo with hi on the TF32 grid (round to nearest, ties away -- what cvt.rna.tf32.f32 does, but on the integer
// pipe: the conversion instruction runs on the quarter-rate XU pipe and was the producers' bottleneck) and lo = x - hi
// exact in FP32 (|lo| <= 2^-11 |x|); the tensor core reads the upper 19 bits of lo (error <= 2^-21 |x|).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo)
{
    hi = (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}

// ---------------------------------------------------------------------------------------------------------
// Y = X * Omega.  grid (gx, row blocks of 256): CTA (bx, by) takes the 32-column chunks bx, bx + gx, ... of its
// rows and writes partial[bx][m][32]; tc_reduce_kernel sums the partials in FP64 in a fixed order.
//
// Warp roles (12 warps, 168 registers each = 3 warps per SM sub-partition):
//   warps 0-7   producers: global -> registers (two chunks ahead, three rotating buffers) -> hi/lo split -> swizzled
//               shared-memory stage -> fence.proxy.async -> arrive on full[stage]
//   warp 8      lane 0 issues the 24 tcgen05.mma of a chunk (2 M-tiles x 4 K-steps x 3 split products) and commits
//               to empty[stage] (stage reusable) and tmem_full[buffer] (chunk sum ready)
//   warps 8-11  epilogue: tcgen05.ld the chunk sum (two 128 x 32 tiles, TMEM double-buffered) and add it to FP32
//               register accumulators with round-to-nearest
template <bool VEC, int NPW>
__global__ void __launch_bounds__(NPW * 32 + 128, 1)
sketch_tc_kernel(const float* __restrict__ X, int m, long long n, const float* __restrict__ OmT, int r, int k0,
                 float* __restrict__ partial)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[TC_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[TC_STAGES];
    __shared__ __align__(8) uint64_t tmem_full_bar[2];
    __shared__ uint32_t tmem_base_sh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row_base = blockIdx.y * TC_ROWS;

    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            mbar_init(&full_bar[s], NPW * 32);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(&tmem_full_bar[0], 1);
        mbar_init(&tmem_full_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == NPW) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_sh)),
                     "r"(TC_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;

    const long long nchunk = (n + TC_K - 1) / TC_K;
    // a contiguous range of chunks per CTA: successive loads of a thread walk along one row of X
    const long long per = (nchunk + gridDim.x - 1) / gridDim.x;
    const long long ch_begin = (long long)blockIdx.x * per;
    const int n_my = (int)(ch_begin >= nchunk ? 0 : (nchunk - ch_begin < per ? nchunk - ch_begin : per));
    auto chunk_col = [&](int it) { return (ch_begin + it) * TC_K; };

    if (warp < NPW) {
        // ================= producers =================
        // A staging: warp w, pass u, lane l -> row 32 w + 4 u + l/8, 16-byte K piece l%8 (full 128-byte lines from
        // global, conflict-free STS.128 into the swizzled tile).  B staging: thread t -> Omega row t/8, K piece t%8.
        constexpr int UP = 64 / NPW;                                       // 128-byte row pieces per thread and chunk
        const bool b_thread = tid < 256;                                   // threads that also stage Omega
        const int b_row = (tid >> 3) & 31, b_kc = tid & 7;
        const bool b_ok = b_thread && (k0 + b_row < r);
        const int lrow0 = warp * (4 * UP) + (lane >> 3);                         // local row of pass 0 (pass u: + 4 u)
        const float* xp = X + (size_t)(row_base + lrow0) * n + 4 * (lane & 7);      // + 4 u n + c0
        const float* bp = OmT + (size_t)(k0 + (b_ok ? b_row : 0)) * n + 4 * b_kc;
        const size_t pass_stride = 4 * (size_t)n;
        unsigned row_ok = 0;
#pragma unroll
        for (int u = 0; u < UP; ++u) row_ok |= (row_base + lrow0 + 4 * u < m) ? (1u << u) : 0u;

        auto load_chunk = [&](int it, float (&xv)[UP][4], float (&bv)[4]) {
            const long long c0 = chunk_col(it);
            const float* src0 = xp + c0;
            if (c0 + TC_K <= n) {                               // whole chunk inside the matrix (CTA-uniform)
#pragma unroll
                for (int u = 0; u < UP; ++u) {
                    const float* src = src0 + u * pass_stride;
                    if (!((row_ok >> u) & 1)) {
                        xv[u][0] = 0.f; xv[u][1] = 0.f; xv[u][2] = 0.f; xv[u][3] = 0.f;
                    } else if (VEC) {
                        const float4 q = __ldcs(reinterpret_cast<const float4*>(src));
                        xv[u][0] = q.x; xv[u][1] = q.y; xv[u][2] = q.z; xv[u][3] = q.w;
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) xv[u][j] = __ldcs(src + j);
                    }
                }
                if (!b_ok) {
                    bv[0] = 0.f; bv[1] = 0.f; bv[2] = 0.f; bv[3] = 0.f;
                } else if (VEC) {
                    const float4 q = __ldg(reinterpret_cast<const float4*>(bp + c0));
                    bv[0] = q.x; bv[1] = q.y; bv[2] = q.z; bv[3] = q.w;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) bv[j] = __ldg(bp + c0 + j);
                }
            } else {                                            // ragged last chunk
                const long long col = c0 + 4 * (lane & 7);
#pragma unroll
                for (int u = 0; u < UP; ++u)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        xv[u][j] = (((row_ok >> u) & 1) && col + j < n) ? __ldcs(src0 + u * pass_stride + j) : 0.f;
                const long long colb = c0 + 4 * b_kc;
#pragma unroll
                for (int j = 0; j < 4; ++j) bv[j] = (b_ok && colb + j < n) ? __ldg(bp + c0 + j) : 0.f;
            }
        };
        // one pipeline step: chunk `it` is in (xv, bv); chunk it+2 is loaded into (xl, bl)
        auto step = [&](int it, float (&xv)[UP][4], float (&bv)[4], float (&xl)[UP][4], float (&bl)[4]) {
            if (it >= n_my) return;
            if (it + 2 < n_my) load_chunk(it + 2, xl, bl);
            const int s = it % TC_STAGES;
            if (it >= TC_STAGES) mbar_wait(&empty_bar[s], (uint32_t)((it / TC_STAGES - 1) & 1));   // MMAs of chunk it-3 done
            unsigned char* st = smem_raw + (size_t)s * TC_STAGE_BYTES;
#pragma unroll
            for (int u = 0; u < UP; ++u) {
                const uint32_t lrow = (uint32_t)(lrow0 + 4 * u);
                const uint32_t off = lrow * 128u + (uint32_t)(((lane & 7) ^ (lrow & 7)) * 16);
                uint4 hi, lo;
                split_tf32(xv[u][0], hi.x, lo.x);
                split_tf32(xv[u][1], hi.y, lo.y);
                split_tf32(xv[u][2], hi.z, lo.z);
                split_tf32(xv[u][3], hi.w, lo.w);
                *reinterpret_cast<uint4*>(st + off) = hi;
                *reinterpret_cast<uint4*>(st + TC_A_BYTES + off) = lo;
            }
            if (b_thread) {
                const uint32_t off = (uint32_t)b_row * 128u + (uint32_t)((b_kc ^ (b_row & 7)) * 16);
                uint4 hi, lo;
                split_tf32(bv[0], hi.x, lo.x);
                split_tf32(bv[1], hi.y, lo.y);
                split_tf32(bv[2], hi.z, lo.z);
                split_tf32(bv[3], hi.w, lo.w);
                *reinterpret_cast<uint4*>(st + 2 * TC_A_BYTES + off) = hi;
                *reinterpret_cast<uint4*>(st + 2 * TC_A_BYTES + TC_B_BYTES + off) = lo;
            }
            fence_async_smem();
            mbar_arrive(&full_bar[s]);
        };
        float x0[UP][4], x1[UP][4], x2[UP][4], b0[4], b1[4], b2[4];
        if (n_my > 0) load_chunk(0, x0, b0);
        if (n_my > 1) load_chunk(1, x1, b1);
#pragma unroll 1
        for (int it = 0; it < n_my; it += 3) {
            step(it, x0, b0, x2, b2);
            step(it + 1, x1, b1, x0, b0);
            step(it + 2, x2, b2, x1, b1);
        }
    } else {
        // ================= MMA issue (warp 8, lane 0) + epilogue (warps 8-11) =================
        constexpr uint32_t idesc = umma_idesc_tf32(128, 32);
        const int ew = warp - NPW;                                             // TMEM lanes 32 ew .. 32 ew + 31
        const uint32_t t_lane = (uint32_t)(32 * ew) << 16;
        const uint32_t desc_lo0 = umma_sw128_lo(smem_u32(smem_raw));
        float acc[2][32];
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
            for (int c = 0; c < 32; ++c) acc[t][c] = 0.f;
#pragma unroll 1
        for (int it = 0; it <= n_my; ++it) {
            if (it < n_my && warp == NPW && lane == 0) {
                const int s = it % TC_STAGES;
                mbar_wait(&full_bar[s], (uint32_t)((it / TC_STAGES) & 1));
                tc_fence_after();
                // descriptor low words: base + (byte offset >> 4); A tile t-step: + 2, next M tile: + 1024, lo: + 2048
                const uint32_t a_lo0 = desc_lo0 + (uint32_t)s * (TC_STAGE_BYTES >> 4);
                const uint32_t b_lo0 = a_lo0 + ((2 * TC_A_BYTES) >> 4);
                const uint32_t d0 = tmem_base + (uint32_t)((it & 1) * 64);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint64_t bh = umma_join(b_lo0 + 2 * t, UMMA_SW128_HI);
                    const uint64_t bl = umma_join(b_lo0 + (TC_B_BYTES >> 4) + 2 * t, UMMA_SW128_HI);
#pragma unroll
                    for (int tile = 0; tile < 2; ++tile) {
                        const uint64_t ah = umma_join(a_lo0 + tile * 1024 + 2 * t, UMMA_SW128_HI);
                        const uint64_t al = umma_join(a_lo0 + (TC_A_BYTES >> 4) + tile * 1024 + 2 * t, UMMA_SW128_HI);
                        const uint32_t d = d0 + tile * 32;
                        if (t == 0) umma_tf32<false>(d, al, bh, idesc); else umma_tf32<true>(d, al, bh, idesc);   // small terms first
                        umma_tf32<true>(d, ah, bl, idesc);
                        umma_tf32<true>(d, ah, bh, idesc);
                    }
                }
                umma_commit(&empty_bar[s]);
                umma_commit(&tmem_full_bar[it & 1]);
            }
            __syncwarp();
            if (it >= 1) {
                // chunk it-1 has been multiplied: add its TMEM tiles into the register accumulators
                const int j = it - 1;
                mbar_wait(&tmem_full_bar[j & 1], (uint32_t)((j >> 1) & 1));
                tc_fence_after();
                uint32_t v0[32], v1[32];
                tmem_ld32(tmem_base + t_lane + (uint32_t)((j & 1) * 64), v0);
                tmem_ld32(tmem_base + t_lane + (uint32_t)((j & 1) * 64 + 32), v1);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[0][c] += __uint_as_float(v0[c]);
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[1][c] += __uint_as_float(v1[c]);
                tc_fence_before();
            }
            // all four epilogue warps are done with TMEM buffer (it-1)&1 before the MMAs of chunk it+1 overwrite it
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
#pragma unroll
        for (int tile = 0; tile < 2; ++tile) {
            const int row = row_base + tile * 128 + 32 * ew + lane;
            if (row < m) {
                float4* out = reinterpret_cast<float4*>(partial + ((size_t)blockIdx.x * m + row) * 32);
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    out[c] = make_float4(acc[tile][4 * c], acc[tile][4 * c + 1], acc[tile][4 * c + 2], acc[tile][4 * c + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPW) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS));
    }
}

// ---------------------------------------------------------------------------------------------------------
// Y = X * Omega with the operand tiles brought in by TMA (cp.async.bulk.tensor, SWIZZLE_128B: the hardware writes the
// 256 x 32 tile of X and the 32 x 32 tile of Omega^T straight into the K-major 128-byte-swizzle layout the MMA
// descriptors expect).  Needs a row pitch that is a multiple of 16 bytes (n % 4 == 0) and 16-byte aligned bases; other
// shapes take the register-staged kernel above.  Raw stages (written by TMA) and derived stages (written by the splitters):
//   warp 12     lane 0: per chunk, waits for the stage to be free, arms raw_full[stage] with the byte count and issues the
//               two tensor copies (out-of-range rows / columns are zero-filled by the hardware)
//   warps 0-7   splitters: wait for raw_full, write x - trunc_tf32(x) of every 16-byte piece of X to the lo tile (same
//               swizzled offset) and the hi and lo tiles of Omega, fence.proxy.async, arrive on full[stage]
//   warps 8-11  MMA issue + epilogue
// The hi tile of X is the raw float32 tile as TMA delivered it: the tensor core takes the upper 19 bits of each operand
// element, i.e. tf32(x) by truncation (same accuracy against the float64 product as the rounded split of sketch_tc_kernel).
// The two products that share it, x_hi o_hi and x_hi o_lo, are ONE MMA with N = 64 (the hi and lo tiles of Omega are adjacent,
// i.e. rows 0-31 / 32-63 of one K-major operand), x_lo o_hi is a second one with N = 32: 16 instead of 24 MMAs per chunk, and
// the X tiles are read from shared memory twice instead of three times.  The three partial sums live in separate TMEM columns
// and are added in the epilogue (round-to-nearest FP32).  The result agrees with sketch_tc_kernel to FP32 level, not bitwise.
// Shared memory: a ring of TMA_RAW raw stages [X raw 32 KB | Omega raw 4 KB] that only TMA writes -- four chunks of
// prefetch, 108 KB in flight per SM -- and a ring of two derived stages [X lo 32 KB | Omega hi 4 KB | Omega lo 4 KB].
constexpr int TMA_THREADS = 384 + 32;
constexpr int TMA_RAW = 4;
constexpr int TMA_RAW_BYTES = TC_A_BYTES + TC_B_BYTES;            // 36 KB
constexpr int TMA_LO_BYTES = TC_A_BYTES + 2 * TC_B_BYTES;         // 40 KB
constexpr int TMA_SMEM_BYTES = TMA_RAW * TMA_RAW_BYTES + 2 * TMA_LO_BYTES;   // 224 KB

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

__global__ void __launch_bounds__(TMA_THREADS, 1)
sketch_tma_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapO, int m, long long n,
                  int r, int k0, float* __restrict__ partial)
{
    constexpr int DCOLS = 96;                                   // TMEM columns per 128-row tile and buffer
    constexpr int TCOLS = 512;                                  // 2 buffers x 2 tiles x DCOLS, rounded up to a power of two
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t raw_bar[TMA_RAW];          // TMA bytes of a raw stage have landed
    __shared__ __align__(8) uint64_t rawfree_bar[TMA_RAW];      // MMAs reading a raw stage are done
    __shared__ __align__(8) uint64_t full_bar[2];               // derived stage written by the splitters
    __shared__ __align__(8) uint64_t lofree_bar[2];             // MMAs reading a derived stage are done
    __shared__ __align__(8) uint64_t tmem_full_bar[2];
    __shared__ uint32_t tmem_base_sh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row_base = blockIdx.y * TC_ROWS;
    unsigned char* lo_base = smem_raw + TMA_RAW * TMA_RAW_BYTES;

    if (tid == 0) {
        for (int s = 0; s < TMA_RAW; ++s) { mbar_init(&raw_bar[s], 1); mbar_init(&rawfree_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&full_bar[s], 256); mbar_init(&lofree_bar[s], 1); mbar_init(&tmem_full_bar[s], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_sh)),
                     "r"(TCOLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;

    const long long nchunk = (n + TC_K - 1) / TC_K;
    const long long per = (nchunk + gridDim.x - 1) / gridDim.x;
    const long long ch_begin = (long long)blockIdx.x * per;
    const int n_my = (int)(ch_begin >= nchunk ? 0 : (nchunk - ch_begin < per ? nchunk - ch_begin : per));

    if (warp == 12) {
        // ================= TMA producer (one thread) =================
        // (The pure TMA stream of 256-row x 128-byte boxes, without split and MMA, tops out at 4.0 TB/s = 0.61 of the copy peak.)
        if (lane == 0) {
            for (int it = 0; it < n_my; ++it) {
                const int s = it % TMA_RAW;
                if (it >= TMA_RAW) mbar_wait(&rawfree_bar[s], (uint32_t)((it / TMA_RAW - 1) & 1));
                unsigned char* st = smem_raw + (size_t)s * TMA_RAW_BYTES;
                const int c0 = (int)((ch_begin + it) * TC_K);
                mbar_arrive_expect_tx(&raw_bar[s], (uint32_t)TMA_RAW_BYTES);
                tma_load_2d(st, &mapX, c0, row_base, &raw_bar[s]);
                tma_load_2d(st + TC_A_BYTES, &mapO, c0, k0, &raw_bar[s]);
            }
        }
    } else if (warp < 8) {
        // ================= splitters =================
        for (int it = 0; it < n_my; ++it) {
            const int s = it % TMA_RAW, l = it & 1;
            mbar_wait(&raw_bar[s], (uint32_t)((it / TMA_RAW) & 1));
            if (it >= 2) mbar_wait(&lofree_bar[l], (uint32_t)((it / 2 - 1) & 1));       // MMAs of chunk it-2 done with the slot
            unsigned char* st = smem_raw + (size_t)s * TMA_RAW_BYTES;
            unsigned char* lt = lo_base + (size_t)l * TMA_LO_BYTES;
            // 2048 16-byte pieces of X per stage, 8 per thread; consecutive threads, consecutive pieces (conflict-free);
            // the raw and the lo tile share the (swizzled) offset, so the swizzle never has to be computed here
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t off = (uint32_t)(u * 256 + tid) * 16u;
                const uint4 x = *reinterpret_cast<const uint4*>(st + off);
                uint4 lo;
                lo.x = __float_as_uint(__uint_as_float(x.x) - __uint_as_float(x.x & 0xFFFFE000u));
                lo.y = __float_as_uint(__uint_as_float(x.y) - __uint_as_float(x.y & 0xFFFFE000u));
                lo.z = __float_as_uint(__uint_as_float(x.z) - __uint_as_float(x.z & 0xFFFFE000u));
                lo.w = __float_as_uint(__uint_as_float(x.w) - __uint_as_float(x.w & 0xFFFFE000u));
                *reinterpret_cast<uint4*>(lt + off) = lo;
            }
            {
                const uint32_t off = (uint32_t)tid * 16u;                 // 256 pieces of Omega^T: hi and lo both go to the derived stage
                const uint4 x = *reinterpret_cast<const uint4*>(st + TC_A_BYTES + off);
                uint4 hi, lo;
                split_tf32(__uint_as_float(x.x), hi.x, lo.x);
                split_tf32(__uint_as_float(x.y), hi.y, lo.y);
                split_tf32(__uint_as_float(x.z), hi.z, lo.z);
                split_tf32(__uint_as_float(x.w), hi.w, lo.w);
                *reinterpret_cast<uint4*>(lt + TC_A_BYTES + off) = hi;
                *reinterpret_cast<uint4*>(lt + TC_A_BYTES + TC_B_BYTES + off) = lo;
            }
            fence_async_smem();
            mbar_arrive(&full_bar[l]);
        }
    } else {
        // ================= MMA issue (warp 8, lane 0) + epilogue (warps 8-11) =================
        constexpr uint32_t idesc = umma_idesc_tf32(128, 32);
        constexpr uint32_t idesc64 = umma_idesc_tf32(128, 64);
        const int ew = warp - 8;
        const uint32_t t_lane = (uint32_t)(32 * ew) << 16;
        const uint32_t raw_lo0 = umma_sw128_lo(smem_u32(smem_raw));
        const uint32_t der_lo0 = umma_sw128_lo(smem_u32(lo_base));
        float acc[2][32];
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
            for (int c = 0; c < 32; ++c) acc[t][c] = 0.f;
#pragma unroll 1
        for (int it = 0; it <= n_my; ++it) {
            if (it < n_my && warp == 8 && lane == 0) {
                const int s = it % TMA_RAW, l = it & 1;
                mbar_wait(&full_bar[l], (uint32_t)((it / 2) & 1));
                tc_fence_after();
                // descriptor low words: base + (byte offset >> 4); K step: + 2, next M tile: + 1024
                const uint32_t ah0 = raw_lo0 + (uint32_t)s * (TMA_RAW_BYTES >> 4);
                const uint32_t al0 = der_lo0 + (uint32_t)l * (TMA_LO_BYTES >> 4);
                const uint32_t bh0 = al0 + (TC_A_BYTES >> 4);
                const uint32_t d0 = tmem_base + (uint32_t)((it & 1) * 2 * DCOLS);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint64_t bh = umma_join(bh0 + 2 * t, UMMA_SW128_HI);          // N = 64 spans the hi and the lo tile
#pragma unroll
                    for (int tile = 0; tile < 2; ++tile) {
                        const uint64_t ah = umma_join(ah0 + tile * 1024 + 2 * t, UMMA_SW128_HI);
                        const uint64_t al = umma_join(al0 + tile * 1024 + 2 * t, UMMA_SW128_HI);
                        const uint32_t d = d0 + tile * DCOLS;
                        if (t == 0) { umma_tf32<false>(d, ah, bh, idesc64); umma_tf32<false>(d + 64, al, bh, idesc); }
                        else { umma_tf32<true>(d, ah, bh, idesc64); umma_tf32<true>(d + 64, al, bh, idesc); }
                    }
                }
                umma_commit(&rawfree_bar[s]);
                umma_commit(&lofree_bar[l]);
                umma_commit(&tmem_full_bar[it & 1]);
            }
            __syncwarp();
            if (it >= 1) {
                const int j = it - 1;
                mbar_wait(&tmem_full_bar[j & 1], (uint32_t)((j >> 1) & 1));
                tc_fence_after();
                const uint32_t tb = tmem_base + t_lane + (uint32_t)((j & 1) * 2 * DCOLS);
                // per tile: columns [0, 32) x_hi o_hi, [32, 64) x_hi o_lo, [64, 96) x_lo o_hi: small terms first, then the sum
#pragma unroll
                for (int tile = 0; tile < 2; ++tile)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {                              // 16 columns at a time: register budget
                        uint32_t vh[16], vl[16], vx[16];
                        tmem_ld16(tb + tile * DCOLS + 16 * h, vh);
                        tmem_ld16(tb + tile * DCOLS + 32 + 16 * h, vl);
                        tmem_ld16(tb + tile * DCOLS + 64 + 16 * h, vx);
                        tmem_ld_wait();
#pragma unroll
                        for (int c = 0; c < 16; ++c)
                            acc[tile][16 * h + c] += (__uint_as_float(vl[c]) + __uint_as_float(vx[c])) + __uint_as_float(vh[c]);
                    }
                tc_fence_before();
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
#pragma unroll
        for (int tile = 0; tile < 2; ++tile) {
            const int row = row_base + tile * 128 + 32 * ew + lane;
            if (row < m) {
                float4* out = reinterpret_cast<float4*>(partial + ((size_t)blockIdx.x * m + row) * 32);
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    out[c] = make_float4(acc[tile][4 * c], acc[tile][4 * c + 1], acc[tile][4 * c + 2], acc[tile][4 * c + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TCOLS));
    }
}

// ---- A operand from tensor memory (tcgen05.mma "TS" form): lanes = M rows, one 32-bit column per K element ----
template <bool ACC>
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "n"(ACC ? 1 : 0)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr int TS_STAGES = 3;
constexpr int TS_B_STAGE_BYTES = 2 * TC_B_BYTES;     // Omega / Y chunk, hi + lo (8 KB)
constexpr int TS_TMEM_COLS = 512;                    // 3 stages x 2 tiles x (32 hi + 32 lo) + 2 buffers x 2 tiles x 32
constexpr uint32_t TS_D_COL = 384;

// ---------------------------------------------------------------------------------------------------------
// Bt = Y^T X with the A operand (X^T tile: M = 256 columns of X, K = 32 rows) written by the producers straight
// into tensor memory: lane = column, so every warp load reads 128 contiguous bytes of one row of X and no
// shared-memory staging or transposition of X is needed at all; only the small Y chunk goes through shared memory.
__global__ void __launch_bounds__(TC_THREADS, 1)
xty_ts_kernel(const float* __restrict__ X, int m, long long n, const float* __restrict__ Y, int r, int k0,
              float* __restrict__ Bt)
{
    __shared__ __align__(1024) unsigned char bsm[TS_STAGES * TS_B_STAGE_BYTES];
    __shared__ __align__(8) uint64_t full_bar[TS_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[TS_STAGES];
    __shared__ __align__(8) uint64_t tmem_full_bar[2];
    __shared__ uint32_t tmem_base_sh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
        for (int s = 0; s < TS_STAGES; ++s) {
            mbar_init(&full_bar[s], TC_PRODUCERS);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(&tmem_full_bar[0], 1);
        mbar_init(&tmem_full_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_sh)),
                     "r"(TS_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;

    const int nk = (m + 31) / 32;
    const long long nblk = (n + TC_ROWS - 1) / TC_ROWS;
    const int blk_my = (blockIdx.x < nblk) ? (int)((nblk - 1 - blockIdx.x) / gridDim.x + 1) : 0;
    const int n_my = blk_my * nk;
    auto blk_col = [&](int b) { return ((long long)blockIdx.x + (long long)b * gridDim.x) * TC_ROWS; };

    if (warp < 8) {
        // ================= producers: lane <-> column (warp w: tile w/4, TMEM lanes 32 (w%4) ..) =================
        const int b_n = tid >> 3, b_kc = tid & 7;
        const bool b_ok = (k0 + b_n < r);
        const int col_in_blk = (warp >> 2) * 128 + 32 * (warp & 3) + lane;
        const uint32_t t_lane = (uint32_t)(32 * (warp & 3)) << 16;
        const uint32_t a_col = (uint32_t)((warp >> 2) * 64);                // + stage * 128 (+ 32 for lo)
        auto load_chunk = [&](int it, float (&xv)[32], float (&bv)[4]) {
            const int b = it / nk, kc = it - b * nk;
            const long long col = blk_col(b) + col_in_blk;
            const int i0 = kc * 32;
            const float* src = X + (size_t)i0 * n + col;
            if (col < n && i0 + 32 <= m) {
#pragma unroll
                for (int k = 0; k < 32; ++k) xv[k] = __ldcs(src + (size_t)k * n);
            } else {
#pragma unroll
                for (int k = 0; k < 32; ++k) xv[k] = (col < n && i0 + k < m) ? __ldcs(src + (size_t)k * n) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int row = i0 + 4 * b_kc + j;
                bv[j] = (b_ok && row < m) ? __ldg(Y + (size_t)row * r + k0 + b_n) : 0.f;
            }
        };
        auto step = [&](int it, float (&xv)[32], float (&bv)[4], float (&xl)[32], float (&bl)[4]) {
            if (it >= n_my) return;
            if (it + 2 < n_my) load_chunk(it + 2, xl, bl);
            const int s = it % TS_STAGES;
            if (it >= TS_STAGES) {
                mbar_wait(&empty_bar[s], (uint32_t)((it / TS_STAGES - 1) & 1));     // MMAs of chunk it-3 have read the stage
                tc_fence_after();
            }
            const uint32_t ta = tmem_base + t_lane + (uint32_t)(s * 128) + a_col;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) split_tf32(xv[16 * h + k], hi[k], lo[k]);
                tmem_st16(ta + 16 * h, hi);
                tmem_st16(ta + 32 + 16 * h, lo);
            }
            {
                unsigned char* st = bsm + (size_t)s * TS_B_STAGE_BYTES;
                const uint32_t off = (uint32_t)b_n * 128u + (uint32_t)((b_kc ^ (b_n & 7)) * 16);
                uint4 hi, lo;
                split_tf32(bv[0], hi.x, lo.x);
                split_tf32(bv[1], hi.y, lo.y);
                split_tf32(bv[2], hi.z, lo.z);
                split_tf32(bv[3], hi.w, lo.w);
                *reinterpret_cast<uint4*>(st + off) = hi;
                *reinterpret_cast<uint4*>(st + TC_B_BYTES + off) = lo;
            }
            tmem_wait_st();
            fence_async_smem();
            tc_fence_before();
            mbar_arrive(&full_bar[s]);
        };
        float x0[32], x1[32], x2[32], b0[4], b1[4], b2[4];
        if (n_my > 0) load_chunk(0, x0, b0);
        if (n_my > 1) load_chunk(1, x1, b1);
#pragma unroll 1
        for (int it = 0; it < n_my; it += 3) {
            step(it, x0, b0, x2, b2);
            step(it + 1, x1, b1, x0, b0);
            step(it + 2, x2, b2, x1, b1);
        }
    } else {
        // ================= MMA issue (warp 8, lane 0) + epilogue (warps 8-11) =================
        constexpr uint32_t idesc = umma_idesc_tf32(128, 32);
        const int ew = warp - 8;
        const uint32_t t_lane = (uint32_t)(32 * ew) << 16;
        const uint32_t desc_lo0 = umma_sw128_lo(smem_u32(bsm));
        float acc[2][32];
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
            for (int c = 0; c < 32; ++c) acc[t][c] = 0.f;
#pragma unroll 1
        for (int it = 0; it <= n_my; ++it) {
            if (it < n_my && warp == 8 && lane == 0) {
                const int s = it % TS_STAGES;
                mbar_wait(&full_bar[s], (uint32_t)((it / TS_STAGES) & 1));
                tc_fence_after();
                const uint32_t b_lo0 = desc_lo0 + (uint32_t)s * (TS_B_STAGE_BYTES >> 4);
                const uint32_t d0 = tmem_base + TS_D_COL + (uint32_t)((it & 1) * 64);
                const uint32_t a0 = tmem_base + (uint32_t)(s * 128);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint64_t bh = umma_join(b_lo0 + 2 * t, UMMA_SW128_HI);
                    const uint64_t bl = umma_join(b_lo0 + (TC_B_BYTES >> 4) + 2 * t, UMMA_SW128_HI);
#pragma unroll
                    for (int tile = 0; tile < 2; ++tile) {
                        const uint32_t d = d0 + tile * 32, a_hi = a0 + tile * 64 + 8 * t;
                        if (t == 0) umma_tf32_ts<false>(d, a_hi + 32, bh, idesc); else umma_tf32_ts<true>(d, a_hi + 32, bh, idesc);   // x_lo * y_hi
                        umma_tf32_ts<true>(d, a_hi, bl, idesc);                                    // x_hi * y_lo
                        umma_tf32_ts<true>(d, a_hi, bh, idesc);                                    // x_hi * y_hi
                    }
                }
                umma_commit(&empty_bar[s]);
                umma_commit(&tmem_full_bar[it & 1]);
            }
            __syncwarp();
            if (it >= 1) {
                const int j = it - 1;
                mbar_wait(&tmem_full_bar[j & 1], (uint32_t)((j >> 1) & 1));
                tc_fence_after();
                uint32_t v0[32], v1[32];
                tmem_ld32(tmem_base + t_lane + TS_D_COL + (uint32_t)((j & 1) * 64), v0);
                tmem_ld32(tmem_base + t_lane + TS_D_COL + (uint32_t)((j & 1) * 64 + 32), v1);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[0][c] += __uint_as_float(v0[c]);
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[1][c] += __uint_as_float(v1[c]);
                tc_fence_before();
                if ((j + 1) % nk == 0) {
                    const long long c0 = blk_col(j / nk);
#pragma unroll
                    for (int tile = 0; tile < 2; ++tile) {
                        const long long col = c0 + tile * 128 + 32 * ew + lane;
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            if (col < n && k0 + c < r) __stcs(Bt + (size_t)(k0 + c) * n + col, acc[tile][c]);
                            acc[tile][c] = 0.f;
                        }
                    }
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TS_TMEM_COLS));
    }
}

// fixed-order FP64 sum of the per-CTA partials [nparts][m][32] -> Y[m][r] columns k0 .. k0+31
__global__ void tc_reduce_kernel(const float* __restrict__ partial, int nparts, int m, int r, int k0,
                                 float* __restrict__ Y)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= m * 32) return;
    const int row = idx >> 5, k = idx & 31;
    if (k0 + k >= r) return;
    double s = 0.0;
    for (int p = 0; p < nparts; ++p) s += (double)partial[(size_t)p * m * 32 + idx];
    Y[(size_t)row * r + k0 + k] = (float)s;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
typedef CUresult (*tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static tmap_encode_fn tmap_encoder()
{
    static tmap_encode_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<tmap_encode_fn>(p);
        else
            cudaGetLastError();
    }
    return fn;
}
// row-major float32 [rows][cols], box = box_rows x 32 columns, 128-byte swizzle, zero fill outside.  L2 promotion: a 128-byte
// row piece pulls its 256-byte neighbourhood into L2 -- the other half is the same CTA's next chunk.
static bool make_tmap_f32(CUtensorMap* map, const float* base, long long rows, long long cols, int box_rows)
{
    tmap_encode_fn enc = tmap_encoder();
    if (!enc) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)TC_K, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int tc_sm_count()
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_rsvd_tc_workspace_bytes(int m)
{
    if (m <= 0) return -1;
    return (long long)tc_sm_count() * m * 32 * (long long)sizeof(float);
}

int ggp_rsvd_sketch_tc_f32(const float* X, int m, long long n, const float* OmegaT, int r, float* Y_out, void* workspace,
                           long long workspace_bytes, void* stream)
{
    GGP_ARG(X && OmegaT && Y_out && workspace, "null pointer");
    GGP_ARG(m > 0 && n > 0 && r > 0, "m, n, r must be positive");
    if (workspace_bytes < ggp_rsvd_tc_workspace_bytes(m)) {
        set_error("ggp_rsvd_sketch_tc_f32: workspace too small");
        return GGP_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    float* partial = reinterpret_cast<float*>(workspace);
    const int gy = (m + TC_ROWS - 1) / TC_ROWS;
    const long long nchunk = (n + TC_K - 1) / TC_K;
    long long gx = tc_sm_count() / gy;                       // one CTA per SM (216 KB of shared memory each)
    if (gx < 1) gx = 1;
    if (gx > nchunk) gx = nchunk;
    const size_t smem = (size_t)TC_STAGES * TC_STAGE_BYTES;
    // 16-byte loads of both operands: row pitch a multiple of 16 bytes and 16-byte aligned bases
    const bool vec = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && ((reinterpret_cast<uintptr_t>(OmegaT) & 15) == 0);
    // TMA-fed kernel: additionally, column coordinates within int32 and both tensor maps encode
    CUtensorMap mapX, mapO;
    const bool tma = vec && n < (1LL << 31) && make_tmap_f32(&mapX, X, m, n, TC_ROWS) && make_tmap_f32(&mapO, OmegaT, r, n, 32);
    if (tma) {
        GGP_CUDA(cudaFuncSetAttribute(sketch_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM_BYTES));
        for (int k0 = 0; k0 < r; k0 += 32) {
            sketch_tma_kernel<<<dim3((unsigned)gx, gy), TMA_THREADS, TMA_SMEM_BYTES, st>>>(mapX, mapO, m, n, r, k0, partial);
            GGP_CUDA(cudaGetLastError());
            tc_reduce_kernel<<<(m * 32 + 255) / 256, 256, 0, st>>>(partial, (int)gx, m, r, k0, Y_out);
            GGP_CUDA(cudaGetLastError());
        }
        return GGP_OK;
    }
    GGP_CUDA(cudaFuncSetAttribute(sketch_tc_kernel<true, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GGP_CUDA(cudaFuncSetAttribute(sketch_tc_kernel<false, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int k0 = 0; k0 < r; k0 += 32) {
        if (vec) sketch_tc_kernel<true, 8><<<dim3((unsigned)gx, gy), 384, smem, st>>>(X, m, n, OmegaT, r, k0, partial);
        else sketch_tc_kernel<false, 8><<<dim3((unsigned)gx, gy), 384, smem, st>>>(X, m, n, OmegaT, r, k0, partial);
        GGP_CUDA(cudaGetLastError());
        tc_reduce_kernel<<<(m * 32 + 255) / 256, 256, 0, st>>>(partial, (int)gx, m, r, k0, Y_out);
        GGP_CUDA(cudaGetLastError());
    }
    return GGP_OK;
}

int ggp_rsvd_xty_tc_f32(const float* X, int m, long long n, const float* Y, int r, float* Bt_out, void* stream)
{
    GGP_ARG(X && Y && Bt_out, "null pointer");
    GGP_ARG(m > 0 && n > 0 && r > 0, "m, n, r must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    const long long nblk = (n + TC_ROWS - 1) / TC_ROWS;
    long long gx = tc_sm_count();
    if (gx > nblk) gx = nblk;
    for (int k0 = 0; k0 < r; k0 += 32) {
        xty_ts_kernel<<<(unsigned)gx, TC_THREADS, 0, st>>>(X, m, n, Y, r, k0, Bt_out);
        GGP_CUDA(cudaGetLastError());
    }
    return GGP_OK;
}

}  // extern "C"
