// Fused covariance build + blocked Cholesky + log-determinant + forward solve for ONE matrix per CTA.
//
// Replaces, for one (chain, PC) block evaluation, the reference chain
//   SepiaDistCov.compute_cov_mat -> np.fill_diagonal(nuggets) -> scipy.linalg.cholesky ->
//   scipy.linalg.solve_triangular -> -sum(log diag L) - 0.5 ||L^-1 w||^2
// (SURVEY.md 8a rows a3+a4 / Appendix A.10 cov_self, do_loglik, log_lik; called from
//  /root/reference/src/model.py:234-235 through sepia).
//
// Algorithm: left-looking blocked Cholesky, panel width 32, 128 threads (four warps), four CTAs per SM.  For panel j:
//   1. S = L[rows, 0:32j] * L[panel rows, 0:32j]^T on the FP64 tensor cores (DMMA.8x8x4), accumulators
//      in registers, A/B fragments are 16-byte loads straight from the packed factor;
//   2. covariance entries of the panel computed in the accumulator layout (squared distances as a rank-(d+2) DMMA
//      product, exp fused, nothing read from HBM), P = C - S stays in registers;
//   3. the 32x32 diagonal block goes through shared memory: warp 0 factors it (row per lane), then
//      warp 0 forward-solves the w block and stores the diagonal rows while warp 1 inverts the block;
//   4. X = P * Minv^T again on DMMA: the accumulator fragments of step 2 are valid A fragments under a
//      permutation of the k index, so no data movement is needed; X is stored to the packed factor
//      straight from the fragments and the running forward solve of w is updated.
// The covariance matrix itself never exists in memory.  Two schedules of the same arithmetic (bit-identical results):
//   eval_block_loglik_la       look-ahead (one CTA per matrix): step 3 of panel j+1 runs while panel j is finished;
//   eval_block_loglik<true>    one matrix per thread-block cluster (small batches, large matrices): steps 1-4 per panel.
// eval_block_loglik<false, 1> runs steps 1-4 in one CTA on a given matrix (the prediction path's draw, ggp_chol_draw_f64).
// The serial phase is written as compact loops over shared memory: a fully unrolled register version made the
// kernel 200 KB of SASS and instruction-fetch bound (profiles/README.md).
#pragma once
#include <cstdlib>
#include "ggp_common.cuh"

namespace ggp {

// entries of the shared-memory table of the in-kernel exponential (exp_neg below)
constexpr int ETAB = 64;

// DMMA steps / shared-memory doubles of the covariance distance product (see pair_cov)
__host__ __device__ inline int cov_ksteps(int d) { return (d + 5) >> 2; }
__host__ __device__ inline int sc_doubles(int d) { return 128 * cov_ksteps(d); }

struct EvalSmem {
    double* D;      // [32][D_LD]   diagonal block: P on entry, rows of Ljj after the factorisation
    double* LT;     // [32][LT_LD]  LT[k][i] = L[i][k]
    double* Minv;   // [32][MI_LD]  Minv[c][k] = (Ljj^-1)[c][k]
    double* rdiag;  // [32]
    double* uj;     // [32]
    double* red;    // [8]
    double* etab;   // [ETAB] 2^(j/ETAB)
    double* wres;   // [Mp]
    double* sb;     // [d]     sqrt(beta)
    double* SC;     // [sc_doubles(d)] B fragments of the distance product for the current panel's columns
    int* flag;      // [4]
    int* soff;      // [4*nP] offset (doubles) of sub-slab s = 4*kb + ks such that soff[s] + r*8 + c addresses row r
};

__host__ __device__ inline size_t eval_smem_bytes(int Mp, int d) {
    return (size_t)(32 * D_LD + 32 * LT_LD + 32 * MI_LD + 32 + 32 + 8 + ETAB + Mp + (size_t)sc_doubles(d) + ((d + 1) & ~1)) * sizeof(double) + 16 + (size_t)(Mp / 8) * sizeof(int);
}

// shared-memory carve-out (percent of 228 KB) that just fits CTAS_PER_SM CTAs: the rest stays L1 so that the
// B-operand rows of a panel, shared by the warps of a CTA, are served from L1 instead of L2
inline int eval_carveout_pct(size_t smem) {
    size_t need = CTAS_PER_SM * (smem + 1024);
    int pct = (int)((need * 100 + 228 * 1024 - 1) / (228 * 1024));
    return pct > 100 ? 100 : pct;
}

__device__ inline EvalSmem carve_eval_smem(unsigned char* base, int Mp, int d) {
    EvalSmem s;
    double* p = reinterpret_cast<double*>(base);
    s.Minv = p;     p += 32 * MI_LD;
    s.LT = p;       p += 32 * LT_LD;     // LT and D are contiguous: outside the diagonal-block phase the two
    s.D = p;        p += 32 * D_LD;      // serve as per-warp scratch of the covariance step (NWARP x 2 KB)
    s.rdiag = p;    p += 32;
    s.uj = p;       p += 32;
    s.red = p;      p += 8;
    s.etab = p;     p += ETAB;
    s.wres = p;     p += Mp;
    s.SC = p;       p += (size_t)sc_doubles(d);
    s.sb = p;       p += ((d + 1) & ~1);
    s.flag = reinterpret_cast<int*>(p);
    s.soff = s.flag + 4;
    return s;
}

// exp(y) for y <= 0, ~1 ulp: y = (T n + j) ln2/T + r, |r| <= ln2/(2T), exp(y) = 2^n * 2^(j/T) * p(r), T = ETAB = 64 table
// entries.  |r| <= 0.0054, the r^6/720 term is below 4e-17, so degree 5 is enough: 10 operations on the FP64 pipe the DMMAs
// share (libdevice exp: ~25), and a fraction of its code size.
// Results below 1e-300 flush to 0 (covariance entries that small cannot influence any result at 1e-8).
__device__ __forceinline__ double exp_neg(double y, const double* __restrict__ etab)
{
    const double t = fma(y, 92.33248261689366, 6755399441055744.0);          // T/ln2, 1.5*2^52
    const int nt = __double2loint(t);
    const double fn = t - 6755399441055744.0;
    double r = fma(fn, -0.010830424695086549, y);                               // ln2/T high part (low 20 mantissa bits zero)
    r = fma(fn, -1.162596423439437e-12, r);                                     // ln2/T low part
    double p = 8.3333333333333332e-03;                                          // 1/120
    p = fma(p, r, 4.1666666666666664e-02);
    p = fma(p, r, 1.6666666666666666e-01);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    const double v = p * etab[nt & (ETAB - 1)];
    const int n = nt >> 6;
    const double res = __hiloint2double(__double2hiint(v) + (n << 20), __double2loint(v));
    return (y < -690.0) ? 0.0 : res;
}

__device__ inline void fill_exp_table(double* etab)
{
    if (threadIdx.x < ETAB) etab[threadIdx.x] = exp2((double)threadIdx.x * (1.0 / ETAB));
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

__device__ inline void fill_slab_offsets(int* soff, int Mp)
{
    for (int s = threadIdx.x; s < Mp / 8; s += blockDim.x) {
        const int kb = s >> 2, ks = s & 3;
        soff[s] = (int)(panel_off(kb, Mp) + (long long)ks * (Mp - 32 * kb) * 8 - 32LL * kb * 8);
    }
}

// S += A[rows, 0:32j] * Lb[panel rows, 0:32j]^T for NU 8-row units of one warp (DMMA.8x8x4).
// A-operand rows come from `Ap` (packed factor layout when a_ld == 0, else a [slab][a_ld][8] layout
// indexed by local row), B-operand rows from the packed factor `Lb`.  NU is a template parameter so
// that no predicated-off DMMA is ever issued (a predicated-off DMMA still occupies the pipe).
// Latency: the A fragment of the next sub-slab is loaded one iteration ahead into registers; further
// ahead, lanes 0..4NU-1 pull the A lines of sub-slab s+6 into L2 and lanes 16..31 the B lines of
// sub-slab s+2 into L1 (the B rows are shared by all warps of the CTA).
template <int NU>
static __device__ __forceinline__ void panel_gemm(double (&acc)[2][4][2], const double* __restrict__ Ap,
                                                  const double* __restrict__ Lb, const int* __restrict__ soff, int j,
                                                  int row0, const int (&rb)[2], int g, int q, int a_ld)
{
    constexpr int PD = 2;                    // prefetch distance in k-blocks (4 sub-slabs each)
    constexpr int RA = 2, RB = 2;            // register ring depths (sub-slabs) of the A and B fragments: loads run R - 1 ahead
    const int lane = 4 * g + q;
    const int nsub = 4 * j;
    // sub-slab pointers: packed factor -> soff table; V workspace (a_ld != 0) -> s * a_ld * 8
    auto a_slab = [&](int s) -> const double* { return a_ld ? Ap + (size_t)s * a_ld * 8 : Ap + soff[s]; };
    // prefetch roles, one 128-byte line per lane and sub-slab group:
    //   A: unit (lane>>4)%NU, sub-slab (lane>>2)&3, line lane&3      (NU*16 lines per k-block)
    //   B: sub-slab lane>>3 (two passes: +0 / +... ) see below
    const int pa_unit = ((lane >> 4) < NU) ? (lane >> 4) : 0;
    const int pa_ks = (lane >> 2) & 3;
    const int pa_off = ((pa_unit == 0) ? rb[0] : rb[1]) * 8 + (lane & 3) * 16;
    const int pb_ks = lane >> 3;                                      // 8 lanes per sub-slab, 2 lines each
    const int pb_off = (row0 + 4 * (lane & 7)) * 8;
    int aoff[NU];
#pragma unroll
    for (int i = 0; i < NU; ++i) aoff[i] = (rb[i] + g) * 8 + 2 * q;
    const int boff = (row0 + g) * 8 + 2 * q;
    double2 ar[RA][NU], br[RB][4];          // fragment rings: slot s % R holds sub-slab s
#pragma unroll
    for (int t = 0; t < RA - 1; ++t)
        if (t < nsub) {
            const double* sl = a_slab(t);
#pragma unroll
            for (int i = 0; i < NU; ++i) ar[t][i] = ldcg2(sl + aoff[i]);
        }
#pragma unroll
    for (int t = 0; t < RB - 1; ++t)
        if (t < nsub) {
            const double* sl = Lb + soff[t] + boff;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) br[t][cb] = *reinterpret_cast<const double2*>(sl + 64 * cb);
        }
    for (int kb = 0; kb < j; ++kb) {
        if (kb + PD < j) {
            const int sp = 4 * (kb + PD);
            prefetch_l2(a_slab(sp + pa_ks) + pa_off);
            const double* pb = Lb + soff[sp + pb_ks] + pb_off;
            prefetch_l1(pb);
            prefetch_l1(pb + 16);
        }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            const int s = 4 * kb + ks;
            // loads of sub-slab s + R - 1 go into the slot that sub-slab s - 1 has just left
            if (s + RA - 1 < nsub) {
                const double* sn = a_slab(s + RA - 1);
#pragma unroll
                for (int i = 0; i < NU; ++i) ar[(ks + RA - 1) % RA][i] = ldcg2(sn + aoff[i]);
            }
            if (s + RB - 1 < nsub) {
                const double* sbn = Lb + soff[s + RB - 1] + boff;
#pragma unroll
                for (int cb = 0; cb < 4; ++cb) br[(ks + RB - 1) % RB][cb] = *reinterpret_cast<const double2*>(sbn + 64 * cb);
            }
            const double2 (&a)[NU] = ar[ks % RA];
            const double2 (&b)[4] = br[ks % RB];
            // all even-k DMMAs first, then the odd-k ones: dependent DMMAs on one accumulator are 4*NU apart
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int i = 0; i < NU; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].x, b[cb].x);
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int i = 0; i < NU; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].y, b[cb].y);
        }
    }
}

// ---- asynchronous copies (LDGSTS): global -> shared memory without a register stage ------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Same product as panel_gemm (identical DMMA sequence per accumulator, hence bit-identical results), but the A
// fragments travel global -> shared memory by cp.async (LDGSTS.128, L2 only) DA-1 sub-slabs ahead of their use instead
// of one sub-slab ahead through registers: a warp no longer waits a full L2 / DRAM round trip per sub-slab, and the
// loads in flight cost no registers.  The 16-byte piece a lane needs of an 8-row x 8-column unit block is piece number
// `lane` of that block (row g, columns 2q..2q+1), so every lane copies exactly the pieces it later reads: no
// cross-lane synchronisation, cp.async.wait_group alone orders the copy before the LDS.128 (conflict-free: consecutive
// lanes, consecutive 16-byte pieces).  `ring`: per-warp shared memory, DA * NU * 64 <= 512 doubles (the warp's covariance
// scratch: idle during the product).  Packed-factor A operand only.
template <int NU>
static __device__ __forceinline__ void panel_gemm_cp(double (&acc)[2][4][2], const double* __restrict__ Ap,
                                                     const double* __restrict__ Lb, const int* __restrict__ soff, int j,
                                                     int row0, const int (&rb)[2], int g, int q, double* __restrict__ ring)
{
    constexpr int PD = 2;                    // L2 prefetch distance in k-blocks (4 sub-slabs each)
    constexpr int DA = 4;                    // depth (sub-slabs) of the shared-memory ring of A fragments
    constexpr int RB = 2;                    // register ring depth of the B fragments
    const int lane = 4 * g + q;
    const int nsub = 4 * j;
    const int pa_unit = ((lane >> 4) < NU) ? (lane >> 4) : 0;
    const int pa_ks = (lane >> 2) & 3;
    const int pa_off = ((pa_unit == 0) ? rb[0] : rb[1]) * 8 + (lane & 3) * 16;
    int aoff[NU];
#pragma unroll
    for (int i = 0; i < NU; ++i) aoff[i] = (rb[i] + g) * 8 + 2 * q;
    const int boff = (row0 + g) * 8 + 2 * q;
    double* __restrict__ mine = ring + 2 * lane;              // this lane's piece; slot t, unit i at + (t * NU + i) * 64
    double2 br[RB][4];
    __syncwarp();                                             // previous user of the scratch (covariance step) is done
#pragma unroll
    for (int t = 0; t < DA - 1; ++t) {
        if (t < nsub) {
            const double* sl = Ap + soff[t];
#pragma unroll
            for (int i = 0; i < NU; ++i) cp_async16(mine + (t * NU + i) * 64, sl + aoff[i]);
        }
        cp_async_commit();
    }
#pragma unroll
    for (int t = 0; t < RB - 1; ++t)
        if (t < nsub) {
            const double* sl = Lb + soff[t] + boff;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) br[t][cb] = *reinterpret_cast<const double2*>(sl + 64 * cb);
        }
    for (int kb = 0; kb < j; ++kb) {
        if (kb + PD < j) prefetch_l2(Ap + soff[4 * (kb + PD) + pa_ks] + pa_off);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            const int s = 4 * kb + ks;
            if (s + DA - 1 < nsub) {
                const double* sn = Ap + soff[s + DA - 1];
                const int slot = (ks + DA - 1) % DA;
#pragma unroll
                for (int i = 0; i < NU; ++i) cp_async16(mine + (slot * NU + i) * 64, sn + aoff[i]);
            }
            cp_async_commit();
            if (s + RB - 1 < nsub) {
                const double* sbn = Lb + soff[s + RB - 1] + boff;
#pragma unroll
                for (int cb = 0; cb < 4; ++cb) br[(ks + RB - 1) % RB][cb] = *reinterpret_cast<const double2*>(sbn + 64 * cb);
            }
            cp_async_wait<DA - 1>();                          // sub-slab s has landed (the DA-1 younger groups may be in flight)
            double2 a[NU];
#pragma unroll
            for (int i = 0; i < NU; ++i) a[i] = *reinterpret_cast<const double2*>(mine + (ks * NU + i) * 64);
            const double2 (&b)[4] = br[ks % RB];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int i = 0; i < NU; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].x, b[cb].x);
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int i = 0; i < NU; ++i) dmma884(acc[i][cb][0], acc[i][cb][1], a[i].y, b[cb].y);
        }
    }
}

// One 8-row unit: X = P * Minv^T on DMMA.  p[cb][e] (accumulator layout) doubles as the A fragment.
static __device__ __forceinline__ void unit_trsm(const double (&p)[4][2], double (&x)[4][2],
                                                 const double* __restrict__ Minv, int g, int q)
{
#pragma unroll
    for (int cb = 0; cb < 4; ++cb) {
        x[cb][0] = 0.0; x[cb][1] = 0.0;
#pragma unroll
        for (int kb = 0; kb <= cb; ++kb) {
            const double2 b = *reinterpret_cast<const double2*>(Minv + (8 * cb + g) * MI_LD + 8 * kb + 2 * q);
            dmma884(x[cb][0], x[cb][1], p[kb][0], b.x);
            dmma884(x[cb][0], x[cb][1], p[kb][1], b.y);
        }
    }
}

// Covariance entries of NU units (8 rows x 32 panel columns each) in the accumulator layout: p = C - p.
// The squared distances are a rank-(d+2) product on the FP64 tensor cores:
//   -dist(i, c) = [x~_i, |x~_i|^2, 1] . [2 x~_c, -1, -|x~_c|^2],   x~ = sqrt(beta) o x,
// KS = ceil((d+2)/4) DMMA.8x8x4 steps per 8x8 tile instead of 2d DADD/DFMA per entry (the difference form kept the
// FP64 pipe -- shared with DMMA -- busy with 16x more instructions; profiles/README.md).  The cancellation costs
// a few ulp of |x~|^2 in dist, i.e. ~1e-15 relative in a covariance entry for coordinates in [0, 1].
// Row coordinates come from global memory (Xr[r][d], L1/L2 resident); the panel side (B fragments, shared by all
// units of a panel) sits in shared memory, filled by fill_panel_coords: SCB[s][cb][lane] = B[k = 4s + lane%4][n = 8cb + lane/4].
// self: rows are training points (diagonal / padding rules).  The 8*NU exponentials go through a per-warp
// shared-memory scratch (scr[16][32]) and a 4-way unrolled loop, so the exp code exists 4 times in the kernel
// instead of 32: the fully inlined version made the kernel > 100 KB of SASS and instruction-fetch bound.

// -dist for NU units x 32 panel columns: dn += [x~, |x~|^2, 1] . B.  KS > 0: compile-time step count (the row values
// stay in registers: every global load of the pair is in flight before the first use); KS = 0: runtime loop.
template <int NU, int KS>
static __device__ __forceinline__ void cov_dist(double (&dn)[2][4][2], const double* const (&xr)[2],
                                                const double* __restrict__ SCB, const double* __restrict__ sb,
                                                int d, int q, int lane)
{
    if constexpr (KS > 0) {
        double x[NU][KS];
#pragma unroll
        for (int i = 0; i < NU; ++i)
#pragma unroll
            for (int s = 0; s < KS; ++s) x[i][s] = (4 * s + q < d) ? __ldg(xr[i] + 4 * s + q) : 0.0;
        double rn[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) {
            double part = 0.0;
#pragma unroll
            for (int s = 0; s < KS; ++s) {
                const int k = 4 * s + q;
                x[i][s] = (k < d) ? x[i][s] * sb[k] : 0.0;
                part = fma(x[i][s], x[i][s], part);
            }
            part += __shfl_xor_sync(0xffffffffu, part, 1);
            part += __shfl_xor_sync(0xffffffffu, part, 2);
            rn[i] = part;
        }
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const int k = 4 * s + q;
            double a[NU];
#pragma unroll
            for (int i = 0; i < NU; ++i) a[i] = (k < d) ? x[i][s] : ((k == d) ? rn[i] : ((k == d + 1) ? 1.0 : 0.0));
            const double* bs = SCB + s * 128 + lane;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                const double b = bs[cb * 32];
#pragma unroll
                for (int i = 0; i < NU; ++i) dmma884(dn[i][cb][0], dn[i][cb][1], a[i], b);
            }
        }
    } else {
        const int ks = cov_ksteps(d);
        double rn[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) {
            // squared norm of the scaled row: the four lanes of a row (q = 0..3) each sum the k = q (mod 4) terms
            double part = 0.0;
            for (int s = 0; s < ks; ++s) {
                const int k = 4 * s + q;
                const double x = (k < d) ? __ldg(xr[i] + k) * sb[k] : 0.0;
                part = fma(x, x, part);
            }
            part += __shfl_xor_sync(0xffffffffu, part, 1);
            part += __shfl_xor_sync(0xffffffffu, part, 2);
            rn[i] = part;
        }
#pragma unroll 1
        for (int s = 0; s < ks; ++s) {
            const int k = 4 * s + q;
            double a[NU];
#pragma unroll
            for (int i = 0; i < NU; ++i) {
                const double x = (k < d) ? __ldg(xr[i] + k) * sb[k] : 0.0;
                a[i] = (k < d) ? x : ((k == d) ? rn[i] : ((k == d + 1) ? 1.0 : 0.0));
            }
            const double* bs = SCB + s * 128 + lane;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                const double b = bs[cb * 32];
#pragma unroll
                for (int i = 0; i < NU; ++i) dmma884(dn[i][cb][0], dn[i][cb][1], a[i], b);
            }
        }
    }
}

template <int NU>
static __device__ __forceinline__ void pair_cov(double (&p)[2][4][2], const double* __restrict__ Xr, const int (&r)[2],
                                                const bool (&row_ok)[2], const double* __restrict__ SCB,
                                                const double* __restrict__ sb, int d, int m, int row0, int q,
                                                double inv_lamz, double diag, bool self,
                                                const double* __restrict__ etab, double* __restrict__ scr, int lane)
{
    double dn[2][4][2];
    const double* xr[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) { dn[i][cb][0] = 0.0; dn[i][cb][1] = 0.0; }
        xr[i] = Xr + (size_t)((i < NU && row_ok[i]) ? r[i] : 0) * d;
    }
    switch (cov_ksteps(d)) {       // d <= 18 (every configuration of the reference: d = 2 -> 1 step, 9 -> 3, 17 -> 5): register-resident form
        case 1: cov_dist<NU, 1>(dn, xr, SCB, sb, d, q, lane); break;
        case 2: cov_dist<NU, 2>(dn, xr, SCB, sb, d, q, lane); break;
        case 3: cov_dist<NU, 3>(dn, xr, SCB, sb, d, q, lane); break;
        case 4: cov_dist<NU, 4>(dn, xr, SCB, sb, d, q, lane); break;
        case 5: cov_dist<NU, 5>(dn, xr, SCB, sb, d, q, lane); break;
        default: cov_dist<NU, 0>(dn, xr, SCB, sb, d, q, lane); break;
    }
#pragma unroll
    for (int i = 0; i < NU; ++i)
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            scr[(8 * i + 2 * cb) * 32 + lane] = dn[i][cb][0];
            scr[(8 * i + 2 * cb + 1) * 32 + lane] = dn[i][cb][1];
        }
#pragma unroll 8
    for (int e = 0; e < 8 * NU; ++e) scr[e * 32 + lane] = exp_neg(scr[e * 32 + lane], etab);
#pragma unroll
    for (int i = 0; i < NU; ++i)
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = row0 + 8 * cb + 2 * q + e;
                double v = (row_ok[i] && c < m) ? scr[(8 * i + 2 * cb + e) * 32 + lane] * inv_lamz : 0.0;
                if (self && r[i] == c) v = (r[i] < m) ? diag : 1.0;
                p[i][cb][e] = v - p[i][cb][e];
            }
        }
}

// B fragments of the distance product for the 32 columns of panel `row0` -> SCB[s][cb][lane]; all threads of the CTA
// (contains a __syncthreads: the column norms are summed from the scaled coordinates already in shared memory, not
// from d dependent global loads); caller syncs afterwards
static __device__ __forceinline__ void fill_panel_coords(double* __restrict__ SCB, const double* __restrict__ X,
                                                         const double* __restrict__ sb, int d, int m, int row0)
{
    const int n = sc_doubles(d);
    for (int idx = threadIdx.x; idx < n; idx += blockDim.x) {
        const int s = idx >> 7, cb = (idx >> 5) & 3, ln = idx & 31;
        const int k = 4 * s + (ln & 3), c = row0 + 8 * cb + (ln >> 2);
        double v = 0.0;
        if (c < m) {
            if (k < d) v = 2.0 * (__ldg(X + (size_t)c * d + k) * sb[k]);
            else if (k == d) v = -1.0;
        }
        SCB[idx] = v;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int cc = threadIdx.x;                          // column of the panel: cb = cc / 8, g = cc % 8
        if (row0 + cc < m) {
            double rr = 0.0;
            for (int t = 0; t < d; ++t) {
                const double x = 0.5 * SCB[(t >> 2) * 128 + (cc >> 3) * 32 + (cc & 7) * 4 + (t & 3)];
                rr = fma(x, x, rr);
            }
            const int k = d + 1;
            SCB[(k >> 2) * 128 + (cc >> 3) * 32 + (cc & 7) * 4 + (k & 3)] = -rr;
        }
    }
}

// Whole-CTA evaluation (NT threads).  Returns the block log-likelihood term to every thread;
// *info (if non-null, written by thread 0) = 0 or 1-based index of the failing pivot.
// beta may point to global or shared memory.  Lp is the packed-factor workspace (packed_doubles(Mp)).
// u_out (nullable): receives L^-1 w (Mp entries, zero padded).
// CL = true: the matrix is shared by the CTAs of a thread-block cluster (cluster size G = %cluster_nctarank):
// 8-row units are dealt round-robin to the G*NWARP warps, CTA 0 owns the diagonal block and publishes Minv / u
// through global memory, panels are separated by cluster barriers (release/acquire), the running forward solve
// of w lives in global memory.  Only CTA 0 returns the value.
// SRC = 1 (one CTA per matrix only): the matrix is GIVEN -- X points to a symmetric m x m row-major array instead of
// coordinates (d = 0, beta unused) -- and the vector step is a product instead of a solve: u_out[0:m] = L w (the
// multivariate-normal draw of the prediction path, ggp_chol_draw_f64).  The factorisation arithmetic is the same code.
template <bool CL = false, int SRC = 0>
static __device__ __forceinline__ double eval_block_loglik(const EvalSmem& sm, const double* __restrict__ X, int m, int Mp, int d,
                                    const double* beta, double lamz, double diag_add,
                                    const double* __restrict__ w, double* __restrict__ Lp,
                                    double* __restrict__ u_out, int* info)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int crank = CL ? (int)cluster_ctarank() : 0;
    const int G = CL ? (int)cluster_nctarank() : 1;
    const int gw = crank * NWARP + warp, TW = G * NWARP;       // warp index / warp count over the cluster
    double* __restrict__ aux = Lp + aux_off(Mp);               // [Mp] wres, [32] u block, [32] flag (cluster variant)
    double* __restrict__ wres = CL ? aux : sm.wres;
    const int g = lane >> 2, q = lane & 3;
    const int nP = Mp >> 5;
    const double inv_lamz = 1.0 / lamz;
    const double diag = inv_lamz + diag_add;
    double* __restrict__ D = sm.D;
    double* __restrict__ LT = sm.LT;

    if (CL) cluster_sync_all();   // previous evaluation (and the caller's state update) finished cluster-wide
    __syncthreads();   // previous user of the shared buffers is done
    if (tid < d) sm.sb[tid] = sqrt(beta[tid]);
    static_assert(!(CL && SRC != 0), "given-matrix mode runs one CTA per matrix");
    for (int r = crank * NT + tid; r < Mp; r += G * NT) wres[r] = (SRC == 0 && r < m) ? w[r] : 0.0;
    if (CL && crank == 0 && tid == 0) aux[Mp + 32] = 0.0;
    fill_exp_table(sm.etab);
    fill_slab_offsets(sm.soff, Mp);
    if (tid == 0) sm.flag[0] = 0;
    double logdet = 0.0, quad = 0.0;    // partial sums, live in warp 0
    __syncthreads();

    for (int j = 0; j < nP; ++j) {
        const int row0 = j << 5;
        const int Rj = Mp - row0;
        double* __restrict__ Lpj = Lp + panel_off(j, Mp);
        const int nunits = Rj >> 3;
        // this warp owns units u = warp + NWARP*t (t = 0, 1, ...), processed two at a time; units 0..3 are the
        // diagonal block
        const int nmy = (nunits - gw + TW - 1) / TW;
        const int npairs = max(1, (nmy + 1) >> 1);          // every warp runs pair 0 (it holds the barriers)
        if (CL) cluster_sync_all();                          // panel j-1 (factor rows, wres) visible cluster-wide
        if constexpr (SRC == 0) fill_panel_coords(sm.SC, X, sm.sb, d, m, row0);
        __syncthreads();
        double* __restrict__ scr = LT + warp * 512;          // per-warp scratch of the covariance step (LT and D are idle then)
        static_assert(NWARP * 512 <= 32 * LT_LD + 32 * D_LD, "covariance scratch must fit in LT + D");

#pragma unroll 1
        for (int pr = 0; pr < npairs; ++pr) {
            const int t0 = 2 * pr;
            const int nu = max(0, min(2, nmy - t0));
            double acc[2][4][2];
            int rb[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                rb[i] = row0 + 8 * (gw + TW * (t0 + ((i < nu) ? i : 0)));
#pragma unroll
                for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
            }
            // ------------------------------------------------------------------ 1. DMMA update
            if (j > 0) {
                if (nu == 2) panel_gemm_cp<2>(acc, Lp, Lp, sm.soff, j, row0, rb, g, q, scr);
                else if (nu == 1) panel_gemm_cp<1>(acc, Lp, Lp, sm.soff, j, row0, rb, g, q, scr);
            }
            // ------------------------------------------------------------------ 2. covariance, P = C - S (registers)
            if constexpr (SRC == 0) {
                const int rr[2] = {rb[0] + g, rb[1] + g};
                const bool ok[2] = {rr[0] < m, rr[1] < m};
                if (nu == 2) pair_cov<2>(acc, X, rr, ok, sm.SC, sm.sb, d, m, row0, q, inv_lamz, diag, true, sm.etab, scr, lane);
                else if (nu == 1) pair_cov<1>(acc, X, rr, ok, sm.SC, sm.sb, d, m, row0, q, inv_lamz, diag, true, sm.etab, scr, lane);
            } else {
                // entries of the given matrix (identity in the padding rows and columns)
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    if (i < nu) {
                        const int r = rb[i] + g;
#pragma unroll
                        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int c = row0 + 8 * cb + 2 * q + e;
                                const double v = (r < m && c < m) ? __ldg(X + (size_t)r * m + c) : ((r == c) ? 1.0 : 0.0);
                                acc[i][cb][e] = v - acc[i][cb][e];
                            }
                    }
                }
            }

            // ------------------------------------------------------------------ 3. diagonal block (first pair only)
            if (pr == 0) {
                __syncthreads();          // every warp is done with its covariance scratch (it aliases D)
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int u = gw + TW * i;
                    if (i < nu && u < 4) {
#pragma unroll
                        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                            for (int e = 0; e < 2; ++e)
                                D[(8 * u + g) * D_LD + 8 * cb + 2 * q + e] = acc[i][cb][e];
                    }
                }
                if (!CL || crank == 0) {
                __syncthreads();                                                 // (A)
                if (warp == 0) {
                    // Cholesky of the 32x32 block, lane = row.  Columns in blocks of 8 held in registers; pivots and
                    // multipliers are broadcast through shared memory (a double shuffle is ~25 SASS instructions
                    // with its divergence fallback); trailing columns get one rank-8 update per block.
                    double mypiv = 1.0;
                    int bad = 0;
#pragma unroll 1
                    for (int k0 = 0; k0 < 32; k0 += 8) {
                        double x[8];
#pragma unroll
                        for (int kk = 0; kk < 8; ++kk) x[kk] = D[lane * D_LD + k0 + kk];
#pragma unroll
                        for (int kk = 0; kk < 8; ++kk) {
                            const int k = k0 + kk;
                            if (lane == k) sm.red[2] = x[kk];
                            __syncwarp();
                            const double dk = sm.red[2];
                            if (!(dk > 0.0) || !(dk < 1.0e300)) { if (!bad) bad = row0 + k + 1; }
                            const double rk = rsqrt(dk);
                            const double lik = (lane == k) ? dk * rk : x[kk] * rk;
                            if (lane == k) mypiv = dk;
                            x[kk] = lik;
                            if (lane == 0) sm.rdiag[k] = rk;
                            LT[k * LT_LD + lane] = (lane >= k) ? lik : 0.0;
                            __syncwarp();
#pragma unroll
                            for (int k2 = kk + 1; k2 < 8; ++k2) x[k2] = fma(-lik, LT[k * LT_LD + k0 + k2], x[k2]);
                        }
#pragma unroll
                        for (int kk = 0; kk < 8; ++kk) D[lane * D_LD + k0 + kk] = (lane >= k0 + kk) ? x[kk] : 0.0;
#pragma unroll 2
                        for (int c = k0 + 8; c < 32; ++c) {
                            double a = D[lane * D_LD + c];
#pragma unroll
                            for (int kk = 0; kk < 8; ++kk) a = fma(-x[kk], LT[(k0 + kk) * LT_LD + c], a);
                            D[lane * D_LD + c] = a;
                        }
                        __syncwarp();
                        if (bad) break;
                    }
                    if (bad) { if (lane == 0) { sm.flag[0] = bad; if (CL) aux[Mp + 32] = (double)bad; } }
                    else logdet += 0.5 * log(mypiv);
                }
                __syncthreads();                                                 // (B0)
                const bool failed = sm.flag[0] != 0;
                if (!CL && failed) {
                    if (tid == 0 && info) *info = sm.flag[0];
                    return -INFINITY;
                }
                if (warp == 0 && !failed) {
                    double myu = 0.0;
                    if constexpr (SRC == 0) {
                    // forward solve of the w block: u = Ljj^-1 wres[row0 : row0+32]
                    double b = wres[row0 + lane];
#pragma unroll 1
                    for (int c = 0; c < 32; ++c) {
                        const double uc = __shfl_sync(0xffffffffu, b, c) * sm.rdiag[c];
                        if (lane == c) myu = uc;
                        if (lane > c) b = fma(-D[lane * D_LD + c], uc, b);
                    }
                    sm.uj[lane] = myu;
                    if (CL) aux[Mp + lane] = myu;
                    quad += myu * myu;
                    if (u_out) u_out[row0 + lane] = myu;
                    } else {
                    // product step: (L w)[row0 + lane] = earlier panels (wres) + the diagonal block's row (zeros above the diagonal)
                    sm.uj[lane] = (row0 + lane < m) ? w[row0 + lane] : 0.0;
                    __syncwarp();
                    double b = wres[row0 + lane];
#pragma unroll 4
                    for (int c = 0; c < 32; ++c) b = fma(D[lane * D_LD + c], sm.uj[c], b);
                    if (row0 + lane < m) u_out[row0 + lane] = b;
                    }
                    // store the diagonal rows of L (zeros above the diagonal)
#pragma unroll 1
                    for (int ks = 0; ks < 4; ++ks) {
                        double* dst = Lpj + (long long)ks * Rj * 8 + (long long)lane * 8;
#pragma unroll
                        for (int c = 0; c < 8; c += 2) {
                            const int cc = 8 * ks + c;
                            *reinterpret_cast<double2*>(dst + c) = make_double2(D[lane * D_LD + cc], D[lane * D_LD + cc + 1]);
                        }
                    }
                } else if (warp == 1 && !failed) {
                    // Minv = Ljj^-1: lane k solves Ljj y = e_k.  Rows in blocks of 8: the contribution of all earlier
                    // rows is accumulated for the 8 rows at once (one own-column load + four broadcast LDS.128 of
                    // LT[t][i0..i0+7] per t), then an 8x8 triangular solve in registers.
                    double* gm = Lp + minv_off(Mp) + 1024LL * j;
#pragma unroll 1
                    for (int i0 = 0; i0 < 32; i0 += 8) {
                        double y[8];
#pragma unroll
                        for (int ii = 0; ii < 8; ++ii) y[ii] = (i0 + ii == lane) ? 1.0 : 0.0;
#pragma unroll 2
                        for (int t = 0; t < i0; ++t) {
                            const double yt = sm.Minv[t * MI_LD + lane];
                            const double* lt = LT + t * LT_LD + i0;              // L[i0+ii][t]
#pragma unroll
                            for (int ii = 0; ii < 8; ii += 2) {
                                const double2 l2 = *reinterpret_cast<const double2*>(lt + ii);
                                y[ii] = fma(-l2.x, yt, y[ii]);
                                y[ii + 1] = fma(-l2.y, yt, y[ii + 1]);
                            }
                        }
#pragma unroll
                        for (int ii = 0; ii < 8; ++ii) {
                            y[ii] *= sm.rdiag[i0 + ii];
#pragma unroll
                            for (int i2 = ii + 1; i2 < 8; ++i2) y[i2] = fma(-LT[(i0 + ii) * LT_LD + i0 + i2], y[ii], y[i2]);
                        }
#pragma unroll
                        for (int ii = 0; ii < 8; ++ii) {
                            sm.Minv[(i0 + ii) * MI_LD + lane] = y[ii];          // Minv[i][k = lane]
                            gm[(i0 + ii) * 32 + lane] = y[ii];
                        }
                        __syncwarp();
                    }
                }
                __syncthreads();                                                 // (B)
                }
                if (CL) {
                    cluster_sync_all();                      // Minv, u block, diagonal rows and flag published by CTA 0
                    const int fl = (int)aux[Mp + 32];
                    if (fl != 0) {
                        if (crank == 0 && tid == 0 && info) *info = fl;
                        return -INFINITY;
                    }
                    if (crank != 0) {
                        const double* gm = Lp + minv_off(Mp) + 1024LL * j;
                        for (int idx = tid; idx < 1024; idx += NT) sm.Minv[(idx >> 5) * MI_LD + (idx & 31)] = __ldcg(gm + idx);
                        if (tid < 32) sm.uj[tid] = __ldcg(aux + Mp + tid);
                        __syncthreads();
                    }
                }
            }

            // ------------------------------------------------------------------ 4. X = P Minv^T, store, update w
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i < nu && !(pr == 0 && gw + TW * i < 4)) {
                    double xt[4][2];
                    unit_trsm(acc[i], xt, sm.Minv, g, q);
                    const int r = rb[i] + g;
                    double s0 = 0.0, s1 = 0.0;
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) {
                        const double2 u2 = *reinterpret_cast<const double2*>(sm.uj + 8 * cb + 2 * q);
                        s0 = fma(xt[cb][0], u2.x, s0);
                        s1 = fma(xt[cb][1], u2.y, s1);
                        *reinterpret_cast<double2*>(Lpj + (long long)cb * Rj * 8 + (long long)(r - row0) * 8 + 2 * q) =
                            make_double2(xt[cb][0], xt[cb][1]);
                    }
                    double sdot = s0 + s1;
                    sdot += __shfl_xor_sync(0xffffffffu, sdot, 1);
                    sdot += __shfl_xor_sync(0xffffffffu, sdot, 2);
                    if (q == 0) wres[r] -= (SRC == 0) ? sdot : -sdot;
                }
            }
        }
        if (!CL) __syncthreads();                                                // (C)  (cluster variant: barrier at the top)
    }

    if (warp == 0) {
        double ld = warp_sum(logdet);
        double qd = warp_sum(quad);
        if (lane == 0) sm.red[0] = -ld - 0.5 * qd;
    }
    __syncthreads();
    if (crank == 0 && tid == 0 && info) *info = 0;
    return sm.red[0];
}

// ---------------------------------------------------------------------------------------------
// Look-ahead variant (one CTA per matrix).  The serial part of a panel -- the 32x32 diagonal-block
// factorisation by one warp, its inverse and the w-block solve, ~30 k cycles during which the other warps
// of the CTA used to wait -- is taken off the critical path: the diagonal block of panel j+1 is factored
// while panel j is still being finished.  Stage jc (= j+1):
//   warps 0,1: (a) "priority" pair: the rows of block jc in panel j (GEMM, covariance, TRSM, store), named
//              barrier between the two warps; (b) look-ahead pair: block jc itself over k-blocks 0..j
//              (GEMM, covariance) -> D; warp 0 factors it, then warp 0 solves the w block / stores the diagonal
//              rows while warp 1 inverts the block (into D, copied to Minv at the next stage); (c) join the pool;
//   warps 2,3: pool of the remaining 16-row pairs of panel j, handed out by a shared-memory counter.
// Every matrix entry goes through the same arithmetic in the same order as in eval_block_loglik, so the
// result is bit-identical to it (tests/test_gpu_core.py).  The pair body exists once (a small state machine
// per warp) to keep the kernel's code size -- and instruction fetch -- where it was.
// ---------------------------------------------------------------------------------------------
struct LaSmem {
    double* Minv;   // [32][MI_LD]  inverse of the diagonal block of the panel being finished (TRSM operand)
    double* LT;     // [32][LT_LD]  LT[k][i] = L[i][k] of the block being factored
    double* D;      // [32][D_LD]   P of the look-ahead block, then (after the factorisation) its inverse, D[i][k]
    double* rdiag;  // [32]
    double* uj;     // [2][32]      u blocks (by parity of the block index)
    double* red;    // [8]
    double* etab;   // [ETAB]
    double* wres;   // [Mp]
    double* sb;     // [dpad]
    double* SC;     // [2][sc_doubles(d)] B fragments of the distance product (by parity of the panel index)
    double* scr;    // [NWARP][512] per-warp scratch of the covariance step
    int* flag;      // [4]: 0 failure flag, 1 pool counter
    int* soff;      // [Mp/8]
    int scsz;
};

__host__ __device__ inline size_t la_smem_bytes(int Mp, int d) {
    const int dpad = (d + 1) & ~1;
    return (size_t)(32 * MI_LD + 32 * LT_LD + 32 * D_LD + 32 + 64 + 8 + ETAB + Mp + dpad + 2 * sc_doubles(d) + NWARP * 512) * sizeof(double) +
           16 + (size_t)(Mp / 8) * sizeof(int);
}

__device__ inline LaSmem carve_la_smem(unsigned char* base, int Mp, int d) {
    LaSmem s;
    const int dpad = (d + 1) & ~1;
    double* p = reinterpret_cast<double*>(base);
    s.Minv = p;     p += 32 * MI_LD;
    s.LT = p;       p += 32 * LT_LD;
    s.D = p;        p += 32 * D_LD;
    s.rdiag = p;    p += 32;
    s.uj = p;       p += 64;
    s.red = p;      p += 8;
    s.etab = p;     p += ETAB;
    s.wres = p;     p += Mp;
    s.sb = p;       p += dpad;
    s.SC = p;       p += 2 * sc_doubles(d);
    s.scr = p;      p += NWARP * 512;
    s.flag = reinterpret_cast<int*>(p);
    s.soff = s.flag + 4;
    s.scsz = sc_doubles(d);
    return s;
}

__device__ __forceinline__ void bar_pair01() { asm volatile("bar.sync 1, 64;" ::: "memory"); }
// split producer / consumer forms for warps 0 and 1 (32 threads arrive, 32 wait)
__device__ __forceinline__ void bar01_arrive(int id) { __threadfence_block(); asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void bar01_wait(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

// Role rotation.  Warps are bound to the SM's four sub-partitions by their index (warp w -> sub-partition w % 4), and the
// look-ahead schedule gives the warps of a CTA very different shares of the tensor work (role 0 factors the diagonal
// blocks, roles 2 and 3 do little else than the DMMA product).  With the same role on the same sub-partition in every
// resident CTA, the DMMA pipes of two sub-partitions queue while the other two idle.  Each CTA therefore takes a rotation
// from a per-SM arrival counter: the CTAs resident on one SM get different rotations, and every sub-partition sees the
// same mix of roles.  Roles only decide WHICH warp computes an entry, never how: results are unchanged.
static __device__ unsigned g_role_rot[1024];
__device__ __forceinline__ int cta_role_rotation()          // every thread of the CTA; contains a __syncthreads
{
    __shared__ int rot_sm;
    if (threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        rot_sm = (int)(atomicAdd(&g_role_rot[smid & 1023u], 1u) & (unsigned)(NWARP - 1));
    }
    __syncthreads();
    return rot_sm;
}

static __device__ __forceinline__ double eval_block_loglik_la(const LaSmem& sm, const double* __restrict__ X, int m, int Mp, int d,
                                    const double* beta, double lamz, double diag_add,
                                    const double* __restrict__ w, double* __restrict__ Lp,
                                    double* __restrict__ u_out, int* info, int rot = 0)
{
    static_assert(NWARP >= 2 && (NWARP & (NWARP - 1)) == 0, "look-ahead variant needs a power-of-two number (>= 2) of warps");
    const int tid = threadIdx.x, lane = tid & 31, warp = ((tid >> 5) + rot) & (NWARP - 1);     // warp = role
    const int g = lane >> 2, q = lane & 3;
    const int nP = Mp >> 5;
    const double inv_lamz = 1.0 / lamz;
    const double diag = inv_lamz + diag_add;
    double* __restrict__ D = sm.D;
    double* __restrict__ LT = sm.LT;
    double* __restrict__ wres = sm.wres;
    double* __restrict__ scr = sm.scr + warp * 512;

    __syncthreads();   // previous user of the shared buffers is done
    if (tid < d) sm.sb[tid] = sqrt(beta[tid]);
    for (int r = tid; r < Mp; r += NT) wres[r] = (r < m) ? w[r] : 0.0;
    fill_exp_table(sm.etab);
    fill_slab_offsets(sm.soff, Mp);
    if (tid == 0) sm.flag[0] = 0;
    double logdet = 0.0, quad = 0.0;    // partial sums, live in warp 0
    __syncthreads();

    for (int jc = 0; jc < nP; ++jc) {
        const int j = jc - 1;                       // panel finished in this stage (none in stage 0)
        if (j >= 0)                                 // inverse of block j, produced by the previous stage
            for (int idx = tid; idx < 1024; idx += NT) sm.Minv[(idx >> 5) * MI_LD + (idx & 31)] = D[(idx >> 5) * D_LD + (idx & 31)];
        fill_panel_coords(sm.SC + (jc & 1) * sm.scsz, X, sm.sb, d, m, jc << 5);
        if (tid == 0) sm.flag[1] = 0;
        __syncthreads();                                                         // (T)
        const int nreg = (j >= 0) ? ((Mp - 32 * j) >> 3) - 8 : 0;               // pool units of panel j (multiple of 4)
        const int npair = nreg >> 1;                         // pool tasks: 16-row pairs
        int phase = (warp < 2) ? (j >= 0 ? 0 : 1) : 2;       // 0 priority pair, 1 look-ahead pair, 2 pool, 3 inverse (warp 1)
        int pend = 0;        // warp 1: 1 = inverse of block jc still to do, 2 = do it after the pool pair in hand

#pragma unroll 1
        while (true) {
            int cp = j, r0 = 0;
            if (phase == 2) {
                if (pend == 2) phase = 3;
                else {
                    int idx = 0;
                    if (lane == 0) idx = atomicAdd(&sm.flag[1], 1);
                    idx = __shfl_sync(0xffffffffu, idx, 0);
                    if (idx >= npair) {
                        if (pend == 0) break;
                        phase = 3;
                    } else {
                        if (pend == 1) pend = 2;
                        r0 = 32 * j + 64 + 16 * idx;
                    }
                }
            } else {
                cp = (phase == 0) ? j : jc;
                r0 = 32 * jc + 16 * warp;
            }
            if (phase == 3) {
                // warp 1 (after at most one pool pair, which overlaps warp 0's factorisation): inverse of block jc.
                // Lane k solves Ljj y = e_k, rows in blocks of 8; result D[i][k] and the packed factor's inverse-block
                // area (used by the prediction kernel)
                bar01_wait(2);                                                   // (C) factor (LT, rdiag) or failure flag visible
                if (sm.flag[0] == 0) {
                    double* gm = Lp + minv_off(Mp) + 1024LL * jc;
#pragma unroll 1
                    for (int i0 = 0; i0 < 32; i0 += 8) {
                        double y[8];
#pragma unroll
                        for (int ii = 0; ii < 8; ++ii) y[ii] = (i0 + ii == lane) ? 1.0 : 0.0;
#pragma unroll 2
                        for (int t = 0; t < i0; ++t) {
                            const double yt = D[t * D_LD + lane];
                            const double* lt = LT + t * LT_LD + i0;              // L[i0+ii][t]
#pragma unroll
                            for (int ii = 0; ii < 8; ii += 2) {
                                const double2 l2 = *reinterpret_cast<const double2*>(lt + ii);
                                y[ii] = fma(-l2.x, yt, y[ii]);
                                y[ii + 1] = fma(-l2.y, yt, y[ii + 1]);
                            }
                        }
#pragma unroll
                        for (int ii = 0; ii < 8; ++ii) {
                            y[ii] *= sm.rdiag[i0 + ii];
#pragma unroll
                            for (int i2 = ii + 1; i2 < 8; ++i2) y[i2] = fma(-LT[(i0 + ii) * LT_LD + i0 + i2], y[ii], y[i2]);
                        }
#pragma unroll
                        for (int ii = 0; ii < 8; ++ii) {
                            D[(i0 + ii) * D_LD + lane] = y[ii];
                            gm[(i0 + ii) * 32 + lane] = y[ii];
                        }
                        __syncwarp();
                    }
                }
                pend = 0;
                phase = 2;
                continue;
            }
            const int row0 = cp << 5;
            const int rb[2] = {r0, r0 + 8};
            double acc[2][4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int cb = 0; cb < 4; ++cb) { acc[i][cb][0] = 0.0; acc[i][cb][1] = 0.0; }
            // ------------------------------------------------------------------ 1. DMMA update
            if (cp > 0) panel_gemm_cp<2>(acc, Lp, Lp, sm.soff, cp, row0, rb, g, q, scr);
            // ------------------------------------------------------------------ 2. covariance, P = C - S (registers)
            {
                const int rr[2] = {rb[0] + g, rb[1] + g};
                const bool ok[2] = {rr[0] < m, rr[1] < m};
                pair_cov<2>(acc, X, rr, ok, sm.SC + (cp & 1) * sm.scsz, sm.sb, d, m, row0, q, inv_lamz, diag, true, sm.etab, scr, lane);
            }
            if (phase == 1) {
                // -------------------------------------------------------------- 3. diagonal block jc (look-ahead)
#pragma unroll
                for (int i = 0; i < 2; ++i)
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                        for (int e = 0; e < 2; ++e)
                            D[(16 * warp + 8 * i + g) * D_LD + 8 * cb + 2 * q + e] = acc[i][cb][e];
                if (warp == 1) {
                    bar01_arrive(1);                                             // (B) this half of the block is in D
                    pend = 1;                                                    // inverse after at most one pool pair
                } else {
                    bar01_wait(1);                                               // (B) block complete in D
                    int failed;
                    {
                        // Cholesky of the 32x32 block, lane = row (same arithmetic as eval_block_loglik)
                        double mypiv = 1.0;
                        int bad = 0;
#pragma unroll 1
                        for (int k0 = 0; k0 < 32; k0 += 8) {
                            double x[8];
#pragma unroll
                            for (int kk = 0; kk < 8; ++kk) x[kk] = D[lane * D_LD + k0 + kk];
#pragma unroll
                            for (int kk = 0; kk < 8; ++kk) {
                                const int k = k0 + kk;
                                if (lane == k) sm.red[2] = x[kk];
                                __syncwarp();
                                const double dk = sm.red[2];
                                if (!(dk > 0.0) || !(dk < 1.0e300)) { if (!bad) bad = row0 + k + 1; }
                                const double rk = rsqrt(dk);
                                const double lik = (lane == k) ? dk * rk : x[kk] * rk;
                                if (lane == k) mypiv = dk;
                                x[kk] = lik;
                                if (lane == 0) sm.rdiag[k] = rk;
                                LT[k * LT_LD + lane] = (lane >= k) ? lik : 0.0;
                                __syncwarp();
#pragma unroll
                                for (int k2 = kk + 1; k2 < 8; ++k2) x[k2] = fma(-lik, LT[k * LT_LD + k0 + k2], x[k2]);
                            }
#pragma unroll
                            for (int kk = 0; kk < 8; ++kk) D[lane * D_LD + k0 + kk] = (lane >= k0 + kk) ? x[kk] : 0.0;
#pragma unroll 2
                            for (int c = k0 + 8; c < 32; ++c) {
                                double a = D[lane * D_LD + c];
#pragma unroll
                                for (int kk = 0; kk < 8; ++kk) a = fma(-x[kk], LT[(k0 + kk) * LT_LD + c], a);
                                D[lane * D_LD + c] = a;
                            }
                            __syncwarp();
                            if (bad) break;
                        }
                        if (bad) { if (lane == 0) sm.flag[0] = bad; }
                        else logdet += 0.5 * log(mypiv);
                        failed = bad;
                    }
                    bar01_arrive(2);                                             // (C) factor (LT, rdiag) or failure flag published
                    if (!failed) {
                        // forward solve of the w block: u = Ljj^-1 wres[row0 : row0+32]  (L read from LT: D is being
                        // overwritten with the inverse by warp 1)
                        double b = wres[row0 + lane];
                        double myu = 0.0;
#pragma unroll 1
                        for (int c = 0; c < 32; ++c) {
                            const double uc = __shfl_sync(0xffffffffu, b, c) * sm.rdiag[c];
                            if (lane == c) myu = uc;
                            if (lane > c) b = fma(-LT[c * LT_LD + lane], uc, b);
                        }
                        sm.uj[(jc & 1) * 32 + lane] = myu;
                        quad += myu * myu;
                        if (u_out) u_out[row0 + lane] = myu;
                        // diagonal rows of L (zeros above the diagonal) -> packed factor, panel jc
                        double* __restrict__ Lpc = Lp + panel_off(jc, Mp);
                        const int Rc = Mp - row0;
#pragma unroll 1
                        for (int ks = 0; ks < 4; ++ks) {
                            double* dst = Lpc + (long long)ks * Rc * 8 + (long long)lane * 8;
#pragma unroll
                            for (int c = 0; c < 8; c += 2) {
                                const int cc = 8 * ks + c;
                                *reinterpret_cast<double2*>(dst + c) = make_double2(LT[cc * LT_LD + lane], LT[(cc + 1) * LT_LD + lane]);
                            }
                        }
                    }
                }
                phase = 2;
            } else {
                // -------------------------------------------------------------- 4. X = P Minv^T, store, update w (panel j)
                double* __restrict__ Lpj = Lp + panel_off(j, Mp);
                const int Rj = Mp - row0;
                const double* __restrict__ ujj = sm.uj + (j & 1) * 32;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    double xt[4][2];
                    unit_trsm(acc[i], xt, sm.Minv, g, q);
                    const int r = rb[i] + g;
                    double s0 = 0.0, s1 = 0.0;
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) {
                        const double2 u2 = *reinterpret_cast<const double2*>(ujj + 8 * cb + 2 * q);
                        s0 = fma(xt[cb][0], u2.x, s0);
                        s1 = fma(xt[cb][1], u2.y, s1);
                        *reinterpret_cast<double2*>(Lpj + (long long)cb * Rj * 8 + (long long)(r - row0) * 8 + 2 * q) =
                            make_double2(xt[cb][0], xt[cb][1]);
                    }
                    double sdot = s0 + s1;
                    sdot += __shfl_xor_sync(0xffffffffu, sdot, 1);
                    sdot += __shfl_xor_sync(0xffffffffu, sdot, 2);
                    if (q == 0) wres[r] -= sdot;
                }
                if (phase == 0) {
                    bar_pair01();                                                // (A) rows of block jc complete in panels 0..j
                    phase = 1;
                }
            }
        }
        __syncthreads();                                                         // (E)
        if (sm.flag[0] != 0) {
            if (tid == 0 && info) *info = sm.flag[0];
            return -INFINITY;
        }
    }

    if (warp == 0) {
        double ld = warp_sum(logdet);
        double qd = warp_sum(quad);
        if (lane == 0) sm.red[0] = -ld - 0.5 * qd;
    }
    __syncthreads();
    if (tid == 0 && info) *info = 0;
    return sm.red[0];
}

// Cluster size for `ntasks` independent matrices: one CTA per matrix when the machine is already full, otherwise
// the largest power of two that still fits all clusters in one wave of CL_CTAS_PER_SM resident CTAs per SM: up to 8
// (the portable cluster limit), 16 for matrices of 1024 rows and more (cfg 5: one chain of 20 PCs at m = 4096 runs
// 0.80 -> 0.55 s per step).  GGP_CLUSTER=<n> overrides it, so that one input can run on both sides of the choice (tests).
inline int choose_cluster(long long ntasks, int Mp)
{
    if (const char* e = getenv("GGP_CLUSTER")) {
        int g = atoi(e);
        if (g == 1 || g == 2 || g == 4 || g == 8 || g == 16) return g;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long slots = (long long)sms * CL_CTAS_PER_SM;      // resident CTAs of the cluster kernels
    const int gmax = (Mp >= 1024) ? 16 : 8;
    int g = 1;
    while (g < gmax && ntasks * (g * 2) <= slots) g *= 2;
    return g;
}

// a 16-CTA cluster is beyond the portable size: ask the driver whether this kernel / shared-memory size can be
// co-scheduled that way on this device; otherwise stay at 8
template <typename K>
inline int checked_cluster(K kern, int G, size_t smem)
{
    if (G <= 8) return G;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) { cudaGetLastError(); return 8; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) { cudaGetLastError(); return 8; }
    return G;
}

template <typename K, typename... Args>
inline cudaError_t launch_maybe_cluster(K kern, dim3 grid, dim3 block, size_t smem, cudaStream_t st, int G, Args... args)
{
    if (G > 8) {       // beyond the portable cluster size: opt in (16 CTAs still fit one GPC)
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = (G > 1) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

}  // namespace ggp
