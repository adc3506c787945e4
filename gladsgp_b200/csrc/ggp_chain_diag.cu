// MCMC convergence diagnostics over any number of chains: rank-normalized split R-hat, bulk ESS and tail ESS
// (Vehtari, Gelman, Simpson, Carpenter and Buerkner 2021; ArviZ rhat(method="rank"), ess(method="bulk" / "tail")).
// The conventions are frozen in DESIGN.md section 2 and restated by oracle/chain_diag_oracle.py.
//
// One element = the draws x[c][i] of one scalar (C chains x n draws, FP64).  h = n / 2; split chain sc < C is x[sc][0, h),
// split chain C + c is x[c][n - h, n), so the split array has k = 2C chains and S = k h values.  Elements are independent and
// every element runs the same code with the same thread mapping, so its results do not depend on the rest of the launch.
//
//   chain_diag_rank_kernel   one CTA per element.  The C n draws become order-preserving uint64 keys (-0.0 as +0.0) and are
//                            sorted with their positions by a hand-written stable LSD radix sort: 8-bit digits, digits on
//                            which every key agrees are skipped, each pass a histogram, a scan and an in-order scatter of
//                            2048-key tiles ranked with CUB's block radix sort.  An element of at most 2048 draws is sorted
//                            in shared memory in one go.  A prefix count of the kept (non-middle) draws over sorted order
//                            and a forward max-scan / backward min-scan over tie runs give every kept draw its average rank
//                            r, z = normcdfinv((r - 3/8) / (S + 1/4)) is written in split order.  q05 / q95 (all C n draws,
//                            np.quantile 'linear') and the median of the split values come from the same sorted order; the
//                            folded values |x - median| are sorted and ranked the same way.
//   chain_diag_rhat_kernel   one CTA per element: chain means and variances of both z arrays (a warp per chain, fixed order),
//                            then B, W and R-hat in split-chain order.
//   chain_diag_ess_kernel    one CTA per (element, series): bulk z, 1(x <= q05), 1(x <= q95) (the indicators are regenerated
//                            from the draws).  Lagged sums over all k chains in blocks of 256 lags (one lag per thread, the
//                            chain staged in shared memory), Geyer's initial positive sequence advanced after every block,
//                            stopped as soon as it ends.
//   chain_diag_finish_kernel ess_tail = min of the two indicator series.
#include "ggp_common.cuh"
#include "../../include/gladsgp_b200.h"
#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <climits>

namespace ggp {

typedef unsigned long long u64;

constexpr int CD_NT = 256;
constexpr int CD_IPT = 8;
constexpr int CD_TILE = CD_NT * CD_IPT;   // keys per sort tile (and the largest element sorted in shared memory)
constexpr int CD_LB = CD_NT;              // lags per ESS block, one per thread
constexpr int CD_CH = 1024;               // draws of one chain staged per ESS chunk

__host__ __device__ inline size_t cd_al(size_t b) { return (b + 255) & ~(size_t)255; }

// Per-element workspace carve-up (bytes from the element's base).
struct CdLayout {
    size_t k0, k1, v0, v1, zb, zf, rh, rt, cm, cs, sc, per;
};

__host__ __device__ inline CdLayout cd_layout(int n, int C)
{
    const size_t N = (size_t)n * C, h = (size_t)(n / 2), k = 2 * (size_t)C, S = k * h;
    CdLayout L;
    size_t o = 0;
    L.k0 = o; o += cd_al(8 * N);          // keys, ping
    L.k1 = o; o += cd_al(8 * N);          // keys, pong; (A, B) tie-run pairs while ranking
    L.v0 = o; o += cd_al(4 * N);          // positions, ping
    L.v1 = o; o += cd_al(4 * N);          // positions, pong
    L.zb = o; o += cd_al(8 * S);          // z of the split draws [k][h]
    L.zf = o; o += cd_al(8 * S);          // z of the folded split draws [k][h]
    L.rh = o; o += cd_al(8 * 3 * h);      // rho-hat per series
    L.rt = o; o += cd_al(8 * 3 * h);      // Geyer's sequence per series
    L.cm = o; o += cd_al(8 * 3 * k);      // chain means per series
    L.cs = o; o += cd_al(8 * 4 * k);      // chain means and variances of zb, zf
    L.sc = o; o += 256;                   // q05, q95, non-finite flag, -, ess of series 1, 2
    L.per = o;
    return L;
}

__device__ __forceinline__ u64 dkey(double x)
{
    if (x == 0.0) x = 0.0;                // -0.0 and +0.0 are one value
    const u64 b = (u64)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double dval(u64 k)
{
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

struct CdArgs {
    const double* x;
    long long s_draw, s_chain, s_elem;
    int n, C, h;
    unsigned char* ws;
    size_t per;
};

__device__ __forceinline__ double ld_x(const CdArgs& a, const double* xe, int i, int c)
{
    return xe[(long long)i * a.s_draw + (long long)c * a.s_chain];
}

// split position sc * h + j of draw position p = c n + i, or -1 for a dropped middle draw (odd n)
__device__ __forceinline__ int split_pos(unsigned p, int n, int h, int C)
{
    const int c = (int)(p / (unsigned)n), i = (int)p - c * n;
    if (i < h) return c * h + i;
    if (i >= n - h) return (C + c) * h + (i - (n - h));
    return -1;
}

// draw of split chain sc, position j
__device__ __forceinline__ double split_x(const CdArgs& a, const double* xe, int sc, int j)
{
    return sc < a.C ? ld_x(a, xe, j, sc) : ld_x(a, xe, a.n - a.h + j, sc - a.C);
}

typedef cub::BlockRadixSort<u64, CD_NT, CD_IPT, unsigned> CdSort;
typedef cub::BlockScan<int, CD_NT> CdScanI;
typedef cub::BlockScan<unsigned, CD_NT> CdScanU;
typedef cub::BlockReduce<u64, CD_NT> CdReduceK;

struct CdSmem {
    union {
        typename CdSort::TempStorage sort;
        typename CdScanI::TempStorage scani;
        typename CdScanU::TempStorage scanu;
        typename CdReduceK::TempStorage red;
    } u;
    unsigned hist[256], goff[256], tstart[256];
    unsigned char dig[CD_TILE];
    u64 diff;
    double med[2];
};

// Stable LSD radix sort of n (key, position) pairs held in kb[0] / vb[0].  diff: OR over keys of (key ^ first key), the
// digits on which the keys differ.  Returns the buffer that holds the result.
__device__ int cd_sort(u64* kb[2], unsigned* vb[2], int n, u64 diff, CdSmem& sm)
{
    const int tid = threadIdx.x;
    if (n <= CD_TILE) {
        u64 key[CD_IPT];
        unsigned val[CD_IPT];
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int s = tid * CD_IPT + j;
            key[j] = s < n ? kb[0][s] : ~0ull;
            val[j] = s < n ? vb[0][s] : 0u;
        }
        CdSort(sm.u.sort).Sort(key, val);
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int s = tid * CD_IPT + j;
            if (s < n) { kb[0][s] = key[j]; vb[0][s] = val[j]; }
        }
        __syncthreads();
        return 0;
    }
    static_assert(CD_NT == 256, "one histogram bin per thread");
    int cur = 0;
    for (int d = 0; d < 8; ++d) {
        const int bit = 8 * d;
        if (((diff >> bit) & 0xffull) == 0) continue;            // every key has this digit: the pass is the identity
        const u64* ki = kb[cur];
        const unsigned* vi = vb[cur];
        u64* ko = kb[cur ^ 1];
        unsigned* vo = vb[cur ^ 1];
        sm.hist[tid] = 0;
        __syncthreads();
        for (int base = tid * CD_IPT; base < n; base += CD_TILE) { // runs of equal digits are counted before the atomic
            unsigned prev = 0xffffffffu, cnt = 0;
            const int e = min(base + CD_IPT, n);
            for (int s = base; s < e; ++s) {
                const unsigned g = (unsigned)(ki[s] >> bit) & 0xffu;
                if (g != prev) {
                    if (cnt) atomicAdd(&sm.hist[prev], cnt);
                    prev = g;
                    cnt = 0;
                }
                ++cnt;
            }
            if (cnt) atomicAdd(&sm.hist[prev], cnt);
        }
        __syncthreads();
        {
            unsigned ex;
            CdScanU(sm.u.scanu).ExclusiveSum(sm.hist[tid], ex);
            sm.goff[tid] = ex;
        }
        __syncthreads();
        for (int t0 = 0; t0 < n; t0 += CD_TILE) {
            const int valid = min(CD_TILE, n - t0);
            u64 key[CD_IPT];
            unsigned val[CD_IPT], g[CD_IPT];
#pragma unroll
            for (int j = 0; j < CD_IPT; ++j) {
                const int s = tid * CD_IPT + j;
                key[j] = s < valid ? ki[t0 + s] : ~0ull;        // padding sorts after every real key of digit 0xff
                val[j] = s < valid ? vi[t0 + s] : 0u;
            }
            CdSort(sm.u.sort).Sort(key, val, bit, bit + 8);
#pragma unroll
            for (int j = 0; j < CD_IPT; ++j) {
                g[j] = (unsigned)(key[j] >> bit) & 0xffu;
                sm.dig[tid * CD_IPT + j] = (unsigned char)g[j];
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < CD_IPT; ++j) {
                const int s = tid * CD_IPT + j;
                if (s < valid && (s == 0 || sm.dig[s - 1] != g[j])) sm.tstart[g[j]] = s;
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < CD_IPT; ++j) {
                const int s = tid * CD_IPT + j;
                if (s < valid) {
                    const unsigned pos = sm.goff[g[j]] + (unsigned)s - sm.tstart[g[j]];
                    ko[pos] = key[j];
                    vo[pos] = val[j];
                }
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < CD_IPT; ++j) {
                const int s = tid * CD_IPT + j;
                if (s < valid && (s == valid - 1 || sm.dig[s + 1] != g[j])) sm.goff[g[j]] += (unsigned)(s + 1) - sm.tstart[g[j]];
            }
            __syncthreads();
        }
        cur ^= 1;
    }
    return cur;
}

// Average ranks of the kept draws among the kept draws, over sorted keys k / positions v (n_items of them), and
// z = normcdfinv((r - 3/8) / (S + 1/4)) written to zout in split order.  folded: every item is kept and v is its split
// position; otherwise v is c n + i and split_pos decides.  aux (n_items int2, free memory) holds, per sorted position, A =
// kept count before its tie run and B = kept count through its tie run (B only at run ends after the forward pass).
// With want_median the two middle kept values land in sm.med.
__device__ void cd_rank(const u64* __restrict__ k, const unsigned* __restrict__ v, int2* aux, int n_items, bool folded,
                        const CdArgs& a, int S, double* __restrict__ zout, bool want_median, CdSmem& sm)
{
    const int tid = threadIdx.x;
    int carry_kp = 0, carry_a = -1;
    for (int t0 = 0; t0 < n_items; t0 += CD_TILE) {
        int kept[CD_IPT], kp[CD_IPT], hv[CD_IPT];
        u64 key[CD_IPT];
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int s = t0 + tid * CD_IPT + j;
            key[j] = s < n_items ? k[s] : 0ull;
            kept[j] = (s < n_items && (folded || split_pos(v[s], a.n, a.h, a.C) >= 0)) ? 1 : 0;
        }
        int tile_kept;
        CdScanI(sm.u.scani).ExclusiveSum(kept, kp, tile_kept);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int s = t0 + tid * CD_IPT + j;
            kp[j] += carry_kp;
            const u64 prev = j > 0 ? key[j - 1] : (s > 0 && s < n_items ? k[s - 1] : ~key[j]);
            const bool head = s < n_items && (s == 0 || prev != key[j]);
            hv[j] = head ? kp[j] : -1;
        }
        int tile_max;
        CdScanI(sm.u.scani).InclusiveScan(hv, hv, [](int p, int q) { return max(p, q); }, tile_max);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int s = t0 + tid * CD_IPT + j;
            if (s >= n_items) continue;
            const int A = max(hv[j], carry_a);                   // kp is non-decreasing: the last head's count
            const u64 next = j + 1 < CD_IPT ? key[j + 1] : (s + 1 < n_items ? k[s + 1] : ~key[j]);
            const bool end = s + 1 == n_items || next != key[j];
            aux[s] = make_int2(A, end ? kp[j] + kept[j] : INT_MAX);
            if (want_median && kept[j]) {
                if (kp[j] == S / 2 - 1) sm.med[0] = dval(key[j]);
                if (kp[j] == S / 2) sm.med[1] = dval(key[j]);
            }
        }
        carry_kp += tile_kept;
        carry_a = max(carry_a, tile_max);
    }
    __syncthreads();
    // backward: B of every item = B of the nearest run end at or after it (reverse inclusive min-scan)
    int carry_b = INT_MAX;
    const int ntile = (n_items + CD_TILE - 1) / CD_TILE;
    for (int tt = ntile - 1; tt >= 0; --tt) {
        const int t0 = tt * CD_TILE, valid = min(CD_TILE, n_items - t0);
        int bv[CD_IPT], av[CD_IPT];
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int r = tid * CD_IPT + j;
            const int s = t0 + valid - 1 - r;
            if (r < valid) {
                const int2 p = aux[s];
                av[j] = p.x;
                bv[j] = p.y;
            } else {
                av[j] = 0;
                bv[j] = INT_MAX;
            }
        }
        int tile_min;
        CdScanI(sm.u.scani).InclusiveScan(bv, bv, [](int p, int q) { return min(p, q); }, tile_min);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < CD_IPT; ++j) {
            const int r = tid * CD_IPT + j;
            if (r >= valid) continue;
            const int s = t0 + valid - 1 - r;
            const int sp = folded ? (int)v[s] : split_pos(v[s], a.n, a.h, a.C);
            if (sp < 0) continue;
            const int B = min(bv[j], carry_b);
            const double rank = 0.5 * ((double)av[j] + (double)B + 1.0);
            zout[sp] = normcdfinv((rank - 0.375) / ((double)S + 0.25));
        }
        carry_b = min(carry_b, tile_min);
    }
    __syncthreads();
}

// keys of the draws (folded = false: all C n draws, position c n + i) or of |x - med| over the split draws (folded =
// true, position = split position) into k / v; returns the OR over keys of (key ^ first key).  bad: a draw is not finite.
__device__ u64 cd_keys(const CdArgs& a, const double* xe, bool folded, double med, u64* k, unsigned* v, bool& bad_out,
                       CdSmem& sm)
{
    const int tid = threadIdx.x;
    const int n = a.n, C = a.C, h = a.h;
    const int cnt = folded ? 2 * C * h : n * C;
    const bool chain_fast = llabs(a.s_chain) < llabs(a.s_draw);  // walk the smaller stride between neighbouring threads
    u64 first = 0;
    {
        double x0 = folded ? fabs(split_x(a, xe, 0, 0) - med) : ld_x(a, xe, 0, 0);
        first = dkey(x0);
    }
    u64 diff = 0;
    int bad = 0;
    for (int q = tid; q < cnt; q += CD_NT) {
        int c, i, pos;
        if (folded) {
            int sc, j;
            if (chain_fast) { j = q / (2 * C); sc = q - j * 2 * C; } else { sc = q / h; j = q - sc * h; }
            c = sc < C ? sc : sc - C;
            i = sc < C ? j : n - h + j;
            pos = sc * h + j;
        } else {
            if (chain_fast) { i = q / C; c = q - i * C; } else { c = q / n; i = q - c * n; }
            pos = c * n + i;
        }
        double xv = ld_x(a, xe, i, c);
        bad |= !isfinite(xv);
        if (folded) xv = fabs(xv - med);
        const u64 kk = dkey(xv);
        k[pos] = kk;
        v[pos] = (unsigned)pos;
        diff |= kk ^ first;
    }
    bad_out = __syncthreads_or(bad) != 0;
    if (bad_out) return 0;
    const u64 r = CdReduceK(sm.u.red).Reduce(diff, [](u64 p, u64 q) { return p | q; });
    if (tid == 0) sm.diff = r;
    __syncthreads();
    return sm.diff;
}

__global__ void __launch_bounds__(CD_NT)
chain_diag_rank_kernel(CdArgs a)
{
    __shared__ CdSmem sm;
    const int e = blockIdx.x, tid = threadIdx.x;
    const double* xe = a.x + (long long)e * a.s_elem;
    unsigned char* base = a.ws + (size_t)e * a.per;
    const CdLayout L = cd_layout(a.n, a.C);
    double* sc = reinterpret_cast<double*>(base + L.sc);
    u64* kb[2] = {reinterpret_cast<u64*>(base + L.k0), reinterpret_cast<u64*>(base + L.k1)};
    unsigned* vb[2] = {reinterpret_cast<unsigned*>(base + L.v0), reinterpret_cast<unsigned*>(base + L.v1)};
    const int N = a.n * a.C, S = 2 * a.C * a.h;
    bool bad;
    u64 diff = cd_keys(a, xe, false, 0.0, kb[0], vb[0], bad, sm);
    if (bad) {
        if (tid == 0) sc[2] = 1.0;
        return;
    }
    int cur = cd_sort(kb, vb, N, diff, sm);
    if (tid == 0) {
        sc[2] = 0.0;
        const double qs[2] = {0.05, 0.95};
        for (int t = 0; t < 2; ++t) {                            // np.quantile(x, q), method 'linear'
            const double vi = (double)(N - 1) * qs[t];
            const double fl = floor(vi);
            const int lo = (int)fl, hi = min(lo + 1, N - 1);
            const double tt = vi - fl;
            const double xa = dval(kb[cur][lo]), xb = dval(kb[cur][hi]);
            const double dd = xb - xa;
            sc[t] = (tt >= 0.5) ? xb - dd * (1.0 - tt) : xa + dd * tt;
        }
    }
    cd_rank(kb[cur], vb[cur], reinterpret_cast<int2*>(kb[cur ^ 1]), N, false, a, S,
            reinterpret_cast<double*>(base + L.zb), true, sm);
    const double med = (sm.med[0] + sm.med[1]) / 2.0;            // np.median of the split draws
    diff = cd_keys(a, xe, true, med, kb[0], vb[0], bad, sm);
    cur = cd_sort(kb, vb, S, diff, sm);
    cd_rank(kb[cur], vb[cur], reinterpret_cast<int2*>(kb[cur ^ 1]), S, true, a, S,
            reinterpret_cast<double*>(base + L.zf), false, sm);
}

// chain means and variances (ddof = 1) of z [k][h], one warp per chain -> cs [k][2]; then R-hat in split-chain order
__device__ double cd_rhat(const double* __restrict__ z, double* cs, int k, int h)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int c = warp; c < k; c += CD_NT / 32) {
        const double* zc = z + (size_t)c * h;
        double s = 0.0;
        for (int i = lane; i < h; i += 32) s += zc[i];
        const double m = warp_sum(s) / (double)h;
        double q = 0.0;
        for (int i = lane; i < h; i += 32) {
            const double d = zc[i] - m;
            q += d * d;
        }
        q = warp_sum(q);
        if (lane == 0) {
            cs[2 * c] = m;
            cs[2 * c + 1] = q / (double)(h - 1);
        }
    }
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x == 0) {
        double mm = 0.0, w = 0.0;
        for (int c = 0; c < k; ++c) { mm += cs[2 * c]; w += cs[2 * c + 1]; }
        mm /= (double)k;
        w /= (double)k;
        double vm = 0.0;
        for (int c = 0; c < k; ++c) {
            const double d = cs[2 * c] - mm;
            vm += d * d;
        }
        vm /= (double)(k - 1);
        const double B = (double)h * vm;
        r = (w == 0.0) ? __longlong_as_double(0x7ff8000000000000ll) : sqrt((B / w + (double)h - 1.0) / (double)h);
    }
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(CD_NT)
chain_diag_rhat_kernel(CdArgs a, double* __restrict__ rhat_out)
{
    const int e = blockIdx.x;
    unsigned char* base = a.ws + (size_t)e * a.per;
    const CdLayout L = cd_layout(a.n, a.C);
    const double* sc = reinterpret_cast<const double*>(base + L.sc);
    if (sc[2] != 0.0) {
        if (threadIdx.x == 0) rhat_out[e] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    const int k = 2 * a.C;
    double* cs = reinterpret_cast<double*>(base + L.cs);
    const double rb = cd_rhat(reinterpret_cast<const double*>(base + L.zb), cs, k, a.h);
    const double rf = cd_rhat(reinterpret_cast<const double*>(base + L.zf), cs + 2 * k, k, a.h);
    if (threadIdx.x == 0) rhat_out[e] = (rf > rb) ? rf : rb;      // Python's max(bulk, folded)
}

// value j of split chain sc of a series: bulk z, or the indicator 1(x <= q)
__device__ __forceinline__ double cd_series(const CdArgs& a, const double* xe, const double* zb, int series, double q,
                                            int sc, int j)
{
    if (series == 0) return zb[(size_t)sc * a.h + j];
    return split_x(a, xe, sc, j) <= q ? 1.0 : 0.0;
}

__global__ void __launch_bounds__(CD_NT)
chain_diag_ess_kernel(CdArgs a, double* __restrict__ ess_bulk_out)
{
    __shared__ double sa[CD_CH];
    __shared__ double sb[CD_CH + CD_LB];
    __shared__ double s_meanvar, s_varplus;
    __shared__ int s_more;
    __shared__ typename cub::BlockReduce<double, CD_NT>::TempStorage red;
    const int e = blockIdx.x, series = blockIdx.y, tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const double* xe = a.x + (long long)e * a.s_elem;
    unsigned char* base = a.ws + (size_t)e * a.per;
    const CdLayout L = cd_layout(a.n, a.C);
    double* sc = reinterpret_cast<double*>(base + L.sc);
    double* out = series == 0 ? ess_bulk_out + e : sc + 3 + series;
    if (sc[2] != 0.0) {
        if (tid == 0) *out = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    const double* zb = reinterpret_cast<const double*>(base + L.zb);
    const double q = series == 0 ? 0.0 : sc[series - 1];
    const int h = a.h, k = 2 * a.C;
    const double kh = (double)k * (double)h;
    double* cm = reinterpret_cast<double*>(base + L.cm) + (size_t)series * k;
    double* rh = reinterpret_cast<double*>(base + L.rh) + (size_t)series * h;
    double* rt = reinterpret_cast<double*>(base + L.rt) + (size_t)series * h;

    // all values equal: ESS = k h
    double lo = INFINITY, hi = -INFINITY;
    for (long long p = tid; p < (long long)k * h; p += CD_NT) {
        const double v = cd_series(a, xe, zb, series, q, (int)(p / h), (int)(p % h));
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
    lo = cub::BlockReduce<double, CD_NT>(red).Reduce(lo, [](double p, double r) { return fmin(p, r); });
    __syncthreads();
    hi = cub::BlockReduce<double, CD_NT>(red).Reduce(hi, [](double p, double r) { return fmax(p, r); });
    if (tid == 0) s_more = (lo == hi);
    __syncthreads();
    if (s_more) {
        if (tid == 0) *out = kh;
        return;
    }
    // chain means, one warp per chain
    for (int c = warp; c < k; c += CD_NT / 32) {
        double s = 0.0;
        for (int j = lane; j < h; j += 32) s += cd_series(a, xe, zb, series, q, c, j);
        s = warp_sum(s);
        if (lane == 0) cm[c] = s / (double)h;
    }
    __syncthreads();
    double varm = 0.0;
    if (tid == 0) {
        double mm = 0.0;
        for (int c = 0; c < k; ++c) mm += cm[c];
        mm /= (double)k;
        for (int c = 0; c < k; ++c) {
            const double d = cm[c] - mm;
            varm += d * d;
        }
        varm /= (double)(k - 1);
    }

    // Geyer's initial positive sequence, advanced after every block of lags (thread 0's registers)
    int t = 1;
    double even = 1.0, odd = 0.0;
    for (int t0 = 0; t0 < h; t0 += CD_LB) {
        const int lag = t0 + tid;
        double acc = 0.0;
        for (int c = 0; c < k; ++c) {
            const double m = cm[c];
            double raw = 0.0;
            for (int i0 = 0; i0 < h - t0; i0 += CD_CH) {             // lag >= t0: only i < h - t0 contributes
                const int cnt = min(CD_CH, h - t0 - i0);
                for (int jj = tid; jj < CD_CH; jj += CD_NT)
                    sa[jj] = jj < cnt ? cd_series(a, xe, zb, series, q, c, i0 + jj) - m : 0.0;
                for (int jj = tid; jj < CD_CH + CD_LB; jj += CD_NT) {
                    const int i = i0 + t0 + jj;
                    sb[jj] = i < h ? cd_series(a, xe, zb, series, q, c, i) - m : 0.0;
                }
                __syncthreads();
#pragma unroll 8
                for (int ii = 0; ii < cnt; ++ii) raw = fma(sa[ii], sb[ii + tid], raw);   // sb is zero from h on
                __syncthreads();
            }
            acc += raw / (double)h;                              // acov_c[lag], summed in chain order
        }
        const double macov = acc / (double)k;
        if (t0 == 0 && tid == 0) {
            s_meanvar = macov * (double)h / ((double)h - 1.0);
            s_varplus = s_meanvar * ((double)h - 1.0) / (double)h + varm;
        }
        __syncthreads();
        if (lag < h) rh[lag] = 1.0 - (s_meanvar - macov) / s_varplus;
        __syncthreads();
        if (tid == 0) {
            const int end = min(t0 + CD_LB, h);
            if (t0 == 0) {
                odd = rh[1];
                rt[0] = 1.0;
                rt[1] = odd;
            }
            int more = 0;
            while (t < h - 3 && even + odd > 0.0) {
                if (t + 2 >= end) { more = 1; break; }
                even = rh[t + 1];
                odd = rh[t + 2];
                const bool keep = even + odd >= 0.0;
                rt[t + 1] = keep ? even : 0.0;
                rt[t + 2] = keep ? odd : 0.0;
                t += 2;
            }
            s_more = more;
        }
        __syncthreads();
        if (!s_more) break;
    }
    if (tid == 0) {
        const int max_t = t - 2;
        if (even > 0.0) rt[max_t + 1] = even;                    // improve estimation
        for (int u = 1; u <= max_t - 2; u += 2) {                // initial monotone sequence
            if (rt[u + 1] + rt[u + 2] > rt[u - 1] + rt[u]) {
                rt[u + 1] = (rt[u - 1] + rt[u]) / 2.0;
                rt[u + 2] = rt[u + 1];
            }
        }
        double s = 0.0;
        for (int u = 0; u <= max_t; ++u) s += rt[u];
        double tau = -1.0 + 2.0 * s + (max_t + 1 < h ? rt[max_t + 1] : 0.0);
        const double floor_tau = 1.0 / log10(kh);
        tau = tau > floor_tau ? tau : floor_tau;
        *out = kh / tau;
    }
}

__global__ void chain_diag_finish_kernel(CdArgs a, int n_elem, double* __restrict__ ess_tail_out)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_elem) return;
    const CdLayout L = cd_layout(a.n, a.C);
    const double* sc = reinterpret_cast<const double*>(a.ws + (size_t)e * a.per + L.sc);
    const double e05 = sc[4], e95 = sc[5];
    ess_tail_out[e] = sc[2] != 0.0 ? __longlong_as_double(0x7ff8000000000000ll) : (e95 < e05 ? e95 : e05);
}

}  // namespace ggp

using namespace ggp;

extern "C" {

long long ggp_chain_diag_workspace_bytes(int n_draws, int n_chains, int n_elem)
{
    if (n_draws < 4 || n_chains < 1 || n_elem < 1 || (long long)n_chains * n_draws >= (1LL << 31)) return -1;
    return (long long)cd_layout(n_draws, n_chains).per * n_elem;
}

int ggp_chain_diag_f64(const double* x, int n_draws, int n_chains, int n_elem, long long s_draw, long long s_chain,
                       long long s_elem, double* rhat_out, double* ess_bulk_out, double* ess_tail_out, void* workspace,
                       long long workspace_bytes, void* stream)
{
    GGP_ARG(x && rhat_out && ess_bulk_out && ess_tail_out && workspace, "null pointer");
    GGP_ARG(n_draws >= 4, "n_draws must be at least 4");
    GGP_ARG(n_chains >= 1 && n_elem >= 1, "n_chains and n_elem must be positive");
    GGP_ARG((long long)n_chains * n_draws < (1LL << 31), "n_chains * n_draws must be below 2^31");
    GGP_ARG(workspace_bytes >= ggp_chain_diag_workspace_bytes(n_draws, n_chains, n_elem), "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    CdArgs a;
    a.x = x;
    a.s_draw = s_draw;
    a.s_chain = s_chain;
    a.s_elem = s_elem;
    a.n = n_draws;
    a.C = n_chains;
    a.h = n_draws / 2;
    a.ws = (unsigned char*)workspace;
    a.per = cd_layout(n_draws, n_chains).per;
    chain_diag_rank_kernel<<<n_elem, CD_NT, 0, st>>>(a);
    chain_diag_rhat_kernel<<<n_elem, CD_NT, 0, st>>>(a, rhat_out);
    chain_diag_ess_kernel<<<dim3(n_elem, 3), CD_NT, 0, st>>>(a, ess_bulk_out);
    chain_diag_finish_kernel<<<(n_elem + 127) / 128, 128, 0, st>>>(a, n_elem, ess_tail_out);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
