// Device-resident Metropolis-within-Gibbs sampler for the sim-only SEPIA model.
//
// Replaces SepiaModel.mcmc_step / do_mcmc / logPost (SURVEY.md 8a row a5, Appendix A.4-A.6,
// A.10; driven from /root/reference/src/model.py:234-235).  One step is ONE launch:
//   step kernel (1 CTA or cluster / (PC,chain)):
//     sweep     the d betaU sites, lamUz and lamWs of one PC, sequentially; each site is one fused
//               cov+Cholesky evaluation.  PCs are independent for these sites (the log-likelihood is a
//               sum of per-PC terms, priors are per element), so all PCs of all chains run at once;
//     lamWOs    the per-PC term under the candidate lamWOs (known since the start of the step);
//     close     the last CTA of a chain to finish (per-chain arrival counter) sums the pu candidate terms in
//               fixed order, accepts / rejects lamWOs, records the draw and the log-posterior, and draws
//               the candidates of the NEXT step from the uniform stream (or copies them from the replay
//               tables): candidates, bounds and the PropMH correction depend only on start-of-step values.
//   plan kernel (1 thread / chain) runs once, before the first step.
#include "ggp_chol.cuh"
#include "../../include/gladsgp_b200.h"

namespace ggp {

enum { PRIOR_UNIFORM = 0, PRIOR_GAMMA = 1, PRIOR_BETA = 2, PRIOR_NORMAL = 3 };
enum { PROP_UNIFORM = 0, PROP_BETARHO = 1, PROP_PROPMH = 2 };

__device__ inline double elem_log_prior(int kind, double a, double b, double x)
{
    switch (kind) {
        case PRIOR_GAMMA: return (a - 1.0) * log(x) - b * x;
        case PRIOR_BETA: {
            double rho = exp(-x / 4.0);
            if (rho > 0.999) rho = 0.999;
            return (a - 1.0) * log(rho) + (b - 1.0) * log(1.0 - rho);
        }
        case PRIOR_NORMAL: {
            double z = (x - a) / b;
            return -0.5 * (z * z);
        }
        default: return 0.0;
    }
}

// pl.valid of a site: what the step kernel does there
enum { SITE_REJECT = 0,      // nothing to evaluate: out of bounds, fixed, aCorr = 0, or a neutral site whose candidate the plan rejected
       SITE_EVAL = 1,        // evaluate the candidate, then accept / reject
       SITE_ACCEPT = 2 };    // neutral site whose candidate the plan accepted: th[s] = cand, the PC's term is unchanged
enum { FIXED_NEUTRAL = 3 };  // fixed table: sampled betaU element of a constant input column (include/gladsgp_b200.h)

struct Plan {
    double* cand;      // [n_chains][P]
    double* lacorr;    // [n_chains][P]
    double* logu;      // [n_chains][P]
    int* valid;        // [n_chains][P]  SITE_*
};

__device__ __forceinline__ size_t chain_prior_off(const ggp_mcmc_args& a, int c)
{
    return a.per_chain_data ? (size_t)c * ((size_t)a.d * a.pu + 2 * a.pu + 1) : 0;
}

// candidates of step t for chain c (one thread)
__device__ inline void plan_chain(const ggp_mcmc_args& a, const Plan& pl, int t, int c)
{
    const int P = a.d * a.pu + 2 * a.pu + 1;
    const double* th = a.theta + (size_t)c * P;
    const double* step = a.step + (size_t)t * a.step_stride_t + (size_t)c * a.step_stride_c;
    long long pos = a.upos ? a.upos[c] : 0;
    const double* us = a.uniforms ? a.uniforms + (size_t)c * a.n_uniform : nullptr;
    for (int s = 0; s < P; ++s) {
        const size_t o = (size_t)c * P + s;
        double cand, lac = 0.0, lu = 0.0;
        int valid;
        if (a.fixed[s] == 2) {            // block not in mcmcList: never visited, consumes no randomness
            pl.cand[o] = th[s]; pl.lacorr[o] = 0.0; pl.logu[o] = 0.0; pl.valid[o] = SITE_REJECT;
            continue;
        }
        const bool neutral = a.fixed[s] == FIXED_NEUTRAL && s < a.d * a.pu;
        const bool sampled = a.fixed[s] == 0 || neutral;
        if (a.replay) {
            const size_t ro = ((size_t)t * a.n_chains + c) * P + s;
            cand = a.r_cand[ro];
            lac = a.r_logacorr[ro];
            lu = a.r_logu[ro];
            valid = a.r_valid[ro] && sampled;
        } else {
            const double x = th[s];
            const double st = step[s];
            const double u = us[pos++];
            double acorr = 1.0;
            int kind = a.prop_kind[s];
            if (kind == PROP_PROPMH && !a.do_propMH) kind = PROP_UNIFORM;
            if (kind == PROP_UNIFORM) {
                cand = __dadd_rn(x, __dmul_rn(st, __dadd_rn(-0.5, u)));
            } else if (kind == PROP_BETARHO) {
                const double rho = __dadd_rn(exp(-x / 4.0), __dmul_rn(st, __dadd_rn(-0.5, u)));
                cand = (rho <= 0.0) ? INFINITY : -4.0 * log(rho);
            } else {
                const double w = fmax(1.0, x / 3.0);
                cand = __dadd_rn(x, __dmul_rn(w, __dadd_rn(-1.0, __dmul_rn(2.0, u))));
                const double w1 = fmax(1.0, cand / 3.0);
                acorr = (x > cand + w1) ? 0.0 : w / w1;
            }
            valid = sampled && (acorr > 0.0) && (cand >= a.lo[s]) && (cand <= a.hi[s]);
            if (valid) {
                lu = log(us[pos++]);
                lac = log(acorr);
            }
        }
        // Neutral site: the column is constant, so the candidate leaves the covariance and the PC's term exactly as they
        // are (ll_new == ll_old) and the step kernel's rule ((ll_new - ll_old) + dprior) + lacorr reduces to the one below.
        // th[s] is still its start-of-step value when the sweep reaches s (only site s writes it).  An infinite candidate
        // (BetaRho, rho <= 0) would put inf * 0 into the covariance: it is evaluated as before.
        if (valid && neutral && isfinite(cand)) {
            const size_t po = chain_prior_off(a, c) + s;
            const double dprior = elem_log_prior(a.prior_kind[s], a.prior_a[po], a.prior_b[po], cand) -
                                  elem_log_prior(a.prior_kind[s], a.prior_a[po], a.prior_b[po], th[s]);
            valid = (lu < dprior + lac) ? SITE_ACCEPT : SITE_REJECT;
        }
        pl.cand[o] = cand;
        pl.lacorr[o] = lac;
        pl.logu[o] = lu;
        pl.valid[o] = valid;
    }
    if (a.upos) a.upos[c] = pos;
}

__global__ void plan_kernel(ggp_mcmc_args a, Plan pl, int t)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < a.n_chains) plan_chain(a, pl, t, c);
}

// per-chain model data (per_chain_data != 0: chain c is its own model on the shared design)
__device__ __forceinline__ const double* chain_w(const ggp_mcmc_args& a, int c, int j)
{
    return a.W + ((size_t)(a.per_chain_data ? c : 0) * a.pu + j) * a.m;
}
__device__ __forceinline__ double chain_lamsim(const ggp_mcmc_args& a, int c, int j)
{
    return a.lamsim[(size_t)(a.per_chain_data ? c : 0) * a.pu + j];
}
// parameters of PC j under the current state, optionally with one site replaced by its candidate
__device__ inline void gather_block_params(const ggp_mcmc_args& a, const double* th, int c, int j, int site, double cand,
                                           double* beta_sm, double& lamz, double& diag_add)
{
    const int d = a.d, pu = a.pu, P = d * pu + 2 * pu + 1;
    if (threadIdx.x < d) {
        const int s = j * d + threadIdx.x;
        beta_sm[threadIdx.x] = (s == site) ? cand : th[s];
    }
    const int sz = d * pu + j, ss = d * pu + pu + j, so = P - 1;
    lamz = (sz == site) ? cand : th[sz];
    const double lamws = (ss == site) ? cand : th[ss];
    const double lamwos = (so == site) ? cand : th[so];
    diag_add = 1.0 / (chain_lamsim(a, c, j) * lamwos) + 1.0 / lamws;
}

// Look-ahead variant: NOT inlined on purpose.  Inside the site loop of the step kernel the inlined body shared its register
// budget with the loop's live state (a dozen pointers and indices) and spilled in the DMMA loops; as a function of its own
// it gets the whole budget (the caller's few live values are saved once per evaluation), as in the batched log-likelihood
// kernel.  (The cluster variant, 168 registers, has no spills when inlined and gets them as a function: it stays inline.)
#ifndef GGP_EVAL_INLINE
#define GGP_EVAL_INLINE 0
#endif
#if GGP_EVAL_INLINE
#define GGP_EVAL_ATTR __forceinline__
#else
#define GGP_EVAL_ATTR __noinline__
#endif
static __device__ GGP_EVAL_ATTR double eval_la_call(unsigned char* smem_raw, const double* __restrict__ X, int m, int Mp, int d,
                                                    const double* beta, double lamz, double diag_add,
                                                    const double* __restrict__ w, double* __restrict__ Lp, int rot)
{
    LaSmem sm = carve_la_smem(smem_raw, Mp, d);
    return eval_block_loglik_la(sm, X, m, Mp, d, beta, lamz, diag_add, w, Lp, nullptr, nullptr, rot);
}

// one evaluation by the CTA (cluster): CL = cluster variant, LA = look-ahead variant (one CTA per matrix)
template <bool CL, bool LA, int RA>
static __device__ __forceinline__ double eval_dispatch(unsigned char* smem_raw, const double* __restrict__ X, int m, int Mp, int d,
                                                       const double* beta, double lamz, double diag_add,
                                                       const double* __restrict__ w, double* __restrict__ Lp, int rot = 0)
{
    if constexpr (LA) {
        return eval_la_call(smem_raw, X, m, Mp, d, beta, lamz, diag_add, w, Lp, rot);
    } else {
        EvalSmem sm = carve_eval_smem(smem_raw, Mp, d);
        return eval_block_loglik<CL, RA>(sm, X, m, Mp, d, beta, lamz, diag_add, w, Lp, nullptr, nullptr);
    }
}

// close of step t for chain c (one thread: the lead of the last CTA of the chain to arrive): lamWOs accept / reject from
// the candidate terms summed in PC order, log-posterior, record.  Same arithmetic as SepiaModel.mcmc_step's last site.
__device__ inline void finalize_chain(const ggp_mcmc_args& a, const Plan& pl, const double* __restrict__ sig_cand, int t, int c)
{
    const int d = a.d, pu = a.pu, P = d * pu + 2 * pu + 1;
    double* th = a.theta + (size_t)c * P;
    double* sig = a.sigwl + (size_t)c * pu;
    const int s = P - 1;
    const size_t o = (size_t)c * P + s;
    int acc = 0;
    if (pl.valid[o]) {
        double sn = 0.0, so = 0.0;
        for (int j = 0; j < pu; ++j) {
            sn += sig_cand[(size_t)c * pu + j];
            so += sig[j];
        }
        const double cand = pl.cand[o];
        const size_t po = chain_prior_off(a, c) + s;
        const double dprior = elem_log_prior(a.prior_kind[s], a.prior_a[po], a.prior_b[po], cand) -
                              elem_log_prior(a.prior_kind[s], a.prior_a[po], a.prior_b[po], th[s]);
        acc = pl.logu[o] < ((sn - so) + dprior) + pl.lacorr[o];
        if (acc) {
            th[s] = cand;
            for (int j = 0; j < pu; ++j) sig[j] = sig_cand[(size_t)c * pu + j];
        }
    }
    if (a.accepted) a.accepted[((size_t)t * a.n_chains + c) * P + s] = (unsigned char)acc;
    // log posterior of the state at the end of the step: sum_j SigWl[j] + prior sums of the blocks in mcmcList
    // (a block removed from mcmcList -- fixed flag 2 -- contributes nothing, as in SepiaModel.logPost)
    if (a.lp_draws) {
        double ll = 0.0;
        for (int j = 0; j < pu; ++j) ll += sig[j];
        double lpr = 0.0;
        const int bounds[5] = {0, d * pu, d * pu + pu, d * pu + 2 * pu, P};
        for (int blk = 0; blk < 4; ++blk) {
            if (a.fixed[bounds[blk]] == 2) continue;
            double sblk = 0.0;
            for (int e = bounds[blk]; e < bounds[blk + 1]; ++e)
                sblk += elem_log_prior(a.prior_kind[e], a.prior_a[chain_prior_off(a, c) + e], a.prior_b[chain_prior_off(a, c) + e], th[e]);
            lpr += sblk;
        }
        a.lp_draws[(size_t)t * a.n_chains + c] = ll + lpr;
    }
    if (a.draws) {
        double* dr = a.draws + ((size_t)t * a.n_chains + c) * P;
        for (int e = 0; e < P; ++e) dr[e] = th[e];
    }
}

// One mcmc_step of every chain in one launch (see the header of this file).
template <bool CL, bool LA = false, int RA = GGP_RA>
__global__ void __launch_bounds__(NT, CL ? GGP_CL_CTAS_PER_SM : GGP_CTAS_PER_SM)
sweep_kernel(ggp_mcmc_args a, Plan pl, double* __restrict__ Lws, long long l_stride, double* __restrict__ sig_cand,
             unsigned* __restrict__ arrive, int t)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Mp = round_up32(a.m);
    __shared__ double beta_sm[64];
    const int j = a.pc_begin + (CL ? blockIdx.x / cluster_nctarank() : blockIdx.x), c = blockIdx.y;
    const bool lead = (threadIdx.x == 0) && (!CL || cluster_ctarank() == 0);    // the one thread that owns the state
    const int d = a.d, pu = a.pu, P = d * pu + 2 * pu + 1;
    double* th = a.theta + (size_t)c * P;
    double* sig = a.sigwl + (size_t)c * pu;
    double* Lp = Lws + ((size_t)c * pu + j) * l_stride;
    const double* wj = chain_w(a, c, j);
    unsigned char* accd = a.accepted ? a.accepted + ((size_t)t * a.n_chains + c) * P : nullptr;
    const int rot = LA ? cta_role_rotation() : 0;
    const bool shard = a.pc_count > 0;                         // PC shard: results leave through a.xchg, no close here
    double* xrow = shard ? a.xchg + ((size_t)j * a.n_chains + c) * (2 * d + 6) : nullptr;
    if (shard && lead) {
        xrow[d + 3] = sig[j];                                  // no valid lamWOs candidate: the term is not used
        for (int e = 0; e < d + 2; ++e) xrow[d + 4 + e] = 0.0;
    }

    // sites of PC j: d betaU elements, lamUz[j], lamWs[j]; then (sl == d + 2) the PC's term under the candidate lamWOs
    for (int sl = 0; sl < d + 3; ++sl) {
        const bool wos = (sl == d + 2);
        const int s = wos ? P - 1 : ((sl < d) ? j * d + sl : (sl == d ? d * pu + j : d * pu + pu + j));
        const size_t o = (size_t)c * P + s;
        const int valid = pl.valid[o];
        if (valid != SITE_EVAL) {                  // decided by the plan (the lamWOs candidate is never SITE_ACCEPT)
            const bool acc = valid == SITE_ACCEPT;
            if (lead && !wos) {
                if (acc) th[s] = pl.cand[o];
                if (accd) accd[s] = acc ? 1 : 0;
                if (shard) xrow[d + 4 + sl] = acc ? 1.0 : 0.0;
            }
            if (CL && acc) cluster_sync_all();     // the other CTAs of the cluster gather th[s] for the next evaluation
            continue;
        }
        const double cand = pl.cand[o];
        double lamz, diag_add;
        __syncthreads();
        gather_block_params(a, th, c, j, s, cand, beta_sm, lamz, diag_add);
        __syncthreads();
        const double ll_new = eval_dispatch<CL, LA, RA>(smem_raw, a.X, a.m, Mp, d, beta_sm, lamz, diag_add, wj, Lp, rot);
        if (lead) {
            if (a.eval_count) atomicAdd(a.eval_count + (wos ? 1 : 0), 1ULL);
            if (wos) {
                sig_cand[(size_t)c * pu + j] = ll_new;
            } else {
                const double ll_old = sig[j];
                const double xold = th[s];
                const size_t po = chain_prior_off(a, c) + s;
                const double dprior = elem_log_prior(a.prior_kind[s], a.prior_a[po], a.prior_b[po], cand) -
                                      elem_log_prior(a.prior_kind[s], a.prior_a[po], a.prior_b[po], xold);
                const bool acc = pl.logu[o] < ((ll_new - ll_old) + dprior) + pl.lacorr[o];
                if (acc) {
                    th[s] = cand;
                    sig[j] = ll_new;
                }
                if (accd) accd[s] = acc ? 1 : 0;
                if (shard) xrow[d + 4 + sl] = acc ? 1.0 : 0.0;
            }
        }
        if (CL) cluster_sync_all();        // the accepted state is visible to every CTA of the cluster
        else __syncthreads();
    }
    // close of the step: the last PC of the chain to arrive decides lamWOs, records, and plans the next step.  Its reads
    // of the other PCs' results are ordered by the fence / atomic pair; the sums run in PC order whoever arrives last.
    if (lead && shard) {
        for (int e = 0; e < d; ++e) xrow[e] = th[j * d + e];
        xrow[d] = th[d * pu + j];
        xrow[d + 1] = th[d * pu + pu + j];
        xrow[d + 2] = sig[j];
        if (pl.valid[(size_t)c * P + (P - 1)]) xrow[d + 3] = sig_cand[(size_t)c * pu + j];
    } else if (lead) {
        __threadfence();
        const unsigned prev = atomicAdd(&arrive[c], 1u);
        if (prev == (unsigned)pu - 1u) {
            arrive[c] = 0u;
            __threadfence();
            finalize_chain(a, pl, sig_cand, t, c);
            if (t + 1 < a.n_steps) plan_chain(a, pl, t + 1, c);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Speculative step kernel for FEW chains (the reference's own workload is ONE chain, src/model.py:234-235): the sites of a
// PC are inherently sequential, and with a handful of matrices in flight most of the GPU idles.  Three thread-block
// clusters ("lanes") per (PC, chain) evaluate, in every round, the next TWO evaluations of the PC's sequence:
//   lane 0: evaluation e0 under the current state;
//   lane 1: evaluation e1 under the state in which e0's candidate was accepted;  lane 2: e1 under the unchanged state.
// After the round every lane reads the three results, takes e0's decision, picks the matching e1 result, takes e1's
// decision -- the arithmetic of the sequential sweep, evaluation by evaluation, so the chain is bit-identical -- and
// updates its private copy of the PC's state.  A round costs one evaluation's latency and retires two.  (SURVEY 7.1 step 9.)
// The lanes of a PC meet at a counter in global memory once per round; all clusters of the launch must be resident at the
// same time (the host checks cudaOccupancyMaxActiveClusters before choosing this kernel, and the wait is bounded).
// Sequence of a PC: its valid betaU sites, lamUz, lamWs (validity is known from the plan), then its term under the candidate
// lamWOs (no decision here: that is the close of the step).
// ---------------------------------------------------------------------------------------------
constexpr int SPEC_LANES = 3;
constexpr int SPEC_MAXEV = 72;          // d + 3 <= 67

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// st = private state of one lane: [0, d) betaU[:, j], [d] lamUz[j], [d + 1] lamWs[j], [d + 2] SigWl[j];  evaluation index
// e: e < d betaU element, d lamUz, d + 1 lamWs, d + 2 lamWOs.  Up to two entries are replaced by candidates.  Neutral
// sites the plan accepted (bits of nacc, candidates in ncand) are not in st until the end of the step: an evaluation
// at index lim sees the candidates of those before it.
__device__ inline void gather_spec(const ggp_mcmc_args& a, const double* st, double lamwos_cur, int c, int j,
                                   int ea, double ca, int eb, double cb, unsigned long long nacc, const double* ncand, int lim,
                                   double* beta_sm, double& lamz, double& diag_add)
{
    const int d = a.d;
    if (threadIdx.x < d) {
        const int e = threadIdx.x;
        beta_sm[e] = (e == ea) ? ca : ((e == eb) ? cb : ((e < lim && ((nacc >> e) & 1ULL)) ? ncand[e] : st[e]));
    }
    lamz = (ea == d) ? ca : ((eb == d) ? cb : st[d]);
    const double lamws = (ea == d + 1) ? ca : ((eb == d + 1) ? cb : st[d + 1]);
    const double lamwos = (ea == d + 2) ? ca : ((eb == d + 2) ? cb : lamwos_cur);
    diag_add = 1.0 / (chain_lamsim(a, c, j) * lamwos) + 1.0 / lamws;
}

struct SpecWs {
    double* res;        // [n_chains][pu][2][4]   results of a round, by round parity and lane
    unsigned* cnt;      // [n_chains][pu]         arrivals (3 per round; zeroed by the host before every run)
    double* state;      // [n_chains][pu][3][d + 3]
    double* Lws;        // [n_chains][pu][3] factor workspaces
};

template <int RA>
__global__ void __launch_bounds__(NT, GGP_CL_CTAS_PER_SM)
sweep_spec_kernel(ggp_mcmc_args a, Plan pl, SpecWs sw, long long l_stride, double* __restrict__ sig_cand,
                  unsigned* __restrict__ arrive, int t, unsigned round_base)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double beta_sm[64];
    __shared__ int ev_sm[SPEC_MAXEV];
    __shared__ int nev_sm;
    __shared__ unsigned long long nacc_sm;
    const int Mp = round_up32(a.m);
    const int G = (int)cluster_nctarank();
    const int cl = blockIdx.x / G;                       // cluster index along x: (PC, lane)
    const int jl = cl / SPEC_LANES, lane_id = cl - jl * SPEC_LANES, c = blockIdx.y;
    const int j = a.pc_begin + jl;                       // (PC shard: this launch covers PCs [pc_begin, pc_begin + pc_count))
    const bool lead = (threadIdx.x == 0) && (cluster_ctarank() == 0);
    const bool shard = a.pc_count > 0;
    const int d = a.d, pu = a.pu, P = d * pu + 2 * pu + 1;
    const int E = d + 3;                                  // evaluations of the PC's sequence (last = lamWOs term)
    double* th = a.theta + (size_t)c * P;
    double* st = sw.state + (((size_t)c * pu + j) * SPEC_LANES + lane_id) * (d + 3);
    double* Lp = sw.Lws + (((size_t)c * pu + j) * SPEC_LANES + lane_id) * l_stride;
    double* res = sw.res + ((size_t)c * pu + j) * 8;
    unsigned* cnt = sw.cnt + (size_t)c * pu + j;
    const double* wj = chain_w(a, c, j);
    unsigned char* accd = a.accepted ? a.accepted + ((size_t)t * a.n_chains + c) * P : nullptr;
    const double lamwos_cur = th[P - 1];
    double* xrow = shard ? a.xchg + ((size_t)j * a.n_chains + c) * (2 * d + 6) : nullptr;
    if (shard && lead && lane_id == 0) {
        xrow[d + 3] = a.sigwl[(size_t)c * pu + j];
        for (int e = 0; e < d + 2; ++e) xrow[d + 4 + e] = 0.0;
    }
    auto site_of = [&](int e) { return e < d ? j * d + e : (e == d ? d * pu + j : (e == d + 1 ? d * pu + pu + j : P - 1)); };
    const double* ncand = pl.cand + (size_t)c * P + (size_t)j * d;       // candidates of the PC's betaU sites

    // private state, the list of evaluations and the neutral sites the plan accepted (identical in the three lanes)
    if (threadIdx.x == 0) {
        int n = 0;
        unsigned long long nacc = 0ULL;
        for (int e = 0; e < E; ++e) {
            const int v = pl.valid[(size_t)c * P + site_of(e)];
            if (v == SITE_EVAL) {
                ev_sm[n++] = e;
                continue;
            }
            if (v == SITE_ACCEPT) nacc |= 1ULL << e;
            if (lead && lane_id == 0 && e < d + 2) {
                if (accd) accd[site_of(e)] = (v == SITE_ACCEPT) ? 1 : 0;
                if (shard) xrow[d + 4 + e] = (v == SITE_ACCEPT) ? 1.0 : 0.0;
            }
        }
        nev_sm = n;
        nacc_sm = nacc;
        if (cluster_ctarank() == 0) {
            for (int e = 0; e < d; ++e) st[e] = th[j * d + e];
            st[d] = th[d * pu + j];
            st[d + 1] = th[d * pu + pu + j];
            st[d + 2] = a.sigwl[(size_t)c * pu + j];
        }
    }
    cluster_sync_all();
    const int nev = nev_sm;
    const unsigned long long nacc = nacc_sm;
    const int nrounds = (nev + 1) >> 1;

    for (int r = 0; r < nrounds; ++r) {
        const int e0 = ev_sm[2 * r];
        const int e1 = (2 * r + 1 < nev) ? ev_sm[2 * r + 1] : -1;
        const size_t o0 = (size_t)c * P + site_of(e0);
        const size_t o1 = (e1 >= 0) ? (size_t)c * P + site_of(e1) : 0;
        const double c0 = pl.cand[o0];
        const double c1 = (e1 >= 0) ? pl.cand[o1] : 0.0;
        // this lane's evaluation of the round
        const bool work = (lane_id == 0) || (e1 >= 0);
        double ll = 0.0;
        if (work) {
            double lamz, diag_add;
            __syncthreads();
            if (lane_id == 0) gather_spec(a, st, lamwos_cur, c, j, e0, c0, -1, 0.0, nacc, ncand, e0, beta_sm, lamz, diag_add);
            else if (lane_id == 1) gather_spec(a, st, lamwos_cur, c, j, e0, c0, e1, c1, nacc, ncand, e1, beta_sm, lamz, diag_add);
            else gather_spec(a, st, lamwos_cur, c, j, e1, c1, -1, 0.0, nacc, ncand, e1, beta_sm, lamz, diag_add);
            __syncthreads();
            ll = eval_dispatch<true, false, RA>(smem_raw, a.X, a.m, Mp, d, beta_sm, lamz, diag_add, wj, Lp, 0);
        }
        if (lead) {
            if (work && a.eval_count) atomicAdd(a.eval_count, 1ULL);
            double* slot = res + (r & 1) * 4;
            slot[lane_id] = ll;
            __threadfence();
            atomicAdd(cnt, 1u);
            const unsigned target = (round_base + (unsigned)r + 1u) * SPEC_LANES;
            const long long t0 = clock64();
            bool ok = true;
            while ((int)(ld_acquire_u32(cnt) - target) < 0) {
                if (clock64() - t0 > (1LL << 33)) { ok = false; break; }          // ~4 s: a lane is not resident (never expected)
            }
            const double l0 = __ldcg(slot + 0), l1a = __ldcg(slot + 1), l1r = __ldcg(slot + 2);
            if (!ok && a.lp_draws) a.lp_draws[(size_t)t * a.n_chains + c] = NAN;
            // decision of e0, then of e1: the sequential sweep's arithmetic
            bool acc0 = false;
            if (e0 == d + 2) {
                if (lane_id == 0) sig_cand[(size_t)c * pu + j] = l0;
            } else {
                const int s0 = site_of(e0);
                const size_t po = chain_prior_off(a, c) + s0;
                const double dprior = elem_log_prior(a.prior_kind[s0], a.prior_a[po], a.prior_b[po], c0) -
                                      elem_log_prior(a.prior_kind[s0], a.prior_a[po], a.prior_b[po], st[e0]);
                acc0 = pl.logu[o0] < ((l0 - st[d + 2]) + dprior) + pl.lacorr[o0];
                if (acc0) { st[e0] = c0; st[d + 2] = l0; }
                if (accd && lane_id == 0) accd[s0] = acc0 ? 1 : 0;
                if (shard && lane_id == 0) xrow[d + 4 + e0] = acc0 ? 1.0 : 0.0;
            }
            if (e1 >= 0) {
                const double l1 = acc0 ? l1a : l1r;
                if (e1 == d + 2) {
                    if (lane_id == 0) sig_cand[(size_t)c * pu + j] = l1;
                } else {
                    const int s1 = site_of(e1);
                    const size_t po = chain_prior_off(a, c) + s1;
                    const double dprior = elem_log_prior(a.prior_kind[s1], a.prior_a[po], a.prior_b[po], c1) -
                                          elem_log_prior(a.prior_kind[s1], a.prior_a[po], a.prior_b[po], st[e1]);
                    const bool acc1 = pl.logu[o1] < ((l1 - st[d + 2]) + dprior) + pl.lacorr[o1];
                    if (acc1) { st[e1] = c1; st[d + 2] = l1; }
                    if (accd && lane_id == 0) accd[s1] = acc1 ? 1 : 0;
                    if (shard && lane_id == 0) xrow[d + 4 + e1] = acc1 ? 1.0 : 0.0;
                }
            }
        }
        cluster_sync_all();              // the lane's state is visible to every CTA of its cluster
    }
    if (lead) {
        // every launch adds the same number of arrivals to the counter, whatever the number of valid evaluations
        const int rcap = (E + 1) >> 1;
        if (nrounds < rcap) atomicAdd(cnt, (unsigned)(rcap - nrounds));
        if (lane_id == 0)
            for (int e = 0; e < d; ++e)
                if ((nacc >> e) & 1ULL) st[e] = ncand[e];
        if (lane_id == 0 && shard) {
            for (int e = 0; e < d + 3; ++e) xrow[e] = st[e];                     // betaU[:, j], lamUz[j], lamWs[j], SigWl[j]
            if (pl.valid[(size_t)c * P + (P - 1)]) xrow[d + 3] = sig_cand[(size_t)c * pu + j];
        } else if (lane_id == 0) {
            for (int e = 0; e < d; ++e) th[j * d + e] = st[e];
            th[d * pu + j] = st[d];
            th[d * pu + pu + j] = st[d + 1];
            a.sigwl[(size_t)c * pu + j] = st[d + 2];
            __threadfence();
            const unsigned prev = atomicAdd(&arrive[c], 1u);
            if (prev == (unsigned)pu - 1u) {
                arrive[c] = 0u;
                __threadfence();
                finalize_chain(a, pl, sig_cand, t, c);
                if (t + 1 < a.n_steps) plan_chain(a, pl, t + 1, c);
            }
        }
    }
}

// mode 0: sigwl <- per-PC terms of the current state.  mode 1: sigwl_cand <- terms under candidate lamWOs.
template <bool CL, bool LA = false, int RA = GGP_RA>
__global__ void __launch_bounds__(NT, CL ? GGP_CL_CTAS_PER_SM : GGP_CTAS_PER_SM)
eval_all_kernel(ggp_mcmc_args a, Plan pl, double* __restrict__ Lws, long long l_stride,
                double* __restrict__ sig_cand, int mode)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Mp = round_up32(a.m);
    __shared__ double beta_sm[64];
    const int j = CL ? blockIdx.x / cluster_nctarank() : blockIdx.x, c = blockIdx.y;
    const int d = a.d, pu = a.pu, P = d * pu + 2 * pu + 1;
    const double* th = a.theta + (size_t)c * P;
    double* Lp = Lws + ((size_t)c * pu + j) * l_stride;
    int site = -1;
    double cand = 0.0;
    if (mode == 1) {
        const size_t o = (size_t)c * P + (P - 1);
        if (!pl.valid[o]) return;
        site = P - 1;
        cand = pl.cand[o];
    }
    double lamz, diag_add;
    const int rot = LA ? cta_role_rotation() : 0;
    gather_block_params(a, th, c, j, site, cand, beta_sm, lamz, diag_add);
    __syncthreads();
    const double ll = eval_dispatch<CL, LA, RA>(smem_raw, a.X, a.m, Mp, d, beta_sm, lamz, diag_add, chain_w(a, c, j), Lp, rot);
    if (threadIdx.x == 0 && (!CL || cluster_ctarank() == 0)) {
        if (mode == 0) a.sigwl[(size_t)c * pu + j] = ll;
        else sig_cand[(size_t)c * pu + j] = ll;
        if (a.eval_count) atomicAdd(a.eval_count + 1, 1ULL);
    }
}

// PC-sharded stepping: close of step t on every rank from the gathered rows (one thread per chain)
__global__ void close_kernel(ggp_mcmc_args a, Plan pl, double* __restrict__ sig_cand, int t, int plan_next)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chains) return;
    const int d = a.d, pu = a.pu, P = d * pu + 2 * pu + 1;
    double* th = a.theta + (size_t)c * P;
    double* sig = a.sigwl + (size_t)c * pu;
    unsigned char* accd = a.accepted ? a.accepted + ((size_t)t * a.n_chains + c) * P : nullptr;
    for (int j = 0; j < pu; ++j) {
        const double* row = a.xchg + ((size_t)j * a.n_chains + c) * (2 * d + 6);
        for (int e = 0; e < d; ++e) th[j * d + e] = row[e];
        th[d * pu + j] = row[d];
        th[d * pu + pu + j] = row[d + 1];
        sig[j] = row[d + 2];
        sig_cand[(size_t)c * pu + j] = row[d + 3];
        if (accd) {
            for (int e = 0; e < d; ++e) accd[j * d + e] = (unsigned char)(row[d + 4 + e] != 0.0);
            accd[d * pu + j] = (unsigned char)(row[d + 4 + d] != 0.0);
            accd[d * pu + pu + j] = (unsigned char)(row[d + 4 + d + 1] != 0.0);
        }
    }
    finalize_chain(a, pl, sig_cand, t, c);
    if (plan_next) plan_chain(a, pl, t + 1, c);
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Cluster size of the speculative step kernel (0: not used).  It needs 3 clusters per (PC, chain), all resident at once;
// a round retires two evaluations, so it pays when its clusters are more than half as large as those of the plain cluster
// kernel would be (cfg3, one chain: 30 clusters of 8 CTAs against 10 of 8; cfg5, one chain: 60 of 4 against 20 of 16 -- no).
// GGP_SPEC=0 in the environment switches it off.
static int spec_cluster_size(int pu, int n_chains, int Mp, int d)
{
    if (const char* e = getenv("GGP_SPEC")) { if (atoi(e) == 0) return 0; }
    if (d + 3 > SPEC_MAXEV) return 0;
    const int g_plain = choose_cluster((long long)pu * n_chains, Mp);
    if (g_plain <= 1) return 0;
    const int g_spec = choose_cluster((long long)SPEC_LANES * pu * n_chains, Mp);
    return (g_spec >= 2 && 2 * g_spec > g_plain) ? g_spec : 0;
}

// workspace carve-up shared by the entry points
struct McmcWs {
    double* Lws; Plan pl; double* sig_cand; unsigned* arrive; SpecWs spec;
};
long long workspace_bytes_impl(int m, int d, int pu, int n_chains, bool with_spec);

static McmcWs carve_ws(const ggp_mcmc_args& a)
{
    const int Mp = round_up32(a.m);
    const size_t P = (size_t)a.d * a.pu + 2 * a.pu + 1;
    McmcWs w;
    unsigned char* p = reinterpret_cast<unsigned char*>(a.workspace);
    w.Lws = reinterpret_cast<double*>(p);
    p += align256((size_t)a.n_chains * a.pu * packed_doubles(Mp) * sizeof(double));
    w.pl.cand = reinterpret_cast<double*>(p);   p += align256((size_t)a.n_chains * P * sizeof(double));
    w.pl.lacorr = reinterpret_cast<double*>(p); p += align256((size_t)a.n_chains * P * sizeof(double));
    w.pl.logu = reinterpret_cast<double*>(p);   p += align256((size_t)a.n_chains * P * sizeof(double));
    w.pl.valid = reinterpret_cast<int*>(p);     p += align256((size_t)a.n_chains * P * sizeof(int));
    w.sig_cand = reinterpret_cast<double*>(p);  p += align256((size_t)a.n_chains * a.pu * sizeof(double));
    w.arrive = reinterpret_cast<unsigned*>(p);  p += align256((size_t)a.n_chains * sizeof(unsigned));
    w.spec.res = nullptr; w.spec.cnt = nullptr; w.spec.state = nullptr; w.spec.Lws = nullptr;
    // (a workspace sized while the speculative kernel was switched off simply runs without it)
    if (spec_cluster_size(1, a.n_chains, Mp, a.d) > 0 &&
        (long long)a.workspace_bytes >= workspace_bytes_impl(a.m, a.d, a.pu, a.n_chains, true)) {
        w.spec.res = reinterpret_cast<double*>(p);   p += align256((size_t)a.n_chains * a.pu * 8 * sizeof(double));
        w.spec.cnt = reinterpret_cast<unsigned*>(p); p += align256((size_t)a.n_chains * a.pu * sizeof(unsigned));
        w.spec.state = reinterpret_cast<double*>(p); p += align256((size_t)a.n_chains * a.pu * SPEC_LANES * (a.d + 3) * sizeof(double));
        w.spec.Lws = reinterpret_cast<double*>(p);
    }
    return w;
}

}  // namespace ggp

using namespace ggp;

extern "C" {

int ggp_sizeof_mcmc_args(void) { return (int)sizeof(ggp_mcmc_args); }

}  // extern "C"

long long ggp::workspace_bytes_impl(int m, int d, int pu, int n_chains, bool with_spec)
{
    if (m <= 0 || d <= 0 || pu <= 0 || n_chains <= 0) return -1;
    const int Mp = round_up32(m);
    const size_t P = (size_t)d * pu + 2 * pu + 1;
    size_t b = 0;
    b += align256((size_t)n_chains * pu * packed_doubles(Mp) * sizeof(double));   // factor workspaces
    b += 3 * align256((size_t)n_chains * P * sizeof(double));                      // cand, lacorr, logu
    b += align256((size_t)n_chains * P * sizeof(int));                             // valid
    b += align256((size_t)n_chains * pu * sizeof(double));                         // sigwl_cand
    b += align256((size_t)n_chains * sizeof(unsigned));                            // per-chain arrival counters
    if (with_spec) {                                                               // speculative step kernel (few chains)
        b += align256((size_t)n_chains * pu * 8 * sizeof(double));
        b += align256((size_t)n_chains * pu * sizeof(unsigned));
        b += align256((size_t)n_chains * pu * SPEC_LANES * (d + 3) * sizeof(double));
        b += align256((size_t)n_chains * pu * SPEC_LANES * packed_doubles(Mp) * sizeof(double));
    }
    return (long long)b;
}

extern "C" {

long long ggp_mcmc_workspace_bytes(int m, int d, int pu, int n_chains)
{
    if (m <= 0 || d <= 0 || pu <= 0 || n_chains <= 0) return -1;
    // few chains: room for the speculative step kernel (eligible for the whole chain or for a PC shard of it)
    return workspace_bytes_impl(m, d, pu, n_chains, spec_cluster_size(1, n_chains, round_up32(m), d) > 0);
}

int ggp_mcmc_run_f64(const ggp_mcmc_args* args, void* stream)
{
    GGP_ARG(args, "null args");
    const ggp_mcmc_args a = *args;
    GGP_ARG(a.m > 0 && a.d > 0 && a.pu > 0 && a.n_chains > 0 && a.n_steps >= 0, "sizes must be positive");
    GGP_ARG(a.d <= 64, "d must be <= 64");
    GGP_ARG(a.X && a.W && a.lamsim && a.theta && a.sigwl, "null model/state pointer");
    GGP_ARG(a.prior_kind && a.prior_a && a.prior_b && a.lo && a.hi && a.prop_kind && a.fixed && a.step, "null table pointer");
    GGP_ARG(a.workspace, "null workspace");
    GGP_ARG(a.pc_count >= 0 && a.pc_begin >= 0 && a.pc_begin + a.pc_count <= a.pu, "PC shard out of range");
    if (a.pc_count > 0) {
        GGP_ARG(a.n_steps == 1 && a.xchg, "a PC shard runs one step per call and needs xchg");
        GGP_ARG(a.step_index >= 0, "step_index must be >= 0");
    } else {
        GGP_ARG(a.pc_begin == 0, "pc_begin without pc_count");
    }
    if (a.replay) GGP_ARG(a.r_cand && a.r_logacorr && a.r_logu && a.r_valid, "replay tables missing");
    else GGP_ARG(a.uniforms && a.upos && a.n_uniform > 0, "uniform stream missing");
    const long long need = workspace_bytes_impl(a.m, a.d, a.pu, a.n_chains, false);
    if ((long long)a.workspace_bytes < need) {
        set_error("ggp_mcmc_run_f64: workspace too small (%lld < %lld)", (long long)a.workspace_bytes, need);
        return GGP_ERR_WORKSPACE;
    }
    if (!a.replay && a.pc_count == 0) {
        const long long P = (long long)a.d * a.pu + 2 * a.pu + 1;
        GGP_ARG(a.n_uniform >= 2 * P * a.n_steps, "uniform stream shorter than 2*P*n_steps");
    }
    const int Mp = round_up32(a.m);
    int G = choose_cluster((long long)a.pu * a.n_chains, round_up32(a.m));
    int Gs = 0;                                    // cluster size of the speculative step kernel (0: not used)
    const bool la = (G == 1) && use_lookahead();
    const size_t smem = la ? la_smem_bytes(Mp, a.d) : eval_smem_bytes(Mp, a.d);
    if (smem > 227 * 1024) {
        set_error("ggp_mcmc_run_f64: m=%d d=%d needs %zu B of shared memory (> 227 KB)", a.m, a.d, smem);
        return GGP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int cpct = eval_carveout_pct(smem);
    const bool deep = Mp <= 1024;          // cluster kernels: A-fragment ring depth 4 (see eval_block_loglik)
    if (G > 1) {
        auto prep = [&](auto sweep, auto evall) -> int {
            GGP_CUDA(cudaFuncSetAttribute(sweep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            GGP_CUDA(cudaFuncSetAttribute(sweep, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
            GGP_CUDA(cudaFuncSetAttribute(evall, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            GGP_CUDA(cudaFuncSetAttribute(evall, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
            G = checked_cluster(sweep, G, smem);
            G = checked_cluster(evall, G, smem);
            return GGP_OK;
        };
        const int rc = deep ? prep(sweep_kernel<true, false, 4>, eval_all_kernel<true, false, 4>)
                            : prep(sweep_kernel<true, false, 2>, eval_all_kernel<true, false, 2>);
        if (rc != GGP_OK) return rc;
        // speculative step kernel: three clusters per (PC, chain), every one of them resident at the same time
        const int npc = a.pc_count > 0 ? a.pc_count : a.pu;                 // PCs swept by this call
        if (carve_ws(a).spec.Lws != nullptr) Gs = spec_cluster_size(npc, a.n_chains, Mp, a.d);
        if (Gs > 0) {
            auto prep_spec = [&](auto kern) -> int {
                GGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                GGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
                if (Gs > 8 && cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
                    cudaGetLastError(); Gs = 0; return GGP_OK;
                }
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3(SPEC_LANES * npc * Gs, a.n_chains); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = smem;
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = (unsigned)Gs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.attrs = at; cfg.numAttrs = 1;
                int nact = 0;
                if (cudaOccupancyMaxActiveClusters(&nact, kern, &cfg) != cudaSuccess || nact < SPEC_LANES * npc * a.n_chains) {
                    cudaGetLastError(); Gs = 0;
                }
                return GGP_OK;
            };
            const int rs = deep ? prep_spec(sweep_spec_kernel<4>) : prep_spec(sweep_spec_kernel<2>);
            if (rs != GGP_OK) return rs;
        }
    } else if (la) {
        GGP_CUDA(cudaFuncSetAttribute(sweep_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GGP_CUDA(cudaFuncSetAttribute(sweep_kernel<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
        GGP_CUDA(cudaFuncSetAttribute(eval_all_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GGP_CUDA(cudaFuncSetAttribute(eval_all_kernel<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
    } else {
        GGP_CUDA(cudaFuncSetAttribute(sweep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GGP_CUDA(cudaFuncSetAttribute(sweep_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
        GGP_CUDA(cudaFuncSetAttribute(eval_all_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GGP_CUDA(cudaFuncSetAttribute(eval_all_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cpct));
    }

    const McmcWs wsp = carve_ws(a);
    double* Lws = wsp.Lws;
    Plan pl = wsp.pl;
    double* sig_cand = wsp.sig_cand;
    unsigned* arrive = wsp.arrive;
    const long long l_stride = packed_doubles(Mp);
    const bool shard = a.pc_count > 0;
    const dim3 grid_all(a.pu * G, a.n_chains);
    const dim3 grid((shard ? a.pc_count : a.pu) * G, a.n_chains);
    const int cb = (a.n_chains + 31) / 32;

    auto launch_eval_all = [&](int mode) -> cudaError_t {
        if (G > 1) return deep ? launch_maybe_cluster(eval_all_kernel<true, false, 4>, grid_all, dim3(NT), smem, st, G, a, pl, Lws, l_stride, sig_cand, mode)
                               : launch_maybe_cluster(eval_all_kernel<true, false, 2>, grid_all, dim3(NT), smem, st, G, a, pl, Lws, l_stride, sig_cand, mode);
        if (la) eval_all_kernel<false, true><<<grid_all, NT, smem, st>>>(a, pl, Lws, l_stride, sig_cand, mode);
        else eval_all_kernel<false><<<grid_all, NT, smem, st>>>(a, pl, Lws, l_stride, sig_cand, mode);
        return cudaGetLastError();
    };
    const SpecWs specws = wsp.spec;
    const int rcap = (a.d + 3 + 1) / 2;            // rounds of the speculative kernel per step (arrivals per step: 3 * rcap)
    auto launch_sweep = [&](int t, int tbase = -1) -> cudaError_t {
        if (Gs > 0) {
            const dim3 gs(SPEC_LANES * (a.pc_count > 0 ? a.pc_count : a.pu) * Gs, a.n_chains);
            const unsigned base = (unsigned)(tbase >= 0 ? tbase : t) * (unsigned)rcap;   // rounds since the counters were zeroed
            return deep ? launch_maybe_cluster(sweep_spec_kernel<4>, gs, dim3(NT), smem, st, Gs, a, pl, specws, l_stride, sig_cand, arrive, t, base)
                        : launch_maybe_cluster(sweep_spec_kernel<2>, gs, dim3(NT), smem, st, Gs, a, pl, specws, l_stride, sig_cand, arrive, t, base);
        }
        if (G > 1) return deep ? launch_maybe_cluster(sweep_kernel<true, false, 4>, grid, dim3(NT), smem, st, G, a, pl, Lws, l_stride, sig_cand, arrive, t)
                               : launch_maybe_cluster(sweep_kernel<true, false, 2>, grid, dim3(NT), smem, st, G, a, pl, Lws, l_stride, sig_cand, arrive, t);
        if (la) sweep_kernel<false, true><<<grid, NT, smem, st>>>(a, pl, Lws, l_stride, sig_cand, arrive, t);
        else sweep_kernel<false><<<grid, NT, smem, st>>>(a, pl, Lws, l_stride, sig_cand, arrive, t);
        return cudaGetLastError();
    };
    if (a.init_sigwl) GGP_CUDA(launch_eval_all(0));
    if (shard) {
        // one step of a PC shard: candidates come from ggp_mcmc_plan_f64 / ggp_mcmc_close_f64, the close is the caller's
        if (Gs > 0) GGP_CUDA(cudaMemsetAsync(specws.cnt, 0, (size_t)a.n_chains * a.pu * sizeof(unsigned), st));
        GGP_CUDA(launch_sweep(a.step_index, 0));
        return GGP_OK;
    }
    if (a.n_steps > 0) {
        GGP_CUDA(cudaMemsetAsync(arrive, 0, (size_t)a.n_chains * sizeof(unsigned), st));
        if (Gs > 0) GGP_CUDA(cudaMemsetAsync(specws.cnt, 0, (size_t)a.n_chains * a.pu * sizeof(unsigned), st));
        plan_kernel<<<cb, 32, 0, st>>>(a, pl, 0);
        GGP_CUDA(cudaGetLastError());
    }
    // optional device timing of the step kernels (CUDA events on the launching stream)
    const bool timed = a.kernel_ms != nullptr && a.n_steps > 0;
    cudaEvent_t* ev = nullptr;
    if (timed) {
        ev = new cudaEvent_t[2 * (size_t)a.n_steps];
        for (int i = 0; i < 2 * a.n_steps; ++i) cudaEventCreate(&ev[i]);
    }
    cudaError_t le = cudaSuccess;
    for (int t = 0; t < a.n_steps && le == cudaSuccess; ++t) {
        if (timed) cudaEventRecord(ev[2 * t + 0], st);
        le = launch_sweep(t);
        if (timed) cudaEventRecord(ev[2 * t + 1], st);
    }
    if (timed) {
        cudaStreamSynchronize(st);
        double sw = 0.0;
        if (le == cudaSuccess)
            for (int t = 0; t < a.n_steps; ++t) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, ev[2 * t + 0], ev[2 * t + 1]); sw += ms;
            }
        a.kernel_ms[0] = sw;      // total step-kernel time (ms): sweep + lamWOs terms + close of the step
        a.kernel_ms[1] = 0.0;     // (the lamWOs wave was a launch of its own before version 2)
        for (int i = 0; i < 2 * a.n_steps; ++i) cudaEventDestroy(ev[i]);
        delete[] ev;
    }
    if (le != cudaSuccess) return cuda_fail(le, "mcmc launches");
    return GGP_OK;
}

static int check_shard_args(const ggp_mcmc_args* args)
{
    GGP_ARG(args, "null args");
    const ggp_mcmc_args& a = *args;
    GGP_ARG(a.m > 0 && a.d > 0 && a.pu > 0 && a.n_chains > 0, "sizes must be positive");
    GGP_ARG(a.d <= 64, "d must be <= 64");
    GGP_ARG(a.theta && a.sigwl && a.workspace && a.fixed && a.step, "null state / table pointer");
    GGP_ARG((long long)a.workspace_bytes >= workspace_bytes_impl(a.m, a.d, a.pu, a.n_chains, false), "workspace too small");
    if (a.replay) GGP_ARG(a.r_cand && a.r_logacorr && a.r_logu && a.r_valid, "replay tables missing");
    else GGP_ARG(a.uniforms && a.upos && a.n_uniform > 0, "uniform stream missing");
    return GGP_OK;
}

int ggp_mcmc_plan_f64(const ggp_mcmc_args* args, int t, void* stream)
{
    const int rc = check_shard_args(args);
    if (rc != GGP_OK) return rc;
    const ggp_mcmc_args a = *args;
    GGP_ARG(t >= 0, "t must be >= 0");
    const McmcWs w = carve_ws(a);
    plan_kernel<<<(a.n_chains + 31) / 32, 32, 0, (cudaStream_t)stream>>>(a, w.pl, t);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

int ggp_mcmc_close_f64(const ggp_mcmc_args* args, int t, int plan_next, void* stream)
{
    const int rc = check_shard_args(args);
    if (rc != GGP_OK) return rc;
    const ggp_mcmc_args a = *args;
    GGP_ARG(t >= 0 && a.xchg, "t must be >= 0 and xchg non-null");
    const McmcWs w = carve_ws(a);
    close_kernel<<<(a.n_chains + 31) / 32, 32, 0, (cudaStream_t)stream>>>(a, w.pl, w.sig_cand, t, plan_next);
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

}  // extern "C"
