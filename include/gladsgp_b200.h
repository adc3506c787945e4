/* gladsgp_b200 -- C ABI of the B200-native GP-emulator hot path (libgladsgp_b200.so).
 *
 * The reference (timghill/GladsGP) has no FFI of its own: the path sits behind the Python package
 * `sepia` (imports at /root/reference/src/model.py:13-15 and
 * experiments/synthetic/analysis/assess_all_models.py:30-32).  Each entry point below names the
 * reference-side routine it replaces; the SEPIA routines are un-vendored (requirements-cc.txt:42),
 * so they are cited by the call site that drives them and by SURVEY.md Appendix A.
 *
 * Conventions: extern "C"; every function returns 0 on success or a negative GGP_ERR_* code
 * (text via ggp_last_error_string(), thread-local); no exceptions cross the boundary; all array
 * pointers are DEVICE pointers unless the name ends in _host; row-major; `stream` is a
 * cudaStream_t passed as void* (NULL = default stream); the caller owns every buffer; calls are
 * asynchronous on `stream`.
 */
#ifndef GLADSGP_B200_H
#define GLADSGP_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GGP_VERSION 202

int ggp_version(void);
const char* ggp_last_error_string(void);
int ggp_device_info(int* sm_count, int* cc_major, int* cc_minor, long long* smem_optin);

/* ---- (1) covariance ---------------------------------------------------------------------
 * SepiaDistCov.compute_cov_mat type 1 (SURVEY 8a row a3; A.10 cov_self + nugget fill, as used by
 * compute_log_lik under src/model.py:234-235):
 *   C[b][i][j] = exp(-sum_k beta[b][k] (X[i][k]-X[j][k])^2) / lamz[b]   (i != j)
 *   C[b][i][i] = 1/lamz[b] + diag_add[b]
 * X[m][d], beta[B][d], lamz[B], diag_add[B], C_out[B][m][m]. */
int ggp_cov_build_f64(const double* X, int m, int d, const double* beta, const double* lamz,
                      const double* diag_add, int B, double* C_out, void* stream);

/* SepiaDistCov type 2 (cross covariance; SURVEY A.10 cov_cross, used by wPred under
 * assess_all_models.py:489-490):  S21[b][i][t] = exp(-sum_k beta[b][k](X[i][k]-Xp[t][k])^2)/lamz[b]
 * X[m][d], Xp[n][d], S21_out[B][m][n]. */
int ggp_cross_cov_f64(const double* X, int m, const double* Xp, int n, int d, const double* beta,
                      const double* lamz, int B, double* S21_out, void* stream);

/* ---- (2) fused covariance + Cholesky + log-determinant + forward solve ------------------------
 * doLogLik / compute_log_lik (SURVEY 8a row a4; A.10 do_loglik): for each b
 *   loglik[b] = -sum_i log L_ii - 0.5 ||L^-1 W[b]||^2 ,  L = chol(C[b]) (C as above, never stored)
 * info[b] = 0, or the 1-based index of the first non-positive pivot (then loglik[b] = -inf; the
 * reference maps a failed Cholesky to -inf the same way).
 * W: vector b starts at W + b*w_stride.  factor_ws[B][ggp_factor_doubles(m)] receives the packed
 * factor (layout in DESIGN.md; unpack with ggp_factor_unpack_f64).  u_out (nullable)
 * [B][ggp_padded_m(m)] receives L^-1 W[b], zero padded.  info_out nullable.  A matrix runs on one CTA
 * (look-ahead schedule) or on a thread-block cluster, chosen from B and m: both give bit-identical results. */
/* test hook: out[i] = exp(y[i]) for y <= 0 with the kernel-internal exponential (about 1 ulp) */
int ggp_debug_exp_neg_f64(const double* y, double* out, int n, void* stream);
long long ggp_factor_doubles(int m);
int ggp_padded_m(int m);
int ggp_loglik_batched_f64(const double* X, int m, int d, const double* W, long long w_stride,
                           const double* beta, const double* lamz, const double* diag_add, int B,
                           double* factor_ws, double* u_out, double* loglik_out, int* info_out, void* stream);
int ggp_factor_unpack_f64(const double* factor_ws, int m, int B, double* L_dense, void* stream);

/* ---- Metropolis-within-Gibbs sampler ------------------------------------------------------------
 * SepiaModel.mcmc_step / do_mcmc (SURVEY 8a row a5; A.4-A.6, A.10 mcmc_step), n_chains independent
 * chains of one model.  Parameter vector theta[P], P = d*pu + 2*pu + 1, in SEPIA's sampling order:
 * betaU in Fortran order (all d inputs of PC 0, then PC 1, ...), lamUz[pu], lamWs[pu], lamWOs.
 * Per-element tables have length P.  fixed: 0 sampled, 1 fixed (SEPIA still draws the candidate, then
 * rejects), 2 not in mcmcList (never visited, no draw), 3 sampled and likelihood-neutral: a betaU element
 * (k, j) whose input column k of X holds the same finite value in every row (the dummy x of a model without
 * x_sim).  Its beta multiplies (x_ik - x_jk)^2 = 0, so the PC's term does not depend on it; the sampler draws
 * the candidate and the uniforms as for 0 and decides from the prior ratio alone, without an evaluation.
 * Code 3 on any other element reads as 0.  Enumerations:
 *   prior_kind: 0 Uniform, 1 Gamma(a, b = rate), 2 Beta(a, b) on rho = exp(-x/4) (rho clamped to
 *               0.999), 3 Normal(a = mean, b = sd)
 *   prop_kind : 0 Uniform  x + step*U(-.5,.5);  1 BetaRho;  2 PropMH (Uniform when !do_propMH)
 * Two ways to feed randomness:
 *   replay = 0: uniforms[n_chains][n_uniform] is a pre-drawn U[0,1) stream per chain, consumed
 *               exactly like SEPIA consumes np.random (one draw per visited site, one more iff the
 *               candidate is in bounds and aCorr > 0); upos[n_chains] (in/out) = draws consumed.
 *   replay = 1: r_cand / r_logacorr / r_logu / r_valid [n_steps][n_chains][P] give every
 *               candidate, log(aCorr), log(u) and validity explicitly (bit-exact replays).
 * step: element s of chain c at step t is step[t*step_stride_t + c*step_stride_c + s].
 * Outputs (nullable): draws[n_steps][n_chains][P], lp_draws[n_steps][n_chains],
 * accepted[n_steps][n_chains][P].  theta and sigwl[n_chains][pu] are updated in place;
 * init_sigwl != 0 recomputes sigwl from theta first. */
typedef struct ggp_mcmc_args {
    int m, d, pu, n_chains, n_steps;
    int do_propMH, replay, init_sigwl;
    int per_chain_data;    /* 0: every chain samples the same model.  1: chain c is its own model on the shared design X
                              (e.g. the per-threshold scalar models of fit_scalar_models.py:457-473 fitted together):
                              W is [n_chains][pu][m], lamsim [n_chains][pu], prior_a / prior_b [n_chains][P] */
    const double* X;       /* [m][d]   zt = [dummy x | t]           */
    const double* W;       /* [pu][m]  PC weights                   */
    const double* lamsim;  /* [pu]     diag(K K^T)                  */
    const int* prior_kind;
    const double* prior_a;
    const double* prior_b;
    const double* lo;
    const double* hi;
    const int* prop_kind;
    const unsigned char* fixed;
    const double* step;
    long long step_stride_t, step_stride_c;
    double* theta;         /* [n_chains][P] in/out */
    double* sigwl;         /* [n_chains][pu] in/out */
    const double* uniforms;
    long long n_uniform;
    long long* upos;
    const double* r_cand;
    const double* r_logacorr;
    const double* r_logu;
    const unsigned char* r_valid;
    double* draws;
    double* lp_draws;
    unsigned char* accepted;
    void* workspace;
    size_t workspace_bytes;
    unsigned long long* eval_count; /* device, nullable: [2] += block evaluations done by the sweep launches
                              and by the init / lamWOs-wave launches */
    double* kernel_ms;     /* HOST pointer, nullable: [0] receives the total device time (ms, CUDA events on
                              `stream`) of the step kernels, [1] = 0 (the lamWOs terms are part of the step
                              kernel since version 2); makes the call synchronous */
    /* PC shard (SURVEY 8e ii: one chain's PCs spread over several GPUs).  pc_count == 0: all PCs, every step is
     * closed inside the step kernel.  pc_count > 0: this call sweeps only PCs [pc_begin, pc_begin + pc_count) of
     * ONE step (n_steps must be 1; step_index = its index into step / replay / draws / accepted) and leaves, per
     * (PC j, chain c), the row  xchg[(j * n_chains + c) * (2 d + 6)] = { betaU[:, j] (d), lamUz[j], lamWs[j],
     * SigWl[j], SigWl[j] under the candidate lamWOs, accept flags of the d + 2 sites }.  The caller gathers the rows
     * of all shards (e.g. NCCL all_gather) and closes the step on every rank with ggp_mcmc_close_f64, which unpacks
     * all pu rows, decides lamWOs, records, and draws the candidates of the next step; ggp_mcmc_plan_f64 draws those
     * of the first step.  Every rank holds the full state and reaches bit-identical decisions. */
    int pc_begin, pc_count, step_index, reserved0;
    double* xchg;          /* device, [pu][n_chains][2 d + 6]; used iff pc_count > 0 */
} ggp_mcmc_args;

int ggp_sizeof_mcmc_args(void);   /* sizeof(ggp_mcmc_args), for binding self-checks */
long long ggp_mcmc_workspace_bytes(int m, int d, int pu, int n_chains);
int ggp_mcmc_run_f64(const ggp_mcmc_args* args, void* stream);
/* PC-sharded stepping (see ggp_mcmc_args.pc_count): candidates of step t; close of step t from the gathered rows
 * (plan_next != 0: also the candidates of step t + 1). */
int ggp_mcmc_plan_f64(const ggp_mcmc_args* args, int t, void* stream);
int ggp_mcmc_close_f64(const ggp_mcmc_args* args, int t, int plan_next, void* stream);

/* ---- (3) posterior prediction ------------------------------------------------------------------
 * SepiaPredict.wPred (SURVEY 8a row a7; A.7, A.10 w_pred; callers assess_all_models.py:489-490,
 * plot_test_error.py:77, time_predictions.py:76).  For every (posterior sample, PC) pair b the
 * caller first factors S22 once with ggp_loglik_batched_f64 (factor + u = L^-1 w); then
 *   V[b]      = S21[b]^T L[b]^-T                         (n x m, rows = test designs)
 *   mean[b]   = V[b] u[b]                                = S21^T S22^-1 w
 *   var[b][t] = s11_diag[b] - sum_k V[b][t][k]^2         = diag(S11 - S21^T S22^-1 S21)
 * factor[B][ggp_factor_doubles(m)], u[B][ggp_padded_m(m)], beta[B][d], lamz[B], s11_diag[B]
 * (= 1/lamUz + 1/lamWs), Xp[n][d].  V_out nullable: [B][n][ggp_padded_m(m)].
 * workspace: ggp_predict_workspace_bytes(m, n, B). */
long long ggp_predict_workspace_bytes(int m, int n, int B);
int ggp_predict_f64(const double* X, int m, int d, const double* factor, const double* u, const double* beta,
                    const double* lamz, const double* s11_diag, const double* Xp, int n, int B,
                    double* mean_out, double* var_out, double* V_out, void* workspace, long long workspace_bytes,
                    void* stream);
/* Joint predictive covariance of n designs (the per-PC block of SEPIA's Syhat):
 *   Sigma[b] = S11[b] - V[b] V[b]^T,  S11 off-diagonal = cov(xp_s, xp_t), diagonal = s11_diag[b]. */
int ggp_pred_cov_f64(const double* Xp, int n, int d, const double* beta, const double* lamz,
                     const double* s11_diag, const double* V, int m, int B, double* Sigma_out, void* stream);
/* The draw step of SEPIA's wPred (rmultnormsvd on the per-PC blocks of Syhat, SURVEY A.7): one multivariate-normal
 * deviate per block, dev_out[b] = L[b] z[b] with Sigma[b] = L[b] L[b]^T.  SEPIA multiplies by U sqrt(s) of an SVD; the
 * Cholesky factor gives the same distribution (neither is bit-comparable across implementations).
 *   Sigma (B, n, n) row-major symmetric (as written by ggp_pred_cov_f64), z and dev_out (B, n), info_out (B):
 *   0 or the 1-based index of a non-positive pivot (dev_out[b] is then undefined; the caller falls back).
 * workspace: scratch factors; any size >= ggp_chol_draw_workspace_bytes(n, 1) works (blocks are processed in as many
 * launches as the workspace requires), ggp_chol_draw_workspace_bytes(n, B) gives one launch. */
long long ggp_chol_draw_workspace_bytes(int n, int B);
int ggp_chol_draw_f64(const double* Sigma, int n, int B, const double* z, double* dev_out, int* info_out,
                      void* workspace, long long workspace_bytes, void* stream);
/* Cross-validation from the factor of the FULL training covariance (SepiaXvalEmulatorPrediction; SEPIA refits a
 * sub-model per fold instead).  For every block b and held-out training row i = idx[t]:
 *   z = L[b]^-1 e_i   (zero above row i),   alpha_out[b][t] = z . u[b],   pdiag_out[b][t] = z . z = (S22^-1)_ii
 * and, if Z_out is not null, Z_out[b][t][0:ggp_padded_m(m)] = z (zero padded).  A leave-one-out fold needs only these:
 * mean = w_i - alpha / p, variance = 1 / p - 1 / (LamSim lamWOs); a larger fold F needs the rows z_i, i in F
 * ((S22^-1)_FF = Z_F Z_F^T).  factor / u as for ggp_predict_f64; idx[nidx] int32 in any order (ascending order lets each
 * row skip the panels above its index: about m^3/3 flop per block instead of m^3); an entry outside [0, m) gives a zero
 * row.  Sums are in a fixed order (deterministic).  workspace: ggp_xval_workspace_bytes(m, nidx, B). */
long long ggp_xval_workspace_bytes(int m, int nidx, int B);
int ggp_xval_solve_f64(const double* factor, const double* u, int m, int B, const int* idx, int nidx,
                       double* alpha_out, double* pdiag_out, double* Z_out, void* workspace, long long workspace_bytes,
                       void* stream);

/* SepiaEmulatorPrediction.get_y (SURVEY 8a row a8; assess_all_models.py:492), float32:
 *   y[r][c] = (sum_p w[r][p] K[p][c]) * sd[c] + mean[c],  r < R (= nsamp*npred), c < n_y.
 * sd_len / mean_len are 1 (scalar) or n_y. */
int ggp_reconstruct_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                        int mean_len, int R, int pu, long long n_y, float* y_out, void* stream);

/* Fused predictive-distribution statistics (SURVEY 8f rank 1; what every caller does right after get_y:
 * assess_all_models.py:493-500, plot_test_error.py:81-87), float32.  Over the posterior samples s, for design t
 * and output c:  y_s = (w[s][t] . K[:,c]) * sd[c] + mean[c],  z_s = y_s + sd[c] * noise[s][t]  (noise nullable):
 *   ymean = mean_s y_s;  ylo / yhi = q and 1-q quantiles of z_s (np.quantile, linear interpolation).
 * w[nsamp][npred][pu], noise[nsamp][npred], outputs [npred][n_y].  Needs floor(q (nsamp-1)) + 2 <= 8 and pu <= 16
 * (GGP_ERR_UNSUPPORTED otherwise). */
int ggp_reconstruct_stats_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                              int mean_len, const float* noise, int nsamp, int npred, int pu, long long n_y, double q,
                              float* ymean_out, float* ylo_out, float* yhi_out, void* stream);
/* 1 if ggp_reconstruct_stats_f32 / ggp_reconstruct_errstats_f32 serve (nsamp, pu, q) -- the order statistic
 * floor(q (nsamp-1)) + 2 <= 8 and <= nsamp, pu <= 16, the staged samples within 200 KB -- else 0 (they return
 * GGP_ERR_UNSUPPORTED).  Argument errors are not judged here. */
int ggp_reconstruct_stats_supported(int nsamp, int pu, double q);

/* Exact quantile fields over the posterior samples, for any sample count up to 16 384, up to 32 quantiles and pu <= 32
 * (csrc/ggp_quantile.cu).  y_s, z_s as above (noise nullable; without it z_s = y_s), formed with the same float32
 * operations as ggp_reconstruct_f32 and `y + sd * noise`:
 *   ymean_out[t][c] = mean_s y_s (FP64 sum in a fixed order, rounded once; nullable),
 *   yq_out[k][t][c] = np.quantile(z, q_host[k]) of the float32 z_s (NumPy 2.x, method 'linear', float32 arithmetic:
 *                     pos = float32(nsamp-1) float32(q), i = floor(pos), t = pos - i, j = min(i+1, nsamp-1),
 *                     d = x_j - x_i, x_j - d (1-t) if t >= 0.5 else x_i + d t); a NaN sample makes every quantile NaN.
 * q_host[nq] is a HOST array of values in [0, 1], 1 <= nq <= 32.  Any npred.  GGP_ERR_UNSUPPORTED for nsamp > 16384 or
 * pu > 32. */
int ggp_reconstruct_quantiles_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                                  int mean_len, const float* noise, int nsamp, int npred, int pu, long long n_y,
                                  const double* q_host, int nq, float* ymean_out, float* yq_out, void* stream);

/* Same pass with the test-error statistics of assess_all_models.py:523-538 fused in: for every test design t
 *   err[t] = { sum (ymean - y_test)^2,  sum |ymean - y_test| / y_test over y_test >= mape_floor,  count(y_test >= mape_floor),
 *              count(ylo <= y_test <= yhi),  sum ylo,  sum yhi }        (FP64 sums over the n_y outputs, fixed order)
 * from which RMSE, MAPE (the reference masks y_test below its 10 % quantile: mape_floor), coverage, mean limits and the
 * integrated interval width follow.  ymean_out / ylo_out / yhi_out may all be null: then no field is written at all.
 * y_test[npred][n_y]; err_out[npred][6]; workspace: ggp_errstats_workspace_bytes(npred, n_y). */
long long ggp_errstats_workspace_bytes(int npred, long long n_y);
int ggp_reconstruct_errstats_f32(const float* w, const float* K, const float* sd, int sd_len, const float* mean,
                                 int mean_len, const float* noise, int nsamp, int npred, int pu, long long n_y, double q,
                                 const float* y_test, float mape_floor, float* ymean_out, float* ylo_out, float* yhi_out,
                                 double* err_out, void* workspace, long long workspace_bytes, void* stream);
/* The same six sums from stored fields (e.g. those of ggp_reconstruct_quantiles_f32): ymean, ylo, yhi, y_test [npred][n_y].
 * The column tiles and the summation order are those of ggp_reconstruct_errstats_f32, so fed that function's own fields
 * it returns its err bit for bit.  workspace: ggp_errstats_workspace_bytes(npred, n_y). */
int ggp_fields_errstats_f32(const float* ymean, const float* ylo, const float* yhi, const float* y_test, int npred,
                            long long n_y, float mape_floor, double* err_out, void* workspace, long long workspace_bytes,
                            void* stream);

/* ---- Sobol' / Saltelli sensitivity statistics (SURVEY 8f rank 3) --------------------------------
 * src/utils.py:80-92 (point estimates), :97-118 and :213-243 (the statistics scipy.stats.bootstrap evaluates 9999 times and
 * the BCa jackknife N times; callers sensitivity_indices.py:96,214).  For each of R index sets ids (n entries of 0..N-1;
 * idx null = the identity set 0..n-1):
 *   var = population variance of [f_A[ids], f_B[ids]] per output;  V = mean(f_A (f_AB - f_B));  E = mean((f_B - f_AB)^2)/2
 *   first[r][out][i] = V/var,  total[r][out][i] = E/var   (V, E clamped at 0 iff clamp, as in the reference's bootstrap statistics)
 * fA, fB [N][p]; fAB [n_dim][N][p]; idx [R][idx_stride] int32; outputs [R][p][n_dim]. */
int ggp_sobol_stats_f64(const double* fA, const double* fB, const double* fAB, int N, int p, int n_dim,
                        const int* idx, long long idx_stride, int n, int R, int clamp,
                        double* first_out, double* total_out, void* stream);

/* ---- Closed-form GP sensitivity (csrc/ggp_gp_sens.cu) -------------------------------------------
 * Exact Sobol' moments of f(x) = sum_n a_n prod_k exp(-beta_nk (x_k - z_nk)^2) with independent inputs uniform on
 * [0,1]^q (the emulator's predictive mean of a PC weight: a = S22^-1 w / lamUz).  Blocks b = s * pu + j carry beta[b][q]
 * and the weights a[b][m] of the m training rows Z[m][q] (the inputs only: no dummy-x column).
 *   mode 0: one function per block, terms n = i (F = S pu functions);
 *   mode 1: one function per PC j, terms n = (s, i) over every sample (F = pu; scale a by 1/S for the posterior mean).
 * Per function f, with M(u) = E_{x_u}[(E_{x_~u} f)^2]:
 *   M_out[f][k] = M({k}),  M_out[f][q + k] = M(all \ k)  (k < q),  M_out[f][2q] = M(all);   E0_out[f] = E[f].
 * Then V = M(all) - E0^2, first-order S_k = (M({k}) - E0^2) / V, total T_k = 1 - (M(all\k) - E0^2) / V.
 * ggp_main_effects_f64: out[f][k][g] = E[f | x_k = grid[g]] for a device grid[ngrid].
 * FP64 libdevice erf / exp; sums in a fixed order (bit-identical between identical calls).  Both entry points take
 * workspace_bytes >= ggp_gp_sens_workspace_bytes(m, q, S, pu, mode) (-1 for arguments the calls refuse).  GGP_ERR_ARG: a
 * null pointer, m, S, pu or ngrid < 1, q outside [1, 32], mode not 0 or 1, S pu or S m >= 2^31. */
long long ggp_gp_sens_workspace_bytes(int m, int q, int S, int pu, int mode);
int ggp_gp_sens_f64(const double* Z, int m, int q, const double* beta, const double* a, int S, int pu, int mode,
                    double* M_out, double* E0_out, void* workspace, long long workspace_bytes, void* stream);
int ggp_main_effects_f64(const double* Z, int m, int q, const double* beta, const double* a, int S, int pu, int mode,
                         const double* grid, int ngrid, double* out, void* workspace, long long workspace_bytes,
                         void* stream);

/* ---- Closed-form gradient outer products (csrc/ggp_grad_sens.cu; DESIGN.md section 2 item 12) ----------------------
 * C = E[grad g grad g^T] over independent inputs uniform on [0,1]^q, for g a weighted combination of the functions
 * mu_b(x) = sum_i a[b][i] prod_k exp(-beta[b][k] (x_k - Z[i][k])^2) of blocks b = s * pu + j (the layout of
 * ggp_gp_sens_f64): C = sum over pairs of terms (n, n') of a_n a_n' Omega_{j(n) j(n')} int grad phi_n grad phi_n'^T.
 *   mode 0: one function per block (F = S pu, Omega = 1);   mode 1: one per PC j over every sample's terms (F = pu,
 *   Omega = 1; scale a by 1/S for the posterior mean);   mode 2: one per sample s over every PC's terms (F = S,
 *   Omega = omega[pu][pu], symmetric);   mode 3: one function over every (s, j) (F = 1, omega; a scaled by 1/S).
 * C_out[f][k][l] (F x q x q, exactly symmetric): the active-subspace matrix; its diagonal is the derivative-based
 * sensitivity E[(d_k g)^2].  An input whose beta is 0 in every term gets row and column k exactly 0.  FP64 libdevice
 * erf / exp, the off-diagonal pair sums on DMMA m8n8k4; every sum in a fixed order (bit-identical between identical
 * calls).  workspace_bytes >= ggp_grad_sens_workspace_bytes(m, q, S, pu, mode) (-1 for arguments the call refuses), else
 * GGP_ERR_WORKSPACE.  GGP_ERR_ARG: a null pointer (omega in modes 2 and 3), m, S or pu < 1, q outside [1, 32], mode
 * outside 0-3, S pu or a function's term count (m, S m, pu m or S pu m) >= 2^31. */
long long ggp_grad_sens_workspace_bytes(int m, int q, int S, int pu, int mode);
int ggp_grad_sens_f64(const double* Z, int m, int q, const double* beta, const double* a, int S, int pu, int mode,
                      const double* omega, double* C_out, void* workspace, long long workspace_bytes, void* stream);

/* ---- Emulator-based calibration (csrc/ggp_calib.cu; DESIGN.md section 2 item 9) ------------------------------------
 * Log-likelihood of observed outputs at n input points, from the predictive moments of ggp_predict_f64 at the points'
 * designs: mean, var (S pu, n), block s * pu + j (posterior sample s, PC j), var clamped at 0.  Per-sample observation
 * terms, precomputed by the caller: G (S, pu, pu) symmetric = K_O D_s^-1 K_O^T, b (S, pu) = K_O D_s^-1 r and
 * c0 (S) = r^T D_s^-1 r + sum log D_s,ii + n_o log 2 pi.  With A = I + V^1/2 G V^1/2, V = diag(var), h = b - G mu:
 *   l_s = -1/2 (c0 - 2 mu^T b + mu^T G mu - h^T V^1/2 A^-1 V^1/2 h + log det A),
 *   ll_out[p] = log((1/S) sum_s exp l_s)   (running maximum, s ascending),   ll_s_out[s][p] = l_s (nullable).
 * Deterministic (fixed summation orders, no atomics).  GGP_ERR_ARG: a null pointer, S or n < 1, pu outside [1, 32],
 * S pu >= 2^31. */
int ggp_calib_loglik_f64(const double* mean, const double* var, int S, int pu, int n, const double* G, const double* b,
                         const double* c0, double* ll_out, double* ll_s_out, void* stream);
/* One Metropolis step of C chains on the uniform box [lo, hi] (q inputs, transformed units).  The candidate of chain c is
 * the last q columns of Xp[c] (C, d), and mean / var are the output of ggp_predict_f64 on Xp issued before this call.
 * valid = every candidate coordinate in [lo, hi] (inclusive); accept = valid && logu[c] < l' - ll[c] (false for a NaN
 * l').  theta (C, q) and ll (C) are updated; rec_theta (C, q), rec_ll (C), rec_acc (C) receive the step's state, l and
 * accepted flag.  If z_next (C, q) is not null, the next candidate theta + L_prop z_next[c] (L_prop (q, q) lower
 * triangular, sums over k ascending) is written to the last q columns of Xp[c]; an input whose row and column of L_prop
 * are zero keeps its value.  GGP_ERR_ARG: a null pointer (z_next may be null), S or C < 1, pu or q outside [1, 32],
 * d < q, S pu >= 2^31. */
int ggp_calib_step_f64(const double* mean, const double* var, int S, int pu, int C, const double* G, const double* b,
                       const double* c0, double* Xp, int d, int q, const double* lo, const double* hi,
                       const double* L_prop, const double* z_next, const double* logu, double* theta, double* ll,
                       double* rec_theta, double* rec_ll, unsigned char* rec_acc, void* stream);

/* ---- Sequential design (csrc/ggp_design.cu; DESIGN.md section 2 item 10) --------------------------------------------
 * Greedy ALC over B (sample, PC) blocks.  XR (n_ref, d) reference and XC (n_cand, d) candidate designs; beta (B, d),
 * lamz, dadd (the S22 nugget), s11 (B); V_R (B, n_ref, Mp) and V_C (B, n_cand, Mp) as ggp_predict_f64 writes V
 * (Mp = ggp_padded_m(m), zero padding); A_R (B, n_ref, Kp), A_C (B, n_cand, Kp): one column per chosen run, columns >= t
 * zero; Kp a multiple of 8.  With k_b(x, x') = exp(-sum_k beta_bk (x_k - x'_k)^2) / lamz_b,
 *   Sigma(r, c) = k_b(r, c) - V_r . V_c - A_r . A_c,   den(c) = 1/lamz_b + dadd_b - |V_c|^2 - |A_c|^2,
 *   score_out[c] = start + sum_b wgt[b] sum_r Sigma(r, c)^2 / den(c),
 *   imse_out[0]  = start + sum_b wgt[b] sum_r max(s11_b - |V_r|^2 - |A_r|^2, 0),
 * blocks summed in ascending order; start is 0, or the output's value when accumulate != 0 (so a split of the blocks
 * over several calls gives the same bits).  score_out may be null (imse only).  The product runs on the FP64 tensor
 * cores, the n_ref x n_cand matrix is never stored.  workspace: ggp_design_workspace_bytes(n_cand, B).
 * ggp_design_condition_f64 writes column t of A_R and A_C after choosing candidate `index`:
 *   A_x[t] = (k_b(x, c*) - V_x . V_c* - A_x[0:t] . A_c*[0:t]) / sqrt(den(c*))   for every reference and candidate x.
 * Passing the same XR / XC, V_R / V_C and A_R / A_C pointers (reference set = candidate set) conditions each point once.
 * Deterministic.  GGP_ERR_ARG: a null pointer, a size <= 0, Kp not a multiple of 8, m > 8192, t outside [0, Kp] (score)
 * or [0, Kp) (condition), index outside [0, n_cand), a short workspace. */
long long ggp_design_workspace_bytes(int n_cand, int B);
int ggp_design_score_f64(const double* XR, int n_ref, const double* XC, int n_cand, int d, const double* beta,
                         const double* lamz, const double* dadd, const double* s11, const double* wgt, const double* V_R,
                         const double* V_C, int m, const double* A_R, const double* A_C, int Kp, int t, int B,
                         int accumulate, double* score_out, double* imse_out, void* workspace, long long workspace_bytes,
                         void* stream);
int ggp_design_condition_f64(const double* XR, int n_ref, const double* XC, int n_cand, int d, const double* beta,
                             const double* lamz, const double* dadd, const double* V_R, const double* V_C, int m,
                             double* A_R, double* A_C, int Kp, int t, int B, int index, void* stream);

/* ---- History matching (csrc/ggp_hm.cu; DESIGN.md section 2 item 11) -------------------------------------------------
 * Implausibility of n input points against n_o observed outputs.  mean, var (S pu, n): block s * pu + j as
 * ggp_predict_f64 writes them, var clamped at 0.  Over the samples, m_j = (1/S) sum_s mean_sj and
 * M_jk = (1/S) sum_s [delta_jk var_sj + (mean_sj - m_j)(mean_sk - m_k)].  K_O (pu, n_o), r and c (n_o) in standardized
 * units, c_i = rho + tau_i^2 + delta_i^2 (truncation residual, observation and discrepancy variances).  Per output
 *   e_i = r_i - sum_j K_ji m_j,   V_i = sum_jk K_ji M_jk K_ki + c_i,   I_i = |e_i| / sqrt(V_i)
 * (V_i = 0: +inf for e_i != 0, 0 for e_i = 0; a NaN counts as +inf).  impl_out (n, order) receives each point's `order`
 * largest I_i in descending order, nover_out (n) the number of outputs with I_i > cutoff.  The two products run on the
 * FP64 tensor cores; the n x n_o matrices are never stored.  Deterministic (the outputs' split over CTAs does not change
 * a result).  workspace: ggp_hm_workspace_bytes(n, n_o, pu, S) (-1 for arguments the call refuses).  GGP_ERR_ARG: a null
 * pointer, S, n or n_o < 1, pu outside [1, 32], order outside [1, min(8, n_o)], a non-finite or non-positive cutoff,
 * S pu >= 2^31, a short workspace. */
long long ggp_hm_workspace_bytes(int n, int n_o, int pu, int S);
int ggp_hm_impl_f64(const double* mean, const double* var, int S, int pu, int n, const double* K_O, const double* r,
                    const double* c, int n_o, int order, double cutoff, double* impl_out, int* nover_out,
                    void* workspace, long long workspace_bytes, void* stream);

/* ---- MCMC convergence diagnostics (csrc/ggp_chain_diag.cu; DESIGN.md section 2 "Chain diagnostics") ----------------
 * Rank-normalized split R-hat, bulk ESS and tail ESS of Vehtari et al. (2021), as ArviZ computes rhat(method="rank"),
 * ess(method="bulk") and ess(method="tail"), with the autocovariance as a direct sum.  Draw i of chain c of element e is
 * x[i*s_draw + c*s_chain + e*s_elem] (strides in doubles), which covers the sampler's (n_steps, n_chains, P) draws, its
 * (n_steps, n_chains) logPost and one-chain-per-model layouts.  Per element: rhat_out[e], ess_bulk_out[e], ess_tail_out[e]
 * (device, FP64; all three NaN if a draw is NaN or +-inf; R-hat NaN and ESS = 2 n_chains floor(n_draws/2) for a constant
 * element).  Deterministic; an element's results do not depend on the other elements of the call.
 * GGP_ERR_ARG: a null pointer, n_draws < 4, n_chains < 1, n_elem < 1, n_chains * n_draws >= 2^31, or workspace_bytes below
 * ggp_chain_diag_workspace_bytes(n_draws, n_chains, n_elem) (which is -1 for arguments the call refuses). */
long long ggp_chain_diag_workspace_bytes(int n_draws, int n_chains, int n_elem);
int ggp_chain_diag_f64(const double* x, int n_draws, int n_chains, int n_elem, long long s_draw, long long s_chain,
                       long long s_elem, double* rhat_out, double* ess_bulk_out, double* ess_tail_out, void* workspace,
                       long long workspace_bytes, void* stream);

/* ---- (4) randomized SVD passes -----------------------------------------------------------------
 * src/svd.py:52  Y = X @ omega           -> ggp_rsvd_sketch_tc_f32 (OmegaT = omega^T, [r][n])
 * src/svd.py:56  Y = X @ X.T @ Y         -> ggp_rsvd_xty_tc_f32 then ggp_rsvd_sketch_tc_f32 (X (X^T Y))
 * src/svd.py:60  B = Q.T @ X             -> ggp_rsvd_xty_tc_f32 (Bt_out[r][n] = Y^T X)
 * X[m][n] float32 row-major, any m.  The products run on the tcgen05 tensor cores (3xTF32 split, FP32-level accuracy;
 * csrc/ggp_rsvd_tc.cu), bound by the HBM read of X.  workspace: ggp_rsvd_tc_workspace_bytes(m). */
long long ggp_rsvd_tc_workspace_bytes(int m);
int ggp_rsvd_sketch_tc_f32(const float* X, int m, long long n, const float* OmegaT, int r, float* Y_out,
                           void* workspace, long long workspace_bytes, void* stream);
int ggp_rsvd_xty_tc_f32(const float* X, int m, long long n, const float* Y, int r, float* Bt_out, void* stream);

/* ---- (5) ensemble ingest and initialisation passes (SURVEY 8f rank 2) ------------------------------
 * The streaming work of init_model / fit_models around the PCA, on the (m x n) float32 ensemble:
 *   src/model.py:60-64    mu = mean(y, 0); sd = std(y, ddof=1, 0); sd[sd < thr] = thr   -> ggp_colstats_f32
 *   src/model.py:71-72    y_std = (y - mu) / sd          (SepiaData.standardize_y)       -> ggp_standardize_f32
 *   src/model.py:219-223  w = (pinv(K)^T y_std^T)^T; var(y_std - w K); SepiaModel.__init__ (w, LamSim, lamWOs prior)
 *                                                                                         -> ggp_project_f32
 * transposed != 0: the input is stored [n][m] (the ensemble file layout of src/aggregate_outputs.py:61-68, which
 * the reference transposes on the host, src/model.py:133); outputs are always [m][n].  ld: row stride of the input in
 * elements (0 = dense), so that the first m simulations of a larger ensemble can be used in place (y_sim[:m]).
 * mean_len / sd_len: 1 (SEPIA's default scalar standardisation) or n.  sd < sd_floor is replaced by sd_floor.
 * ggp_project_f32: P_out[m][pu+2] (double) = { X Kt^T (pu columns), row sums of X, row sums of X^2 }, accumulated in
 * FP64 in a fixed order (deterministic).  With X = y_std it yields w = (y_std K^T)(K K^T)^-1, ||y_std - w K||^2 and
 * sum(y_std - w K) without a second pass; with X = K it yields K K^T.  pu <= 32. */
int ggp_colstats_f32(const float* Y, long long ld, int m, long long n, int transposed, int ddof, float sd_floor,
                     float* mean_out, float* sd_out, void* stream);
int ggp_standardize_f32(const float* Y, long long ld, int m, long long n, int transposed, const float* mean,
                        long long mean_len, const float* sd, long long sd_len, float* Ystd_out, void* stream);
long long ggp_project_workspace_bytes(int m, int pu);
int ggp_project_f32(const float* X, int m, long long n, const float* Kt, int pu, double* P_out, void* workspace,
                    long long workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GLADSGP_B200_H */
