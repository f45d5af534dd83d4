/* rfsurfhmc.h — C ABI of librfsurf_b200.so (hand-written sm_100a CUDA behind plain C).
 *
 * Drop-in boundary for the hot path of nqdu/RfSurfHmc.  Every entry point names the reference
 * interface it replaces (paths relative to the reference repository root):
 *
 *   libsurf.forward / libsurf.adjoint_kernel      src/SWD/main.cpp:14-82  (pybind11 module :84-94)
 *     -> surfdisp96_, sregn96_, sregnpu_, slegn96_, slegnpu_   src/SWD/surfdisp.hpp:17-93
 *   librf.forward / librf.kernel / librf.kernel_all             src/RF/main.cpp:17-189 (:191-213)
 *     -> cal_rf_freq_, cal_rf_par_freq_, cal_rf_par_freq_all_   src/RF/rf_cal.hpp:10-51
 *   Joint_RF_SWD.misfit_and_grad (+ SurfWD / ReceiverFunc)      model/model_rf_swd_vs_thk.py:66-86,
 *                                                               model/model_surf.py:155-228,
 *                                                               model/model_rf.py:137-197
 *   HamitonianMC.sample / HMCDualAveraging.sample               pyhmc/hmc.py:228-276,
 *                                                               pyhmc/hmcda.py:280-369
 *
 * Conventions
 *   - all entry points return 0 on success, a negative RFS_E_* code otherwise;
 *     rfs_last_error(ctx) returns a human-readable message for the last failure on that context.
 *   - no torch / C++ types cross the boundary: plain pointers, sizes and an opaque context.
 *   - *_dev functions take DEVICE pointers and a cudaStream_t (passed as void*); they never
 *     allocate in steady state (workspace is grown on the first call for a given batch size) and
 *     are stream-ordered.  *_host functions take HOST pointers and perform the H2D/D2H copies.
 *   - arrays are row-major, float64 unless stated; batch index first.
 *   - wave types: 0 "Rc", 1 "Rg", 2 "Lc", 3 "Lg".  rf_type: 1 P, 2 S.  method: 0 time, 1 freq.
 *   - there is NO CPU fallback: if no CUDA device is usable rfs_create fails.
 */
#ifndef RFSURFHMC_H
#define RFSURFHMC_H

#ifdef __cplusplus
extern "C" {
#endif

#define RFS_OK 0
#define RFS_E_CUDA -1      /* CUDA runtime error (message has the detail) */
#define RFS_E_ARG -2       /* invalid argument (bad wave type / rf type / sizes) */
#define RFS_E_UNSUPPORTED -3 /* reference feature not built (currently unused) */
#define RFS_E_CONFIG -4    /* context not configured for this call */

typedef struct rfs_ctx rfs_ctx;

/* ---- lifetime ------------------------------------------------------------------------------ */
int rfs_create(rfs_ctx **out, int device);
void rfs_destroy(rfs_ctx *ctx);
const char *rfs_last_error(rfs_ctx *ctx);
/* version string of the library, e.g. "rfsurf_b200 0.1 sm_100a" */
const char *rfs_version(void);
/* number of kernels launched by this context since creation (bench.py's gpu_launches) */
long long rfs_launch_count(rfs_ctx *ctx);

/* ---- configuration (replaces SurfWD.__init__, ReceiverFunc.__init__, Joint_RF_SWD.__init__ +
 *      set_obsdata: model/model_surf.py:5-29, model/model_rf.py:5-18,
 *      model/model_rf_swd_vs_thk.py:6-25) -------------------------------------------------------- */
/* period lists may be empty (n*=0).  mode: 0 fundamental.  sphere: 1 = earth-flattening transformation.
 * stale_group_kernel=1 reproduces sregnpu/slegnpu's stale first term (sregn96.f90:1841-1844). */
int rfs_config_swd(rfs_ctx *ctx, int nlayer, int ntRc, const double *tRc, int ntRg,
                   const double *tRg, int ntLc, const double *tLc, int ntLg, const double *tLg,
                   int mode, int sphere, int stale_group_kernel);
int rfs_config_rf(rfs_ctx *ctx, int nlayer, double ray_p, int nt, double dt, double gauss,
                  double time_shift, double water, int rf_type, int method);
/* Extensions of the two calls above for objectives with several modes / several ray parameters
 * (BASELINE configs 2 and 3; the reference's classes hold one `mode` and one `ray_p`, so such data
 * sets need one model object per mode / ray parameter there).  modes[] ascending; the SWD data
 * vector becomes [mode][Rc,Rg,Lc,Lg], the RF data vector [ray parameter][nt].  All modes are solved
 * in ONE chained root-search pass (surfdisp96.f:232-368 solves modes 1..mode+1 anyway). */
int rfs_config_swd_modes(rfs_ctx *ctx, int nlayer, int ntRc, const double *tRc, int ntRg,
                         const double *tRg, int ntLc, const double *tLc, int ntLg, const double *tLg,
                         int nmodes, const int *modes, int sphere, int stale_group_kernel);
int rfs_config_rf_rays(rfs_ctx *ctx, int nlayer, int nray, const double *ray_p, int nt, double dt,
                       double gauss, double time_shift, double water, int rf_type, int method);
/* Receiver functions at several Gaussian widths in one objective (RFs are usually inverted at two or
 * three widths together, e.g. gauss = 1.0, 2.5, 5.0: low widths give stable traces, high widths resolve
 * thin layers; the reference's ReceiverFunc holds one `gauss`).  gauss [ngauss] (host pointer), 1 <= ngauss
 * <= 16, every width finite and > 0.  The RF data vector becomes [ray parameter][gauss][nt], so
 * n_rf = nray * ngauss * nt (also in the joint weight); misfit and gradient are the sums over all (ray,
 * width) traces.  nt, dt, time shift, water level, RF type and method are shared by every width.  Each
 * trace equals the trace of a one-width configuration; the frequency method deconvolves every width of a
 * ray on the same spectra and contracts the summed adjoint weights with the derivative spectra once.
 * rfs_config_rf_rays is this call with ngauss = 1 (and, as before, no check of its one width).
 * Returns RFS_E_ARG for a bad width list, and for everything rfs_config_rf_rays rejects.  Lifetime: see
 * "Per-set tables" below (an rfs_config_rf* call). */
int rfs_config_rf_gauss(rfs_ctx *ctx, int nlayer, int nray, const double *ray_p, int ngauss,
                        const double *gauss, int nt, double dt, double time_shift, double water,
                        int rf_type, int method);
/* dobs (host pointer): [nt_rf + n_swd] joint, or the matching sub-vector for which=1/2 */
int rfs_config_obs(rfs_ctx *ctx, double sigma1, double sigma2, const double *dobs, int ndobs);
/* S observation sets ("stations", no reference counterpart: the reference inverts one station per run):
 * dobs [S][ndobs], sigma1/sigma2 [S] (host pointers).  Every set shares the forward configuration above
 * (layer count, periods, modes, ray parameters, RF sampling); each has its own data vector and its own
 * joint weight (sigma1[s]/sigma2[s])^2 n_rf/n_swd.  rfs_config_obs is this call with S = 1.
 * On a context holding S > 1 sets, every call without a set array (rfs_misfit_grad_dev/_host,
 * rfs_hmc_run) returns RFS_E_CONFIG. */
int rfs_config_obs_sets(rfs_ctx *ctx, int S, const double *sigma1, const double *sigma2,
                        const double *dobs, int ndobs);
/* Per-set tables.  The four calls below give each of the S observation sets held its own ray
 * parameters, SWD period lists, receiver-function samples or Gaussian widths.  Each table belongs to the
 * sets held and to the configuration it refines, and its lifetime follows one rule:
 *   - rfs_config_obs_sets and rfs_config_obs drop all four tables;
 *   - a successful rfs_config_rf, rfs_config_rf_rays or rfs_config_rf_gauss drops the ray table, the
 *     RF-sample table and the width table, and keeps the period table;
 *   - a successful rfs_config_swd or rfs_config_swd_modes drops the period table, and keeps the other three;
 *   - each of the four calls below drops its own table first, so a call of it that fails leaves no such
 *     table, and it keeps the other three;
 *   - a failed rfs_config_swd* or rfs_config_rf* changes nothing: the configuration and every table stay.
 * Without a table the context evaluates every set on the shared configuration.  Each call returns
 * RFS_E_CONFIG without the configuration its table refines or when S differs from the number of
 * observation sets held.  A row whose device set index lies outside [0, S) reads no table entry; it is
 * failed as described below.  Like every rfs_config_* call, these copy synchronously into the context's
 * device buffers: an evaluation still running on a caller's stream must have finished before the
 * context is reconfigured. */
/* Per-set ray parameters of the RF objective (each station's stack has its own mean slowness; the
 * reference's ReceiverFunc.ray_p is per station): ray_p [S][nray] (host pointer, copied to the device
 * here, never during an evaluation).  Row b's pass ir then uses ray_p[set[b]][ir] in place of the
 * shared list of rfs_config_rf*, for every Gaussian width of that ray; everything else (nt, dt, gauss, time shift, water
 * level, RF type, method, layers, periods, modes) stays shared.  The evaluations and the HMC use the
 * table whenever it is present; their signatures do not change.  The librf drop-ins keep their own
 * ray_p argument.  A row with an out-of-range set index computes with the shared value.
 * Returns RFS_E_ARG when nray differs from the configured ray count, ray_p is NULL or a value is not
 * finite and > 0.  Lifetime: see "Per-set tables" above. */
int rfs_config_obs_rays(rfs_ctx *ctx, int S, int nray, const double *ray_p);
/* Per-set SWD period lists (dispersion curves are rarely measured on the same periods at every
 * station): the four lists of rfs_config_swd[_modes] form a common period grid, and use [S][nper]
 * (host pointer, values 0 or 1, nper = ntRc + ntRg + ntLc + ntLg, one mode block of the data vector in
 * its order) marks the grid periods each set observes.  The same mask applies to every mode block.
 * Row b of set s then gives exactly U, grad and flag of a one-set context configured with
 * rfs_config_swd[_modes] on set s's subset lists (everything else unchanged): every root search runs
 * the set's own compact period list.  dsyn keeps the grid layout: the subset context's values at the
 * observed positions, NaN at the others in every mode block; a failed row returns dobs as before.  The
 * joint weight of set s is (sigma1[s]/sigma2[s])^2 n_rf/(nmodes * observed periods of s).  RF-only
 * evaluations (which = 1) ignore the table; the libsurf drop-ins are not affected.  A row with an
 * out-of-range set index runs the grid lists.
 * Returns RFS_E_ARG when nper is wrong, use is NULL, a value is not 0 or 1, or a set observes no period.
 * Lifetime: see "Per-set tables" above. */
int rfs_config_obs_periods(rfs_ctx *ctx, int S, int nper, const unsigned char *use);
/* Per-set receiver-function samples (missing ray-parameter bins, station-dependent fitting windows):
 * use [S][nrf] (host pointer, values 0 or 1, nrf = nray * ngauss * nt, the RF block of the data vector in
 * its order [ray][gauss][sample]) marks the samples each set fits.  For a row of set s the RF misfit is
 * 0.5 sum over observed samples (d - dobs)^2 and the adjoint source is zero at the others: the residual
 * there is selected as 0, never formed, so dobs may hold anything at unobserved samples (missing data
 * may be stored as NaN).  dsyn keeps the full synthetic trace at every sample; a failed row returns
 * dobs as before.  A set whose mask keeps whole traces gives exactly U, grad and flag of a one-set
 * context configured with rfs_config_rf_rays on its observed rays.  The joint weight of set s is
 * (sigma1[s]/sigma2[s])^2 n1_s/nsw_s with n1_s = sum of use[s].  SWD-only evaluations (which = 2) ignore
 * the table; the librf drop-ins are not affected.
 * Returns RFS_E_ARG when nrf is wrong, use is NULL, a value is not 0 or 1, or a set observes no sample
 * (its joint weight would be zero).  Lifetime: see "Per-set tables" above. */
int rfs_config_obs_rf_samples(rfs_ctx *ctx, int S, int nrf, const unsigned char *use);
/* Per-set Gaussian widths (an observed receiver function can only be fitted by a synthetic filtered with
 * the Gaussian its data were processed with, and stations from different networks or catalogues come at
 * different widths): gauss [S][ngauss] (host pointer, copied to the device here), ngauss the width count
 * of rfs_config_rf*.  Trace (ray ir, width g) of a row of set s is deconvolved with gauss[s][g] in place
 * of the shared width g, at every ray; the data vector keeps its layout [ray][gauss][nt].  A set that
 * fits fewer widths drops the others with its RF-sample mask.  Row b of set s gives exactly (bit for bit)
 * U, grad, dsyn and flag of a one-set context configured with rfs_config_rf_gauss on set s's widths, in
 * that order, with everything else unchanged (ray table and RF-sample table included).  The joint weight
 * does not change (n_rf counts samples, not widths).  SWD-only evaluations (which = 2) ignore the table;
 * the librf drop-ins keep their scalar gauss.  A row with an out-of-range set index reads no width and
 * is failed as described below.
 * Returns RFS_E_ARG when ngauss differs from the configured width count, gauss is NULL or a value is not
 * finite and > 0.  Lifetime: see "Per-set tables" above. */
int rfs_config_obs_gauss(rfs_ctx *ctx, int S, int ngauss, const double *gauss);

/* Parameterisation of the model vector (no reference counterpart: model_rf_swd_vs_thk.py fixes
 * [vs, thk]).  Receiver functions constrain Vp through the Ps delays, which trade thickness against
 * Vp/Vs (the H-kappa trade-off); with Vp tied to vs by Brocher's curve that trade-off cannot be sampled.
 *   RFS_PARAM_VS_THK      (0, the default at rfs_create): x = [vs(n), thk(n)], vp and rho from Brocher's
 *                         polynomials of vs.
 *   RFS_PARAM_VS_THK_VPVS (1): x = [vs(n), thk(n), k(n)], k the Vp/Vs ratio of each layer (half-space
 *                         included): vp = k vs, rho = Brocher's density polynomial of that vp.  grad is
 *                         [dU/dvs | dU/dthk | dU/dk] with, per layer, g_vs = K_b + k (K_a + drho/dvp K_r)
 *                         and g_k = vs (K_a + drho/dvp K_r).
 * With param 1 every x, grad, samples and initmodel row below has P n = 3n columns instead of 2n, and the
 * HMC bounds are [nb][3n][2]; the failure convention writes grad zeros of width 3n.  This covers
 * rfs_misfit_grad_{dev,host}, rfs_misfit_grad_sets_{dev,host} (every which), rfs_profile_eval,
 * rfs_hmc_run and rfs_hmc_run_sets; the libsurf/librf drop-ins are not affected.  The setting belongs to
 * the context and is shared by every observation set: no other rfs_config_* call changes it and it
 * changes no per-set table.  It copies nothing to the device, but like every rfs_config_* call it must
 * not be made while an evaluation on the context is in flight.  Any other value returns RFS_E_ARG. */
#define RFS_PARAM_VS_THK 0
#define RFS_PARAM_VS_THK_VPVS 1
int rfs_config_param(rfs_ctx *ctx, int param);

/* ---- the hot path: batched misfit + gradient ------------------------------------------------
 * x [B][2n] = [vs(n), thk(n)];  U [B];  grad [B][2n];  dsyn [B][ndata];  flag [B] (1 ok / 0 fail)
 * (P n = 3n columns for x and grad under RFS_PARAM_VS_THK_VPVS, see rfs_config_param)
 * which: 0 Joint_RF_SWD.misfit_and_grad, 1 ReceiverFunc.misfit_and_grad, 2 SurfWD.misfit_and_grad */
int rfs_misfit_grad_dev(rfs_ctx *ctx, long long B, const double *x, int which, double *U,
                        double *grad, double *dsyn, unsigned char *flag, void *stream);
int rfs_misfit_grad_host(rfs_ctx *ctx, long long B, const double *x, int which, double *U,
                         double *grad, double *dsyn, unsigned char *flag);
/* The same over several observation sets: row b is compared with set[b]'s data vector (and weighted
 * with its sigma1/sigma2).  set [B] int32: a DEVICE pointer for _dev, a HOST pointer for _host; NULL
 * only when the context holds one set (then these are the two calls above).  The failure convention
 * (U 0, grad 0, dsyn = dobs, flag 0) returns the row's own set's dobs.
 * _host rejects an index outside [0, S) with RFS_E_ARG.  _dev cannot check without synchronising: a
 * row whose index is outside [0, S) reads no observation and gets flag 0, U 0, grad 0 and NaN dsyn;
 * every other row is unaffected. */
int rfs_misfit_grad_sets_dev(rfs_ctx *ctx, long long B, const double *x, const int *set, int which,
                             double *U, double *grad, double *dsyn, unsigned char *flag, void *stream);
int rfs_misfit_grad_sets_host(rfs_ctx *ctx, long long B, const double *x, const int *set, int which,
                              double *U, double *grad, double *dsyn, unsigned char *flag);

/* ---- libsurf drop-ins, batched over B models (host pointers) --------------------------------
 * thk,vp,vs,rho [B][n] (cast to float32 inside, as src/SWD/main.cpp:9);  period [nT]
 * c [B][nT];  dcda,dcdb,dcdr,dcdh [B][nT][n];  ok [B] */
int rfs_surf_forward(rfs_ctx *ctx, long long B, int n, const double *thk, const double *vp,
                     const double *vs, const double *rho, int nT, const double *period,
                     int wavetype, int mode, int sphere, double *c, unsigned char *ok);
int rfs_surf_adjoint_kernel(rfs_ctx *ctx, long long B, int n, const double *thk, const double *vp,
                            const double *vs, const double *rho, int nT, const double *period,
                            int wavetype, int mode, int sphere, int stale_group_kernel, double *c,
                            double *dcda, double *dcdb, double *dcdr, double *dcdh,
                            unsigned char *ok);
/* all modes 0..mode at once (BASELINE config 2): c [B][mode+1][nT], kernels [B][mode+1][nT][n] */
int rfs_surf_adjoint_kernel_modes(rfs_ctx *ctx, long long B, int n, const double *thk,
                                  const double *vp, const double *vs, const double *rho, int nT,
                                  const double *period, int wavetype, int mode,
                                  int stale_group_kernel, double *c, double *dcda, double *dcdb,
                                  double *dcdr, double *dcdh, unsigned char *ok);

/* ---- librf drop-ins, batched over B models (host pointers) ----------------------------------
 * thk,rho,vp,vs,qa,qb [B][n] (RF argument order, src/RF/main.cpp:17-19);  rf [B][nt]
 * par_type: 1 rho, 2 vp, 3 vs, 4 thickness;  drf [B][n][nt] (kernel) or [B][4][n][nt] (kernel_all) */
int rfs_rf_forward(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                   const double *vp, const double *vs, const double *qa, const double *qb,
                   double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                   double water, int rf_type, double *rf);
int rfs_rf_kernel(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                  const double *vp, const double *vs, const double *qa, const double *qb,
                  double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                  double water, int rf_type, int par_type, double *rf, double *drf);
int rfs_rf_kernel_all(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                      const double *vp, const double *vs, const double *qa, const double *qb,
                      double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                      double water, int rf_type, double *rf, double *drf);

/* ---- device-resident HMC (replaces the Python loops of pyhmc/hmc.py:140-276 and
 *      pyhmc/hmcda.py:170-369; chain i uses NumPy-legacy MT19937 seeded with seed+chain_id[i]) ---
 * which  : objective sampled, as in rfs_misfit_grad_dev (0 Joint_RF_SWD, 1 ReceiverFunc, 2 SurfWD:
 *          the reference samplers take any object with misfit_and_grad, pyhmc/hmc.py:113-119).
 * sampler: 0 HamitonianMC (fixed dt, L ~ randint[Lmin,Lmax]), 1 HMCDualAveraging (L0, target;
 *          Lmax > 0 caps L = max(1,int(lambda/dt)) — an extension, 0 = unlimited as the reference).
 * bounds [2n][2] (low, high), shared by all chains (host pointer).
 * Outputs (host pointers, may be NULL): samples [C][nsamples][2n], misfit [C][nsamples],
 * syn [C][nsamples][ndata], initmodel [C][2n], n_iter [C] (trajectories run), n_acc [C],
 * dt_final [C], accept_seq [C][max_iter_log] (1/0 per trajectory, -1 padding; for RNG parity tests).
 * max_iters bounds the number of trajectories per chain (0 = unlimited). */
int rfs_hmc_run(rfs_ctx *ctx, int sampler, int which, long long C, const long long *chain_id,
                const double *bounds, double dt, int Lmin, int Lmax, int L0, double target_ratio,
                long long seed, int nsamples, int ndraws, long long max_iters, double *samples,
                double *misfit, double *syn, double *initmodel, long long *n_iter,
                long long *n_acc, double *dt_final, signed char *accept_seq,
                long long max_iter_log);
/* The same over several observation sets: chain c samples set chain_set[c]'s objective (host pointer
 * [C]; NULL only when the context holds one set) inside its box, bounds [nb][2n][2] with nb = 1 (one
 * box for all chains) or S (one box per set).  An index outside [0, S) returns RFS_E_ARG.  Chain ids
 * may repeat across sets: chain c is seeded seed + chain_id[c] and the id is used for nothing else, so
 * set s's chains 0..K-1 give exactly what a one-set run of chains 0..K-1 on set s gives.
 * rfs_hmc_run is this call with chain_set = NULL and nb = 1. */
int rfs_hmc_run_sets(rfs_ctx *ctx, int sampler, int which, long long C, const long long *chain_id,
                     const int *chain_set, const double *bounds, int nb, double dt, int Lmin, int Lmax,
                     int L0, double target_ratio, long long seed, int nsamples, int ndraws,
                     long long max_iters, double *samples, double *misfit, double *syn, double *initmodel,
                     long long *n_iter, long long *n_acc, double *dt_final, signed char *accept_seq,
                     long long max_iter_log);
/* number of misfit_and_grad evaluations / of global steps (one batched evaluation each) performed by
 * the last rfs_hmc_run */
long long rfs_hmc_last_evals(rfs_ctx *ctx);
long long rfs_hmc_last_steps(rfs_ctx *ctx);
/* Options of rfs_hmc_run (no reference counterpart).  resident_slots > 0: at most that many chains are
 * resident on the device at a time; a finished chain hands its slot to the next queued chain on the
 * device, so the evaluated batch stays full (results do not depend on it).  max_seconds > 0: stop the
 * run after that wall-clock time; unfinished chains keep what they have (rfs_hmc_run returns 1). */
int rfs_set_hmc_options(rfs_ctx *ctx, long long resident_slots, double max_seconds);

/* ---- measurement helpers (no reference counterpart; used by bench.py) --------------------------
 * rfs_count_evals(ctx,1) zeroes and enables a device counter of secular-function evaluations
 * (the algorithmic work of the root-search kernel); rfs_read_evals synchronises and reads it.
 * rfs_measure_fp64_peak runs a DFMA micro-benchmark: the roofline denominator of the FP64 path. */
int rfs_count_evals(rfs_ctx *ctx, int enable);
/* Root-search mapping (no reference counterpart; results are bit-identical for every mapping):
 * T < 0 automatic by batch size (default), T = 0 one thread per (model, period sequence),
 * T in {2,4,8,16,32}: a team of T lanes per sequence, S speculative scan points per round
 * (csrc/swd_roots_team.cuh).  Environment override at rfs_create: RFS_ROOTS_TEAM="T,S". */
int rfs_set_roots_team(rfs_ctx *ctx, int T, int S);
int rfs_last_roots_team(rfs_ctx *ctx, int *T, int *S);
/* Length-sorted job order of the thread-mapped root search (no reference counterpart): large batches
 * are solved longest-job-first through a permutation built on the device (a bisection estimate of the
 * phase velocity at the longest period predicts the scan length of every (model, sequence) job).  The
 * order changes which lane solves which job and nothing else: results are bit-identical.
 * mode < 0 automatic (on for large, throughput-bound batches; default), 0 off, 1 on.
 * rfs_last_roots_sched: 1 if the last root search ran in sorted order.  Environment override at
 * rfs_create: RFS_ROOTS_SCHED. */
int rfs_set_roots_sched(rfs_ctx *ctx, int mode);
int rfs_last_roots_sched(rfs_ctx *ctx);
long long rfs_read_evals(rfs_ctx *ctx);
int rfs_read_eval_stats(rfs_ctx *ctx, long long *out3); /* total, slowest thread, threads > 2000 */
int rfs_measure_fp64_peak(rfs_ctx *ctx, double *tflops);
/* One rfs_misfit_grad_dev call with CUDA events around every kernel launch (the RF branch is
 * serialised behind the SWD branch for this call, so each kernel is timed alone).  ms[RFS_PROF_NK] =
 * milliseconds per kernel class, launches[RFS_PROF_NK] (may be NULL) = launch counts;
 * rfs_profile_kernel_name(i) names class i.  bench.py derives every roofline figure from this. */
#define RFS_PROF_NK 10
int rfs_profile_eval(rfs_ctx *ctx, long long B, const double *x, int which, double *U, double *grad,
                     double *dsyn, unsigned char *flag, void *stream, double *ms,
                     long long *launches);
const char *rfs_profile_kernel_name(int i);
/* self-test: the constant-bank exp / sincos / rsqrt of the root search against the CUDA math library
 * on n device-generated arguments; mismatches[6] = exp, sin/cos (large args), sin/cos (small), rsqrt */
int rfs_selftest_math(rfs_ctx *ctx, long long n, long long *mismatches);

#ifdef __cplusplus
}
#endif
#endif /* RFSURFHMC_H */
