// C ABI of librfsurf_b200.so — see include/rfsurfhmc.h for the contract and the reference
// interfaces each entry point replaces.  Host-side orchestration only: plan building, workspace,
// kernel launches.  No CPU fallback: every numerical result comes from the sm_100a kernels.
#include "../../include/rfsurfhmc.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <memory>
#include <string>
#include <vector>

#include "hmc_kernels.cuh"
#include "joint_kernels.cuh"
#include "rf_kernels.cuh"
#include "rf_time_kernels.cuh"
#include "swd_kernels.cuh"
#include "swd_roots_launch.h"

using namespace rfs;

namespace {

// device allocation owned by the context (grown by ensure); freed with its owner, on the owner's device
struct Buf {
  void *p = nullptr;
  size_t cap = 0;
  Buf() = default;
  Buf(const Buf &) = delete;
  Buf &operator=(const Buf &) = delete;
  ~Buf() {
    if (p) cudaFree(p);
  }
};

// settings of one receiver-function run: the fused objective's (rfs_config_rf*) or one drop-in call's
// (one Gaussian width).  t0: the time shift, negated for S receiver functions (src/RF/main.cpp:35);
// sigma: the damping of the frequency method, 0 for the time method.  The ray parameter is passed on
// its own (RayView): the fused objective has a list of them, and may have one list per observation set.
struct RfCfg {
  int n = 0, nt = 0, nft = 0, logn = 0, n2 = 0, rf_type = 1, method = 1;
  double dt = 0, water = 0.001, t0 = 0, sigma = 0;
  GaussList gauss{1, {0.0}};
};

// Per-set observation tables of the sets held (rfs_config_obs_rays / _periods / _rf_samples / _gauss).  Each one
// belongs to the sets and to one configuration; drop_tables is the only code that clears one.
struct ObsTables {
  // ray parameters [nsets][nray], used in place of the shared list
  bool has_rays = false;
  Buf d_rays;
  // period lists: the plan the table was built for (the grid's, or the grid's without the Rc/Rg sequence
  // sharing when a set observes other Rg than Rc periods), its period table (the grid lists, then each
  // set's compact lists) and the SwdSetView table [nsets][ld], whose column use_col starts the observed
  // flags; nobs: each set's observed periods per mode block
  bool has_periods = false;
  SwdPlan plan;
  Buf d_periods, d_tab;
  int ld = 0, use_col = 0;
  std::vector<int> nobs;
  // RF samples: the mask [nsets][nray * nt] (read through ObsSets::observed) and each set's sample count
  bool has_rf = false;
  Buf d_rf;
  std::vector<int> n1;
  // Gaussian widths [nsets][ngauss], used in place of the shared list (read through GaussView)
  bool has_gauss = false;
  Buf d_gauss;
};

}  // namespace

// "Front" buffers of one chunk of a batch: model blocks and everything the root search produces.  They
// are small (35 KB per model at n = 200), so a chunked batch keeps one set per chunk and runs the root
// searches of ALL chunks concurrently before the memory-hungry eigen / RF stages go chunk by chunk.
struct Front {
  Buf w_sph[4];  // spherical earth: rootR, rootL, eigR, eigL model blocks
  Buf w_rstat;
  Buf w_swd, w_rfm, w_chain, w_croot, w_cwork, w_ierr;
  Buf w_key, w_perm;  // length-sorted job order of the thread-mapped root search
  cudaEvent_t ev_prep = nullptr;   // model blocks of this chunk written, its root search about to be enqueued
  bool prep_pending = false;       // ev_prep still to be recorded (release_rf_branch)
  cudaEvent_t ev_ready = nullptr;  // root search of this chunk finished
  ~Front() {
    if (ev_ready) cudaEventDestroy(ev_ready);
    if (ev_prep) cudaEventDestroy(ev_prep);
  }
};

struct rfs_ctx {
  int device = 0;
  std::string err;
  long long launches = 0;
  cudaStream_t stream = nullptr;  // used by the *_host entry points
  cudaStream_t stream2 = nullptr; // RF branch of the joint evaluation runs concurrently with SWD
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_asm = nullptr;
  // ---- SWD configuration
  bool has_swd = false;
  int n_swd = 0, mode = 0, stale = 1, sphere = 0;
  std::vector<int> modes;  // modes of the fused SWD objective (reference: one mode)
  // the period grid (plan, its four lists and their lengths tRc, tRg, tLc, tLg): written only by a
  // successful rfs_config_swd*
  SwdPlan plan;
  std::vector<double> periods;
  Buf d_periods;
  int swd_nts[4] = {0, 0, 0, 0};
  // ---- RF configuration
  bool has_rf = false;
  RfCfg rf;                    // its Gaussian widths: rf.gauss (reference: one)
  std::vector<double> ray_ps;  // ray parameters of the fused RF objective (reference: one)
  // ---- parameterisation (rfs_config_param): npar blocks of n per model, [vs, thk] with Brocher vp and
  // rho (2) or [vs, thk, Vp/Vs] with vp = k vs and Brocher rho (3).  Shared by every set.
  int npar = 2;
  // ---- observations: nsets data vectors ("stations") of ndobs values each, and their per-set tables
  bool has_obs = false;
  int nsets = 0, ndobs = 0;
  std::vector<double> sigma1, sigma2;  // [nsets]
  Buf d_dobs;                          // [nsets][ndobs]
  ObsTables tables;
  // SWD weight of the joint objective per set, (sigma1/sigma2)^2 n1/nsw: computed on the host for the
  // data lengths (wt_n1, wt_nsw) of the last joint call and uploaded again when they change or when
  // drop_tables resets them
  std::vector<double> wt;
  Buf d_wt;
  int wt_n1 = -1, wt_nsw = -1;
  // ---- workspace (grown on demand, never shrunk)
  std::vector<std::unique_ptr<Front>> fronts;  // one per chunk; fronts[0] always exists (drop-ins use it)
  cudaStream_t stream_front[3] = {nullptr, nullptr, nullptr};  // root searches (high priority)
  Buf w_rfl;  // RfLayer table [B][n]
  Buf d_tw;   // FFT twiddle factors exp(-i pi j/(nft/2)), j < nft/2, of transform length tw_nft
  int tw_nft = 0;
  Buf w_ugr, w_kern, w_spec, w_dspec, w_urf, w_grf, w_rftr;
  Buf io_x, io_U, io_grad, io_dsyn, io_flag, io_set, io_a, io_b, io_c, io_d, io_e, io_f;
  // ---- HMC
  long long hmc_evals = 0, hmc_steps = 0;
  long long hmc_resident = 0;    // resident chain slots of rfs_hmc_run (0 = all chains at once)
  double hmc_max_seconds = 0.0;  // wall-clock budget of rfs_hmc_run (0 = none)
  Buf h_state, h_misc, h_out;
  size_t ws_budget = (size_t)24 << 30;  // workspace budget per chunk (bytes)
  Buf d_counter;                 // [0] secular-function evaluations (algorithmic-work counter)
  bool count_evals = false;
  // root-search mapping: team_T < 0 automatic (by batch size), 0 thread-mapped, else T lanes per
  // (model, sequence) with team_S speculative scan slots (swd_roots_team.cuh)
  int team_T = -1, team_S = 1;
  int last_team_T = 0, last_team_S = 1;  // what the last launch used (reported by bench.py)
  // length-sorted job order of the thread-mapped search: -1 automatic (large batches), 0 off, 1 on
  int sched = -1;
  int last_sched = 0;
  int nsm = 148;  // SMs of the device
  // per-kernel timing (rfs_profile_eval): CUDA events around every launch while `prof` is set
  struct ProfRec {
    const char *name;
    cudaEvent_t e0, e1;
  };
  bool prof = false;
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;
  size_t prof_used = 0;
};

namespace {

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                     \
      return RFS_E_CUDA;                                                                 \
    }                                                                                    \
  } while (0)

cudaEvent_t prof_event(rfs_ctx *ctx) {
  if (ctx->prof_used == ctx->prof_pool.size()) {
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    ctx->prof_pool.push_back(e);
  }
  return ctx->prof_pool[ctx->prof_used++];
}
inline void prof_begin(rfs_ctx *ctx, const char *name, cudaStream_t st) {
  if (!ctx->prof) return;
  rfs_ctx::ProfRec r{name, prof_event(ctx), prof_event(ctx)};
  cudaEventRecord(r.e0, st);
  ctx->prof_recs.push_back(r);
}
inline void prof_end(rfs_ctx *ctx, cudaStream_t st) {
  if (!ctx->prof) return;
  cudaEventRecord(ctx->prof_recs.back().e1, st);
}

#define LAUNCH(kern, grid, block, smem, st, ...)                 \
  do {                                                           \
    prof_begin(ctx, #kern, (st));                                \
    kern<<<(grid), (block), (smem), (st)>>>(__VA_ARGS__);        \
    ctx->launches++;                                             \
    prof_end(ctx, (st));                                         \
    CK(cudaGetLastError());                                      \
  } while (0)

int ensure(rfs_ctx *ctx, Buf &b, size_t bytes) {
  if (bytes <= b.cap) return RFS_OK;
  if (b.p) CK(cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  size_t want = bytes + bytes / 8 + 256;
  CK(cudaMalloc(&b.p, want));
  b.cap = want;
  return RFS_OK;
}

int fail(rfs_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg;
  return code;
}

enum { TAB_RAYS = 1, TAB_PERIODS = 2, TAB_RF = 4, TAB_GAUSS = 8, TAB_ALL = 15 };

// The only code that clears a per-set table.  The joint weights follow the period and RF-sample tables,
// so their cache goes with any table.
void drop_tables(rfs_ctx *ctx, int which) {
  ObsTables &ot = ctx->tables;
  if (which & TAB_RAYS) ot.has_rays = false;
  if (which & TAB_PERIODS) ot.has_periods = false;
  if (which & TAB_RF) ot.has_rf = false;
  if (which & TAB_GAUSS) ot.has_gauss = false;
  ctx->wt_n1 = ctx->wt_nsw = -1;
}

// Prologue of the table setters.  It drops the table first, so that a call that fails leaves none.
int begin_table(rfs_ctx *ctx, int table, const std::string &name, bool configured, const char *config, int S) {
  drop_tables(ctx, table);
  if (!configured) return fail(ctx, RFS_E_CONFIG, name + " needs " + config);
  if (!ctx->has_obs || S != ctx->nsets)
    return fail(ctx, RFS_E_CONFIG, name + " for " + std::to_string(S) + " sets, the context holds " +
                                       std::to_string(ctx->has_obs ? ctx->nsets : 0));
  return RFS_OK;
}

// A per-set 0/1 mask use [S][width] over the `want` entries of one data block, in which every set keeps
// at least one entry ("set s observes no <what>"); cnt: each set's count of ones.
int check_mask(rfs_ctx *ctx, const std::string &name, const char *what, const unsigned char *use, int S,
               int width, int want, std::vector<int> &cnt) {
  if (width != want)
    return fail(ctx, RFS_E_ARG, name + " has " + std::to_string(width) + " entries per set, the configuration has " +
                                    std::to_string(want));
  if (!use) return fail(ctx, RFS_E_ARG, "no " + name);
  cnt.assign(S, 0);
  for (int s = 0; s < S; s++) {
    for (int j = 0; j < width; j++) {
      const unsigned char u = use[(size_t)s * width + j];
      if (u > 1) return fail(ctx, RFS_E_ARG, name + " values must be 0 or 1");
      cnt[s] += u;
    }
    if (cnt[s] == 0) return fail(ctx, RFS_E_ARG, "set " + std::to_string(s) + " observes no " + what);
  }
  return RFS_OK;
}

// Length of one set's data vector for `which` (0 joint, 1 RF, 2 SWD): the RF block [ray][gauss][nt],
// then the SWD block [mode][grid periods].
int ndata_of(const rfs_ctx *ctx, int which) {
  return (which != 2 ? ctx->rf.nt * (int)ctx->ray_ps.size() * ctx->rf.gauss.n : 0) +
         (which != 1 ? ctx->plan.ndata * (int)ctx->modes.size() : 0);
}

// The plan and device period table the SWD stage runs: the period table's when present, else the grid's.
struct SwdGrid {
  const SwdPlan &plan;
  const double *periods;
};
SwdGrid swd_grid(const rfs_ctx *ctx) {
  const ObsTables &ot = ctx->tables;
  if (ot.has_periods) return {ot.plan, (const double *)ot.d_periods.p};
  return {ctx->plan, (const double *)ctx->d_periods.p};
}

inline unsigned gridFor(long long total, int block) { return (unsigned)((total + block - 1) / block); }

int nmax_for(int n) {
  if (n <= 8) return 8;
  if (n <= 16) return 16;
  if (n <= 48) return 48;
  if (n <= 208) return 208;
  return -1;
}

bool same_periods(const double *a, int na, const double *b, int nb) {
  if (na != nb) return false;
  for (int i = 0; i < na; i++)
    if (a[i] != b[i]) return false;
  return true;
}

// Build the sequence / row plan for the requested wave types (see swd_kernels.cuh).
// want_kernels: group-velocity rows need the 1.05 T / 0.95 T sequences (surfdisp.cpp:234-241).
// share: a group-velocity row on the same periods as the phase-velocity row reuses its T sequence
int build_plan(rfs_ctx *ctx, SwdPlan &P, std::vector<double> &periods, const int nts[4],
               const double *ts[4], int mode, bool want_kernels, bool share = true) {
  memset(&P, 0, sizeof(P));
  periods.clear();
  P.nmode = mode + 1;
  int per_off[4] = {0, 0, 0, 0};
  for (int w = 0; w < 4; w++) {
    per_off[w] = (int)periods.size();
    for (int i = 0; i < nts[w]; i++) {
      if (!(ts[w][i] > 0.0)) return fail(ctx, RFS_E_ARG, "periods must be positive");
      if (i > 0 && !(ts[w][i] > ts[w][i - 1]))
        return fail(ctx, RFS_E_ARG, "periods must be strictly ascending (surfdisp96.f:356-362)");
      periods.push_back(ts[w][i]);
    }
  }
  auto add_seq = [&](int ifunc, int poff, int nper, double scale) {
    SwdSeq &s = P.seq[P.nseq];
    s.ifunc = ifunc;
    s.per_off = poff;
    s.nper = nper;
    s.out_off = P.nsolve;
    s.scale = scale;
    P.nsolve += nper;
    return P.nseq++;
  };
  int d_off = 0;
  for (int fam = 0; fam < 2; fam++) {  // 0 Rayleigh (types 0,1), 1 Love (types 2,3)
    const int wc = fam * 2, wg = fam * 2 + 1;
    const int ifunc = fam == 0 ? 2 : 1;
    int sc = -1;
    if (nts[wc] > 0) {
      sc = add_seq(ifunc, per_off[wc], nts[wc], 1.0);
      SwdRow &r = P.row[P.nrow++];
      r.type = wc;
      r.nper = nts[wc];
      r.per_off = per_off[wc];
      r.s0 = sc;
      r.s1 = r.s2 = -1;
      r.d_off = d_off;
      d_off += nts[wc];
    }
    if (nts[wg] > 0) {
      int s0;
      if (share && sc >= 0 && same_periods(ts[wc], nts[wc], ts[wg], nts[wg]))
        s0 = sc;  // the reference recomputes these roots (surfdisp.cpp:239); they are identical
      else
        s0 = add_seq(ifunc, per_off[wg], nts[wg], 1.0);
      SwdRow &r = P.row[P.nrow++];
      r.type = wg;
      r.nper = nts[wg];
      r.per_off = per_off[wg];
      r.s0 = s0;
      r.s1 = r.s2 = -1;
      if (want_kernels) {
        r.s1 = add_seq(ifunc, per_off[wg], nts[wg], 1.0 + 0.05);
        r.s2 = add_seq(ifunc, per_off[wg], nts[wg], 1.0 - 0.05);
      }
      r.d_off = d_off;
      d_off += nts[wg];
    }
  }
  P.ndata = d_off;
  return RFS_OK;
}

// flat block -> SwdBlocks (runs the earth-flattening prep when sphere)
int make_blocks(rfs_ctx *ctx, Front &F, const double *d_flat, long long B, int n, int sphere,
                SwdBlocks &blk, cudaStream_t st) {
  blk.sphere = sphere;
  if (!sphere) {
    blk.root[0] = blk.root[1] = blk.eig[0] = blk.eig[1] = d_flat;
    return RFS_OK;
  }
  int rc;
  for (int i = 0; i < 4; i++)
    if ((rc = ensure(ctx, F.w_sph[i], sizeof(double) * SWD_NF * (size_t)n * B))) return rc;
  LAUNCH(prep_sphere_kernel, gridFor(B, 128), 128, 0, st, d_flat, B, n, (double *)F.w_sph[0].p,
         (double *)F.w_sph[1].p, (double *)F.w_sph[2].p, (double *)F.w_sph[3].p);
  blk.root[0] = (const double *)F.w_sph[0].p;
  blk.root[1] = (const double *)F.w_sph[1].p;
  blk.eig[0] = (const double *)F.w_sph[2].p;
  blk.eig[1] = (const double *)F.w_sph[3].p;
  return RFS_OK;
}

// ---- root-search mapping (K1 thread-mapped / K1t team-mapped), chosen by the number of sequences in
// flight.  Thread-mapped needs ~25 k sequences to fill 148 SMs; below that a team of T lanes per
// sequence cuts the latency of every secular evaluation (layer-parallel) and of the bracketing scan
// (S speculative grid points).  Thresholds measured on B200 (profiles/r02_roots_sweep.json).
void pick_team(const rfs_ctx *ctx, long long jobs, int n, int &T, int &S) {
  if (ctx->team_T >= 0) {
    T = ctx->team_T;
    S = ctx->team_T ? ctx->team_S : 1;
    return;
  }
  T = 0;
  S = 1;
  // jobs = (model, sequence) pairs in flight; thresholds: fastest mapping in the measured sweep
  if (n <= 16) {
    if (jobs >= 32768) return;                      // thread-mapped
    if (jobs >= 9216) { T = 2; S = 2; return; }     // two lanes, one scan point each, no layer split
    if (jobs >= 4608) { T = 8; S = 2; return; }
    if (jobs >= 1536) { T = 16; S = 2; return; }
    T = 32; S = 4;
    return;
  }
  // many layers (n = 40 ... 200): the sequential 5-vector chain dominates; wide teams pay off longer
  if (jobs >= 12288) return;
  if (jobs >= 1536) { T = 16; S = (n <= 48) ? 2 : 1; return; }
  T = 32; S = 2;
}

bool team_supported(int T, int S) { return team_shape_supported(T, S); }

// launch through the root-search translation unit (swd_roots_tu.cu), with the bookkeeping of LAUNCH
#define LAUNCH_TU(name, call)                                   \
  do {                                                          \
    prof_begin(ctx, name, st);                                  \
    cudaError_t e_ = (call);                                    \
    ctx->launches++;                                            \
    prof_end(ctx, st);                                          \
    if (e_ != cudaSuccess) {                                    \
      ctx->err = std::string(name) + ": " + cudaGetErrorString(e_); \
      return RFS_E_CUDA;                                        \
    }                                                           \
  } while (0)

// The RF branch of a chunk (second stream) is released by the event ev_prep.  It is recorded right
// before the root-search kernel is launched, not right after the model preparation: the RF kernels
// have large grids and would otherwise take every SM while the short scheduling kernels of the sorted
// order run, leaving the latency-bound root search to trickle in behind them.
static inline void release_rf_branch(Front &F, cudaStream_t st) {
  if (F.prep_pending && F.ev_prep) {
    cudaEventRecord(F.ev_prep, st);
    F.prep_pending = false;
  }
}

// batches from this many (model, sequence) jobs on are throughput-bound in the thread mapping: below,
// the job order does not matter (tools/gpu_r2_s.sh: no gain at 36 864 jobs, 8 % at 49 152, 11 % at 196 608)
#ifndef RFS_SCHED_MIN_JOBS
#define RFS_SCHED_MIN_JOBS 32768
#endif
int launch_roots(rfs_ctx *ctx, Front &F, const SwdPlan &P, const SwdSetView &sv, const double *d_periods,
                 const SwdBlocks &d_swd, long long B, int n, int all_modes, cudaStream_t st) {
  unsigned long long *cnt = ctx->count_evals ? (unsigned long long *)ctx->d_counter.p : nullptr;
  int T, S;
  const long long jobs = B * P.nseq;
  pick_team(ctx, jobs, n, T, S);
  ctx->last_team_T = T;
  ctx->last_team_S = S;
  ctx->last_sched = 0;
  if (T == 0) {
    const int *perm = nullptr;
    // automatic: only where the kernel stages the models in shared memory (n <= RFS_ROOTS_STAGE_NMAX).
    // With more layers every evaluation reads the model block from global memory, coalesced over
    // consecutive models; the sorted order scatters those reads (C2, n = 40: 716 -> 1 110 ms).
    const bool auto_on = ctx->sched < 0 && jobs >= RFS_SCHED_MIN_JOBS && n <= RFS_ROOTS_STAGE_NMAX;
    if ((ctx->sched > 0 || auto_on) && jobs < 2147483647LL) {
      int rc;
      if ((rc = ensure(ctx, F.w_key, sizeof(unsigned int) * (size_t)jobs))) return rc;
      if ((rc = ensure(ctx, F.w_perm, sizeof(int) * (size_t)jobs))) return rc;
      LAUNCH_TU("swd_roots_sched_key_kernel",
                launch_sched_keys(P, d_swd, sv, B, n, d_periods, (unsigned int *)F.w_key.p, st));
      LAUNCH_TU("swd_roots_sched_sort_kernel",
                launch_sched_sort(P, B, (const unsigned int *)F.w_key.p, (int *)F.w_perm.p, st));
      perm = (const int *)F.w_perm.p;
      ctx->last_sched = 1;
    }
    release_rf_branch(F, st);
    LAUNCH_TU("swd_roots_kernel",
              launch_roots_thread(P, d_swd, sv, B, n, d_periods, all_modes, (double *)F.w_croot.p,
                                  (double *)F.w_cwork.p, (int *)F.w_ierr.p, cnt, perm, ctx->nsm, st));
    return RFS_OK;
  }
  if (!team_shape_supported(T, S)) return fail(ctx, RFS_E_ARG, "unsupported root-search team shape");
  release_rf_branch(F, st);
  LAUNCH_TU("swd_roots_team_kernel",
            launch_roots_team(T, S, P, d_swd, sv, B, n, d_periods, all_modes, (double *)F.w_croot.p,
                              (double *)F.w_cwork.p, (int *)F.w_ierr.p, cnt, st));
  return RFS_OK;
}

// ---- SWD pipeline on a prepared model block: roots + eigen solves
// roots (+ retries) into the front set F, then (run_swd_eigen) the eigen solves
// sv: each row's own period lists (SwdSetView; tab NULL for the plan's)
int run_swd_roots(rfs_ctx *ctx, Front &F, const SwdPlan &P, const SwdSetView &sv, const double *d_periods,
                  const SwdBlocks &d_swd, long long B, int n, bool all_modes, cudaStream_t st) {
  const int nmo = all_modes ? P.nmode : 1;
  int rc;
  // the kernels index the model block with 32-bit element offsets (SwdModel::ld)
  if ((long long)SWD_NF * n * B > 2147483647LL)
    return fail(ctx, RFS_E_ARG, "SWD batch too large: 10*layers*models must stay below 2^31 per call");
  if ((rc = ensure(ctx, F.w_croot, sizeof(double) * (size_t)nmo * P.nsolve * B))) return rc;
  if ((rc = ensure(ctx, F.w_cwork, sizeof(double) * (size_t)P.nsolve * B))) return rc;
  if ((rc = ensure(ctx, F.w_ierr, sizeof(int) * (size_t)P.nseq * B))) return rc;
  if ((rc = launch_roots(ctx, F, P, sv, d_periods, d_swd, B, n, all_modes ? 1 : 0, st))) return rc;
  // per-period retries of failed fundamental-mode searches (rare; idle warps exit at once)
  if ((rc = ensure(ctx, F.w_rstat, sizeof(int) * (size_t)P.nsolve * B))) return rc;
  LAUNCH_TU("swd_retry_kernel",
            launch_roots_retry(P, d_swd, sv, B, n, d_periods, all_modes ? 1 : 0, (double *)F.w_croot.p,
                               (double *)F.w_cwork.p, (const int *)F.w_ierr.p, (int *)F.w_rstat.p,
                               ctx->count_evals ? (unsigned long long *)ctx->d_counter.p : nullptr, st));
  LAUNCH(swd_retry_finish_kernel, gridFor(B * P.nseq, 128), 128, 0, st, P, sv, B, all_modes ? 1 : 0,
         (double *)F.w_croot.p, (int *)F.w_ierr.p, (const int *)F.w_rstat.p);
  return RFS_OK;
}

int run_swd_eigen(rfs_ctx *ctx, const Front &F, const SwdPlan &P, const SwdSetView &sv, const double *d_periods,
                  const SwdBlocks &d_swd, long long B, int n, bool all_modes, cudaStream_t st) {
  const int nmo = all_modes ? P.nmode : 1;
  int rc;
  if ((rc = ensure(ctx, ctx->w_ugr, sizeof(double) * (size_t)nmo * P.nsolve * B))) return rc;
  if ((rc = ensure(ctx, ctx->w_kern, sizeof(double) * (size_t)nmo * P.nsolve * 4 * n * B)))
    return rc;
  const long long tot = B * P.nsolve * nmo;
  // NMAX = 8: the Rayleigh up-sweep vectors live in shared memory ([48][128] doubles per block)
#define EIG(NM)                                                                                 \
  LAUNCH(swd_eigen_kernel<NM>, gridFor(tot, 128), 128, (NM <= 8 ? 128 * NM * 6 * sizeof(double) : 0), st, \
         P, d_swd, sv, B, n, d_periods, nmo, (const double *)F.w_croot.p, (double *)ctx->w_ugr.p,         \
         (double *)ctx->w_kern.p)
  switch (nmax_for(n)) {
    case 8: EIG(8); break;
    case 16: EIG(16); break;
    case 48: EIG(48); break;
    case 208: EIG(208); break;
    default: return fail(ctx, RFS_E_ARG, "too many layers (max 208)");
  }
#undef EIG
  return RFS_OK;
}

int run_swd(rfs_ctx *ctx, Front &F, const SwdPlan &P, const double *d_periods, const SwdBlocks &d_swd,
            long long B, int n, bool all_modes, bool want_eigen, cudaStream_t st) {
  const SwdSetView sv{nullptr, nullptr, 0, 0};  // the drop-ins: one period list for every model
  int rc = run_swd_roots(ctx, F, P, sv, d_periods, d_swd, B, n, all_modes, st);
  if (rc || !want_eigen) return rc;
  return run_swd_eigen(ctx, F, P, sv, d_periods, d_swd, B, n, all_modes, st);
}

// ---- RF pipeline on a prepared model block (freq method)
// nq: 0 forward only, 2 chain-rule rows (vs, thk), 3 (vs, thk, Vp/Vs), 4 all parameters.  Brings the twiddle table that the
// FFTs of run_rf_decon / run_rf_time read to cfg.nft, in order on `st`.
int run_rf_spectra(rfs_ctx *ctx, const RfCfg &cfg, const RayView &ray, const double *d_rfm,
                   const double *d_chain, const double *d_qa, const double *d_qb, long long B, int n,
                   int nq, cudaStream_t st, double pi_used = RFS_PI32) {
  int rc;
  if (ctx->tw_nft != cfg.nft) {  // not counted in rfs_launch_count
    fft_twiddle_kernel<<<(cfg.nft / 2 + 127) / 128, 128, 0, st>>>(cfg.nft, (double2 *)ctx->d_tw.p);
    CK(cudaGetLastError());
    ctx->tw_nft = cfg.nft;
  }
  const int n2 = cfg.n2;
  if ((rc = ensure(ctx, ctx->w_spec, sizeof(double2) * (size_t)B * 2 * n2))) return rc;
  if (nq > 0)
    if ((rc = ensure(ctx, ctx->w_dspec, sizeof(double2) * (size_t)B * nq * n * n2))) return rc;
  double2 *dsp = nq > 0 ? (double2 *)ctx->w_dspec.p : nullptr;
  // frequency-independent layer constants, once per (model, layer)
  if ((rc = ensure(ctx, ctx->w_rfl, sizeof(RfLayer) * (size_t)B * n))) return rc;
  LAUNCH(rf_layer_kernel, gridFor(B * n, 128), 128, 0, st, d_rfm, d_qa, d_qb, B, n, ray,
         (RfLayer *)ctx->w_rfl.p);
  const long long tot = B * n2;
#define PROP(NM, NQ)                                                                             \
  LAUNCH((rf_propagate_kernel<NM, NQ>), gridFor(tot, 128), 128, 0, st,                           \
         (const RfLayer *)ctx->w_rfl.p, d_chain, B, n, n2, cfg.nft, cfg.dt, ray, cfg.sigma,      \
         pi_used, cfg.rf_type, (double2 *)ctx->w_spec.p, dsp)
#define PROPQ(NM)    \
  if (nq == 2) {     \
    PROP(NM, 2);     \
  } else if (nq == 3) { \
    PROP(NM, 3);     \
  } else {           \
    PROP(NM, 4);     \
  }
  switch (nmax_for(n)) {
    case 8: PROPQ(8); break;
    case 16: PROPQ(16); break;
    case 48: PROPQ(48); break;
    case 208: PROPQ(208); break;
    default: return fail(ctx, RFS_E_ARG, "too many layers (max 208)");
  }
#undef PROPQ
#undef PROP
  return RFS_OK;
}

// Dynamic shared memory above the default 48 KB needs an opt-in per kernel.  It also asks for the full
// shared-memory carve-out (rf_time_kernel at nft = 2048: two ~100 KB blocks per SM instead of one).
template <class K>
int allow_smem(rfs_ctx *ctx, K kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  }
  return RFS_OK;
}

// rf_decon_kernel's layout; more than one Gaussian width adds the weight accumulator (n2 complex)
size_t decon_smem(int nft, int n2, int ngauss = 1) {
  return sizeof(double) * (2 * (size_t)nft + (ngauss > 1 ? 8 : 6) * (size_t)n2 + 64);
}
int decon_threads(int nft) { return std::max(64, std::min(512, nft / 2)); }

template <bool MULTI>
int launch_rf_decon(rfs_ctx *ctx, const RfCfg &cfg, const GaussView &gv, long long B, int nrow, const ObsSets &obs,
                    double *d_rf, long long ldrf, double *d_U, double *d_grad, unsigned char *d_flag, cudaStream_t st,
                    int accumulate) {
  const size_t sm = decon_smem(cfg.nft, cfg.n2, cfg.gauss.n);
  int rc;
  if ((rc = allow_smem(ctx, rf_decon_kernel<MULTI>, sm))) return rc;
  LAUNCH(rf_decon_kernel<MULTI>, (unsigned)B, decon_threads(cfg.nft), sm, st,
         (const double2 *)ctx->w_spec.p, (const double2 *)ctx->w_dspec.p, B, nrow, cfg.nt, cfg.nft,
         cfg.logn, cfg.dt, cfg.gauss, gv, cfg.t0, cfg.water, cfg.sigma, obs, d_rf, ldrf, d_U, d_grad, d_flag,
         (const double2 *)ctx->d_tw.p, accumulate);
  return RFS_OK;
}
// every width of cfg.gauss (or of each row's set, gv), each one trace of d_rf / obs
int run_rf_decon(rfs_ctx *ctx, const RfCfg &cfg, const GaussView &gv, long long B, int nrow, const ObsSets &obs,
                 double *d_rf, long long ldrf, double *d_U, double *d_grad, unsigned char *d_flag, cudaStream_t st,
                 int accumulate = 0) {
  if (cfg.gauss.n > 1)
    return launch_rf_decon<true>(ctx, cfg, gv, B, nrow, obs, d_rf, ldrf, d_U, d_grad, d_flag, st, accumulate);
  return launch_rf_decon<false>(ctx, cfg, gv, B, nrow, obs, d_rf, ldrf, d_U, d_grad, d_flag, st, accumulate);
}

size_t time_smem(int nft, int n2) { return sizeof(double) * (2 * (size_t)nft + 5 * (size_t)n2 + 64); }
// one radix-4 butterfly per thread in the half-length transform (two at nft = 4096); 256-thread blocks
// of 74 KB: three per SM at nft = 2048
int time_threads(int nft) { return std::max(64, std::min(256, nft / 8)); }

// time-domain method: iterative deconvolution of the spectra in w_spec / w_dspec (sigma = 0)
// nrow = 0 (receiver function only) or 4n (plus all Frechet traces -> w_rftr [B][4n][nt]); ig: the
// Gaussian width of this pass (cfg.gauss.a[ig], or each row's set's width ig of gv)
int run_rf_time(rfs_ctx *ctx, const RfCfg &cfg, const GaussView &gv, int ig, long long B, int nrow, double *d_rf,
                long long ldrf, cudaStream_t st) {
  int rc;
  if (nrow > 0)
    if ((rc = ensure(ctx, ctx->w_rftr, sizeof(double) * (size_t)B * nrow * cfg.nt))) return rc;
  const size_t sm = time_smem(cfg.nft, cfg.n2);
  if ((rc = allow_smem(ctx, rf_time_kernel, sm))) return rc;
  LAUNCH(rf_time_kernel, (unsigned)(B * (nrow + 1)), time_threads(cfg.nft), sm, st,
         (const double2 *)ctx->w_spec.p, (const double2 *)ctx->w_dspec.p, B, nrow, cfg.nt, cfg.nft,
         cfg.logn, cfg.dt, gv, ig, cfg.gauss.a[ig], cfg.t0, d_rf, ldrf, (double *)ctx->w_rftr.p,
         (const double2 *)ctx->d_tw.p);
  return RFS_OK;
}

// validated RF settings with the transform length, the signed time shift and the damping derived;
// ctx only receives the error message.  The frequency method deconvolves every width of `gauss` per block.
int make_rf_cfg(rfs_ctx *ctx, RfCfg &cfg, int n, int nt, double dt, const GaussList &gauss, double time_shift,
                double water, int rf_type, int method) {
  if (rf_type != 1 && rf_type != 2) return fail(ctx, RFS_E_ARG, "rf_type should be one of [P,p,S,s]");
  if (method != 0 && method != 1) return fail(ctx, RFS_E_ARG, "method should be time or freq");
  if (nt < 1 || !(dt > 0.0) || n < 2) return fail(ctx, RFS_E_ARG, "bad nt/dt/nlayer");
  if (nmax_for(n) < 0) return fail(ctx, RFS_E_ARG, "too many layers (max 208)");
  int lg = 1;  // nft: the smallest power of two >= max(nt, 2)
  while ((1 << lg) < nt) lg++;
  const int nft = 1 << lg, n2 = nft / 2 + 1;
  // this cap also bounds the twiddle table allocated in rfs_create (nft / 2 <= 2048 entries); at nft = 4096
  // rf_decon_kernel takes 197 184 bytes with several widths, so the cap is the same for every width count
  if (std::max(decon_smem(nft, n2, gauss.n), time_smem(nft, n2)) > 220 * 1024)
    return fail(ctx, RFS_E_ARG, "nt too large (max 4096 samples after padding)");
  const double t0 = rf_type == 2 ? -time_shift : time_shift;  // src/RF/main.cpp:35
  const double sigma = method == 0 ? 0.0 : 1.0 / dt / nft * 4.;
  cfg = RfCfg{n, nt, nft, lg, n2, rf_type, method, dt, water, t0, sigma, gauss};
  return RFS_OK;
}

// The checks of every evaluation of the objective (rfs_misfit_grad_sets_dev / _host, rfs_hmc_run_sets); entry
// names the caller in the message about a missing set array.  n: layers, ndata: one set's data length.
int check_objective(rfs_ctx *ctx, int which, bool has_set, const char *entry, int &n, int &ndata) {
  if (which < 0 || which > 2) return fail(ctx, RFS_E_ARG, "which must be 0,1,2");
  const bool use_swd = which != 1, use_rf = which != 2;
  if ((use_swd && !ctx->has_swd) || (use_rf && !ctx->has_rf) || !ctx->has_obs)
    return fail(ctx, RFS_E_CONFIG, "objective not configured (rfs_config_swd/rf/obs)");
  if (!has_set && ctx->nsets > 1)
    return fail(ctx, RFS_E_CONFIG, "the context holds " + std::to_string(ctx->nsets) +
                                       " observation sets: call " + entry + " with a set array");
  if (use_swd && use_rf && ctx->n_swd != ctx->rf.n) return fail(ctx, RFS_E_CONFIG, "SWD and RF layer counts differ");
  n = use_swd ? ctx->n_swd : ctx->rf.n;
  ndata = ndata_of(ctx, which);
  if (ctx->ndobs != ndata) return fail(ctx, RFS_E_CONFIG, "dobs length != ndata");
  return RFS_OK;
}

// Constants of one fused evaluation, shared by its stages.  overlap: the RF branch of a joint evaluation
// runs on stream2 and root searches on the front streams (false in rfs_profile_eval: every kernel alone).
struct Eval {
  long long B;
  const double *x;
  int which, n, P, ndata, n1, nsw, nray;  // P: parameter blocks per model (rfs_ctx::npar)
  double *U, *grad, *dsyn;
  unsigned char *flag;
  cudaStream_t st;
  bool overlap, use_swd, use_rf;
  SwdGrid grid;  // the period table's plan when there is one (rfs_config_obs_periods)
  ObsSets obs;   // the RF sample mask rides along for the RF residual kernels (ld n1: one set's RF block)
  SwdSetView sv;  // each row's own period lists (rfs_config_obs_periods)
  // several modes in one objective: solve all modes 0..max in one chained pass and pick the listed ones
  bool multi_mode;
  ModeSel msel;
  int nch = 1;  // chunks of Bch rows (plan_chunks)
  long long Bch = 0;

  Eval(const rfs_ctx *ctx, long long B, const double *x, const int *set, int which, int n, int ndata, double *U,
       double *grad, double *dsyn, unsigned char *flag, cudaStream_t st, bool overlap)
      : B(B), x(x), which(which), n(n), P(ctx->npar), ndata(ndata), U(U), grad(grad), dsyn(dsyn), flag(flag), st(st),
        overlap(overlap), use_swd(which != 1), use_rf(which != 2), grid(swd_grid(ctx)) {
    n1 = use_rf ? ndata_of(ctx, 1) : 0;
    nsw = ndata - n1;
    nray = use_rf ? (int)ctx->ray_ps.size() : 0;
    const ObsTables &ot = ctx->tables;
    obs = ObsSets{(const double *)ctx->d_dobs.p, set, ctx->nsets, ndata,
                  use_rf && ot.has_rf ? (const unsigned char *)ot.d_rf.p : nullptr, n1};
    sv = SwdSetView{ot.has_periods ? (const int *)ot.d_tab.p : nullptr, set, ctx->nsets, ot.ld};
    const int nmsel = use_swd ? (int)ctx->modes.size() : 0;
    multi_mode = nmsel > 1;
    msel.n = use_swd ? nmsel : 1;
    for (int i = 0; i < RFS_MAX_MODES; i++) msel.m[i] = multi_mode && i < nmsel ? ctx->modes[i] : 0;
  }
  // chunk k: rows [off, off + B) of the batch; obs and sv as its rows read them (set indices from off on)
  struct Chunk {
    int k;
    long long off, B;
    ObsSets obs;
    SwdSetView sv;
  };
  Chunk chunk(int k) const {
    Chunk c{k, (long long)k * Bch, 0, obs, sv};
    c.B = std::min(Bch, B - c.off);
    if (obs.set) c.obs.set = c.sv.set = obs.set + c.off;
    return c;
  }
};

// Trace (ray ir, width ig) of the RF block [ray][gauss][nt]: its observations, sample mask and synthetics
struct RfTrace {
  ObsSets obs;
  double *dsyn;
};
RfTrace rf_trace(const RfCfg &rf, ObsSets obs, double *dsyn, int ir, int ig) {
  const size_t o = ((size_t)ir * rf.gauss.n + ig) * rf.nt;
  obs.dobs += o;
  if (obs.use) obs.use += o;
  return {obs, dsyn + o};
}

// Chunking.  Bytes of workspace per model: pmf for the front buffers (model blocks and root-search
// results), kept for the whole batch; pm for the eigen / RF workspaces, sized per chunk against what is
// left of the budget.  Chunks are balanced.
void plan_chunks(const rfs_ctx *ctx, Eval &E) {
  size_t pmf = sizeof(double) * E.P * (size_t)E.n, pm = 64;
  if (E.use_swd) {
    const SwdPlan &P = E.grid.plan;
    const size_t nmo = E.multi_mode ? (size_t)P.nmode : 1;
    pmf += sizeof(double) * ((size_t)SWD_NF * E.n * (ctx->sphere ? 5 : 1) + (1 + nmo) * (size_t)P.nsolve) +
           sizeof(int) * ((size_t)3 * P.nseq + P.nsolve);  // ierr, sched key + perm, rstat
    pm += sizeof(double) * (nmo * (size_t)P.nsolve + nmo * (size_t)P.nsolve * 4 * E.n);
  }
  if (E.use_rf) {
    const RfCfg &rf = ctx->rf;
    pmf += sizeof(double) * (4 * (size_t)rf.n);
    pm += sizeof(RfLayer) * (size_t)rf.n + sizeof(double2) * ((size_t)2 * rf.n2 + (size_t)E.P * rf.n * rf.n2) +
          sizeof(double) * (1 + E.P * (size_t)rf.n);
    if (rf.method == 0)  // all four derivative rows, and the Frechet traces
      pm += sizeof(double2) * ((size_t)(4 - E.P) * rf.n * rf.n2) + sizeof(double) * ((size_t)4 * rf.n * rf.nt);
  }
  const size_t front_total = pmf * (size_t)E.B + (pmf * (size_t)E.B) / 8;
  const size_t budget = std::max(ctx->ws_budget > front_total ? ctx->ws_budget - front_total : (size_t)0,
                                 ctx->ws_budget / 4);
  long long Bmax = (long long)std::max<size_t>(32, budget / (pm + pm / 8));
  Bmax = std::min(Bmax, 2147483647LL / ((long long)SWD_NF * E.n));  // 32-bit offsets in SwdModel::ld
  E.nch = (int)((E.B + Bmax - 1) / Bmax);
  E.Bch = (E.B + E.nch - 1) / E.nch;
}

// the SWD weight of the joint objective per set, uploaded again when the data lengths change
int upload_weights(rfs_ctx *ctx, const Eval &E) {
  if (ctx->wt_n1 == E.n1 && ctx->wt_nsw == E.nsw) return RFS_OK;
  const ObsTables &ot = ctx->tables;
  ctx->wt.resize(ctx->nsets);
  for (int k = 0; k < ctx->nsets; k++) {
    const double q = ctx->sigma1[k] / ctx->sigma2[k];
    // with per-set period lists: the data count of set k's own lists, as a one-set context has it
    const int nsw_k = ot.has_periods ? E.msel.n * ot.nobs[k] : E.nsw;
    // likewise the set's own observed RF samples (rfs_config_obs_rf_samples)
    const int n1_k = ot.has_rf ? ot.n1[k] : E.n1;
    ctx->wt[k] = q * q * n1_k / nsw_k;
  }
  int rc;
  if ((rc = ensure(ctx, ctx->d_wt, sizeof(double) * ctx->nsets))) return rc;
  CK(cudaMemcpyAsync(ctx->d_wt.p, ctx->wt.data(), sizeof(double) * ctx->nsets, cudaMemcpyHostToDevice, E.st));
  ctx->wt_n1 = E.n1;
  ctx->wt_nsw = E.nsw;
  return RFS_OK;
}

// Pass A of chunk k: model blocks and root search.  The search runs on a (high-priority) front stream
// for every chunk after the first, and for the first one too when an RF branch competes with it for the SMs.
int front_pass(rfs_ctx *ctx, const Eval &E, const Eval::Chunk &c, Front &F, SwdBlocks &blk) {
  const int n = E.n;
  const bool side = E.overlap && (E.nch > 1 || (E.use_swd && E.use_rf));
  cudaStream_t sk = side ? ctx->stream_front[c.k % 3] : E.st;
  if (sk != E.st) CK(cudaStreamWaitEvent(sk, ctx->ev_fork, 0));
  int rc;
  const size_t nB = (size_t)n * c.B;
  if (E.use_swd && (rc = ensure(ctx, F.w_swd, sizeof(double) * SWD_NF * nB))) return rc;
  if (E.use_rf && (rc = ensure(ctx, F.w_rfm, sizeof(double) * 4 * nB))) return rc;
  if ((rc = ensure(ctx, F.w_chain, sizeof(double) * E.P * nB))) return rc;
#define PREP(P)                                                                                        \
  LAUNCH(prep_models_kernel<P>, gridFor(c.B * n, 256), 256, 0, sk, E.x + c.off * P * n, c.B, n,         \
         E.use_swd ? (double *)F.w_swd.p : nullptr, E.use_rf ? (double *)F.w_rfm.p : nullptr,           \
         (double *)F.w_chain.p)
  if (E.P == 3)
    PREP(3);
  else
    PREP(2);
#undef PREP
  if (!F.ev_prep) CK(cudaEventCreateWithFlags(&F.ev_prep, cudaEventDisableTiming));
  if (!F.ev_ready) CK(cudaEventCreateWithFlags(&F.ev_ready, cudaEventDisableTiming));
  F.prep_pending = true;  // recorded by launch_roots right before the search kernel, or just below
  if (E.use_swd) {
    if ((rc = make_blocks(ctx, F, (const double *)F.w_swd.p, c.B, n, ctx->sphere, blk, sk))) return rc;
    if ((rc = run_swd_roots(ctx, F, E.grid.plan, c.sv, E.grid.periods, blk, c.B, n, E.multi_mode, sk)))
      return rc;
  }
  release_rf_branch(F, sk);
  CK(cudaEventRecord(F.ev_ready, sk));
  return RFS_OK;
}

// RF branch of chunk k: one pass per ray parameter; misfit and gradient accumulate over the passes (the
// reference's ReceiverFunc has one ray parameter, model/model_rf.py:5-18; the list is BASELINE config 3).
// A ray pass covers every Gaussian width: its traces are [gauss][nt] of the data vector.
int rf_branch(rfs_ctx *ctx, const Eval &E, const Eval::Chunk &c, const Front &F) {
  const int n = E.n;
  const RfCfg &rf = ctx->rf;
  int rc;
  // the RF branch only needs the chunk's model blocks: it runs on a second stream, beside the
  // (latency-bound, < 1 wave) root search and the eigen solves
  const bool side = E.use_swd && E.overlap;
  cudaStream_t sr = side ? ctx->stream2 : E.st;
  // RF workspaces and outputs are shared by the chunks: wait for the previous chunk's assemble
  if (side) CK(cudaStreamWaitEvent(sr, c.k == 0 ? ctx->ev_fork : ctx->ev_asm, 0));
  CK(cudaStreamWaitEvent(sr, F.ev_prep, 0));
  if (side) {
    // The RF branch starts behind a 25 us hold kernel, so that the root search's blocks are placed on
    // the SMs before the RF kernels' large grids.  Measured on a B200 in round 2 (tools/gpu_r2_x.sh at
    // commit d506195; ms per step / e2e / HMC evaluations per s), first chunk's search on the caller's
    // stream: 7.99-8.13 / 2.19 M / 1.86 M without the hold, 7.98 / 2.20 M / 1.92 M with it; on a front
    // stream: 10.6 / 2.25 M / 1.87 M without, 8.00 / 2.31 M / 1.92 M with it (the arrangement used).
    LAUNCH(rf_branch_hold_kernel, 1, 32, 0, sr, 25000u);
  }
  if ((rc = ensure(ctx, ctx->w_urf, sizeof(double) * c.B))) return rc;
  if ((rc = ensure(ctx, ctx->w_grf, sizeof(double) * E.P * (size_t)n * c.B))) return rc;
  double *Uo = (E.which == 1) ? E.U + c.off : (double *)ctx->w_urf.p;
  double *go = (E.which == 1) ? E.grad + c.off * E.P * n : (double *)ctx->w_grf.p;
  // RF only: every row succeeds except one whose set index is out of range (the RF kernels write its 0)
  unsigned char *fo = (E.which == 1) ? E.flag + c.off : nullptr;
  if (fo) CK(cudaMemsetAsync(fo, 1, c.B, sr));
  double *dsyn = E.dsyn + c.off * E.ndata;
  const bool rf_time = rf.method == 0;
  const GaussView gv{ctx->tables.has_gauss ? (const double *)ctx->tables.d_gauss.p : nullptr, c.obs.set, ctx->nsets,
                     rf.gauss.n};
  for (int ir = 0; ir < E.nray; ir++) {
    const RayView ray{ctx->tables.has_rays ? (const double *)ctx->tables.d_rays.p : nullptr, c.obs.set, ctx->nsets,
                      E.nray, ir, ctx->ray_ps[ir]};
    if ((rc = run_rf_spectra(ctx, rf, ray, (const double *)F.w_rfm.p, (const double *)F.w_chain.p, nullptr,
                             nullptr, c.B, n, rf_time ? 4 : E.P, sr, rf_time ? RFS_PI64 : RFS_PI32)))
      return rc;
    if (!rf_time) {
      const RfTrace t = rf_trace(rf, c.obs, dsyn, ir, 0);
      if ((rc = run_rf_decon(ctx, rf, gv, c.B, E.P * n, t.obs, t.dsyn, E.ndata, Uo, go, fo, sr, ir > 0))) return rc;
      continue;
    }
    // deconit is nonlinear (argmax spike picking): no adjoint shortcut, materialise the traces of each
    // width in turn from the same spectra
    for (int ig = 0; ig < rf.gauss.n; ig++) {
      const RfTrace t = rf_trace(rf, c.obs, dsyn, ir, ig);
      if ((rc = run_rf_time(ctx, rf, gv, ig, c.B, 4 * n, t.dsyn, E.ndata, sr))) return rc;
#define TGRAD(P)                                                                                         \
  LAUNCH(rf_trace_grad_kernel<P>, gridFor(c.B * n, 128), 128, 0, sr, (const double *)ctx->w_rftr.p,        \
         (const double *)F.w_chain.p, t.dsyn, (long long)E.ndata, t.obs, c.B, n, rf.nt, Uo, go, fo, \
         ir > 0 || ig > 0)
      if (E.P == 3)
        TGRAD(3);
      else
        TGRAD(2);
#undef TGRAD
    }
  }
  if (sr != E.st) CK(cudaEventRecord(ctx->ev_join, sr));
  return RFS_OK;
}

// SWD back pass of chunk k on the caller's stream: the eigen solves, then (after the chunk's RF branch)
// the assembly of the objective
int swd_back_pass(rfs_ctx *ctx, const Eval &E, const Eval::Chunk &c, const Front &F, const SwdBlocks &blk) {
  const int n = E.n;
  CK(cudaStreamWaitEvent(E.st, F.ev_ready, 0));
  int rc;
  if ((rc = run_swd_eigen(ctx, F, E.grid.plan, c.sv, E.grid.periods, blk, c.B, n, E.multi_mode, E.st))) return rc;
  const SwdView V{(const double *)F.w_croot.p, (const double *)ctx->w_ugr.p, (const double *)ctx->w_kern.p,
                  E.grid.periods, c.B, n, blk, 0};
  if (E.use_rf && E.overlap) CK(cudaStreamWaitEvent(E.st, ctx->ev_join, 0));
#define ASM(P)                                                                                                  \
  LAUNCH(joint_assemble_kernel<P>, dim3(gridFor(c.B, 32), (unsigned)n), 32 * RFS_ASM_Q, 0, E.st, E.grid.plan, V, \
         c.sv, (const int *)F.w_ierr.p, (const double *)F.w_chain.p, ctx->stale, E.which, E.n1, c.obs,          \
         (const double *)ctx->w_urf.p, (const double *)ctx->w_grf.p, (const double *)ctx->d_wt.p, E.U + c.off,  \
         E.grad + c.off * P * n, E.dsyn + c.off * E.ndata, E.flag + c.off, E.msel)
  if (E.P == 3)
    ASM(3);
  else
    ASM(2);
#undef ASM
  CK(cudaEventRecord(ctx->ev_asm, E.st));
  return RFS_OK;
}

// the fused evaluation behind rfs_misfit_grad_sets_dev (overlap) and rfs_profile_eval (no overlap)
int misfit_grad(rfs_ctx *ctx, long long B, const double *x, const int *set, int which, double *U, double *grad,
                double *dsyn, unsigned char *flag, cudaStream_t st, bool overlap) {
  if (B <= 0) return RFS_OK;
  int n, ndata, rc;
  if ((rc = check_objective(ctx, which, set != nullptr, "rfs_misfit_grad_sets_dev", n, ndata))) return rc;
  CK(cudaSetDevice(ctx->device));
  Eval E(ctx, B, x, set, which, n, ndata, U, grad, dsyn, flag, st, overlap);
  plan_chunks(ctx, E);
  if (which == 0 && (rc = upload_weights(ctx, E))) return rc;
  while ((int)ctx->fronts.size() < E.nch) ctx->fronts.push_back(std::make_unique<Front>());
  std::vector<SwdBlocks> blks((size_t)E.nch);
  // ---- pass A: model blocks and root search of EVERY chunk.  A chunk's root search is latency-bound
  // when the chunk is small against the machine (n = 200: ~290 ms for anything up to ~25 k models), so
  // the chunks' searches run concurrently instead of one after the other.
  CK(cudaEventRecord(ctx->ev_fork, st));  // everything this call launches comes after what is on `st`
  for (int k = 0; k < E.nch; k++)
    if ((rc = front_pass(ctx, E, E.chunk(k), *ctx->fronts[k], blks[k]))) return rc;
  // ---- pass B: the memory-hungry stages chunk by chunk (RF branch beside the SWD branch)
  for (int k = 0; k < E.nch; k++) {
    const Eval::Chunk c = E.chunk(k);
    if (E.use_rf && (rc = rf_branch(ctx, E, c, *ctx->fronts[k]))) return rc;
    if (E.use_swd && (rc = swd_back_pass(ctx, E, c, *ctx->fronts[k], blks[k]))) return rc;
  }
  return RFS_OK;
}

}  // namespace

extern "C" {

const char *rfs_version(void) { return "rfsurf_b200 0.1 sm_100a"; }

int rfs_create(rfs_ctx **out, int device) {
  if (!out) return RFS_E_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return RFS_E_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return RFS_E_CUDA;
  rfs_ctx *ctx = new rfs_ctx();
  ctx->device = device;
  // the root search runs on high-priority streams: when its blocks and the RF branch's blocks are
  // pending together, the latency-bound search is placed first
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_asm, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithPriority(&ctx->stream_front[0], cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      cudaStreamCreateWithPriority(&ctx->stream_front[1], cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      cudaStreamCreateWithPriority(&ctx->stream_front[2], cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      // FFT twiddle table at its largest size (nft = 4096); run_rf_spectra fills it for each run's nft
      ensure(ctx, ctx->d_tw, sizeof(double2) * 2048) != RFS_OK) {
    rfs_destroy(ctx);
    return RFS_E_CUDA;
  }
  ctx->fronts.push_back(std::make_unique<Front>());
  if (const char *e = getenv("RFS_ROOTS_SCHED")) ctx->sched = atoi(e) < 0 ? -1 : (atoi(e) > 0 ? 1 : 0);
  {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) ctx->nsm = v;
  }
  // RFS_ROOTS_TEAM="T,S" pins the root-search mapping (0 = thread-mapped); default: by batch size
  if (const char *e = getenv("RFS_ROOTS_TEAM")) {
    int t = -1, s2 = 1;
    if (sscanf(e, "%d,%d", &t, &s2) >= 1 && (t == 0 || team_supported(t, s2))) {
      ctx->team_T = t;
      ctx->team_S = s2;
    }
  }
  // workspace budget per chunk of the fused path; batches larger than what fits are chunked.  Default:
  // 60 % of the memory free on this GPU now (a B200 has 180 GB: the Jacobians of 8 192 models of 200
  // layers fit in two chunks), overridden in MiB by RFS_WS_BUDGET_MB
  {
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) == cudaSuccess && fr > ((size_t)8 << 30))
      ctx->ws_budget = std::max<size_t>((size_t)4 << 30, (size_t)(0.6 * (double)fr));
  }
  if (const char *e = getenv("RFS_WS_BUDGET_MB")) {
    const long long mb = atoll(e);
    if (mb > 0) ctx->ws_budget = (size_t)mb << 20;
  }
  *out = ctx;
  return RFS_OK;
}

void rfs_destroy(rfs_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);  // the buffers and fronts free themselves with the context, on this device
  for (cudaStream_t sf : ctx->stream_front)
    if (sf) cudaStreamDestroy(sf);
  for (cudaEvent_t e : ctx->prof_pool) cudaEventDestroy(e);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_asm) cudaEventDestroy(ctx->ev_asm);
  delete ctx;
}

const char *rfs_last_error(rfs_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
long long rfs_launch_count(rfs_ctx *ctx) { return ctx ? ctx->launches : 0; }

int rfs_config_swd_modes(rfs_ctx *ctx, int nlayer, int ntRc, const double *tRc, int ntRg,
                         const double *tRg, int ntLc, const double *tLc, int ntLg, const double *tLg,
                         int nmodes, const int *modes, int sphere, int stale) {
  if (!ctx) return RFS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  if (nlayer < 2 || nmax_for(nlayer) < 0) return fail(ctx, RFS_E_ARG, "bad layer count");
  if (nmodes < 1 || nmodes > RFS_MAX_MODES || !modes) return fail(ctx, RFS_E_ARG, "bad mode list");
  int mode = 0;
  for (int i = 0; i < nmodes; i++) {
    if (modes[i] < 0 || modes[i] > 16) return fail(ctx, RFS_E_ARG, "bad mode");
    if (i > 0 && modes[i] <= modes[i - 1]) return fail(ctx, RFS_E_ARG, "modes must be ascending");
    mode = std::max(mode, modes[i]);
  }
  const int nts[4] = {ntRc, ntRg, ntLc, ntLg};
  const double *ts[4] = {tRc, tRg, tLc, tLg};
  // the new grid is built aside, and a larger period table is uploaded into a new buffer before the old
  // one is released: a call that fails leaves the context as it was
  SwdPlan plan;
  std::vector<double> periods;
  int rc = build_plan(ctx, plan, periods, nts, ts, mode, true);
  if (rc) return rc;
  if (plan.ndata == 0) return fail(ctx, RFS_E_ARG, "no periods given");
  const size_t bytes = sizeof(double) * periods.size();
  Buf grown;
  Buf &dst = bytes <= ctx->d_periods.cap ? ctx->d_periods : grown;
  if ((rc = ensure(ctx, dst, bytes))) return rc;
  CK(cudaMemcpy(dst.p, periods.data(), bytes, cudaMemcpyHostToDevice));
  if (grown.p) {
    std::swap(ctx->d_periods.p, grown.p);
    std::swap(ctx->d_periods.cap, grown.cap);
  }
  ctx->plan = plan;
  ctx->periods.swap(periods);
  for (int w = 0; w < 4; w++) ctx->swd_nts[w] = nts[w];
  ctx->n_swd = nlayer;
  ctx->mode = mode;
  ctx->modes.assign(modes, modes + nmodes);
  ctx->stale = stale ? 1 : 0;
  ctx->sphere = sphere ? 1 : 0;
  ctx->has_swd = true;
  drop_tables(ctx, TAB_PERIODS);  // it marks periods of the previous grid
  return RFS_OK;
}

int rfs_config_swd(rfs_ctx *ctx, int nlayer, int ntRc, const double *tRc, int ntRg,
                   const double *tRg, int ntLc, const double *tLc, int ntLg, const double *tLg,
                   int mode, int sphere, int stale) {
  return rfs_config_swd_modes(ctx, nlayer, ntRc, tRc, ntRg, tRg, ntLc, tLc, ntLg, tLg, 1, &mode,
                              sphere, stale);
}

// Gaussian widths must be finite and > 0 (rfs_config_rf_gauss, rfs_config_obs_gauss)
static int check_widths(rfs_ctx *ctx, const double *gauss, size_t cnt) {
  for (size_t i = 0; i < cnt; i++)
    if (!(isfinite(gauss[i]) && gauss[i] > 0.0)) return fail(ctx, RFS_E_ARG, "Gaussian widths must be finite and > 0");
  return RFS_OK;
}

// The one implementation of the rfs_config_rf* calls; the width list is checked by rfs_config_rf_gauss
// (rfs_config_rf and rfs_config_rf_rays accept any one width, as they always have).
static int config_rf(rfs_ctx *ctx, int nlayer, int nray, const double *ray_p, int ngauss, const double *gauss,
                     int nt, double dt, double time_shift, double water, int rf_type, int method) {
  if (nray < 1 || nray > 64 || !ray_p) return fail(ctx, RFS_E_ARG, "bad ray-parameter list");
  GaussList widths{ngauss, {}};
  std::copy(gauss, gauss + ngauss, widths.a);
  RfCfg cfg;
  int rc = make_rf_cfg(ctx, cfg, nlayer, nt, dt, widths, time_shift, water, rf_type, method);
  if (rc) return rc;
  ctx->rf = cfg;
  ctx->ray_ps.assign(ray_p, ray_p + nray);
  ctx->has_rf = true;
  drop_tables(ctx, TAB_RAYS | TAB_RF | TAB_GAUSS);  // laid out by the previous ray and width lists and nt
  return RFS_OK;
}

int rfs_config_rf_gauss(rfs_ctx *ctx, int nlayer, int nray, const double *ray_p, int ngauss,
                        const double *gauss, int nt, double dt, double time_shift, double water,
                        int rf_type, int method) {
  if (!ctx) return RFS_E_ARG;
  if (ngauss < 1 || ngauss > RFS_MAX_GAUSS || !gauss)
    return fail(ctx, RFS_E_ARG, "bad Gaussian-width list (1 to " + std::to_string(RFS_MAX_GAUSS) + " widths)");
  int rc = check_widths(ctx, gauss, ngauss);
  if (rc) return rc;
  return config_rf(ctx, nlayer, nray, ray_p, ngauss, gauss, nt, dt, time_shift, water, rf_type, method);
}

int rfs_config_rf_rays(rfs_ctx *ctx, int nlayer, int nray, const double *ray_p, int nt, double dt,
                       double gauss, double time_shift, double water, int rf_type, int method) {
  if (!ctx) return RFS_E_ARG;
  return config_rf(ctx, nlayer, nray, ray_p, 1, &gauss, nt, dt, time_shift, water, rf_type, method);
}

int rfs_config_rf(rfs_ctx *ctx, int nlayer, double ray_p, int nt, double dt, double gauss,
                  double time_shift, double water, int rf_type, int method) {
  return rfs_config_rf_rays(ctx, nlayer, 1, &ray_p, nt, dt, gauss, time_shift, water, rf_type,
                            method);
}

int rfs_config_obs_sets(rfs_ctx *ctx, int S, const double *sigma1, const double *sigma2,
                        const double *dobs, int ndobs) {
  if (!ctx || S < 1 || !sigma1 || !sigma2 || !dobs || ndobs <= 0) return RFS_E_ARG;
  drop_tables(ctx, TAB_ALL);  // every table belongs to the sets held
  CK(cudaSetDevice(ctx->device));
  const size_t bytes = sizeof(double) * (size_t)S * ndobs;
  int rc = ensure(ctx, ctx->d_dobs, bytes);
  if (rc) return rc;
  CK(cudaMemcpy(ctx->d_dobs.p, dobs, bytes, cudaMemcpyHostToDevice));
  ctx->sigma1.assign(sigma1, sigma1 + S);
  ctx->sigma2.assign(sigma2, sigma2 + S);
  ctx->nsets = S;
  ctx->ndobs = ndobs;
  ctx->has_obs = true;
  return RFS_OK;
}

int rfs_config_obs(rfs_ctx *ctx, double sigma1, double sigma2, const double *dobs, int ndobs) {
  return rfs_config_obs_sets(ctx, 1, &sigma1, &sigma2, dobs, ndobs);
}

int rfs_config_param(rfs_ctx *ctx, int param) {
  if (!ctx) return RFS_E_ARG;
  if (param != RFS_PARAM_VS_THK && param != RFS_PARAM_VS_THK_VPVS)
    return fail(ctx, RFS_E_ARG, "param must be RFS_PARAM_VS_THK (0) or RFS_PARAM_VS_THK_VPVS (1)");
  ctx->npar = param == RFS_PARAM_VS_THK_VPVS ? 3 : 2;
  return RFS_OK;
}

int rfs_config_obs_rays(rfs_ctx *ctx, int S, int nray, const double *ray_p) {
  if (!ctx) return RFS_E_ARG;
  int rc = begin_table(ctx, TAB_RAYS, "ray-parameter table", ctx->has_rf, "an RF configuration (rfs_config_rf)", S);
  if (rc) return rc;
  if (nray != (int)ctx->ray_ps.size())
    return fail(ctx, RFS_E_ARG, "ray-parameter table has " + std::to_string(nray) + " rays per set, the RF " +
                                    "objective has " + std::to_string(ctx->ray_ps.size()));
  if (!ray_p) return fail(ctx, RFS_E_ARG, "no ray-parameter table");
  const size_t cnt = (size_t)S * nray;
  for (size_t i = 0; i < cnt; i++)
    if (!(isfinite(ray_p[i]) && ray_p[i] > 0.0))
      return fail(ctx, RFS_E_ARG, "ray parameters must be finite and > 0");
  CK(cudaSetDevice(ctx->device));
  ObsTables &ot = ctx->tables;
  if ((rc = ensure(ctx, ot.d_rays, sizeof(double) * cnt))) return rc;
  CK(cudaMemcpy(ot.d_rays.p, ray_p, sizeof(double) * cnt, cudaMemcpyHostToDevice));
  ot.has_rays = true;
  return RFS_OK;
}

int rfs_config_obs_periods(rfs_ctx *ctx, int S, int nper, const unsigned char *use) {
  if (!ctx) return RFS_E_ARG;
  int rc = begin_table(ctx, TAB_PERIODS, "period table", ctx->has_swd, "an SWD configuration (rfs_config_swd)", S);
  if (rc) return rc;
  ObsTables &ot = ctx->tables;
  const SwdPlan &G = ctx->plan;
  const int ng = G.ndata;  // one mode block of the data vector
  if ((rc = check_mask(ctx, "period mask", "period", use, S, nper, ng, ot.nobs))) return rc;
  // the T sequence of Rc may serve Rg only where every set observes the same Rc and Rg periods
  bool share = true;
  for (int fam = 0; fam < 2; fam++) {
    int rc_row = -1, rg_row = -1;
    for (int r = 0; r < G.nrow; r++) {
      if (G.row[r].type == 2 * fam) rc_row = r;
      if (G.row[r].type == 2 * fam + 1) rg_row = r;
    }
    if (rc_row < 0 || rg_row < 0 || G.row[rc_row].s0 != G.row[rg_row].s0) continue;
    const SwdRow &a = G.row[rc_row], &g = G.row[rg_row];
    for (int st = 0; st < S && share; st++)
      share = memcmp(use + (size_t)st * ng + a.d_off, use + (size_t)st * ng + g.d_off, a.nper) == 0;
  }
  // the table's plan on the grid lists (the grid plan itself when sharing stays)
  const double *ts[4];
  for (int w = 0, o = 0; w < 4; o += ctx->swd_nts[w], w++) ts[w] = ctx->periods.data() + o;
  std::vector<double> per;  // the grid lists, then each set's compact lists
  if ((rc = build_plan(ctx, ot.plan, per, ctx->swd_nts, ts, ctx->mode, true, share))) return rc;
  const SwdPlan &P = ot.plan;
  const int ld = 2 * P.nseq + 2 * ng;
  std::vector<int> tab((size_t)S * ld, 0);
  for (int st = 0; st < S; st++) {
    const unsigned char *u = use + (size_t)st * ng;
    int *t = tab.data() + (size_t)st * ld;
    for (int r = 0; r < P.nrow; r++) {
      const SwdRow &rw = P.row[r];
      const int off = (int)per.size();
      int nk = 0;
      for (int g = 0; g < rw.nper; g++)
        if (u[rw.d_off + g]) {
          per.push_back(ctx->periods[rw.per_off + g]);
          t[2 * P.nseq + rw.d_off + nk++] = g;
        }
      for (int q : {rw.s0, rw.s1, rw.s2})
        if (q >= 0) {
          t[q] = off;
          t[P.nseq + q] = nk;
        }
    }
    for (int j = 0; j < ng; j++) t[2 * P.nseq + ng + j] = u[j];
  }
  CK(cudaSetDevice(ctx->device));
  if ((rc = ensure(ctx, ot.d_periods, sizeof(double) * per.size())) ||
      (rc = ensure(ctx, ot.d_tab, sizeof(int) * tab.size())))
    return rc;
  CK(cudaMemcpy(ot.d_periods.p, per.data(), sizeof(double) * per.size(), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ot.d_tab.p, tab.data(), sizeof(int) * tab.size(), cudaMemcpyHostToDevice));
  ot.ld = ld;
  ot.use_col = 2 * P.nseq + ng;
  ot.has_periods = true;
  return RFS_OK;
}

int rfs_config_obs_rf_samples(rfs_ctx *ctx, int S, int nrf, const unsigned char *use) {
  if (!ctx) return RFS_E_ARG;
  int rc = begin_table(ctx, TAB_RF, "RF sample mask", ctx->has_rf, "an RF configuration (rfs_config_rf)", S);
  if (rc) return rc;
  ObsTables &ot = ctx->tables;
  // a set without RF samples would get a zero joint weight, silently dropping its dispersion data
  if ((rc = check_mask(ctx, "RF sample mask", "RF sample", use, S, nrf, ndata_of(ctx, 1), ot.n1))) return rc;
  CK(cudaSetDevice(ctx->device));
  const size_t bytes = (size_t)S * nrf;
  if ((rc = ensure(ctx, ot.d_rf, bytes))) return rc;
  CK(cudaMemcpy(ot.d_rf.p, use, bytes, cudaMemcpyHostToDevice));
  ot.has_rf = true;
  return RFS_OK;
}

int rfs_config_obs_gauss(rfs_ctx *ctx, int S, int ngauss, const double *gauss) {
  if (!ctx) return RFS_E_ARG;
  int rc = begin_table(ctx, TAB_GAUSS, "Gaussian-width table", ctx->has_rf, "an RF configuration (rfs_config_rf)", S);
  if (rc) return rc;
  if (ngauss != ctx->rf.gauss.n)
    return fail(ctx, RFS_E_ARG, "Gaussian-width table has " + std::to_string(ngauss) + " widths per set, the RF " +
                                    "objective has " + std::to_string(ctx->rf.gauss.n));
  if (!gauss) return fail(ctx, RFS_E_ARG, "no Gaussian-width table");
  const size_t cnt = (size_t)S * ngauss;
  if ((rc = check_widths(ctx, gauss, cnt))) return rc;
  CK(cudaSetDevice(ctx->device));
  ObsTables &ot = ctx->tables;
  if ((rc = ensure(ctx, ot.d_gauss, sizeof(double) * cnt))) return rc;
  CK(cudaMemcpy(ot.d_gauss.p, gauss, sizeof(double) * cnt, cudaMemcpyHostToDevice));
  ot.has_gauss = true;
  return RFS_OK;
}

int rfs_misfit_grad_sets_dev(rfs_ctx *ctx, long long B, const double *x, const int *set, int which,
                             double *U, double *grad, double *dsyn, unsigned char *flag, void *stream) {
  if (!ctx) return RFS_E_ARG;
  return misfit_grad(ctx, B, x, set, which, U, grad, dsyn, flag, (cudaStream_t)stream, true);
}

int rfs_misfit_grad_dev(rfs_ctx *ctx, long long B, const double *x, int which, double *U,
                        double *grad, double *dsyn, unsigned char *flag, void *stream) {
  return rfs_misfit_grad_sets_dev(ctx, B, x, nullptr, which, U, grad, dsyn, flag, stream);
}

int rfs_misfit_grad_sets_host(rfs_ctx *ctx, long long B, const double *x, const int *set, int which,
                              double *U, double *grad, double *dsyn, unsigned char *flag) {
  if (!ctx) return RFS_E_ARG;
  if (B <= 0) return RFS_OK;
  int n, ndata, rc;
  if ((rc = check_objective(ctx, which, set != nullptr, "rfs_misfit_grad_sets_host", n, ndata))) return rc;
  if (set)
    for (long long b = 0; b < B; b++)
      if (set[b] < 0 || set[b] >= ctx->nsets)
        return fail(ctx, RFS_E_ARG, "set index " + std::to_string(set[b]) + " of row " + std::to_string(b) +
                                        " outside [0, " + std::to_string(ctx->nsets) + ")");
  CK(cudaSetDevice(ctx->device));
  const int np = ctx->npar * n;  // x and grad columns
  if ((rc = ensure(ctx, ctx->io_x, sizeof(double) * B * np))) return rc;
  if ((rc = ensure(ctx, ctx->io_U, sizeof(double) * B))) return rc;
  if ((rc = ensure(ctx, ctx->io_grad, sizeof(double) * B * np))) return rc;
  if ((rc = ensure(ctx, ctx->io_dsyn, sizeof(double) * B * ndata))) return rc;
  if ((rc = ensure(ctx, ctx->io_flag, B))) return rc;
  if (set && (rc = ensure(ctx, ctx->io_set, sizeof(int) * B))) return rc;
  cudaStream_t st = ctx->stream;
  CK(cudaMemcpyAsync(ctx->io_x.p, x, sizeof(double) * B * np, cudaMemcpyHostToDevice, st));
  if (set) CK(cudaMemcpyAsync(ctx->io_set.p, set, sizeof(int) * B, cudaMemcpyHostToDevice, st));
  rc = rfs_misfit_grad_sets_dev(ctx, B, (const double *)ctx->io_x.p, set ? (const int *)ctx->io_set.p : nullptr,
                                which, (double *)ctx->io_U.p, (double *)ctx->io_grad.p, (double *)ctx->io_dsyn.p,
                                (unsigned char *)ctx->io_flag.p, st);
  if (rc) return rc;
  if (U) CK(cudaMemcpyAsync(U, ctx->io_U.p, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
  if (grad)
    CK(cudaMemcpyAsync(grad, ctx->io_grad.p, sizeof(double) * B * np, cudaMemcpyDeviceToHost, st));
  if (dsyn)
    CK(cudaMemcpyAsync(dsyn, ctx->io_dsyn.p, sizeof(double) * B * ndata, cudaMemcpyDeviceToHost, st));
  if (flag) CK(cudaMemcpyAsync(flag, ctx->io_flag.p, B, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return RFS_OK;
}

int rfs_misfit_grad_host(rfs_ctx *ctx, long long B, const double *x, int which, double *U,
                         double *grad, double *dsyn, unsigned char *flag) {
  return rfs_misfit_grad_sets_host(ctx, B, x, nullptr, which, U, grad, dsyn, flag);
}

// ------------------------------------------------------------------------------ libsurf drop-ins
static int surf_common(rfs_ctx *ctx, long long B, int n, const double *thk, const double *vp,
                       const double *vs, const double *rho, int nT, const double *period,
                       int wavetype, int mode, int sphere, int stale, bool want_kernels,
                       bool all_modes, double *c, double *dcda, double *dcdb, double *dcdr,
                       double *dcdh, unsigned char *ok) {
  if (!ctx) return RFS_E_ARG;
  if (wavetype < 0 || wavetype > 3)
    return fail(ctx, RFS_E_ARG, "wavetype should be one of [Rc,Rg,Lc,Lg]");
  if (B <= 0 || nT <= 0) return RFS_OK;
  if (n < 2 || nmax_for(n) < 0) return fail(ctx, RFS_E_ARG, "bad layer count");
  if (mode < 0 || mode > 16) return fail(ctx, RFS_E_ARG, "bad mode");
  CK(cudaSetDevice(ctx->device));
  // a fluid layer is accepted at the top of the stack only (surfdisp96.f:138-139 handles b(1)<=0)
  for (long long b = 0; b < B; b++)
    for (int m = 1; m < n; m++)
      if (!((float)vs[b * n + m] > 0.0f))
        return fail(ctx, RFS_E_ARG, "vs <= 0 is only supported for the top (water) layer");
  SwdPlan P;
  std::vector<double> periods;
  int nts[4] = {0, 0, 0, 0};
  const double *ts[4] = {nullptr, nullptr, nullptr, nullptr};
  nts[wavetype] = nT;
  ts[wavetype] = period;
  int rc = build_plan(ctx, P, periods, nts, ts, mode, want_kernels);
  if (rc) return rc;
  const bool group = (wavetype & 1) != 0;
  const bool want_eigen = want_kernels || group;
  // libsurf.forward(...,"Lg") goes through _LoveGroup, which replaces vp by 1.732*vs
  // (surfdisp.cpp:127,132); only the float32 start value of the root search sees it.
  const bool love_group_vp = (wavetype == 3) && !want_kernels;
  cudaStream_t st = ctx->stream;
  Front &F = *ctx->fronts[0];
  // pack the model block on the host: [SWD_NF][n][B] float32-rounded (src/SWD/main.cpp:9,62)
  std::vector<double> blk((size_t)SWD_NF * n * B);
  const size_t nB = (size_t)n * B;
  for (long long b = 0; b < B; b++)
    for (int m = 0; m < n; m++) {
      const double d32 = (double)(float)thk[b * n + m], b32 = (double)(float)vs[b * n + m],
                   r32 = (double)(float)rho[b * n + m];
      const double a32 = love_group_vp ? (double)(float)(1.732 * (double)(float)vs[b * n + m])
                                       : (double)(float)vp[b * n + m];
      blk[F_D * nB + (size_t)m * B + b] = d32;
      blk[F_A * nB + (size_t)m * B + b] = a32;
      blk[F_B * nB + (size_t)m * B + b] = b32;
      blk[F_RHO * nB + (size_t)m * B + b] = r32;
      blk[F_IA * nB + (size_t)m * B + b] = 1.0 / a32;
      blk[F_IB * nB + (size_t)m * B + b] = 1.0 / b32;
      blk[F_IRHO * nB + (size_t)m * B + b] = 1.0 / r32;
      blk[F_VTP * nB + (size_t)m * B + b] = 1.0;
      blk[F_DTP * nB + (size_t)m * B + b] = 1.0;
      blk[F_RTP * nB + (size_t)m * B + b] = 1.0;
    }
  if ((rc = ensure(ctx, F.w_swd, sizeof(double) * blk.size()))) return rc;
  if ((rc = ensure(ctx, ctx->io_a, sizeof(double) * periods.size()))) return rc;
  CK(cudaMemcpyAsync(F.w_swd.p, blk.data(), sizeof(double) * blk.size(), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->io_a.p, periods.data(), sizeof(double) * periods.size(),
                     cudaMemcpyHostToDevice, st));
  SwdBlocks dblk;
  if ((rc = make_blocks(ctx, F, (const double *)F.w_swd.p, B, n, sphere ? 1 : 0, dblk, st))) return rc;
  if ((rc = run_swd(ctx, F, P, (const double *)ctx->io_a.p, dblk, B, n, all_modes, want_eigen, st)))
    return rc;
  const int nmo = all_modes ? P.nmode : 1;
  const size_t nc = (size_t)B * nT, nk = (size_t)B * nT * n;
  if ((rc = ensure(ctx, ctx->io_b, sizeof(double) * nc))) return rc;
  if (want_kernels) {
    if ((rc = ensure(ctx, ctx->io_c, sizeof(double) * nk))) return rc;
    if ((rc = ensure(ctx, ctx->io_d, sizeof(double) * nk))) return rc;
    if ((rc = ensure(ctx, ctx->io_e, sizeof(double) * nk))) return rc;
    if ((rc = ensure(ctx, ctx->io_f, sizeof(double) * nk))) return rc;
  }
  for (int mo = 0; mo < nmo; mo++) {
    SwdView V;
    V.croot = (const double *)F.w_croot.p + (size_t)mo * P.nsolve * B;
    V.ugr = want_eigen ? (const double *)ctx->w_ugr.p + (size_t)mo * P.nsolve * B : nullptr;
    V.kern = want_eigen ? (const double *)ctx->w_kern.p + (size_t)mo * P.nsolve * 4 * n * B : nullptr;
    V.periods = (const double *)ctx->io_a.p;
    V.B = B;
    V.n = n;
    V.blk = dblk;
    V.fwd = want_kernels ? 0 : 1;
    LAUNCH(swd_export_row_kernel, gridFor(B * nT * n, 256), 256, 0, st, P, 0, V, stale,
           (double *)ctx->io_b.p, want_kernels ? (double *)ctx->io_c.p : nullptr,
           (double *)ctx->io_d.p, (double *)ctx->io_e.p, (double *)ctx->io_f.p);
    // outputs are [B][nmo][nT](...) : strided copy per model when nmo > 1
    if (nmo == 1) {
      CK(cudaMemcpyAsync(c, ctx->io_b.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, st));
      if (want_kernels) {
        CK(cudaMemcpyAsync(dcda, ctx->io_c.p, sizeof(double) * nk, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(dcdb, ctx->io_d.p, sizeof(double) * nk, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(dcdr, ctx->io_e.p, sizeof(double) * nk, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(dcdh, ctx->io_f.p, sizeof(double) * nk, cudaMemcpyDeviceToHost, st));
      }
    } else {
      const size_t wc = sizeof(double) * nT, wk = sizeof(double) * nT * n;
      CK(cudaMemcpy2DAsync(c + (size_t)mo * nT, wc * nmo, ctx->io_b.p, wc, wc, B,
                           cudaMemcpyDeviceToHost, st));
      if (want_kernels) {
        CK(cudaMemcpy2DAsync(dcda + (size_t)mo * nT * n, wk * nmo, ctx->io_c.p, wk, wk, B,
                             cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpy2DAsync(dcdb + (size_t)mo * nT * n, wk * nmo, ctx->io_d.p, wk, wk, B,
                             cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpy2DAsync(dcdr + (size_t)mo * nT * n, wk * nmo, ctx->io_e.p, wk, wk, B,
                             cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpy2DAsync(dcdh + (size_t)mo * nT * n, wk * nmo, ctx->io_f.p, wk, wk, B,
                             cudaMemcpyDeviceToHost, st));
      }
      CK(cudaStreamSynchronize(st));
    }
  }
  std::vector<int> ierr((size_t)P.nseq * B);
  CK(cudaMemcpyAsync(ierr.data(), F.w_ierr.p, sizeof(int) * ierr.size(), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (ok)
    for (long long b = 0; b < B; b++) {
      bool good = true;
      for (int s = 0; s < P.nseq; s++) good = good && ierr[(size_t)s * B + b] == 0;
      ok[b] = good ? 1 : 0;
    }
  return RFS_OK;
}

int rfs_surf_forward(rfs_ctx *ctx, long long B, int n, const double *thk, const double *vp,
                     const double *vs, const double *rho, int nT, const double *period,
                     int wavetype, int mode, int sphere, double *c, unsigned char *ok) {
  return surf_common(ctx, B, n, thk, vp, vs, rho, nT, period, wavetype, mode, sphere, 1, false,
                     false, c, nullptr, nullptr, nullptr, nullptr, ok);
}

int rfs_surf_adjoint_kernel(rfs_ctx *ctx, long long B, int n, const double *thk, const double *vp,
                            const double *vs, const double *rho, int nT, const double *period,
                            int wavetype, int mode, int sphere, int stale, double *c, double *dcda,
                            double *dcdb, double *dcdr, double *dcdh, unsigned char *ok) {
  return surf_common(ctx, B, n, thk, vp, vs, rho, nT, period, wavetype, mode, sphere, stale, true,
                     false, c, dcda, dcdb, dcdr, dcdh, ok);
}

int rfs_surf_adjoint_kernel_modes(rfs_ctx *ctx, long long B, int n, const double *thk,
                                  const double *vp, const double *vs, const double *rho, int nT,
                                  const double *period, int wavetype, int mode, int stale,
                                  double *c, double *dcda, double *dcdb, double *dcdr,
                                  double *dcdh, unsigned char *ok) {
  return surf_common(ctx, B, n, thk, vp, vs, rho, nT, period, wavetype, mode, 0, stale, true, true,
                     c, dcda, dcdb, dcdr, dcdh, ok);
}

// -------------------------------------------------------------------------------- librf drop-ins
static int rf_common(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                     const double *vp, const double *vs, const double *qa, const double *qb,
                     double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                     double water, int rf_type, int par_type, int nq, double *rf, double *drf) {
  if (!ctx) return RFS_E_ARG;
  RfCfg cfg;  // this call's settings; the fused objective's (ctx->rf) stay as they are
  int rc = make_rf_cfg(ctx, cfg, n, nt, dt, GaussList{1, {gauss}}, time_shift, water, rf_type, method);
  if (rc) return rc;
  if (nq == 1 && (par_type < 1 || par_type > 4))
    return fail(ctx, RFS_E_ARG, "par_type should be one of [vp,vs,rho,thick]");
  if (B <= 0) return RFS_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  Front &F = *ctx->fronts[0];
  const size_t nB = (size_t)n * B;
  std::vector<double> blk(6 * nB);
  for (long long b = 0; b < B; b++)
    for (int m = 0; m < n; m++) {
      blk[0 * nB + (size_t)m * B + b] = thk[b * n + m];
      blk[1 * nB + (size_t)m * B + b] = rho[b * n + m];
      blk[2 * nB + (size_t)m * B + b] = vp[b * n + m];
      blk[3 * nB + (size_t)m * B + b] = vs[b * n + m];
      blk[4 * nB + (size_t)m * B + b] = qa[b * n + m];
      blk[5 * nB + (size_t)m * B + b] = qb[b * n + m];
    }
  if ((rc = ensure(ctx, F.w_rfm, sizeof(double) * 6 * nB))) return rc;
  CK(cudaMemcpyAsync(F.w_rfm.p, blk.data(), sizeof(double) * 6 * nB, cudaMemcpyHostToDevice, st));
  const double *d_rfm = (const double *)F.w_rfm.p;
  if ((rc = run_rf_spectra(ctx, cfg, RayView{nullptr, nullptr, 0, 1, 0, ray_p}, d_rfm, nullptr, d_rfm + 4 * nB, d_rfm + 5 * nB, B, n,
                           nq > 0 ? 4 : 0, st, (method == 0 && nq == 4) ? RFS_PI64 : RFS_PI32)))
    return rc;
  if ((rc = ensure(ctx, ctx->io_b, sizeof(double) * B * nt))) return rc;
  const int nrow = 4 * n;
  const GaussView one{nullptr, nullptr, 1, 1};  // the call's one width, gauss
  if (method == 0) {
    if ((rc = run_rf_time(ctx, cfg, one, 0, B, nq > 0 ? nrow : 0, (double *)ctx->io_b.p, nt, st))) return rc;
  } else {
    if ((rc = run_rf_decon(ctx, cfg, one, B, 0, ObsSets{nullptr, nullptr, 1, 0}, (double *)ctx->io_b.p, nt, nullptr,
                           nullptr, nullptr, st)))
      return rc;
  }
  CK(cudaMemcpyAsync(rf, ctx->io_b.p, sizeof(double) * B * nt, cudaMemcpyDeviceToHost, st));
  if (nq > 0) {
    if (method != 0) {
      if ((rc = ensure(ctx, ctx->w_rftr, sizeof(double) * (size_t)B * nrow * nt))) return rc;
      const size_t sm = decon_smem(cfg.nft, cfg.n2);
      if ((rc = allow_smem(ctx, rf_trace_kernel, sm))) return rc;
      LAUNCH(rf_trace_kernel, (unsigned)(B * nrow), decon_threads(cfg.nft), sm, st,
             (const double2 *)ctx->w_spec.p, (const double2 *)ctx->w_dspec.p, B, nrow, nt, cfg.nft,
             cfg.logn, cfg.dt, cfg.gauss.a[0], cfg.t0, cfg.water, cfg.sigma, (double *)ctx->w_rftr.p,
             (const double2 *)ctx->d_tw.p);
    }
    if (nq == 4) {
      CK(cudaMemcpyAsync(drf, ctx->w_rftr.p, sizeof(double) * (size_t)B * nrow * nt,
                         cudaMemcpyDeviceToHost, st));
    } else {
      const size_t w = sizeof(double) * (size_t)n * nt;
      CK(cudaMemcpy2DAsync(drf, w, (const double *)ctx->w_rftr.p + (size_t)(par_type - 1) * n * nt,
                           w * 4, w, B, cudaMemcpyDeviceToHost, st));
    }
  }
  CK(cudaStreamSynchronize(st));
  return RFS_OK;
}

int rfs_rf_forward(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                   const double *vp, const double *vs, const double *qa, const double *qb,
                   double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                   double water, int rf_type, double *rf) {
  return rf_common(ctx, B, n, thk, rho, vp, vs, qa, qb, ray_p, nt, dt, gauss, time_shift, method,
                   water, rf_type, 0, 0, rf, nullptr);
}
int rfs_rf_kernel(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                  const double *vp, const double *vs, const double *qa, const double *qb,
                  double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                  double water, int rf_type, int par_type, double *rf, double *drf) {
  return rf_common(ctx, B, n, thk, rho, vp, vs, qa, qb, ray_p, nt, dt, gauss, time_shift, method,
                   water, rf_type, par_type, 1, rf, drf);
}
int rfs_rf_kernel_all(rfs_ctx *ctx, long long B, int n, const double *thk, const double *rho,
                      const double *vp, const double *vs, const double *qa, const double *qb,
                      double ray_p, int nt, double dt, double gauss, double time_shift, int method,
                      double water, int rf_type, double *rf, double *drf) {
  return rf_common(ctx, B, n, thk, rho, vp, vs, qa, qb, ray_p, nt, dt, gauss, time_shift, method,
                   water, rf_type, 0, 4, rf, drf);
}


// ---- measurement helpers (bench.py) ---------------------------------------------------------
// kernel classes of rfs_profile_eval
static const char *const kProfNames[RFS_PROF_NK] = {
    "prep_models",  "swd_roots", "swd_retry",      "swd_eigen", "rf_layer",
    "rf_propagate", "rf_decon",  "rf_time_domain", "assemble",  "other"};
static int prof_class(const char *name) {
  if (strstr(name, "prep_")) return 0;
  if (strstr(name, "swd_roots")) return 1;
  if (strstr(name, "swd_retry")) return 2;
  if (strstr(name, "swd_eigen")) return 3;
  if (strstr(name, "rf_layer")) return 4;
  if (strstr(name, "rf_propagate")) return 5;
  if (strstr(name, "rf_decon")) return 6;
  if (strstr(name, "rf_time") || strstr(name, "rf_trace")) return 7;
  if (strstr(name, "joint_assemble")) return 8;
  return 9;
}
const char *rfs_profile_kernel_name(int i) {
  return (i >= 0 && i < RFS_PROF_NK) ? kProfNames[i] : "";
}
int rfs_profile_eval(rfs_ctx *ctx, long long B, const double *x, int which, double *U, double *grad,
                     double *dsyn, unsigned char *flag, void *stream, double *ms,
                     long long *launches) {
  if (!ctx || !ms) return RFS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->prof = true;
  ctx->prof_recs.clear();
  ctx->prof_used = 0;
  // without overlap: the RF branch serialised, so that every kernel is timed alone
  int rc = misfit_grad(ctx, B, x, nullptr, which, U, grad, dsyn, flag, (cudaStream_t)stream, false);
  ctx->prof = false;
  if (rc) return rc;
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  for (int i = 0; i < RFS_PROF_NK; i++) ms[i] = 0.0;
  if (launches)
    for (int i = 0; i < RFS_PROF_NK; i++) launches[i] = 0;
  for (const auto &r : ctx->prof_recs) {
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, r.e0, r.e1));
    const int c = prof_class(r.name);
    ms[c] += (double)t;
    if (launches) launches[c]++;
  }
  return RFS_OK;
}

int rfs_set_roots_team(rfs_ctx *ctx, int T, int S) {
  if (!ctx) return RFS_E_ARG;
  if (T > 0 && !team_supported(T, S)) return fail(ctx, RFS_E_ARG, "unsupported root-search team shape");
  ctx->team_T = T;
  ctx->team_S = T > 0 ? S : 1;
  return RFS_OK;
}
int rfs_set_roots_sched(rfs_ctx *ctx, int mode) {
  if (!ctx || mode < -1 || mode > 1) return RFS_E_ARG;
  ctx->sched = mode;
  return RFS_OK;
}
int rfs_last_roots_sched(rfs_ctx *ctx) { return ctx ? ctx->last_sched : 0; }
int rfs_last_roots_team(rfs_ctx *ctx, int *T, int *S) {
  if (!ctx || !T || !S) return RFS_E_ARG;
  *T = ctx->last_team_T;
  *S = ctx->last_team_S;
  return RFS_OK;
}
int rfs_count_evals(rfs_ctx *ctx, int enable) {
  if (!ctx) return RFS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  int rc = ensure(ctx, ctx->d_counter, 64);
  if (rc) return rc;
  CK(cudaMemset(ctx->d_counter.p, 0, 64));
  ctx->count_evals = enable != 0;
  return RFS_OK;
}
long long rfs_read_evals(rfs_ctx *ctx) {
  if (!ctx || !ctx->d_counter.p) return -1;
  unsigned long long v = 0;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  if (cudaMemcpy(&v, ctx->d_counter.p, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (long long)v;
}
// [0] total secular evaluations, [1] evaluations of the slowest thread, [2] threads above 2000
int rfs_read_eval_stats(rfs_ctx *ctx, long long *out3) {
  if (!ctx || !ctx->d_counter.p || !out3) return RFS_E_ARG;
  unsigned long long v[3] = {0, 0, 0};
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(v, ctx->d_counter.p, sizeof(v), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 3; i++) out3[i] = (long long)v[i];
  return RFS_OK;
}

// see rfs_selftest_math
__global__ void math_selftest_kernel(long long n, unsigned long long *bad) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  // splitmix64 -> u in [0,1)
  unsigned long long z = (unsigned long long)i * 0x9E3779B97F4A7C15ULL + 0x1234567ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  z = z ^ (z >> 31);
  const double u = (double)(z >> 11) * (1.0 / 9007199254740992.0);
  const double v = (i & 1) ? 708.0 * u : 40.0 * u * u;  // dense near 0, covers the fast-path range
  const double e0 = exp(-v), e1 = rfs::exp_neg(v);
  if (__double_as_longlong(e0) != __double_as_longlong(e1)) atomicAdd(bad + 0, 1ULL);
  const double x0 = exp(v - 300.0), x1 = rfs::exp_cb(v - 300.0);
  if (__double_as_longlong(x0) != __double_as_longlong(x1)) atomicAdd(bad + 0, 1ULL);
  double s0, c0, s1, c1;
  const double t = v * 1531.7;  // up to ~1.1e6 rad
  sincos(t, &s0, &c0);
  rfs::sincos_cb(t, &s1, &c1);
  if (__double_as_longlong(s0) != __double_as_longlong(s1)) atomicAdd(bad + 1, 1ULL);
  if (__double_as_longlong(c0) != __double_as_longlong(c1)) atomicAdd(bad + 2, 1ULL);
  sincos(v * 0.01, &s0, &c0);
  rfs::sincos_cb(v * 0.01, &s1, &c1);
  if (__double_as_longlong(s0) != __double_as_longlong(s1)) atomicAdd(bad + 3, 1ULL);
  if (__double_as_longlong(c0) != __double_as_longlong(c1)) atomicAdd(bad + 4, 1ULL);
  const double w = v * v * 1e-6 + 1e-290 + t * 1e-9;
  const double q0 = rsqrt(w), q1 = rfs::rsqrt_pos(w);
  if (__double_as_longlong(q0) != __double_as_longlong(q1)) atomicAdd(bad + 5, 1ULL);
}

__global__ void dfma_peak_kernel(double *out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
         a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c);
    a1 = fma(a1, m, c);
    a2 = fma(a2, m, c);
    a3 = fma(a3, m, c);
    a4 = fma(a4, m, c);
    a5 = fma(a5, m, c);
    a6 = fma(a6, m, c);
    a7 = fma(a7, m, c);
  }
  out[blockIdx.x * (long long)blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// Measured FP64 FMA peak of this GPU in TFLOP/s (1 FMA = 2 flop): the roofline denominator for
// the FP64-pipe-bound kernels (MEASURED_PEAKS.json carries no FP64 figure).
int rfs_measure_fp64_peak(rfs_ctx *ctx, double *tflops) {
  if (!ctx || !tflops) return RFS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, ctx->device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 15;
  int rc = ensure(ctx, ctx->io_a, sizeof(double) * (size_t)blocks * threads);
  if (rc) return rc;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    CK(cudaEventRecord(e0, ctx->stream));
    dfma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>((double *)ctx->io_a.p, iters);
    CK(cudaEventRecord(e1, ctx->stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
    if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops = best;
  return RFS_OK;
}

// Self-test of the constant-bank math used by the root search: exp_neg / sincos_cb / rsqrt_pos must be
// bit-identical to the CUDA math library on their fast-path ranges.  n pseudo-random arguments are
// generated on the device; mismatches[0..5] = exp, sin (large), cos (large), sin (small),
// cos (small), rsqrt.
int rfs_selftest_math(rfs_ctx *ctx, long long n, long long *mismatches) {
  if (!ctx || !mismatches || n <= 0) return RFS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  int rc = ensure(ctx, ctx->io_a, sizeof(unsigned long long) * 6);
  if (rc) return rc;
  CK(cudaMemsetAsync(ctx->io_a.p, 0, sizeof(unsigned long long) * 6, ctx->stream));
  math_selftest_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(
      n, (unsigned long long *)ctx->io_a.p);
  ctx->launches++;
  unsigned long long h[6];
  CK(cudaMemcpyAsync(h, ctx->io_a.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < 6; i++) mismatches[i] = (long long)h[i];
  return RFS_OK;
}

}  // extern "C"

#include "hmc_host.inl"
