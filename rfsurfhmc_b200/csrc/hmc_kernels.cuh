// K6 — device-resident Hamiltonian Monte Carlo: one thread per chain, chain state resident in HBM.
//
// Replaces the Python loops of
//   /root/reference/pyhmc/hmc.py    set_initial_model :74-99, _mirror :121-137, _leapfrog :140-201,
//                                   sample :228-276
//   /root/reference/pyhmc/hmcda.py  _find_initial_dt :170-220, _leapfrog :222-278, sample :280-369
// and NumPy's legacy RandomState stream they draw from (MT19937 init_genrand, 53-bit doubles,
// polar Box-Muller with a cached deviate, masked-rejection randint), so that accept/reject
// sequences are identical to the reference under the same seed.
//
// B200 design: every chain is a small state machine; one "global step" = one advance kernel
// (consume the previous evaluation, do momentum/position updates, reflections, Metropolis,
// dual averaging, and emit the next point to evaluate) followed by ONE batched misfit+gradient
// evaluation of all chains.  Chains with different L, different accepted counts and failed
// trajectories never wait for each other inside a trajectory.  The initial potential/gradient of
// a trajectory is the cached value of the current state (result-neutral, SURVEY Q11).
#pragma once
#include "common.cuh"

namespace rfs {

enum { HP_INIT = 0, HP_FD = 1, HP_LEAP = 2, HP_DONE = 3 };
// status: 0 running/finished normally, 2 max_iters reached, 3 current state cannot be evaluated
// (the reference would loop forever), 4 failure inside _find_initial_dt (reference: exit(1)),
// 5 stopped by the wall-clock budget of rfs_set_hmc_options

// n2: columns of x, P n for P parameter blocks of n layers ([vs, thk] or [vs, thk, Vp/Vs])
struct HmcCfg {
  int n2, n, ndata, sampler, Lmin, Lmax, L0, nsamples, ndraws;
  double dt0, target, lambda, mu;
  long long max_iters, max_log;
};

// Chains live in SLOTS: R <= C slots are resident on the device; when the chain of a slot finishes, the
// slot is refilled with the next queued chain (device-side queue head), so the evaluated batch stays
// full until the queue is empty.  Trajectory state is per slot, results are per chain.
struct HmcDev {
  // trajectory state, per slot
  double *xcur, *xnew, *pnew, *gcur, *dcur;  // [R][n2] x4, [R][ndata]
  double *Ucur, *Hcur, *dt, *dtbar, *h0, *fdH;
  int *phase, *istep, *L, *okcur, *fd_it, *fd_a;
  long long *iacc, *ncount;
  // per chain results [C]
  int *status;
  long long *nevals, *o_iter, *o_acc;
  double *o_dt;
  // slot -> chain, queue of chains not started yet
  int *chain;        // [R] chain index of the slot
  int *queue_head;   // next chain index to start (device counter)
  long long C_total; // number of chains
  const long long *chain_id;  // [C] the reference's MPI rank of each chain (seed offset)
  long long seed;
  // RNG (NumPy legacy MT19937), mt laid out [624][C]
  unsigned int *mt;
  int *mti, *has_gauss;
  double *gauss;
  // evaluation I/O
  double *xeval;               // [C][n2]
  const double *Ue, *ge, *de;  // [C], [C][n2], [C][ndata]
  const unsigned char *fe;     // [C]
  // outputs (may be null)
  double *samples, *misfit, *syn, *initmodel;
  signed char *alog;
  const double *bounds;  // [nb][n2][2]: one box for all chains (box_ld 0) or one per set (box_ld 2 n2)
  long long box_ld;
  // observation sets: set [C] of each chain (NULL: one set), rowset [R] = set of the chain a slot runs,
  // setg [Ba] = rowset gathered for the packed batch (evaluated with the rows' own observations)
  const int *set;
  int *rowset, *setg;
  // per-set period lists (rfs_config_obs_periods): obs_use + rowset[c] * use_ld is the grid mask of the
  // slot's set over one SWD mode block (data values use_n1 + k * use_ng + j); the synthetics at the
  // periods a set does not observe are NaN and are not a failure.  NULL: every value is checked.
  const int *obs_use;
  int use_ld, use_n1, use_ng;
  int *n_active;         // [0] slots still running after the last advance, [1] compaction counter
  // compaction of the evaluation batch once slots have run dry: slot[s] = row of slot s in the
  // evaluated batch (-1: finished), idx[j] = slot of row j, xg = gathered positions [Ba][n2]
  int *slot, *idx;
  double *xg;
};

struct Rng {
  unsigned int *mt;
  long long C, c;
  int mti, has_gauss;
  double gauss;
  RFS_DEVINL unsigned int &M(int i) { return mt[(long long)i * C + c]; }
  RFS_DEVINL void seed(unsigned int s) {
    M(0) = s;
    for (int i = 1; i < 624; i++) {
      const unsigned int p = M(i - 1);
      M(i) = 1812433253u * (p ^ (p >> 30)) + (unsigned int)i;
    }
    mti = 624;
    has_gauss = 0;
    gauss = 0.0;
  }
  RFS_DEVINL void gen() {
    const unsigned int UP = 0x80000000u, LO = 0x7fffffffu, MA = 0x9908b0dfu;
    int kk;
    unsigned int y;
    for (kk = 0; kk < 624 - 397; kk++) {
      y = (M(kk) & UP) | (M(kk + 1) & LO);
      M(kk) = M(kk + 397) ^ (y >> 1) ^ ((y & 1u) ? MA : 0u);
    }
    for (; kk < 623; kk++) {
      y = (M(kk) & UP) | (M(kk + 1) & LO);
      M(kk) = M(kk + (397 - 624)) ^ (y >> 1) ^ ((y & 1u) ? MA : 0u);
    }
    y = (M(623) & UP) | (M(0) & LO);
    M(623) = M(396) ^ (y >> 1) ^ ((y & 1u) ? MA : 0u);
    mti = 0;
  }
  RFS_DEVINL unsigned int u32() {
    if (mti >= 624) gen();
    unsigned int y = M(mti++);
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
  }
  RFS_DEVINL double rand() {  // np.random.rand()
    const unsigned int a = u32() >> 5, b = u32() >> 6;
    return (a * 67108864.0 + b) / 9007199254740992.0;
  }
  RFS_DEVINL double randn() {  // np.random.randn(): legacy_gauss
    if (has_gauss) {
      const double t = gauss;
      has_gauss = 0;
      gauss = 0.0;
      return t;
    }
    double x1, x2, r2;
    do {
      x1 = 2.0 * rand() - 1.0;
      x2 = 2.0 * rand() - 1.0;
      r2 = x1 * x1 + x2 * x2;
    } while (r2 >= 1.0 || r2 == 0.0);
    const double f = sqrt(-2.0 * log(r2) / r2);
    gauss = f * x1;
    has_gauss = 1;
    return f * x2;
  }
  RFS_DEVINL long long randint(long long low, long long high) {  // np.random.randint(low, high)
    const unsigned long long rng = (unsigned long long)(high - 1 - low);
    if (rng == 0) return low;
    unsigned long long mask = rng;
    mask |= mask >> 1;
    mask |= mask >> 2;
    mask |= mask >> 4;
    mask |= mask >> 8;
    mask |= mask >> 16;
    mask |= mask >> 32;
    if (rng <= 0xFFFFFFFFull) {
      if (rng == 0xFFFFFFFFull) return low + (long long)u32();
      unsigned int v;
      do {
        v = u32() & (unsigned int)mask;
      } while (v > rng);
      return low + (long long)v;
    }
    unsigned long long v;
    do {
      v = (((unsigned long long)u32() << 32) | u32()) & mask;
    } while (v > rng);
    return low + (long long)v;
  }
};

RFS_DEVINL Rng rng_load(const HmcDev &D, long long C, long long c) {
  Rng r;
  r.mt = D.mt;
  r.C = C;
  r.c = c;
  r.mti = D.mti[c];
  r.has_gauss = D.has_gauss[c];
  r.gauss = D.gauss[c];
  return r;
}
RFS_DEVINL void rng_store(const HmcDev &D, const Rng &r) {
  D.mti[r.c] = r.mti;
  D.has_gauss[r.c] = r.has_gauss;
  D.gauss[r.c] = r.gauss;
}

// _mirror (hmc.py:121-137) applied to (xnew, pnew) of slot c, in the box of the chain it runs; returns
// false if x is not finite
RFS_DEVINL bool hmc_mirror(const HmcDev &D, const HmcCfg &cfg, long long c) {
  bool fin = true;
  const double *box = D.bounds + D.rowset[c] * D.box_ld;
  for (int j = 0; j < cfg.n2; j++) {
    double x = D.xnew[c * cfg.n2 + j], p = D.pnew[c * cfg.n2 + j];
    const double lo = box[2 * j], hi = box[2 * j + 1];
    int it = 0;
    while (x > hi || x < lo) {
      if (x > hi) {
        x = 2 * hi - x;
        p = -p;
      } else {
        x = 2 * lo - x;
        p = -p;
      }
      if (++it >= 64 && (x > hi || x < lo)) {
        // A state with a huge gradient throws x out by many box widths; the reference would bounce
        // |x|/(hi-lo) times (effectively forever).  After 64 exact bounces fold the rest in closed
        // form: same position up to rounding, same momentum sign, and the trajectory carries on to
        // its (certain) rejection with the RNG stream intact.  +-inf and hi==lo give NaN here
        // (the reference never returns).
        const double w = hi - lo;
        double u = x - lo;
        if (u < 0.0) {
          u = -u;
          p = -p;
        }
        double y = fmod(u, 2.0 * w);
        if (y > w) {
          y = 2.0 * w - y;
          p = -p;
        }
        x = lo + y;
        if (!(x >= lo && x <= hi)) x = nan("");
        break;
      }
    }
    if (isnan(x)) fin = false;
    D.xnew[c * cfg.n2 + j] = x;
    D.pnew[c * cfg.n2 + j] = p;
  }
  return fin;
}

// chain initialisation: seed, set_initial_model until in bounds (hmc.py:74-99,231-235).
// Starts chain `ch` in slot `c` (R = number of slots: the stride of the MT19937 state).  The chain id
// only offsets the seed: chains of different sets may share an id and then draw the same stream.
RFS_DEVINL void hmc_chain_start(const HmcDev &D, const HmcCfg &cfg, long long R, long long c,
                                long long ch) {
  const int set = D.set ? D.set[ch] : 0;
  const double *box = D.bounds + set * D.box_ld;
  D.rowset[c] = set;
  Rng r;
  r.mt = D.mt;
  r.C = R;
  r.c = c;
  r.seed((unsigned int)((D.seed + D.chain_id[ch]) & 0xffffffffLL));
  const int n2 = cfg.n2, n = cfg.n;
  const bool vpvs = n2 == 3 * n;
  double *x = D.xcur + c * n2;
  for (;;) {
    for (int i = 0; i < n2; i++) {
      const double lo = box[2 * i], hi = box[2 * i + 1];
      x[i] = lo + (hi - lo) * r.rand();
    }
    // sort vs ascending, permute thk (and Vp/Vs) alike (insertion sort; values are distinct a.s.)
    for (int i = 1; i < n; i++) {
      const double v = x[i], h = x[n + i], k = vpvs ? x[2 * n + i] : 0.0;
      int j = i - 1;
      while (j >= 0 && x[j] > v) {
        x[j + 1] = x[j];
        x[n + j + 1] = x[n + j];
        if (vpvs) x[2 * n + j + 1] = x[2 * n + j];
        j--;
      }
      x[j + 1] = v;
      x[n + j + 1] = h;
      if (vpvs) x[2 * n + j + 1] = k;
    }
    // every entry in its box except the half-space thickness (index 2n - 1)
    bool ok = true;
    for (int i = 0; i < n2; i++)
      if (i != 2 * n - 1 && (x[i] < box[2 * i] || x[i] > box[2 * i + 1])) ok = false;
    if (ok) break;
  }
  for (int i = 0; i < n2; i++) {
    D.xeval[c * n2 + i] = x[i];
    if (D.initmodel) D.initmodel[ch * n2 + i] = x[i];
  }
  D.chain[c] = (int)ch;
  D.phase[c] = HP_INIT;
  D.istep[c] = 0;
  D.L[c] = 0;
  D.okcur[c] = 0;
  D.fd_it[c] = 0;
  D.fd_a[c] = 0;
  D.status[ch] = 0;
  D.iacc[c] = 0;
  D.ncount[c] = 0;
  D.nevals[ch] = 0;
  D.dt[c] = cfg.dt0;
  D.dtbar[c] = cfg.dt0;
  D.h0[c] = 0.0;
  D.Ucur[c] = 0.0;
  D.Hcur[c] = 0.0;
  D.fdH[c] = 0.0;
  rng_store(D, r);
}
__global__ void hmc_init_kernel(HmcDev D, HmcCfg cfg, long long R) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c >= R) return;
  D.slot[c] = (int)c;
  hmc_chain_start(D, cfg, R, c, c);  // slots 0..R-1 start chains 0..R-1; the queue head starts at R
}

// Chains finish at different times (random L, rejections, stuck chains): re-pack the running ones so
// that the forward model is only evaluated for them.  Row order is arbitrary (atomic counter); every
// chain's results are independent of its row.
__global__ void hmc_compact_kernel(HmcDev D, long long C) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (D.phase[c] != HP_DONE) {
    const int j = atomicAdd(D.n_active + 1, 1);
    D.slot[c] = j;
    D.idx[j] = (int)c;
  } else {
    D.slot[c] = -1;
  }
}
__global__ void hmc_gather_kernel(HmcDev D, int n2, long long Ba) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t >= Ba * n2) return;
  const long long j = t / n2;
  const int i = (int)(t % n2);
  D.xg[t] = D.xeval[(long long)D.idx[j] * n2 + i];
  if (D.setg && i == 0) D.setg[j] = D.rowset[D.idx[j]];
}

// Wall-clock budget exhausted (rfs_set_hmc_options): stop every running slot where it stands and mark
// its chain, and every chain still queued, with status 5.
__global__ void hmc_abort_kernel(HmcDev D, long long R) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c < R && D.phase[c] != HP_DONE) {
    const long long ch = D.chain[c];
    D.status[ch] = 5;
    D.o_iter[ch] = D.ncount[c];
    D.o_acc[ch] = D.iacc[c];
    D.o_dt[ch] = D.dt[c];
    D.phase[c] = HP_DONE;
  }
  // chains that never started
  const long long first = min((long long)*D.queue_head, D.C_total);
  for (long long ch = first + c; ch < D.C_total; ch += R) {
    D.status[ch] = 5;
    D.o_iter[ch] = 0;
    D.o_acc[ch] = 0;
    D.o_dt[ch] = 0.0;
  }
}

RFS_DEVINL bool any_nan(const double *v, int n) {
  bool f = false;
  for (int i = 0; i < n; i++) f = f || isnan(v[i]);
  return f;
}

// NaN in the data values slot c's set observes (a failed forward model)
RFS_DEVINL bool any_nan_obs(const HmcDev &D, long long c, const double *v, int n) {
  if (!D.obs_use) return any_nan(v, n);
  const int *u = D.obs_use + (long long)D.rowset[c] * D.use_ld;
  bool f = false;
  for (int i = 0; i < n; i++) f = f || (isnan(v[i]) && (i < D.use_n1 || u[(i - D.use_n1) % D.use_ng]));
  return f;
}

// One global step of every slot (c = slot, ch = the chain it currently runs; C = number of slots).
__global__ void hmc_advance_kernel(HmcDev D, HmcCfg cfg, long long C) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c >= C) return;
  int phase = D.phase[c];
  if (phase == HP_DONE) return;
  const long long ch = D.chain[c];
  const int n2 = cfg.n2, nd = cfg.ndata;
  Rng r = rng_load(D, C, c);
  double *xcur = D.xcur + c * n2, *xnew = D.xnew + c * n2, *pnew = D.pnew + c * n2,
         *gcur = D.gcur + c * n2, *dcur = D.dcur + c * nd, *xev = D.xeval + c * n2;
  const long long e = D.slot[c];  // row of this chain in the evaluated batch
  const double *ge = D.ge + e * n2, *de = D.de + e * nd;
  const double Ue = D.Ue[e];
  const bool fe = D.fe[e] != 0;
  D.nevals[ch] += 1;
  double dt = D.dt[c];
  const double log_half = log(0.5);

  bool begin = false;      // start a new trajectory after handling the result
  bool traj_end = false;   // a trajectory finished in this step
  bool failed = false;
  double Hnew = 0.0;

  if (phase == HP_INIT) {
    D.Ucur[c] = Ue;
    for (int j = 0; j < n2; j++) gcur[j] = ge[j];
    for (int j = 0; j < nd; j++) dcur[j] = de[j];
    D.okcur[c] = (fe && !any_nan_obs(D, c, de, nd)) ? 1 : 0;
    if (cfg.sampler == 1) {
      // ---- _find_initial_dt prologue (hmcda.py:170-184)
      if (!D.okcur[c]) {
        D.status[ch] = 3;
        phase = HP_DONE;
      } else {
        double K = 0.0;
        for (int j = 0; j < n2; j++) {
          const double p = r.randn() * 0.5;
          pnew[j] = p;
          K += p * p;  // np.dot(p, p)
        }
        K *= 0.5;
        D.fdH[c] = Ue + K;
        dt = cfg.dt0;
        for (int j = 0; j < n2; j++) {
          pnew[j] -= 0.5 * dt * gcur[j];
          xnew[j] = xcur[j] + dt * pnew[j];
        }
        hmc_mirror(D, cfg, c);
        for (int j = 0; j < n2; j++) xev[j] = xnew[j];
        D.fd_it[c] = 0;
        D.fd_a[c] = 0;
        phase = HP_FD;
      }
    } else {
      begin = true;
    }
  } else if (phase == HP_FD) {
    // ---- _find_initial_dt loop body (hmcda.py:186-215)
    if (!fe) {
      D.status[ch] = 4;
      phase = HP_DONE;
    } else {
      double K = 0.0;
      for (int j = 0; j < n2; j++) {
        pnew[j] -= 0.5 * dt * ge[j];
        K += pnew[j] * pnew[j];
      }
      K *= 0.5;
      const double Hn = Ue + K;
      const double ediff = -(Hn - D.fdH[c]);
      int it = D.fd_it[c];
      if (it == 0) D.fd_a[c] = 2 * (ediff > log_half ? 1 : 0) - 1;
      bool fin = false;
      if (ediff < log_half) {
        fin = true;
      } else {
        for (int j = 0; j < n2; j++) pnew[j] -= 0.5 * dt * ge[j];
        D.fdH[c] = Hn;
        dt = dt * ((D.fd_a[c] > 0) ? 2.0 : 0.5);
        it++;
        D.fd_it[c] = it;
        if (it >= 20) {
          fin = true;
        } else {
          for (int j = 0; j < n2; j++) xnew[j] = xnew[j] + dt * pnew[j];
          hmc_mirror(D, cfg, c);
          for (int j = 0; j < n2; j++) xev[j] = xnew[j];
        }
      }
      if (fin) {
        D.dtbar[c] = dt;
        D.h0[c] = 0.0;
        begin = true;
      }
    }
  } else {  // HP_LEAP
    const int L = D.L[c];
    int istep = D.istep[c];
    if (any_nan(ge, n2) || !fe || any_nan_obs(D, c, de, nd)) {
      traj_end = true;
      failed = true;
    } else if (istep < L - 1) {
      for (int j = 0; j < n2; j++) {
        pnew[j] -= dt * ge[j];
        xnew[j] += dt * pnew[j];
      }
      const bool fin = hmc_mirror(D, cfg, c);
      if (!fin) {
        traj_end = true;
        failed = true;
      } else {
        D.istep[c] = istep + 1;
        for (int j = 0; j < n2; j++) xev[j] = xnew[j];
      }
    } else {
      double K = 0.0;
      for (int j = 0; j < n2; j++) {
        pnew[j] -= dt * ge[j] * 0.5;
        K += pnew[j] * pnew[j];
      }
      K *= 0.5;
      Hnew = K + Ue;
      traj_end = true;
    }
  }

  // trajectories may also end immediately inside `begin` (non-finite first drift), hence the loop
  for (int guard = 0; guard < 64 && (traj_end || begin); guard++) {
    if (traj_end) {
      traj_end = false;
      bool accept = false;
      double alpha = 0.0;
      if (cfg.sampler == 0) {
        if (!failed) {
          const double u = r.rand();
          accept = u < exp(-(Hnew - D.Hcur[c]));
        }
      } else {
        if (!failed) {
          const double e = exp(-(Hnew - D.Hcur[c]));
          alpha = (e < 1.0) ? e : 1.0;  // Python min(1., e)
        }
        const double u = r.rand();
        accept = u < alpha;
      }
      long long iacc = D.iacc[c];
      const long long nc = D.ncount[c];
      if (accept) {
        D.Ucur[c] = Ue;
        for (int j = 0; j < n2; j++) {
          xcur[j] = xnew[j];
          gcur[j] = ge[j];
        }
        for (int j = 0; j < nd; j++) dcur[j] = de[j];
        D.okcur[c] = 1;
        if (iacc >= cfg.ndraws) {
          const long long s = iacc - cfg.ndraws;
          if (D.misfit) D.misfit[ch * cfg.nsamples + s] = Ue;
          if (D.samples)
            for (int j = 0; j < n2; j++) D.samples[(ch * cfg.nsamples + s) * n2 + j] = xnew[j];
          if (D.syn)
            for (int j = 0; j < nd; j++) D.syn[(ch * cfg.nsamples + s) * nd + j] = de[j];
        }
        iacc++;
        D.iacc[c] = iacc;
      }
      if (cfg.sampler == 1) {
        // dual averaging (hmcda.py:328-345)
        if (nc < cfg.ndraws) {
          const double m = (double)(nc + 1);
          double fac = 1. / (m + 10.0);
          double h0 = (1 - fac) * D.h0[c] + fac * (cfg.target - alpha);
          const double logdt = cfg.mu - sqrt(m) / 0.05 * h0;
          dt = exp(logdt);
          fac = pow(m, -0.75);
          const double logdtbar = fac * logdt + (1 - fac) * log(D.dtbar[c]);
          D.dtbar[c] = exp(logdtbar);
          D.h0[c] = h0;
        } else {
          dt = D.dtbar[c] * 1.;
        }
      }
      if (D.alog && nc < cfg.max_log) D.alog[ch * cfg.max_log + nc] = accept ? 1 : 0;
      D.ncount[c] = nc + 1;
      failed = false;
      begin = true;
    }
    if (begin) {
      begin = false;
      // ---- start of a trajectory (hmc.py:246-249,146-164 / hmcda.py:305-309,228-245)
      if (D.iacc[c] >= (long long)cfg.ndraws + cfg.nsamples) {
        phase = HP_DONE;
        break;
      }
      if (cfg.max_iters > 0 && D.ncount[c] >= cfg.max_iters) {
        D.status[ch] = 2;
        phase = HP_DONE;
        break;
      }
      if (!D.okcur[c]) {
        D.status[ch] = 3;
        phase = HP_DONE;
        break;
      }
      int L;
      if (cfg.sampler == 0) {
        L = (int)r.randint(cfg.Lmin, (long long)cfg.Lmax + 1);
      } else {
        const double q = cfg.lambda / dt;
        L = (q >= 2147483647.0) ? 2147483647 : (int)q;
        if (L < 1) L = 1;
        // extension (off when Lmax = 0): cap the trajectory length.  The reference lets L explode
        // (L = int(lambda/dt) ~ 4e5 after one rejected warm-up trajectory because gamma = 0.05);
        // with thousands of chains some chain always hits that and the run never ends.
        if (cfg.Lmax > 0 && L > cfg.Lmax) L = cfg.Lmax;
      }
      D.L[c] = L;
      double K = 0.0;
      for (int j = 0; j < n2; j++) {
        const double p = r.randn() * 0.5;
        pnew[j] = p;
        K += p * p;
      }
      K *= 0.5;
      D.Hcur[c] = K + D.Ucur[c];
      for (int j = 0; j < n2; j++) {
        pnew[j] -= dt * gcur[j] * 0.5;
        xnew[j] = xcur[j] + dt * pnew[j];
      }
      const bool fin = hmc_mirror(D, cfg, c);
      if (!fin) {
        traj_end = true;
        failed = true;
        continue;
      }
      for (int j = 0; j < n2; j++) xev[j] = xnew[j];
      D.istep[c] = 0;
      phase = HP_LEAP;
    }
  }
  D.dt[c] = dt;
  D.phase[c] = phase;
  rng_store(D, r);
  if (phase == HP_DONE) {
    // chain finished: publish its counters and hand the slot to the next queued chain, if any
    D.o_iter[ch] = D.ncount[c];
    D.o_acc[ch] = D.iacc[c];
    D.o_dt[ch] = dt;
    const int next = atomicAdd(D.queue_head, 1);
    if ((long long)next < D.C_total) {
      hmc_chain_start(D, cfg, C, c, next);
      phase = HP_INIT;
    }
  }
  if (phase != HP_DONE) atomicAdd(D.n_active, 1);
}

}  // namespace rfs
