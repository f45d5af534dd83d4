// K1t — latency-optimised, warp-cooperative phase-velocity root search: a TEAM of T lanes per
// (model, period-sequence) instead of one thread (swd_roots.cuh).  Selected by batch size: with few
// sequences in flight (small batches, the tail of an HMC run, many-layer models) the thread-mapped
// kernel leaves most SMs idle and is bound by the latency of one secular evaluation after the other.
//
// Same algorithm, same operations, same bits (surfdisp96.f: surfdisp96 :54-368, getsol :398-491,
// nevill :568-687, dltar1 :727-787, dltar4 :791-891): the returned roots are bit-identical to the
// thread-mapped kernel (GPU test), because both mappings drive the one getsol/nevill state machine
// (SwdRootSearch, swd_roots.cuh) and every secular value is produced by the same inlined functions in
// the same order.  What changes is the schedule:
//
//  * layer parallelism.  A team evaluates the secular function cooperatively.  The Dunkin 5x5 layer
//    matrices (resp. the Love layer terms) — ~4/5 of the arithmetic, independent from layer to layer
//    — are built by GL = T/S lanes at once, one layer per lane, 32 layers per round at most; only
//    the 5-vector propagation e <- normc(e C_m) is sequential, and it is handed from lane to lane
//    with warp shuffles.
//  * speculative scan ("bracket voting").  The bracketing scan of getsol (:457-479) walks the grid
//    c1 + j dc until the secular function changes sign.  With S > 1 a team evaluates S consecutive
//    grid points at once (same repeated additions, hence the identical grid) and consumes the values
//    in order; a value is consumed only if the state machine really asks for that grid point next
//    (bitwise compare), so mis-speculation (downward scans, resets at clow) just discards work.
//    The Neville/bisection refinement stays sequential (each point depends on the previous value).
//  * the layer parameters of the team's model are staged once in shared memory ([7][n] doubles:
//    d, a, b, rho, 1/a, 1/b, 1/rho) and every evaluation reads them from there.
//
// All lanes of a team carry the same state-machine state (uniform control flow inside a team);
// teams of one warp run their state machines independently (sub-warp masks on every shuffle).
#pragma once
#include "swd_plan.cuh"
#include "swd_roots_launch.h"

namespace rfs {

// model of ONE job in shared memory; same accessor shape as SwdModel (the batch index is ignored)
struct SmemModel {
  const double *p;  // [7][n]
  int n;
  RFS_DEVINL double ld(int f, int m, long long) const { return p[f * n + m]; }
};
#define RFS_TEAM_NF 7  // F_D .. F_IRHO

// layer terms of one warp in shared memory: pairs of entries, pair-major [RFS_TEAM_NP][32 lanes] double2,
// so that the lanes' 128-bit stores are conflict-free and every lane of a slot reads the same 16 bytes
// (broadcast) in the chain
#define RFS_TEAM_NE 19
#define RFS_TEAM_NP 10
RFS_DEVINL void dunkin_st(double2 *cm, int col, const Dunkin &C) {
  const double *v = reinterpret_cast<const double *>(&C);
#pragma unroll
  for (int p = 0; p < RFS_TEAM_NP; p++)
    cm[p * 32 + col] = make_double2(v[2 * p], (2 * p + 1 < RFS_TEAM_NE) ? v[2 * p + 1] : 0.0);
}
RFS_DEVINL Dunkin dunkin_ld(const double2 *cm, int col) {
  Dunkin C;
  double *v = reinterpret_cast<double *>(&C);
#pragma unroll
  for (int p = 0; p < RFS_TEAM_NP; p++) {
    const double2 t = cm[p * 32 + col];
    v[2 * p] = t.x;
    if (2 * p + 1 < RFS_TEAM_NE) v[2 * p + 1] = t.y;
  }
  return C;
}
static_assert(sizeof(Dunkin) == RFS_TEAM_NE * sizeof(double), "Dunkin is stored as 19 doubles");

// Secular function at phase velocity c for this lane's candidate slot; the value is valid in every
// lane of the slot (lanes slot*GL .. slot*GL+GL-1 of the team).
//   build : lane g of the slot forms the layer terms of layer base+g and parks them in shared memory;
//   chain : every lane of the slot then walks the layers in order, reading the parked terms (the next
//           layer's terms are fetched while the current one is applied) — no data moves between lanes,
//           and the 5-vector stays in registers with 4 dependent FP64 operations per layer.
// cm: the warp's [RFS_TEAM_NP][32] double2 parking area; lane: 0..31.
template <int T, int S>
RFS_DEVINL double team_secular(const SmemModel &M, int ifunc, int llw, double omega_in,
                               double iomega_in, double c, unsigned tmask, int tl, double2 *cm,
                               int lane) {
  constexpr int GL = T / S;
  const double wvno = omega_in / c;
  if (GL == 1) {
    return (ifunc == 1) ? dltar1_dev(wvno, omega_in, M, 0, llw)
                        : dltar4_dev<SmemModel, true>(wvno, omega_in, iomega_in, M, 0, llw);
  }
  const int g = tl % GL;
  const int col0 = lane - g;  // column of my slot's first layer lane
  const int mmax = M.n;
  const int nl = mmax - llw;  // finite layers to propagate through: m = mmax-2 ... llw-1
  if (ifunc == 1) {
    double e1, e2;
    love_halfspace(M, 0, wvno, omega_in, e1, e2);
    for (int base = 0; base < nl; base += GL) {
      int li = base + g;
      if (li > nl - 1) li = nl - 1;  // spare lanes rebuild the last layer (never read below)
      const LoveL L = love_layer(M, 0, mmax - 2 - li, wvno, omega_in);
      __syncwarp(tmask);  // the previous round has been read
      cm[0 * 32 + lane] = make_double2(L.xmu, L.cosq);
      cm[1 * 32 + lane] = make_double2(L.y, L.z);
      __syncwarp(tmask);
      const int cnt = min(GL, nl - base);
      for (int s = 0; s < cnt; s++) {
        const double2 a = cm[0 * 32 + col0 + s], bq = cm[1 * 32 + col0 + s];
        LoveL Ls;
        Ls.xmu = a.x;
        Ls.cosq = a.y;
        Ls.y = bq.x;
        Ls.z = bq.y;
        love_apply(Ls, e1, e2);
      }
    }
    return (nl > 0) ? love_finish(e1, e2) : e1;
  }
  double omega = omega_in, iom = iomega_in;
  if (omega < 1.0e-4) {
    omega = 1.0e-4;
    iom = 1.0e4;
  }
  const double wvno2 = wvno * wvno;
  double e0, e1, e2, e3, e4;
  dunkin_halfspace(M, 0, wvno, wvno2, omega, iom, e0, e1, e2, e3, e4);
  for (int base = 0; base < nl; base += GL) {
    int li = base + g;
    if (li > nl - 1) li = nl - 1;
    const Dunkin C = dunkin_layer(M, 0, mmax - 2 - li, wvno, wvno2, omega, iom);
    __syncwarp(tmask);  // the previous round has been read
    dunkin_st(cm, lane, C);
    __syncwarp(tmask);
    const int cnt = min(GL, nl - base);
    // two layers per trip: both layers' terms are fetched first, so the second fetch is in flight while
    // the first layer is applied (no register copies: an odd count peels its first layer)
    int s = 0;
    if (cnt & 1) {
      const Dunkin A = dunkin_ld(cm, col0);
      dunkin_apply(A, e0, e1, e2, e3, e4, true);
      s = 1;
    }
    for (; s < cnt; s += 2) {
      const Dunkin A = dunkin_ld(cm, col0 + s);
      const Dunkin B2 = dunkin_ld(cm, col0 + s + 1);
      dunkin_apply(A, e0, e1, e2, e3, e4, false);
      dunkin_apply(B2, e0, e1, e2, e3, e4, true);
    }
  }
  if (nl > 0) dunkin_finish(e0, e1, e2, e3, e4);
  if (llw != 1) return dunkin_water_top(M, 0, wvno, omega, e0, e1);
  return e0;
}

// A team drives the state machine that the thread mapping drives too (SwdRootSearch, swd_roots.cuh).
// Every lane of the team runs it with identical values.  Global results are written by every lane
// (same address, same value: one transaction), so each lane later reads back its own store of the
// chain values in `cwork`.
template <int T, int S>
RFS_DEVINL int swd_solve_team(const SmemModel &M, long long b, const SwdSeq &sq,
                              const double *__restrict__ periods, int nmode, int all_modes,
                              double *__restrict__ cout, long long cout_mode_stride,
                              double *__restrict__ cwork, long long stride, unsigned int &n_evals,
                              unsigned tmask, int tl, int only_k, double2 *park, int lane) {
  constexpr int GL = T / S;
  SwdNevCol xs, ys;
  SwdRootSearch rs(xs, ys, sq, periods, nmode, all_modes, cout, cout_mode_stride, cwork, stride, b,
                   n_evals);
  rs.start(M, 0, only_k);

  for (;;) {
    if (rs.phase == PH_SETUP) rs.advance();
    if (rs.phase == PH_DONE) break;

    // ---- candidate grid points of this round: ceval, ceval +- dc, ... (same additions as the scan)
    double cand[S];
    cand[0] = rs.ceval;
    double myc = rs.ceval;
    if (S > 1) {
      const bool down = (rs.phase == PH_G_SCAN) && (rs.idir < 0);
      const double stepc = down ? -SwdRootSearch::dc : SwdRootSearch::dc;  // c + (-dc) == c - dc exactly
      const bool spec = (rs.phase == PH_G_FIRST || rs.phase == PH_G_SCAN);
      const int slot = tl / GL;
#pragma unroll
      for (int j = 1; j < S; j++) {
        cand[j] = cand[j - 1] + stepc;
        if (spec && slot == j) myc = cand[j];
      }
    }
    const double myval =
        team_secular<T, S>(M, sq.ifunc, rs.llw, rs.omega, rs.iomega, myc, tmask, tl, park, lane);
    double vals[S];
    vals[0] = myval;
    if (S > 1) {
#pragma unroll
      for (int j = 0; j < S; j++) vals[j] = __shfl_sync(tmask, myval, j * GL, T);
    }
    rs.consume(vals[0]);
    if (S > 1) {
#pragma unroll
      for (int j = 1; j < S; j++) {
        // consumed only if the scan really asks for this grid point next (bitwise the same double)
        if (!(rs.phase == PH_G_SCAN && rs.ceval == cand[j])) break;
        rs.consume(vals[j]);
      }
    }
  }
  return rs.job_ierr;
}

// ---- K1t: T lanes per (model, sequence); blockDim.x / T teams per block
// dynamic shared memory: (blockDim.x / T) * RFS_TEAM_NF * n doubles (staged models)
//                        + (blockDim.x / 32) * RFS_TEAM_NP * 32 double2 (parked layer terms)
template <int T, int S>
__global__ void __launch_bounds__(128)
    swd_roots_team_kernel(SwdPlan plan, SwdBlocks blk, SwdSetView sv, long long B, int n,
                          const double *__restrict__ periods, int all_modes,
                          double *__restrict__ croot, double *__restrict__ cwork,
                          int *__restrict__ ierr, unsigned long long *__restrict__ neval_total) {
  extern __shared__ double team_sm[];
  const int tpb = blockDim.x / T;
  const int team = threadIdx.x / T, tl = threadIdx.x % T;
  const long long job = blockIdx.x * (long long)tpb + team;
  const bool valid = job < B * plan.nseq;
  const long long b = valid ? job % B : 0;
  const int s = valid ? (int)(job / B) : 0;
  const SwdSeq sq = sv.seq(plan, s, b);  // row b's own period list
  // ---- stage the layer parameters of this team's model
  double *lp = team_sm + (size_t)team * RFS_TEAM_NF * n;
  {
    const double *src = blk.root[sq.ifunc == 2 ? 0 : 1];
    const long long nB = (long long)n * B;
    for (int idx = tl; idx < RFS_TEAM_NF * n; idx += T) {
      const int f = idx / n, m = idx - f * n;
      lp[idx] = __ldg(src + f * nB + (long long)m * B + b);
    }
  }
  __syncthreads();
  if (!valid) return;
  const int lane = threadIdx.x & 31;
  const unsigned tmask = (T >= 32) ? 0xffffffffu : (((1u << (T & 31)) - 1u) << (lane & ~(T - 1)));
  // parked layer terms behind the staged models, 16-byte aligned
  const size_t model_doubles = ((size_t)tpb * RFS_TEAM_NF * n + 1) & ~(size_t)1;
  double2 *cm = reinterpret_cast<double2 *>(team_sm + model_doubles) +
                (size_t)(threadIdx.x >> 5) * RFS_TEAM_NP * 32;
  SmemModel M{lp, n};
  unsigned int nev = 0;
  const int e = swd_solve_team<T, S>(M, b, sq, periods, plan.nmode, all_modes, croot,
                                     (long long)plan.nsolve * B, cwork, B, nev, tmask, tl, -1, cm, lane);
  if (tl == 0) {
    ierr[(long long)s * B + b] = e;
    if (neval_total) {
      atomicAdd(neval_total, (unsigned long long)nev);
      atomicMax(neval_total + 1, (unsigned long long)nev);
      if (nev > 2000u) atomicAdd(neval_total + 2, 1ull);
    }
  }
}

}  // namespace rfs
