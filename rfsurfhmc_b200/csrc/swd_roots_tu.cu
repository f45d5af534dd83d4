// Translation unit of the phase-velocity root search (K1 thread-mapped, K1t team-mapped, retry).
// Compiled with -fmad=false (see swd_roots_launch.h): every kernel in here evaluates the secular
// function with the same roundings, so all mappings return the same bits.
#include "swd_roots_team.cuh"

namespace rfs {

// ---- K1: one thread per (model, sequence)
// croot : [nmode_out][nsolve][B]   cwork : [nsolve][B] (only touched when nmode > 1)
// ierr  : [nseq][B] int
#ifndef RFS_ROOTS_MINBLOCKS
#define RFS_ROOTS_MINBLOCKS 4
#endif
#ifndef RFS_ROOTS_BLOCK
#define RFS_ROOTS_BLOCK 128
#endif
// STAGED: the seven root-search fields of the block's models are copied to shared memory first
// ([n][7][128] doubles, n <= RFS_ROOTS_STAGE_NMAX) and every secular evaluation reads them from there
// (one LDS with an immediate offset per value instead of index arithmetic + a global load).
template <bool STAGED>
__global__ void __launch_bounds__(RFS_ROOTS_BLOCK, RFS_ROOTS_MINBLOCKS)
    swd_roots_kernel(SwdPlan plan, SwdBlocks blk, SwdSetView sv, long long B, int n,
                     const double *__restrict__ periods, int all_modes,
                     double *__restrict__ croot, double *__restrict__ cwork,
                     int *__restrict__ ierr, unsigned long long *__restrict__ neval_total,
                     const int *__restrict__ perm, int nsm) {
  __shared__ double wsm_all[RFS_ROOTS_BLOCK / 32][33];
  extern __shared__ double stage[];
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  bool valid = i < B * plan.nseq;
  if (perm) {
    // length-sorted order (see swd_sched_key_kernel): perm lists the jobs longest first; a block takes
    // four adjacent warps of that list, and rounds of nsm blocks (one per SM) alternate between the
    // longest and the shortest blocks left, so that an SM holds long + short + medium blocks of about
    // equal total work and its short block retires early (room for the RF branch beside it)
    const long long J = B * plan.nseq, W = (J + 31) / 32;
    const long long Q = (W + RFS_ROOTS_BLOCK / 32 - 1) / (RFS_ROOTS_BLOCK / 32);
    const long long q = blockIdx.x, t = q / nsm, pos = q % nsm;
    const long long rank = (t & 1) ? (Q - 1 - ((t - 1) / 2) * nsm - pos) : ((t / 2) * nsm + pos);
    const long long j = (rank * (RFS_ROOTS_BLOCK / 32) + (threadIdx.x >> 5)) * 32 + (threadIdx.x & 31);
    valid = j < J;
    i = valid ? __ldg(perm + j) : 0;
  }
  const long long b = valid ? i % B : 0;
  const int s = valid ? (int)(i / B) : 0;
  const SwdSeq sq = sv.seq(plan, s, b);  // row b's own period list
  SwdModel M(blk.root[sq.ifunc == 2 ? 0 : 1], B, n);
  unsigned int nev = 0;
  int e;
  if (STAGED) {
    for (int m = 0; m < n; m++)
#pragma unroll
      for (int f = 0; f < RFS_ROOT_NF; f++)
        stage[(m * RFS_ROOT_NF + f) * RFS_ROOTS_BLOCK + threadIdx.x] = M.ld(f, m, b);
    __syncwarp();  // a lane only ever reads columns of its own warp (its own, or the lane it helps)
    SmemColModel<RFS_ROOTS_BLOCK> Ms{stage, n};
    e = swd_solve_sequence(Ms, b, (long long)threadIdx.x, sq, periods, plan.nmode, all_modes,
                           croot, (long long)plan.nsolve * B, cwork, B, nev, valid,
                           wsm_all[threadIdx.x >> 5], -1);
  } else {
    e = swd_solve_sequence(M, b, b, sq, periods, plan.nmode, all_modes, croot,
                           (long long)plan.nsolve * B, cwork, B, nev, valid,
                           wsm_all[threadIdx.x >> 5], -1);
  }
  if (valid) ierr[(long long)s * B + b] = e;
  if (neval_total) {
    // one aggregated atomic per warp: algorithmic-work counter for the roofline (bench.py)
    unsigned int w = nev;
    for (int o = 16; o > 0; o >>= 1) w += __shfl_down_sync(0xffffffffu, w, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(neval_total, (unsigned long long)w);
    atomicMax(neval_total + 1, (unsigned long long)nev);          // slowest thread
    if (nev > 2000u) atomicAdd(neval_total + 2, 1ull);            // heavy threads (> 2000 evals)
  }
}

// ---- length-sorted scheduling of the thread-mapped search (large, throughput-bound batches).
// A sequence costs about (c(T_longest) - cc) / dc scan steps plus a fixed number of refinement steps
// per period (the scan of period k starts 1.5 dc below the root of period k-1, surfdisp96.f:271), and
// models differ: on the C1 sampler set 830 +- 125 secular evaluations per sequence (556 ... 1 136), so a
// warp of 32 unrelated models waits for its slowest lane.  swd_sched_key_kernel estimates c(T_longest)
// of every job with RFS_SCHED_BISECT bisection steps of the real secular function between the start
// value cc and the fastest layer (7 evaluations against ~830); swd_sched_sort_kernel orders the jobs
// by that estimate, longest first, Rayleigh jobs before Love jobs (a warp must not mix the two secular
// functions); swd_roots_kernel then takes its jobs through that list.  The order changes which lane
// solves which job and nothing else: every job is solved by the same code on the same inputs, so
// the results are bit-identical (GPU test).
#define RFS_SCHED_BISECT 6
#define RFS_SCHED_BINS 1024
__global__ void __launch_bounds__(128)
    swd_sched_key_kernel(SwdPlan plan, SwdBlocks blk, SwdSetView sv, long long B, int n,
                         const double *__restrict__ periods, unsigned int *__restrict__ key) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * plan.nseq) return;
  const long long b = i % B;
  const SwdSeq sq = sv.seq(plan, (int)(i / B), b);
  SwdModel M(blk.root[sq.ifunc == 2 ? 0 : 1], B, n);
  int llw;
  float betmx, cc1;
  swd_start_values(M, b, llw, betmx, cc1);
  double tmax = 0.0;
  for (int k = 0; k < sq.nper; k++) tmax = fmax(tmax, __ldg(periods + sq.per_off + k));
  unsigned int kv = 0;
  if (sq.nper > 0 && tmax > 0.0 && betmx > cc1) {
    const double omega = 2.0 * RFS_PI64 / (tmax * sq.scale), iomega = 1.0 / omega;
    auto f = [&](double c) {
      const double wv = omega / c;
      return (sq.ifunc == 1) ? dltar1_dev(wv, omega, M, b, llw) : dltar4_dev(wv, omega, iomega, M, b, llw);
    };
    double lo = (double)cc1, hi = (double)betmx;
    const bool s0 = neg1(f(lo));
    for (int it = 0; it < RFS_SCHED_BISECT; it++) {
      const double mid = 0.5 * (lo + hi);
      if (neg1(f(mid)) != s0) hi = mid; else lo = mid;
    }
    const double steps = (0.5 * (lo + hi) - (double)cc1) / (double)0.005f;
    kv = (unsigned int)fmin(fmax(steps, 0.0), 1.0e6);
  }
  key[i] = kv;
}

// ONE block: counting sort of the J = nseq * B keys, largest first, Rayleigh (ifunc 2) before Love;
// perm[J] = job ids (sequence * B + model).  With both wave families present each gets half the bins.
__global__ void __launch_bounds__(RFS_SCHED_BINS)
    swd_sched_sort_kernel(SwdPlan plan, const unsigned int *__restrict__ key, long long B,
                          int *__restrict__ perm) {
  __shared__ unsigned int s_lo[2], s_hi[2];
  __shared__ int hist[RFS_SCHED_BINS];
  __shared__ int wsum[32];
  const int t = threadIdx.x;
  const long long J = B * plan.nseq;
  auto cls_of = [&](long long j) { return plan.seq[(int)(j / B)].ifunc == 1 ? 1 : 0; };
  if (t < 2) { s_lo[t] = 0xffffffffu; s_hi[t] = 0u; }
  for (int j = t; j < RFS_SCHED_BINS; j += blockDim.x) hist[j] = 0;
  __syncthreads();
  unsigned int lo[2] = {0xffffffffu, 0xffffffffu}, hi[2] = {0u, 0u};
  for (long long j = t; j < J; j += blockDim.x) {
    const unsigned int v = __ldg(key + j);
    const int c = cls_of(j);
    lo[c] = min(lo[c], v);
    hi[c] = max(hi[c], v);
  }
#pragma unroll
  for (int c = 0; c < 2; c++) {
    for (int o = 16; o > 0; o >>= 1) {
      lo[c] = min(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
      hi[c] = max(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
    }
    if ((t & 31) == 0) {
      atomicMin(&s_lo[c], lo[c]);
      atomicMax(&s_hi[c], hi[c]);
    }
  }
  __syncthreads();
  const bool two = (s_hi[0] >= s_lo[0]) && (s_hi[1] >= s_lo[1]);  // both families have jobs
  const int nb = two ? RFS_SCHED_BINS / 2 : RFS_SCHED_BINS;
  auto bin_of = [&](long long j) {
    const int c = cls_of(j);
    const unsigned int l0 = s_lo[c];
    const unsigned long long span = (unsigned long long)(s_hi[c] - l0) + 1ull;
    const int inner = nb - 1 - (int)(((unsigned long long)(__ldg(key + j) - l0) * nb) / span);
    return (two && c == 1 ? nb : 0) + inner;
  };
  for (long long j = t; j < J; j += blockDim.x) atomicAdd(&hist[bin_of(j)], 1);
  __syncthreads();
  // exclusive prefix sum over the bins (blockDim.x == RFS_SCHED_BINS)
  const int h = hist[t];
  int inc = h;
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if ((t & 31) >= o) inc += u;
  }
  if ((t & 31) == 31) wsum[t >> 5] = inc;
  __syncthreads();
  if (t < 32) {
    int w = wsum[t];
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, w, o);
      if (t >= o) w += u;
    }
    wsum[t] = w;
  }
  __syncthreads();
  hist[t] = inc - h + ((t >> 5) ? wsum[(t >> 5) - 1] : 0);
  __syncthreads();
  for (long long j = t; j < J; j += blockDim.x) perm[atomicAdd(&hist[bin_of(j)], 1)] = (int)j;
}

// ---- per-period retries of _surfdisp (surfdisp.cpp:93-100): when the fundamental mode failed in
// the main pass, every period whose reported value is zero / NaN is searched again as a fresh
// single-period problem (start value cc, scan upward in dc steps: hundreds of evaluations).
// The reference does these one after the other and stops at the first one that fails again; the
// jobs are independent, so they run here as one thread per (model, sequence, period) — in a warp
// that is otherwise idle, whose 31 spare lanes take over the look-ahead scan — and
// swd_retry_finish_kernel re-imposes the sequential stop rule.
//   rstat [nsolve][B] int: -1 not retried, 0 retried ok, 1 retried and failed again
__global__ void __launch_bounds__(RFS_ROOTS_BLOCK, RFS_ROOTS_MINBLOCKS)
    swd_retry_kernel(SwdPlan plan, SwdBlocks blk, SwdSetView sv, long long B, int n,
                     const double *__restrict__ periods, int all_modes,
                     double *__restrict__ croot, double *__restrict__ cwork,
                     const int *__restrict__ ierr, int *__restrict__ rstat,
                     unsigned long long *__restrict__ neval_total) {
  __shared__ double wsm_all[RFS_ROOTS_BLOCK / 32][33];
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const bool inrange = i < B * plan.nsolve;
  const long long b = inrange ? i % B : 0;
  const int solve = inrange ? (int)(i / B) : 0;
  int s = 0;
  for (int q = 0; q < plan.nseq; q++)
    if (solve >= plan.seq[q].out_off && solve < plan.seq[q].out_off + plan.seq[q].nper) s = q;
  const int k = solve - plan.seq[s].out_off;
  const SwdSeq sq = sv.seq(plan, s, b);
  bool valid = false;
  // a solve beyond row b's own list (k >= sq.nper) was never written by the search
  if (inrange && k < sq.nper && ierr[(long long)s * B + b] != 0) {
    const double *clast = croot + (all_modes ? (long long)(plan.nmode - 1) * plan.nsolve * B : 0);
    const double v = clast[(long long)solve * B + b];
    valid = (v == 0.0 || isnan(v));
  }
  // whole warps without work leave (the warp-cooperative loop needs all 32 lanes of a live warp)
  if (__ballot_sync(0xffffffffu, valid) == 0u) {
    if (inrange) rstat[(long long)solve * B + b] = -1;
    return;
  }
  SwdModel M(blk.root[sq.ifunc == 2 ? 0 : 1], B, n);
  unsigned int nev = 0;
  const int e = swd_solve_sequence(M, b, b, sq, periods, plan.nmode, all_modes, croot,
                                   (long long)plan.nsolve * B, cwork, B, nev, valid,
                                   wsm_all[threadIdx.x >> 5], k);
  if (inrange) rstat[(long long)solve * B + b] = valid ? e : -1;
  if (neval_total) {
    unsigned int w = nev;
    for (int o = 16; o > 0; o >>= 1) w += __shfl_down_sync(0xffffffffu, w, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(neval_total, (unsigned long long)w);
  }
}


static inline unsigned grid_for(long long total, int block) {
  return (unsigned)((total + block - 1) / block);
}

cudaError_t launch_roots_thread(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                                const double *periods, int all_modes, double *croot, double *cwork,
                                int *ierr, unsigned long long *counter, const int *perm, int nsm,
                                cudaStream_t st) {
  if (nsm < 1) nsm = 1;
  if (n <= RFS_ROOTS_STAGE_NMAX) {
    const size_t sm = sizeof(double) * RFS_ROOT_NF * (size_t)n * RFS_ROOTS_BLOCK;
    if (sm > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(swd_roots_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
      if (e != cudaSuccess) return e;
    }
    swd_roots_kernel<true><<<grid_for(B * P.nseq, RFS_ROOTS_BLOCK), RFS_ROOTS_BLOCK, sm, st>>>(
        P, blk, sv, B, n, periods, all_modes, croot, cwork, ierr, counter, perm, nsm);
  } else {
    swd_roots_kernel<false><<<grid_for(B * P.nseq, RFS_ROOTS_BLOCK), RFS_ROOTS_BLOCK, 0, st>>>(
        P, blk, sv, B, n, periods, all_modes, croot, cwork, ierr, counter, perm, nsm);
  }
  return cudaGetLastError();
}

cudaError_t launch_sched_keys(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                              const double *periods, unsigned int *key, cudaStream_t st) {
  swd_sched_key_kernel<<<grid_for(B * P.nseq, 128), 128, 0, st>>>(P, blk, sv, B, n, periods, key);
  return cudaGetLastError();
}

cudaError_t launch_sched_sort(const SwdPlan &P, long long B, const unsigned int *key, int *perm,
                              cudaStream_t st) {
  swd_sched_sort_kernel<<<1, RFS_SCHED_BINS, 0, st>>>(P, key, B, perm);
  return cudaGetLastError();
}

cudaError_t launch_roots_retry(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                               const double *periods, int all_modes, double *croot, double *cwork,
                               const int *ierr, int *rstat, unsigned long long *counter,
                               cudaStream_t st) {
  swd_retry_kernel<<<grid_for(B * P.nsolve, RFS_ROOTS_BLOCK), RFS_ROOTS_BLOCK, 0, st>>>(
      P, blk, sv, B, n, periods, all_modes, croot, cwork, ierr, rstat, counter);
  return cudaGetLastError();
}

bool team_shape_supported(int T, int S) {
  static const int ok[][2] = {{2, 2}, {4, 1}, {4, 4}, {8, 1}, {8, 2}, {8, 8}, {16, 1}, {16, 2},
                              {32, 1}, {32, 2}, {32, 4}};
  for (auto &p : ok)
    if (p[0] == T && p[1] == S) return true;
  return false;
}

template <int T, int S>
static cudaError_t launch_team(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                               const double *periods, int all_modes, double *croot, double *cwork,
                               int *ierr, unsigned long long *counter, cudaStream_t st) {
  // threads per block: as many teams as fit ~64 KB of staged layer parameters
  int threads = 128;
  const size_t per_team = sizeof(double) * RFS_TEAM_NF * (size_t)n;
  while (threads > 32 && threads > T && (threads / T) * per_team > 64 * 1024) threads /= 2;
  const size_t sm = (((threads / T) * per_team + 15) & ~(size_t)15) +
                    (size_t)(threads / 32) * RFS_TEAM_NP * 32 * sizeof(double2);
  if (sm > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(swd_roots_team_kernel<T, S>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
  }
  swd_roots_team_kernel<T, S><<<grid_for(B * P.nseq, threads / T), threads, sm, st>>>(
      P, blk, sv, B, n, periods, all_modes, croot, cwork, ierr, counter);
  return cudaGetLastError();
}

cudaError_t launch_roots_team(int T, int S, const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                              const double *periods, int all_modes, double *croot, double *cwork,
                              int *ierr, unsigned long long *counter, cudaStream_t st) {
#define RFS_TEAM(TT, SS) \
  if (T == TT && S == SS) return launch_team<TT, SS>(P, blk, sv, B, n, periods, all_modes, croot, cwork, ierr, counter, st);
  RFS_TEAM(2, 2) RFS_TEAM(4, 1) RFS_TEAM(4, 4) RFS_TEAM(8, 1) RFS_TEAM(8, 2) RFS_TEAM(8, 8) RFS_TEAM(16, 1)
  RFS_TEAM(16, 2)
  RFS_TEAM(32, 1) RFS_TEAM(32, 2) RFS_TEAM(32, 4)
#undef RFS_TEAM
  return cudaErrorInvalidValue;
}

}  // namespace rfs
