// Host-side launchers of the root-search kernels.  The kernels live in their own translation unit
// (swd_roots_tu.cu), compiled with -fmad=false: there ptxas never contracts a*b+c on its own, so the
// thread-mapped, team-mapped and retry kernels -- three different inlining contexts of the same
// secular-function source -- round identically; FMAs appear exactly where the source writes RFS_FMA.
#pragma once
#include <cuda_runtime.h>
#include "swd_plan.cuh"

namespace rfs {

#ifndef RFS_ROOTS_BLOCK
#define RFS_ROOTS_BLOCK 128
#endif
// layer counts up to this one have their root-search model fields staged in shared memory by the
// thread-mapped kernel ([n][7][128] doubles per block)
#ifndef RFS_ROOTS_STAGE_NMAX
#define RFS_ROOTS_STAGE_NMAX 8
#endif

// one thread per (model, sequence); perm != NULL: jobs taken in the length-sorted order of
// launch_sched_sort (nsm = SMs of the device, for the block-to-SM composition)
cudaError_t launch_roots_thread(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                                const double *periods, int all_modes, double *croot, double *cwork,
                                int *ierr, unsigned long long *counter, const int *perm, int nsm,
                                cudaStream_t st);
// length-sorted job order: key[nseq*B] = predicted scan length of every job (bisection estimate of
// c at the longest period); perm[nseq*B] = job ids, longest first, Rayleigh before Love
cudaError_t launch_sched_keys(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                              const double *periods, unsigned int *key, cudaStream_t st);
cudaError_t launch_sched_sort(const SwdPlan &P, long long B, const unsigned int *key, int *perm,
                              cudaStream_t st);
// T lanes per (model, sequence), S speculative scan points; false if (T,S) is not instantiated
bool team_shape_supported(int T, int S);
cudaError_t launch_roots_team(int T, int S, const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                              const double *periods, int all_modes, double *croot, double *cwork,
                              int *ierr, unsigned long long *counter, cudaStream_t st);
// per-period retries of failed fundamental-mode searches (surfdisp.cpp:93-100)
// sv: every launcher runs each row's job on that row's own period list (SwdSetView)
cudaError_t launch_roots_retry(const SwdPlan &P, const SwdBlocks &blk, const SwdSetView &sv, long long B, int n,
                               const double *periods, int all_modes, double *croot, double *cwork,
                               const int *ierr, int *rstat, unsigned long long *counter,
                               cudaStream_t st);

}  // namespace rfs
