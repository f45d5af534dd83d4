// Fused L2 glue on the device: SWD residuals/gradient contraction and the joint weighting.
//
// Replaces the NumPy glue of
//   /root/reference/model/model_surf.py:155-228          (SurfWD.misfit_and_grad)
//   /root/reference/model/model_rf.py:137-197            (ReceiverFunc.misfit_and_grad; its
//                                                          contraction is done inside rf_decon_kernel)
//   /root/reference/model/model_rf_swd_vs_thk.py:66-86   (Joint_RF_SWD.misfit_and_grad)
// The Jacobians are contracted with the residuals on the fly; K = dcdb + dcda*dadb + dcdr*drda*dadb
// (model_surf.py:184) is applied per layer.
#pragma once
#include "swd_kernels.cuh"

namespace rfs {

// modes of one SWD objective (extension of the reference's single `mode`: BASELINE config 2 asks for
// modes 0-2 in one objective).  n == 1 with the mode arrays already offset: the reference's case.
#define RFS_MAX_MODES 8
struct ModeSel {
  int n;                 // modes in the data vector
  int m[RFS_MAX_MODES];  // their indices into the [mode][...] result arrays
};

// which: 0 joint, 1 RF only, 2 SWD only
// RFS_ASM_Q threads per (model, layer): blocks of 32 models x RFS_ASM_Q period slices, one layer per
// blockIdx.y; slice q contracts the periods k = q, q + Q, ... and the slices are summed in a fixed
// order through shared memory (deterministic).  The loop over the Jacobian rows is a chain of dependent
// global loads: four times the threads cut its latency (0.30 -> ~0.1 ms at C1).
// Layout of outputs (row-major per model, as the Python API):
//   U[B], grad[B][P n] (vs, thk, then Vp/Vs when P = 3), dsyn[B][ndata] with ndata = nt_rf + nsw (joint),
//   flag[B] (1 ok, 0 failed SWD root search or observation-set index out of range)
// Row b is compared with observation set obs.row_set(b); wt[S] is each set's SWD weight
// (sigma1/sigma2)^2 n1/nsw of the joint objective.  With per-set period lists (sv) slice q contracts the
// set's compact periods k = q, q + Q, ... (the sums of a one-set context on those lists), dsyn holds
// them at their grid positions and NaN at the grid positions the set does not observe.
// chain [P][n][B]: dadb, drda (P = 3: dadb = k, then dadk = vs; g_k = dadk*(K_a + drda*K_r)).
#define RFS_ASM_Q 4
template <int P>
__global__ void joint_assemble_kernel(SwdPlan plan, SwdView V, SwdSetView sv, const int *__restrict__ ierr,
                                      const double *__restrict__ chain, int stale, int which,
                                      int nt_rf, ObsSets obs, const double *__restrict__ U_rf,
                                      const double *__restrict__ g_rf, const double *__restrict__ wt,
                                      double *__restrict__ U, double *__restrict__ grad,
                                      double *__restrict__ dsyn, unsigned char *__restrict__ flag,
                                      ModeSel ms) {
  __shared__ double red[P + 1][RFS_ASM_Q][32];
  const int bl = threadIdx.x & 31, q = threadIdx.x >> 5;
  const long long B = V.B;
  const int n = V.n;
  const long long b = blockIdx.x * 32LL + bl;
  const int m = blockIdx.y;
  const bool live = b < B;
  const long long nB = (long long)n * B;
  const int nsw = (which == 1) ? 0 : plan.ndata * ms.n;
  const int n1 = (which == 2) ? 0 : nt_rf;
  const int ndata = n1 + nsw;
  const int set = live ? obs.row_set(b) : 0;
  const double *dobs = obs.row(set < 0 ? 0 : set);
  bool ok = set >= 0;
  if (which != 1 && live)
    for (int s = 0; s < plan.nseq; s++) ok = ok && (ierr[(long long)s * B + b] == 0);
  double gv = 0.0, gh = 0.0, gk = 0.0, us = 0.0;
  if (which != 1 && ok && live) {
    const double dadb = chain[0 * nB + m * B + b], drda = chain[1 * nB + m * B + b];
    const double dadk = P == 3 ? chain[2 * nB + m * B + b] : 0.0;
    for (int im = 0; im < ms.n; im++) {
      // view of mode ms.m[im]: results are laid out [mode][solve]...
      SwdView Vm = V;
      const long long mo = ms.m[im];
      Vm.croot = V.croot + mo * plan.nsolve * B;
      Vm.ugr = V.ugr + mo * plan.nsolve * B;
      Vm.kern = V.kern + mo * plan.nsolve * 4 * nB;
      const int doff = n1 + im * plan.ndata;
      for (int r = 0; r < plan.nrow; r++) {
        const int *c2g;
        const SwdRow rw = sv.row(plan, r, b, &c2g);
        for (int k = q; k < rw.nper; k += RFS_ASM_Q) {
          const int j = doff + rw.d_off + (c2g ? c2g[k] : k);  // grid position of compact period k
          const double d = swd_row_value(plan, Vm, rw, k, b);
          const double res = d - dobs[j];
          double K[4];
          swd_row_kernels(plan, Vm, rw, k, m, b, stale, K);
          const double kv = K[1] + K[0] * dadb + K[2] * drda * dadb;
          gv += res * kv;
          gh += res * K[3];
          if (P == 3) gk += res * (K[0] * dadk + K[2] * drda * dadk);
          if (m == 0) {
            us += res * res;
            dsyn[b * ndata + j] = d;
          }
        }
        if (c2g && m == 0) {
          const int *use = c2g - rw.d_off + plan.ndata;  // the set's grid mask
          const int ng = plan.row[r].nper;
          for (int g = q; g < ng; g += RFS_ASM_Q)
            if (!use[rw.d_off + g]) dsyn[b * ndata + doff + rw.d_off + g] = nan("");
        }
      }
    }
  }
  // fixed-order sum over the period slices
  red[0][q][bl] = gv;
  red[1][q][bl] = gh;
  red[2][q][bl] = us;
  if (P == 3) red[3][q][bl] = gk;
  __syncthreads();
  if (q != 0 || !live) return;
  gv = gh = gk = us = 0.0;
#pragma unroll
  for (int j = 0; j < RFS_ASM_Q; j++) {
    gv += red[0][j][bl];
    gh += red[1][j][bl];
    us += red[2][j][bl];
    if (P == 3) gk += red[3][j][bl];
  }
  if (ok) {
    const double w = (which == 0) ? wt[set] : 1.0;
    double g0 = w * gv, g1 = w * gh, g2 = w * gk;
    if (which != 2) {
      g0 += g_rf[b * P * n + m];
      g1 += g_rf[b * P * n + n + m];
      if (P == 3) g2 += g_rf[b * P * n + 2 * n + m];
    }
    grad[b * P * n + m] = g0;
    grad[b * P * n + n + m] = g1;
    if (P == 3) grad[b * P * n + 2 * n + m] = g2;
    if (m == 0) {
      double u = w * 0.5 * us;
      if (which != 2) u += U_rf[b];
      U[b] = u;
      flag[b] = 1;
    }
  } else {
    // model_rf_swd_vs_thk.py:73-74: (0.0, zeros, dobs, False), dobs of the row's own set
    grad[b * P * n + m] = 0.0;
    grad[b * P * n + n + m] = 0.0;
    if (P == 3) grad[b * P * n + 2 * n + m] = 0.0;
    const double fill = (set < 0) ? nan("") : 0.0;
    for (int j = m; j < ndata; j += n) dsyn[b * ndata + j] = (which == 2 || set < 0) ? fill : dobs[j];
    if (m == 0) {
      U[b] = 0.0;
      flag[b] = 0;
    }
  }
}

// Holds a stream for about `ns` nanoseconds (one warp).  Launched ahead of the RF branch of a joint
// evaluation: the RF kernels have grids of thousands of 255-register blocks, the root search one
// partial wave of latency-bound blocks; whichever is placed first keeps the SMs, and the search has to
// be first (10.6 instead of 8.0 ms per step when the RF kernels win the race).
__global__ void rf_branch_hold_kernel(unsigned ns) {
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  do {
    __nanosleep(1000);
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
  } while (t1 - t0 < ns);
}

}  // namespace rfs
