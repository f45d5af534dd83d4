// __global__ kernels of the SWD path and the host-side "plan" that maps the reference's four
// wave types (Rc, Rg, Lc, Lg; /root/reference/src/SWD/surfdisp.cpp:190-297) onto unique
// period sequences and eigen solves.
#pragma once
#include "swd_love.cuh"
#include "swd_rayleigh.cuh"
#include "swd_roots.cuh"
#include "swd_plan.cuh"

namespace rfs {

// ---- model preparation: x=[vs(n),thk(n)] -> Brocher vp/rho (+derivatives) and the two model
// blocks.  Follows model/model_surf.py:47-79 and model/model_rf.py:52-77 (same polynomials) and
// the float32 cast at the SWD boundary (src/SWD/main.cpp:7-9).
// P = 3 (rfs_config_param RFS_PARAM_VS_THK_VPVS): x=[vs(n),thk(n),k(n)] with vp = k vs, rho = Brocher(vp).
// swd  : [SWD_NF][n][B]  float32-rounded values stored as double
// rfm  : [4][n][B]       thk, rho, vp, vs in float64 (RF argument order)
// chain: [P][n][B]       dadb, drda (P = 3: dadb = k, then dadk = vs)
template <int P>
__global__ void prep_models_kernel(const double *__restrict__ x, long long B, int n,
                                   double *__restrict__ swd, double *__restrict__ rfm,
                                   double *__restrict__ chain) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * n) return;
  const long long b = i % B;
  const int m = (int)(i / B);
  const double vs = x[b * P * n + m], thk = x[b * P * n + n + m];
  double vp, dadb;
  if (P == 3) {
    dadb = x[b * P * n + 2 * n + m];
    vp = dadb * vs;
  } else {
    vp = 0.9409 + 2.0947 * vs - 0.8206 * (vs * vs) + 0.2683 * (vs * vs * vs) - 0.0251 * (vs * vs * vs * vs);
    dadb = 2.0947 - 0.8206 * 2 * vs + 0.2683 * 3 * (vs * vs) - 0.0251 * 4 * (vs * vs * vs);
  }
  const double rho = 1.6612 * vp - 0.4721 * (vp * vp) + 0.0671 * (vp * vp * vp) -
                     0.0043 * (vp * vp * vp * vp) + 0.000106 * (vp * vp * vp * vp * vp);
  const double drda = 1.6612 - 0.4721 * 2 * vp + 0.0671 * 3 * (vp * vp) -
                      0.0043 * 4 * (vp * vp * vp) + 0.000106 * 5 * (vp * vp * vp * vp);
  const long long nb = (long long)n * B;
  if (swd) {
    const double d32 = (double)(float)thk, a32 = (double)(float)vp, b32 = (double)(float)vs,
                 r32 = (double)(float)rho;
    swd[F_D * nb + m * B + b] = d32;
    swd[F_A * nb + m * B + b] = a32;
    swd[F_B * nb + m * B + b] = b32;
    swd[F_RHO * nb + m * B + b] = r32;
    swd[F_IA * nb + m * B + b] = 1.0 / a32;
    swd[F_IB * nb + m * B + b] = 1.0 / b32;
    swd[F_IRHO * nb + m * B + b] = 1.0 / r32;
    swd[F_VTP * nb + m * B + b] = 1.0;
    swd[F_DTP * nb + m * B + b] = 1.0;
    swd[F_RTP * nb + m * B + b] = 1.0;
  }
  if (rfm) {
    rfm[0 * nb + m * B + b] = thk;
    rfm[1 * nb + m * B + b] = rho;
    rfm[2 * nb + m * B + b] = vp;
    rfm[3 * nb + m * B + b] = vs;
  }
  if (chain) {
    chain[0 * nb + m * B + b] = dadb;
    chain[1 * nb + m * B + b] = drda;
    if (P == 3) chain[2 * nb + m * B + b] = vs;
  }
}

// ---- earth flattening (sphere=True): build the four flattened model blocks from the flat one.
// One thread per model (the transform accumulates depth layer by layer).
//   root blocks: surfdisp96.f `sphere` (:495-564) — float32 arrays, radius 6370, density exponent
//                -2.275 (Rayleigh) / -5 (Love) applied to the float32 btp;
//   eig blocks : sregn96.f90 `bldsph` (:133-187, radius 6371, rho*tmp^-2.275) and
//                slegn96.f90 `bldsph` (:107-167, rho*tmp^-5), float64 on the float32-cast inputs,
//                plus the factors vtp, dtp, rtp used by sprayl/splove and sregnpu/slegnpu.
__global__ void prep_sphere_kernel(const double *__restrict__ flat, long long B, int n,
                                   double *__restrict__ rootR, double *__restrict__ rootL,
                                   double *__restrict__ eigR, double *__restrict__ eigL) {
  const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (b >= B) return;
  const long long nb = (long long)n * B;
  auto at = [&](int f, int m) { return ((long long)f * n + m) * B + b; };
  // ---- surfdisp96 sphere(): ar = 6370, d(mmax) = 1 while accumulating
  {
    const double ar = 6370.0;
    double dr = 0.0, r0 = ar;
    for (int i = 0; i < n; i++) {
      const float d = (i == n - 1) ? 1.0f : (float)flat[at(F_D, i)];
      const float a = (float)flat[at(F_A, i)], bb = (float)flat[at(F_B, i)], rho = (float)flat[at(F_RHO, i)];
      dr = dr + (double)d;
      const double r1 = ar - dr;
      const double z0 = ar * log(ar / r0), z1 = ar * log(ar / r1);
      const float dn = (i == n - 1) ? 0.0f : (float)(z1 - z0);
      const double tmp = (ar + ar) / (r0 + r1);
      const float an = (float)((double)a * tmp), bn = (float)((double)bb * tmp);
      const float btp = (float)tmp;
      const float b5 = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(btp, btp), btp), btp), btp);
      const float rhoL = __fmul_rn(rho, __fdiv_rn(1.0f, b5));
      const float rhoR = __fmul_rn(rho, powf(btp, -2.275f));
      double *dst[2] = {rootR, rootL};
      const float rr[2] = {rhoR, rhoL};
      for (int f = 0; f < 2; f++) {
        double *o = dst[f];
        o[at(F_D, i)] = (double)dn;
        o[at(F_A, i)] = (double)an;
        o[at(F_B, i)] = (double)bn;
        o[at(F_RHO, i)] = (double)rr[f];
        o[at(F_IA, i)] = 1.0 / (double)an;
        o[at(F_IB, i)] = 1.0 / (double)bn;
        o[at(F_IRHO, i)] = 1.0 / (double)rr[f];
        o[at(F_VTP, i)] = 1.0;
        o[at(F_DTP, i)] = 1.0;
        o[at(F_RTP, i)] = 1.0;
      }
      r0 = r1;
    }
  }
  // ---- bldsph (both wave types): ar = 6371, last layer counts 1 km while accumulating
  {
    const double ar = 6371.0;
    double dr = 0.0, r0 = ar;
    for (int i = 0; i < n; i++) {
      const double zd = (i == n - 1) ? 1.0 : flat[at(F_D, i)];
      dr = dr + zd;
      const double r1 = ar - dr;
      const double z0 = ar * log(ar / r0), z1 = ar * log(ar / r1);
      const double tmp = (2.0 * ar) / (r0 + r1);
      const double dtp = ar / r0;
      const double rtpR = pow(tmp, (double)(-2.275f));
      const double t2 = tmp * tmp;
      const double rtpL = 1.0 / (t2 * t2 * tmp);
      const double dn = (i == n - 1) ? 0.0 : z1 - z0;
      const double a = flat[at(F_A, i)] * tmp, bb = flat[at(F_B, i)] * tmp, rho = flat[at(F_RHO, i)];
      double *dst[2] = {eigR, eigL};
      const double rt[2] = {rtpR, rtpL};
      for (int f = 0; f < 2; f++) {
        double *o = dst[f];
        o[at(F_D, i)] = dn;
        o[at(F_A, i)] = a;
        o[at(F_B, i)] = bb;
        o[at(F_RHO, i)] = rho * rt[f];
        o[at(F_IA, i)] = 1.0 / a;
        o[at(F_IB, i)] = 1.0 / bb;
        o[at(F_IRHO, i)] = 1.0 / (rho * rt[f]);
        o[at(F_VTP, i)] = tmp;
        o[at(F_DTP, i)] = dtp;
        o[at(F_RTP, i)] = rt[f];
      }
      r0 = r1;
    }
  }
  (void)nb;
}

// sequential stop rule of the retry loop: `if(ierr !=0) return ierr;` leaves the later periods
// un-retried (zero) and reports failure; otherwise ierr is that of the last retry (0).
__global__ void swd_retry_finish_kernel(SwdPlan plan, SwdSetView sv, long long B, int all_modes,
                                        double *__restrict__ croot, int *__restrict__ ierr,
                                        const int *__restrict__ rstat) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * plan.nseq) return;
  const long long b = i % B;
  const int s = (int)(i / B);
  if (ierr[(long long)s * B + b] == 0) return;
  const SwdSeq sq = sv.seq(plan, s, b);  // only row b's own periods were searched
  double *clast = croot + (all_modes ? (long long)(plan.nmode - 1) * plan.nsolve * B : 0);
  int e = 1;  // ierr stays 1 if nothing was retried (cannot happen: a failed period is zero)
  bool stopped = false;
  for (int k = 0; k < sq.nper; k++) {
    const long long o = (long long)(sq.out_off + k) * B + b;
    const int r = rstat[o];
    if (r < 0) continue;
    if (stopped) {
      clast[o] = 0.0;  // the reference never retried this period
      continue;
    }
    e = r;
    if (r != 0) stopped = true;
  }
  ierr[(long long)s * B + b] = e;
}

// ---- K2: one thread per (model, solve=(sequence,period)[, mode])
// ugr  : [nmode_out][nsolve][B]     kern : [nmode_out][nsolve][4][n][B]
#ifndef RFS_EIGEN_MINBLOCKS
#define RFS_EIGEN_MINBLOCKS 3
#endif
template <int NMAX>
__global__ void __launch_bounds__(128, RFS_EIGEN_MINBLOCKS)
    swd_eigen_kernel(SwdPlan plan, SwdBlocks blk, SwdSetView setv, long long B, int n,
                     const double *__restrict__ periods, int nmode_out,
                     const double *__restrict__ croot, double *__restrict__ ugr,
                     double *__restrict__ kern) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long tot = B * plan.nsolve * nmode_out;
  if (i >= tot) return;
  const long long b = i % B;
  const long long sv = i / B;  // mode * nsolve + solve
  const int solve = (int)(sv % plan.nsolve);
  // find the sequence of this solve
  int s = 0;
  for (int q = 0; q < plan.nseq; q++)
    if (solve >= plan.seq[q].out_off && solve < plan.seq[q].out_off + plan.seq[q].nper) s = q;
  const SwdSeq sq = setv.seq(plan, s, b);
  const int k = solve - sq.out_off;
  if (k >= sq.nper) return;  // beyond row b's own period list: no root, nothing reads this solve
  const double T = __ldg(periods + sq.per_off + k) * sq.scale;
  const double c = croot[sv * B + b];
  double *kp = kern + sv * 4 * (long long)n * B + b;
  SwdModel M(blk.eig[sq.ifunc == 2 ? 0 : 1], B, n);
  double u;
  if (!(c > 0.0)) {
    // mode does not exist at this period (reference: c = 0 -> NaN kernels downstream, SURVEY Q18)
    const double qnan = nan("");
    for (int j = 0; j < 4 * n; j++) kp[(long long)j * B] = qnan;
    u = qnan;
  } else if (sq.ifunc == 2) {
    if constexpr (NMAX <= 8) {
      // up-sweep vectors of the block in shared memory: [NMAX*6][blockDim.x] doubles (48 KB at 128 threads)
      extern __shared__ double eig_cd[];
      rayleigh_solve<NMAX, true>(M, b, T, c, &u, kp, B, eig_cd + threadIdx.x, (int)blockDim.x);
    } else {
      rayleigh_solve<NMAX, false>(M, b, T, c, &u, kp, B);
    }
  } else {
    love_solve<NMAX>(M, b, T, c, &u, kp, B);
  }
  ugr[sv * B + b] = u;
}

// value + 4 kernels of data row `r`, period k, layer m for model b (drop-in adjoint_kernel
// semantics, surfdisp.cpp:209-294 + sregnpu/slegnpu combination sregn96.f90:1839-1844).
// Returns the datum (phase or group velocity); K[0..3] = d/d(vp,vs,rho,thk).
struct SwdView {
  const double *croot, *ugr, *kern;  // already offset to the reported mode
  const double *periods;
  long long B;
  int n;
  SwdBlocks blk;   // eig[f] carries vtp/dtp/rtp when blk.sphere
  int fwd;         // 1: libsurf.forward semantics (phase velocity through _flat2sphere)
};
// sphericity factor tm of sprayl/splove/sregnpu/slegnpu (float32 pi, radius 6371)
RFS_DEVINL double sph_tm(int love, double t, double c) {
  const double om = (2.0 * RFS_PI32) / t;
  const double x = love ? 3.0 * c / (2. * 6371.0 * om) : c / (2. * 6371.0 * om);
  return sqrt(1. + x * x);
}
RFS_DEVINL double swd_row_value(const SwdPlan &plan, const SwdView &V, const SwdRow &rw, int k,
                                long long b) {
  const int sv0 = plan.seq[rw.s0].out_off + k;
  const double c = V.croot[(long long)sv0 * V.B + b];
  const int love = rw.type >= 2;
  if (rw.type == 0 || rw.type == 2) {
    if (!V.blk.sphere) return c;
    const double t = V.periods[rw.per_off + k];
    if (V.fwd) {
      // _flat2sphere (surfdisp.cpp:16-49): double pi
      const double om = 2.0 * RFS_PI64 / t;
      const double x = (love ? 1.5 : 0.5) * c / (6371.0 * om);
      return c / sqrt(1. + x * x);
    }
    return c / sph_tm(love, t, c);  // csph of sprayl / splove
  }
  const double u = V.ugr[(long long)sv0 * V.B + b];
  if (!V.blk.sphere) return u;
  return u * sph_tm(love, V.periods[rw.per_off + k], c);
}
RFS_DEVINL void swd_row_kernels(const SwdPlan &plan, const SwdView &V, const SwdRow &rw, int k,
                                int m, long long b, int stale, double K[4]) {
  const long long nB = (long long)V.n * V.B;
  const int sv0 = plan.seq[rw.s0].out_off + k;
  const double *k0 = V.kern + (long long)sv0 * 4 * nB + (long long)m * V.B + b;
  const int love = rw.type >= 2;
  double fvt = 1.0, frt = 1.0;
  if (V.blk.sphere) {
    const double *e = V.blk.eig[love];
    fvt = e[((long long)F_VTP * V.n + m) * V.B + b];
    frt = e[((long long)F_RTP * V.n + m) * V.B + b];
  }
  const double t = V.periods[rw.per_off + k];
  const double cp = V.croot[(long long)sv0 * V.B + b];
  if (rw.type == 0 || rw.type == 2) {
    for (int p = 0; p < 4; p++) K[p] = k0[p * nB];
    if (V.blk.sphere) {
      // sprayl (sregn96.f90:1619-1626) / splove: kernels of the ORIGINAL spherical model
      const double tm = sph_tm(love, t, cp);
      const double i3 = 1.0 / (tm * tm * tm);
      K[0] = K[0] * fvt * i3;
      K[1] = K[1] * fvt * i3;
      K[2] = K[2] * frt * i3;
      K[3] = K[3] * i3;  // dtp is already inside the suffix sum
    }
    return;
  }
  const int sv1 = plan.seq[rw.s1].out_off + k, sv2 = plan.seq[rw.s2].out_off + k;
  const double *k1 = V.kern + (long long)sv1 * 4 * nB + (long long)m * V.B + b;
  const double *k2 = V.kern + (long long)sv2 * 4 * nB + (long long)m * V.B + b;
  const double t1 = t * (1.0 + 0.05), t2 = t * (1.0 - 0.05);
  const double cg = V.ugr[(long long)sv0 * V.B + b];
  const double uc1 = cg / cp;
  double tm = 1.0, tm1 = 0.0;
  if (V.blk.sphere) {
    // sregnpu :1847-1868 / slegnpu :881-899
    tm = sph_tm(love, t, cp);
    const double om = (2.0 * RFS_PI32) / t;
    const double y = (love ? 1.5 : 0.5) / (6371.0 * om);
    tm1 = y * y / tm;
  }
  for (int p = 0; p < 4; p++) {
    const double first = stale ? k2[p * nB] : k0[p * nB];
    double du = uc1 * (2.0 - uc1) * first - uc1 * uc1 * t * (k2[p * nB] - k1[p * nB]) / (t2 - t1);
    if (V.blk.sphere) {
      const double f = (p == 2) ? frt : (p == 3 ? 1.0 : fvt);
      du = (tm * du + cg * cp * k0[p * nB] * tm1) * f;
    }
    K[p] = du;
  }
  if (rw.type == 3) K[0] = 0.0;
}

// Materialise the drop-in outputs of libsurf.adjoint_kernel for one row:
//   c[B][nper], dcda/dcdb/dcdr/dcdh [B][nper][n]  (row-major per model, as the pybind returns)
__global__ void swd_export_row_kernel(SwdPlan plan, int r, SwdView V, int stale,
                                      double *__restrict__ c, double *__restrict__ dcda,
                                      double *__restrict__ dcdb, double *__restrict__ dcdr,
                                      double *__restrict__ dcdh) {
  const SwdRow rw = plan.row[r];
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long tot = V.B * rw.nper * V.n;
  if (i >= tot) return;
  const long long b = i % V.B;
  const long long km = i / V.B;
  const int m = (int)(km % V.n);
  const int k = (int)(km / V.n);
  if (m == 0) c[b * rw.nper + k] = swd_row_value(plan, V, rw, k, b);
  if (dcda) {
    double K[4];
    swd_row_kernels(plan, V, rw, k, m, b, stale, K);
    const long long o = (b * rw.nper + k) * V.n + m;
    dcda[o] = K[0];
    dcdb[o] = K[1];
    dcdr[o] = K[2];
    dcdh[o] = K[3];
  }
}

}  // namespace rfs
