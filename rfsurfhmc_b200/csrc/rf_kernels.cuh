// K3 + K4 — receiver functions: Haskell-propagator response per (model, frequency bin) and the
// shared-memory FFT / water-level deconvolution / adjoint gradient per model.
//
// Replaces /root/reference/src/RF/RFModule.f90: cal_rf_freq :193-255, cal_rf_par_freq :258-341,
// cal_rf_par_freq_all :343-430, cal_response :432-478, cal_response_par(_all) :481-707,
// cal_matrix_a :709-764, cal_matrix_a_par :766-879, cal_E_inv :881-922, cal_E_inv_par :924-987,
// and /root/reference/src/RF/fftpack.f90 (FFTW r2c/c2r -> hand-written radix-2 smem FFT).
//
// Re-design (same mathematics, different schedule):
//  * O(n) instead of O(n^2) products per frequency: only one row of E^-1 A(n-1)..A(1) and two
//    columns are consumed (RFModule.f90:653-659), so a bottom-up pass stores the 1x4 suffix rows
//    l_j = e_r^T E^-1 A(n-1)..A(j+1) and a top-down pass carries the 4x2 prefix block
//    r_j = A(j-1)..A(1)[:,1:2]; d/dq_j = l_j (dA_j/dq) r_j.
//  * all layer matrices share the pattern m24=-m13, m33=m22, m34=-m12, m42=-m31, m43=-m21,
//    m44=m11, so 10 instead of 16 entries are formed.
//  * fused misfit+gradient: grad_j = sum_it r[it] K_j[it] is evaluated in the frequency domain
//    from ONE forward FFT of the weighted residual (adjoint form) instead of 4n inverse FFTs;
//    the Brocher chain rule (model/model_rf.py:189) is applied to the spectra.
#pragma once
#include "common.cuh"

namespace rfs {

struct M10 {
  cd m11, m12, m13, m14, m21, m22, m23, m31, m32, m41;
};
RFS_DEVINL void rowmul(const cd l[4], const M10 &M, cd v[4]) {
  v[0] = l[0] * M.m11 + l[1] * M.m21 + l[2] * M.m31 + l[3] * M.m41;
  v[1] = l[0] * M.m12 + l[1] * M.m22 + l[2] * M.m32 - l[3] * M.m31;
  v[2] = l[0] * M.m13 + l[1] * M.m23 + l[2] * M.m22 - l[3] * M.m21;
  v[3] = l[0] * M.m14 - l[1] * M.m13 - l[2] * M.m12 + l[3] * M.m11;
}
RFS_DEVINL void colmul(const M10 &M, const cd r[4], cd o[4]) {
  o[0] = M.m11 * r[0] + M.m12 * r[1] + M.m13 * r[2] + M.m14 * r[3];
  o[1] = M.m21 * r[0] + M.m22 * r[1] + M.m23 * r[2] - M.m13 * r[3];
  o[2] = M.m31 * r[0] + M.m32 * r[1] + M.m22 * r[2] - M.m12 * r[3];
  o[3] = M.m41 * r[0] - M.m31 * r[1] - M.m21 * r[2] + M.m11 * r[3];
}
RFS_DEVINL void scale10(M10 &M, cd s) {
  M.m11 = M.m11 * s;
  M.m12 = M.m12 * s;
  M.m13 = M.m13 * s;
  M.m14 = M.m14 * s;
  M.m21 = M.m21 * s;
  M.m22 = M.m22 * s;
  M.m23 = M.m23 * s;
  M.m31 = M.m31 * s;
  M.m32 = M.m32 * s;
  M.m41 = M.m41 * s;
}

// frequency-independent layer constants; computed once per (model, layer) by rf_layer_kernel and
// read (warp-broadcast, L1-resident) by every frequency bin instead of being re-derived per bin
struct RfLayer {
  cd alpha, beta, miu, gamma, gamma1, va_k, vb_k;
  // reciprocals used by the layer matrices and their derivatives
  cd ialpha, ibeta, ivak, ivbk, imu2, g3, g2, ivak2;  // 1/alpha 1/beta 1/va_k 1/vb_k 1/(2mu) 1/(g-2) g/(alpha p)^2 1/va_k^2
  cd bvs, avp;                                        // beta/vs, alpha/vp (complex -> real velocity factors)
  double thick, rho, vp, vs;
};
static_assert(sizeof(RfLayer) == 38 * sizeof(double), "RfLayer is read as 19 double2");
RFS_DEVINL RfLayer rf_layer(double thick, double rho, double vp, double vs, double qa, double qb,
                            double p) {
  RfLayer L;
  L.thick = thick;
  L.rho = rho;
  L.vp = vp;
  L.vs = vs;
  L.alpha = vp * cd(1.0 + 1.0 / (8.0 * qa * qa), 1.0 / (2.0 * qa));
  L.beta = vs * cd(1.0 + 1.0 / (8.0 * qb * qb), 1.0 / (2.0 * qb));
  const cd b2 = L.beta * L.beta;
  L.miu = rho * b2;
  L.gamma = (2.0 * p * p) * b2;
  L.gamma1 = 1.0 - cinv(L.gamma);
  L.va_k = csqrt(p * p - cinv(L.alpha * L.alpha)) / p;
  L.vb_k = csqrt(p * p - cinv(b2)) / p;
  L.ialpha = cinv(L.alpha);
  L.ibeta = cinv(L.beta);
  L.ivak = cinv(L.va_k);
  L.ivbk = cinv(L.vb_k);
  L.imu2 = cinv(2.0 * L.miu);
  L.g3 = cinv(L.gamma - 2.0);
  const cd ap = L.alpha * p;
  L.g2 = L.gamma * cinv(ap * ap);
  L.ivak2 = cinv(L.va_k * L.va_k);
  L.bvs = L.beta / vs;
  L.avp = L.alpha / vp;
  return L;
}
// Ray parameter of each row in pass `ir` of an RF objective: ray_p[set[b]][ir] of a per-set table, or
// the shared value.  set points at the rows of this launch (NULL: every row is set 0).  A row whose set
// index lies outside [0, nsets) reads nothing from the table and computes with the shared value; the
// residual kernels fail that row (ObsSets::row_set), so no NaN spectrum reaches the spike picking.
struct RayView {
  const double *tab;  // [nsets][nray] or NULL (every row uses `shared`)
  const int *set;     // [B] or NULL
  int nsets, nray, ir;
  double shared;
  RFS_DEVINL double row_p(long long b) const {
    if (!tab) return shared;
    const int s = set ? set[b] : 0;
    return (s >= 0 && s < nsets) ? tab[s * nray + ir] : shared;
  }
};

// Layer constants of row b, layer m, for ray parameter p.  Not inlined, so that p reaches rf_layer as a
// function parameter, as the ray parameter did when it was a kernel argument: inlined next to the table
// lookup, the compiler shares rf_layer's products between their uses and contracts multiply-add pairs
// differently (rf_layer_kernel: 172 instead of 173 DFMA), which changes the last bits of every RF result.
__device__ __noinline__ void rf_layer_row(const double *__restrict__ rfm, const double *__restrict__ qa,
                                          const double *__restrict__ qb, long long B, int n, long long b, int m,
                                          double p, RfLayer *__restrict__ tab) {
  const long long nB = (long long)n * B;
  const double qam = qa ? qa[m * B + b] : 9999.0, qbm = qb ? qb[m * B + b] : 9999.0;
  tab[b * n + m] = rf_layer(rfm[0 * nB + m * B + b], rfm[1 * nB + m * B + b],
                            rfm[2 * nB + m * B + b], rfm[3 * nB + m * B + b], qam, qbm, p);
}
// one thread per (model, layer): rfm [4][n][B] thk, rho, vp, vs -> tab [B][n] RfLayer
__global__ void rf_layer_kernel(const double *__restrict__ rfm, const double *__restrict__ qa,
                                const double *__restrict__ qb, long long B, int n, RayView ray,
                                RfLayer *__restrict__ tab) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * n) return;
  const long long b = i % B;
  rf_layer_row(rfm, qa, qb, B, n, b, (int)(i / B), ray.row_p(b), tab);
}
RFS_DEVINL RfLayer rf_layer_ld(const RfLayer *__restrict__ tab, long long idx) {
  RfLayer L;
  const double2 *src = reinterpret_cast<const double2 *>(tab + idx);
  double2 *dst = reinterpret_cast<double2 *>(&L);
#pragma unroll
  for (int j = 0; j < 19; j++) dst[j] = __ldg(src + j);
  return L;
}

struct RfTrig {
  cd c_a, x_a, y_a, c_b, x_b, y_b;
  cd v_a, v_b;  // vertical wavenumbers (reused by the derivative pass)
};
RFS_DEVINL void ccoshsinh(cd z, cd &ch, cd &sh) {
  // cosh(x+iy) = cosh x cos y + i sinh x sin y ; sinh(x+iy) = sinh x cos y + i cosh x sin y
  double s, c;
  sincos(z.y, &s, &c);
  // one exponential for cosh and sinh; sinh by its series below 0.5 (no cancellation)
  const double ax = fabs(z.x);
  const double e = exp_cb(fmin(ax, 700.0)), ei = 1.0 / e;
  const double chx = 0.5 * (e + ei);
  double shx;
  if (ax < 0.5) {
    const double x2 = ax * ax;
    double q = fma(x2, 1.6059043836821613e-10, 2.5052108385441720e-08);  // 1/13!, 1/11!
    q = fma(x2, q, 2.7557319223985893e-06);                              // 1/9!
    q = fma(x2, q, 1.9841269841269841e-04);                              // 1/7!
    q = fma(x2, q, 8.3333333333333332e-03);                              // 1/5!
    q = fma(x2, q, 1.6666666666666666e-01);                              // 1/3!
    shx = fma(ax * x2, q, ax);
  } else {
    shx = 0.5 * (e - ei);
  }
  shx = copysign(shx, z.x);
  ch = cd(chx * c, shx * s);
  sh = cd(shx * c, chx * s);
}
RFS_DEVINL void rf_trig(const RfLayer &L, cd omega, double p, cd &k, cd &v_alpha, cd &v_beta,
                        RfTrig &t) {
  k = omega * p;
  const cd k_alpha = omega * L.ialpha, k_beta = omega * L.ibeta;
  v_alpha = csqrt(k * k - k_alpha * k_alpha);
  v_beta = csqrt(k * k - k_beta * k_beta);
  cd ch, sh;
  ccoshsinh(v_alpha * L.thick, ch, sh);
  t.c_a = ch;
  t.x_a = L.va_k * sh;
  t.y_a = sh * L.ivak;
  ccoshsinh(v_beta * L.thick, ch, sh);
  t.c_b = ch;
  t.x_b = L.vb_k * sh;
  t.y_b = sh * L.ivbk;
  t.v_a = v_alpha;
  t.v_b = v_beta;
}

// cal_matrix_a (:709-764)
RFS_DEVINL void rf_mat_a(const RfLayer &L, const RfTrig &t, M10 &A) {
  const cd g1 = L.gamma1, mu2 = 2.0 * L.miu, imu2 = L.imu2;
  A.m11 = t.c_a - g1 * t.c_b;
  A.m12 = g1 * t.y_a - t.x_b;
  A.m13 = (t.c_b - t.c_a) * imu2;
  A.m14 = (t.x_b - t.y_a) * imu2;
  A.m21 = g1 * t.y_b - t.x_a;
  A.m22 = t.c_b - g1 * t.c_a;
  A.m23 = (t.x_a - t.y_b) * imu2;
  A.m31 = mu2 * g1 * (t.c_a - t.c_b);
  A.m32 = mu2 * (g1 * g1 * t.y_a - t.x_b);
  A.m41 = mu2 * (g1 * g1 * t.y_b - t.x_a);
  scale10(A, L.gamma);
}

// cal_matrix_a_par (:766-879), including the complex->real velocity factors (:624-628)
RFS_DEVINL void rf_mat_a_par(const RfLayer &L, const RfTrig &t, cd k, cd v_alpha, cd v_beta,
                             double p, int ipar, M10 &D) {
  const cd g = L.gamma, g1 = L.gamma1, miu = L.miu;
  const cd kt = k * L.thick;
  if (ipar == 3) {
    const cd g3 = L.g3;
    const cd ib = L.ibeta;
    const cd ktcb_p = kt * t.c_b + t.y_b, ktcb_m = kt * t.c_b - t.y_b, ktyb = kt * t.y_b;
    const cd imb = (2.0 * L.imu2) * ib;
    D.m11 = (2.0 * ib) * (g * (t.c_a - t.c_b) - g1 * ktyb);
    D.m12 = (2.0 * ib) * (g * (t.y_a - t.x_b) - ktcb_p);
    D.m13 = ktyb * imb;
    D.m14 = ktcb_p * imb;
    D.m21 = ((t.y_b - t.x_a) + g1 * g3 * ktcb_m) * (2.0 * g * ib);
    D.m22 = (2.0 * ib) * (g * (t.c_b - t.c_a) + ktyb);
    D.m23 = -1.0 * (ktcb_m * g * g3 * imb);
    D.m31 = (4.0 * miu * ib) * ((2.0 * g - 1.0) * (t.c_a - t.c_b) - g1 * ktyb);
    D.m32 = (4.0 * miu * ib) * ((2.0 * g) * (g1 * t.y_a - t.x_b) - ktcb_p);
    D.m41 = (4.0 * miu * g * ib) * (2.0 * g1 * t.y_b - 2.0 * t.x_a + g1 * g1 * g3 * ktcb_m);
    scale10(D, L.bvs);
  } else if (ipar == 2) {
    const cd g2 = L.g2;
    const cd ia = L.ialpha;
    const cd ivak2 = L.ivak2;
    const cd ktya = kt * t.y_a, ktca_m = kt * t.c_a - t.y_a, ktca_p = kt * t.c_a + t.y_a;
    const cd i2m = L.imu2;
    D.m11 = ktya * g2 * ia;
    D.m12 = ivak2 * ia * g1 * g2 * ktca_m;
    D.m13 = -1.0 * (ktya * g2 * i2m * ia);
    D.m14 = -1.0 * (ivak2 * ktca_m * g2 * i2m * ia);
    D.m21 = -1.0 * (ktca_p * g2 * ia);
    D.m22 = -1.0 * (ktya * g1 * g2 * ia);
    D.m23 = ktca_p * g2 * i2m * ia;
    D.m31 = ktya * g1 * g2 * (2.0 * miu) * ia;
    D.m32 = (2.0 * miu * ia) * (g1 * g1) * g2 * ktca_m * ivak2;
    D.m41 = -1.0 * ((2.0 * miu * ia) * ktca_p * g2);
    scale10(D, L.avp);
  } else if (ipar == 1) {
    const cd f = -1.0 * (g * L.imu2) / L.rho;
    const cd h = (2.0 / L.rho) * (miu * g);
    D.m11 = cd(0.0);
    D.m12 = cd(0.0);
    D.m21 = cd(0.0);
    D.m22 = cd(0.0);
    D.m13 = f * (t.c_b - t.c_a);
    D.m14 = f * (t.x_b - t.y_a);
    D.m23 = f * (t.x_a - t.y_b);
    D.m31 = h * g1 * (t.c_a - t.c_b);
    D.m32 = h * (g1 * g1 * t.y_a - t.x_b);
    D.m41 = h * (g1 * g1 * t.y_b - t.x_a);
  } else {
    const cd i2m = L.imu2, mu2 = 2.0 * miu;
    const cd vbb = v_beta * L.vb_k, vaa = v_alpha * L.va_k;
    D.m11 = (t.x_a - g1 * t.x_b) * k;
    D.m12 = g1 * k * t.c_a - vbb * t.c_b;
    D.m13 = (t.x_b - t.x_a) * k * i2m;
    D.m14 = (vbb * t.c_b - k * t.c_a) * i2m;
    D.m21 = g1 * k * t.c_b - vaa * t.c_a;
    D.m22 = (t.x_b - g1 * t.x_a) * k;
    D.m23 = (vaa * t.c_a - k * t.c_b) * i2m;
    D.m31 = mu2 * g1 * k * (t.x_a - t.x_b);
    D.m32 = mu2 * (g1 * g1 * k * t.c_a - vbb * t.c_b);
    D.m41 = mu2 * (g1 * g1 * k * t.c_b - vaa * t.c_a);
    scale10(D, g);
  }
}

RFS_DEVINL cd nan0(cd z) { return (isnan(z.x) || isnan(z.y)) ? cd(0.0, 0.0) : z; }

// ---- K3: one thread per (model, frequency bin)
//  rfm  : [4][n][B] thk, rho, vp, vs (float64)     chain: [NQ][n][B] dadb, drda, dadk (NQ==2,3 only)
//  qa,qb: [n][B] or NULL (=> 9999)
//  spec : [B][2][n2] complex  (R21, R22)
//  dspec: [B][NQ*n][n2] complex  D = R22_m R21 - R21_m R22
//         NQ==4: rows rho,vp,vs,h (kernel_all order);  NQ==2: rows vs-chain, thk;
//         NQ==3: rows vs-chain, thk, k-chain (x = [vs, thk, Vp/Vs])
//  sigma: imaginary part of omega is -sigma (freq method) or 0 (time method)
#ifndef RFS_RF_MINBLOCKS
#define RFS_RF_MINBLOCKS 2
#endif
template <int NMAX, int NQ>
__global__ void __launch_bounds__(128, RFS_RF_MINBLOCKS)
    rf_propagate_kernel(const RfLayer *__restrict__ tab, const double *__restrict__ chain,
                        long long B, int n, int n2, int nft, double dt, RayView ray, double sigma,
                        double pi_used, int rf_type, double2 *__restrict__ spec,
                        double2 *__restrict__ dspec) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * n2) return;
  const long long b = i / n2;
  const int kf = (int)(i % n2);
  const long long nB = (long long)n * B;
  // pi_used: float32 pi everywhere except cal_rf_par_time_all (RFModule.f90:94 uses atan(1.0_dp))
  const double w = 1.0 / nft / dt * kf * 2.0 * pi_used;
  const cd omega(w, -sigma);
  const double p = ray.row_p(b);
  const int row = (rf_type == 1) ? 1 : 0;

  cd Ls[NMAX * 4];       // suffix rows l_j
  RfTrig Ts[NMAX];       // cosh/sinh terms of each layer (reused by the top-down pass)

  // ---- half-space row of E^-1 (cal_E_inv :881-922)
  cd l[4];
  {
    const int m = n - 1;
    const RfLayer L = rf_layer_ld(tab, b * n + m);
    const cd hg = 0.5 * L.gamma, i2m = L.imu2;
    if (row == 0) {
      const cd iv = L.ivak;
      l[0] = -1.0 * hg;
      l[1] = -1.0 * (hg * L.gamma1 * iv);
      l[2] = hg * i2m;
      l[3] = hg * i2m * iv;
    } else {
      const cd iv = L.ivbk;
      l[0] = hg * L.gamma1 * iv;
      l[1] = hg;
      l[2] = -1.0 * (hg * i2m * iv);
      l[3] = -1.0 * (hg * i2m);
    }
  }
  // ---- bottom-up: store l_j, then l <- l A_j
  for (int m = n - 2; m >= 0; m--) {
    const RfLayer L = rf_layer_ld(tab, b * n + m);
    cd k, va, vb;
    RfTrig t;
    rf_trig(L, omega, p, k, va, vb, t);
    Ts[m] = t;
    Ls[m * 4 + 0] = l[0];
    Ls[m * 4 + 1] = l[1];
    Ls[m * 4 + 2] = l[2];
    Ls[m * 4 + 3] = l[3];
    M10 A;
    rf_mat_a(L, t, A);
    cd v[4];
    rowmul(l, A, v);
    l[0] = v[0];
    l[1] = v[1];
    l[2] = v[2];
    l[3] = v[3];
  }
  cd R21, R22;
  if (rf_type == 1) {
    R22 = cd(0.0, 1.0) * l[1];
    R21 = l[0];
  } else {
    R22 = cd(0.0, -1.0) * l[0];
    R21 = l[1];
  }
  R22 = nan0(R22);
  R21 = nan0(R21);
  spec[(b * 2 + 0) * n2 + kf] = make_double2(R21.x, R21.y);
  spec[(b * 2 + 1) * n2 + kf] = make_double2(R22.x, R22.y);
  if (dspec == nullptr) return;

  // ---- top-down: r (4x2) and the parameter derivatives
  cd r0[4] = {cd(1.0), cd(0.0), cd(0.0), cd(0.0)};
  cd r1[4] = {cd(0.0), cd(1.0), cd(0.0), cd(0.0)};
  double2 *dout = dspec + (b * (long long)(NQ * n)) * n2 + kf;
  for (int m = 0; m < n; m++) {
    const RfLayer L = rf_layer_ld(tab, b * n + m);
    const cd k = omega * p;
    cd dR[4][2];  // per parameter (rho, vp, vs, h): derivative of (a(row,1), a(row,2))
    if (m < n - 1) {
      const RfTrig t = Ts[m];
      const cd va = t.v_a, vb = t.v_b;
      cd lj[4] = {Ls[m * 4 + 0], Ls[m * 4 + 1], Ls[m * 4 + 2], Ls[m * 4 + 3]};
#pragma unroll
      for (int q = 1; q <= 4; q++) {
        M10 D;
        rf_mat_a_par(L, t, k, va, vb, p, q, D);
        cd v[4];
        rowmul(lj, D, v);
        dR[q - 1][0] = v[0] * r0[0] + v[1] * r0[1] + v[2] * r0[2] + v[3] * r0[3];
        dR[q - 1][1] = v[0] * r1[0] + v[1] * r1[1] + v[2] * r1[2] + v[3] * r1[3];
      }
      M10 A;
      rf_mat_a(L, t, A);
      cd o[4];
      colmul(A, r0, o);
      r0[0] = o[0];
      r0[1] = o[1];
      r0[2] = o[2];
      r0[3] = o[3];
      colmul(A, r1, o);
      r1[0] = o[0];
      r1[1] = o[1];
      r1[2] = o[2];
      r1[3] = o[3];
    } else {
      // half-space: rows of dE^-1/dq (cal_E_inv_par :924-987; intended va_k formula :978-979)
      const cd k_alpha = omega * L.ialpha, k_beta = omega * L.ibeta;
      const cd va = csqrt(k * k - k_alpha * k_alpha), vb = csqrt(k * k - k_beta * k_beta);
      const cd gam = 2.0 * (k * k) * (L.beta * L.beta) / (omega * omega);
      const cd gam1 = 1.0 - cinv(gam);
      const cd gam3 = cinv(gam - 2.0);
      cd v[4][4];
      for (int q = 0; q < 4; q++)
        for (int c = 0; c < 4; c++) v[q][c] = cd(0.0);
      if (row == 0) {
        // beta
        const cd s3 = (gam / L.beta) * (L.beta / L.vs);
        v[2][0] = -1.0 * s3;
        v[2][1] = -1.0 * (k / va) * s3;
        // rho
        const cd s1 = gam / 4.0 / L.rho / L.miu;
        v[0][2] = -1.0 * s1;
        v[0][3] = -1.0 * (k / va) * s1;
        // alpha
        const cd s2 = (L.beta * L.beta) / (L.alpha * L.alpha * L.alpha) /
                      (L.va_k * L.va_k * L.va_k) * (L.alpha / L.vp);
        v[1][1] = gam1 * s2;
        v[1][3] = (-0.5 * cinv(L.miu)) * s2;
      } else {
        const cd s3 = (gam / L.beta) * (L.beta / L.vs);
        v[2][0] = (k / vb) * (1.0 - gam1 * gam3) * s3;
        v[2][1] = s3;
        v[2][2] = (k * gam3 / 2.0 / L.miu / vb) * s3;
        const cd s1 = gam / 4.0 / L.rho / L.miu;
        v[0][2] = (k / vb) * s1;
        v[0][3] = s1;
      }
      for (int q = 0; q < 4; q++) {
        dR[q][0] = v[q][0] * r0[0] + v[q][1] * r0[1] + v[q][2] * r0[2] + v[q][3] * r0[3];
        dR[q][1] = v[q][0] * r1[0] + v[q][1] * r1[1] + v[q][2] * r1[2] + v[q][3] * r1[3];
      }
    }
    // D_q = R22_m R21 - R21_m R22  (:416)
    cd Dq[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      cd r21m, r22m;
      if (rf_type == 1) {
        r22m = cd(0.0, 1.0) * dR[q][1];
        r21m = dR[q][0];
      } else {
        r22m = cd(0.0, -1.0) * dR[q][0];
        r21m = dR[q][1];
      }
      r22m = nan0(r22m);
      r21m = nan0(r21m);
      Dq[q] = r22m * R21 - r21m * R22;
    }
    if (NQ == 4) {
#pragma unroll
      for (int q = 0; q < 4; q++)
        dout[((long long)q * n + m) * n2] = make_double2(Dq[q].x, Dq[q].y);
    } else {
      // chain rule on spectra: kvs + dadb*kvp + drda*dadb*krho  (model_rf.py:189)
      const double dadb = chain[0 * nB + m * B + b], drda = chain[1 * nB + m * B + b];
      const cd Dv = Dq[2] + dadb * Dq[1] + (drda * dadb) * Dq[0];
      dout[((long long)0 * n + m) * n2] = make_double2(Dv.x, Dv.y);
      dout[((long long)1 * n + m) * n2] = make_double2(Dq[3].x, Dq[3].y);
      if (NQ == 3) {
        // Vp/Vs row (vp = k vs): dadk*kvp + drda*dadk*krho, dadk = vs
        const double dadk = chain[2 * nB + m * B + b];
        const cd Dk = dadk * Dq[1] + (drda * dadk) * Dq[0];
        dout[((long long)2 * n + m) * n2] = make_double2(Dk.x, Dk.y);
      }
    }
  }
}

// ------------------------------------------------------------------ shared-memory FFT
// Real <-> Hermitian transforms of length N (power of two) as ONE complex transform of length N/2
// (even/odd packing) with a Stockham autosort radix-4 schedule: log4(N/2) passes (plus one radix-2
// pass when log2(N/2) is odd), no bit-reversal pass, every pass reads a[j + r M/4] with unit stride
// over the threads.  Replaces FFTW's r2c / c2r plans of /root/reference/src/RF/fftpack.f90 (and the
// radix-2 + bit-reversal transform of round 1: half the butterflies, half the passes, a third of the
// barriers).  Unnormalised (FFTW convention).
// tw[j] = exp(-2 pi i j / N), j < N/2 (fft_twiddle_kernel): twiddles are looked up, never evaluated.
__global__ void fft_twiddle_kernel(int N, double2 *__restrict__ tw) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N / 2) return;
  double sn, cs;
  sincospi(-(double)j / (double)(N / 2), &sn, &cs);
  tw[j] = make_double2(cs, sn);
}
// exp(sign 2 pi i q / NT), 0 <= q < NT, from the half-circle table
template <bool TW_SMEM>
RFS_DEVINL cd tw_lookup(const double2 *__restrict__ tw, int q, int NT, int sign) {
  const int h = NT >> 1;
  const bool neg = q >= h;
  const int qq = neg ? q - h : q;
  const double2 t = TW_SMEM ? tw[qq] : __ldg(tw + qq);
  const cd w(t.x, sign < 0 ? t.y : -t.y);
  return neg ? cd(-w.x, -w.y) : w;
}
// Complex transform of length M = 2^logM, ping-pong between a and b (M entries each), executed by the
// whole block; `tw` is the table of length NT/2 for NT = 2M.  Returns the buffer holding the result
// (natural order).  sign = -1 forward (e^{-i..}), +1 backward.
template <bool TW_SMEM>
RFS_DEVINL cd *stockham_fft(cd *a, cd *b, int M, int logM, int sign, const double2 *__restrict__ tw,
                            int NT) {
  const int tid = threadIdx.x, nth = blockDim.x;
  int Ns = 1, lg = logM;
  while (lg >= 2) {
    const int q4 = M >> 2;
    const int tstep = NT / (4 * Ns);  // exp(sign 2 pi i r k / (4 Ns)) = table[r k tstep]
    for (int j = tid; j < q4; j += nth) {
      const int k = j & (Ns - 1);
      cd v0 = a[j], v1 = a[j + q4], v2 = a[j + 2 * q4], v3 = a[j + 3 * q4];
      if (k) {
        v1 = v1 * tw_lookup<TW_SMEM>(tw, k * tstep, NT, sign);
        v2 = v2 * tw_lookup<TW_SMEM>(tw, 2 * k * tstep, NT, sign);
        v3 = v3 * tw_lookup<TW_SMEM>(tw, 3 * k * tstep, NT, sign);
      }
      const cd s02 = v0 + v2, d02 = v0 - v2, s13 = v1 + v3, d13 = v1 - v3;
      const cd jd = (sign < 0) ? cd(d13.y, -d13.x) : cd(-d13.y, d13.x);  // -+ i (v1 - v3)
      const int j0 = ((j - k) << 2) + k;
      b[j0] = s02 + s13;
      b[j0 + Ns] = d02 + jd;
      b[j0 + 2 * Ns] = s02 - s13;
      b[j0 + 3 * Ns] = d02 - jd;
    }
    __syncthreads();
    cd *t = a;
    a = b;
    b = t;
    Ns <<= 2;
    lg -= 2;
  }
  if (lg == 1) {
    const int q2 = M >> 1;
    const int tstep = NT / (2 * Ns);
    for (int j = tid; j < q2; j += nth) {
      const int k = j & (Ns - 1);
      const cd v0 = a[j];
      cd v1 = a[j + q2];
      if (k) v1 = v1 * tw_lookup<TW_SMEM>(tw, k * tstep, NT, sign);
      const int j0 = ((j - k) << 1) + k;
      b[j0] = v0 + v1;
      b[j0 + Ns] = v0 - v1;
    }
    __syncthreads();
    cd *t = a;
    a = b;
    b = t;
  }
  return a;
}
// c2r: Hermitian half spectrum X(k), k = 0..N/2 (imaginary parts of X(0), X(N/2) ignored, as FFTW's
// c2r does) -> real x[0..N): returns z with x[2m] = z[m].x, x[2m+1] = z[m].y.  work: N complex.
template <bool TW_SMEM, class F>
RFS_DEVINL cd *block_irfft(F X, cd *work, int N, int logN, const double2 *__restrict__ tw) {
  const int M = N >> 1;
  for (int k = threadIdx.x; k < M; k += blockDim.x) {
    cd xk = X(k), xm = conj(X(M - k));
    if (k == 0) {
      xk.y = 0.0;
      xm.y = 0.0;
    }
    const cd xe = xk + xm;
    const cd xo = (xk - xm) * tw_lookup<TW_SMEM>(tw, k, N, +1);
    work[k] = cd(xe.x - xo.y, xe.y + xo.x);  // xe + i xo
  }
  __syncthreads();
  return stockham_fft<TW_SMEM>(work, work + M, M, logN - 1, +1, tw, N);
}
RFS_DEVINL double irfft_at(const cd *z, int t) { return (t & 1) ? z[t >> 1].y : z[t >> 1].x; }
// r2c: real x(t), t = 0..N-1 -> z = FFT_{N/2}(x[2m] + i x[2m+1]); the half spectrum is then
// rfft_at(z, k, ..), k = 0..N/2.  work: N complex.
template <bool TW_SMEM, class F>
RFS_DEVINL cd *block_rfft(F x, cd *work, int N, int logN, const double2 *__restrict__ tw) {
  const int M = N >> 1;
  for (int m = threadIdx.x; m < M; m += blockDim.x) work[m] = cd(x(2 * m), x(2 * m + 1));
  __syncthreads();
  return stockham_fft<TW_SMEM>(work, work + M, M, logN - 1, -1, tw, N);
}
template <bool TW_SMEM>
RFS_DEVINL cd rfft_at(const cd *z, int k, int N, const double2 *__restrict__ tw) {
  const int M = N >> 1;
  const cd zk = z[k & (M - 1)], zm = conj(z[(M - k) & (M - 1)]);
  const cd xe = 0.5 * (zk + zm), d = zk - zm;
  const cd xo(0.5 * d.y, -0.5 * d.x);  // (zk - zm) / (2 i)
  if (k == M) return cd(xe.x - xo.x, 0.0);  // e^{-i pi} = -1
  return xe + xo * tw_lookup<TW_SMEM>(tw, k, N, -1);
}

RFS_DEVINL double block_reduce(double v, double *red, bool is_max) {
  // red: >= 32 doubles of shared memory
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    const double t = __shfl_down_sync(0xffffffffu, v, o);
    v = is_max ? fmax(v, t) : v + t;
  }
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    v = (lane < nw) ? red[lane] : (is_max ? -1.0e300 : 0.0);
    for (int o = 16; o > 0; o >>= 1) {
      const double t = __shfl_down_sync(0xffffffffu, v, o);
      v = is_max ? fmax(v, t) : v + t;
    }
    if (lane == 0) red[0] = v;
  }
  __syncthreads();
  const double r = red[0];
  __syncthreads();
  return r;
}

// Gaussian widths of one RF objective (rfs_config_rf_gauss), passed by value: each width is one trace
// of the data vector's [ray][gauss][nt] block
#define RFS_MAX_GAUSS 16
struct GaussList {
  int n;
  double a[RFS_MAX_GAUSS];
};
// Gaussian width g of each row: gauss[set[b]][g] of a per-set table (rfs_config_obs_gauss), or the shared
// width.  Like RayView: set points at the rows of this launch (NULL: every row is set 0), and a row whose
// set index lies outside [0, nsets) reads nothing from the table (the residual kernels fail that row).
struct GaussView {
  const double *tab;  // [nsets][G] or NULL (every row uses `shared`)
  const int *set;     // [B] or NULL
  int nsets, G;
  RFS_DEVINL double row_a(long long b, int g, double shared) const {
    if (!tab) return shared;
    const int s = set ? set[b] : 0;
    return (s >= 0 && s < nsets) ? tab[s * G + g] : shared;
  }
};

// ---- K4: one block per (model, ray pass): water-level deconvolution, c2r FFT, trace, misfit and
// (optional) adjoint gradient, for every Gaussian width of the list on the same staged spectra.
//   dynamic smem: cd buf[nft] + cd s21[n2] + cd s22[n2] + cd wt[n2] + 64 doubles, + cd acc[n2] for G > 1
//   rf   : [B][ldrf >= G*nt], the widths' traces one after the other
//   obs.dobs: [nsets][ld >= G*nt] or NULL   U: [B]   grad: [B][nrow] (nrow = NQ*n)
//   the residual is 0 at the samples the row's set does not fit (ObsSets::observed, sample g*nt + t of
//   width g); rf is written whole
//   flag : [B] or NULL; only written (0) for a row whose observation-set index is out of range
// The spectra, both water levels and the derivative spectra D do not depend on the width, and the
// gradient sum_k Re(W_k D_jk) is linear in the adjoint weights W: the widths' weights are summed in acc
// and contracted with D once.  With one width the weights go straight into wt.
// MULTI = false runs width 0 only: without the width loop's state the kernel keeps 54 registers
// (64 with it), which is the occupancy of the one-width objectives at small nt.
// gv: each set's own widths (rfs_config_obs_gauss) in place of gauss.a; rows of an out-of-range set
// return above, before any width is read.
template <bool MULTI>
__global__ void rf_decon_kernel(const double2 *__restrict__ spec, const double2 *__restrict__ dspec,
                                long long B, int nrow, int nt, int nft, int logn, double dt,
                                GaussList gauss, GaussView gv, double t0, double water, double sigma,
                                ObsSets obs, double *__restrict__ rf, long long ldrf, double *__restrict__ U,
                                double *__restrict__ grad, unsigned char *__restrict__ flag,
                                const double2 *__restrict__ tw, int accumulate) {
  // accumulate != 0: U and grad are added to (second and later ray parameters of one objective)
  extern __shared__ double smem[];
  const int n2 = nft / 2 + 1;
  const int G = MULTI ? gauss.n : 1;
  cd *buf = reinterpret_cast<cd *>(smem);
  cd *s21 = buf + nft;
  cd *s22 = s21 + n2;
  cd *wt = s22 + n2;
  double *red = reinterpret_cast<double *>(wt + n2);
  cd *acc = G > 1 ? reinterpret_cast<cd *>(red + 64) : wt;  // adjoint weights summed over the widths
  const long long b = blockIdx.x;
  const int tid = threadIdx.x, nth = blockDim.x;
  const int set = obs.row_set(b);
  if (set < 0) {
    for (int it = tid; it < G * nt; it += nth) rf[b * ldrf + it] = nan("");
    if (grad)
      for (int rr = tid; rr < nrow; rr += nth) grad[b * nrow + rr] = 0.0;
    if (tid == 0) {
      U[b] = 0.0;
      if (flag) flag[b] = 0;
    }
    return;
  }
  const double *dobs = obs.dobs ? obs.row(set) : nullptr;

  double lmax = 0.0;
  for (int k = tid; k < n2; k += nth) {
    const double2 a = spec[(b * 2 + 0) * n2 + k], c = spec[(b * 2 + 1) * n2 + k];
    s21[k] = cd(a.x, a.y);
    s22[k] = cd(c.x, c.y);
    lmax = fmax(lmax, a.x * a.x + a.y * a.y);
  }
  const double wmax = block_reduce(lmax, red, true);
  // second water level on |R21^2|^2 (:410-413), for the adjoint weights of every width
  double wmax2 = 0.0;
  if (dobs && grad) {
    double lmax2 = 0.0;
    for (int k = tid; k < n2; k += nth) {
      const double wa = norm2(s21[k]);
      lmax2 = fmax(lmax2, wa * wa);
    }
    wmax2 = block_reduce(lmax2, red, true);
  }
  for (int ig = 0; ig < G; ig++) {
    if (ig > 0) __syncthreads();  // the previous width's reads of buf and wt are done
    const double f0 = gv.row_a(b, ig, gauss.a[ig]);
    // spectral division (:393-401) into wt (free until the adjoint pass), then the c2r transform
    for (int k = tid; k < n2; k += nth) {
      const double w = 1.0 / nft / dt * k * 2.0 * RFS_PI32;
      const double gx = w / 2 / f0;
      const double g = exp(-(gx * gx));
      const double wa = norm2(s21[k]);
      const double fai = fmax(wa, water * wmax);
      wt[k] = conj(s21[k]) * s22[k] * g * cis(-w * t0) / fai;
    }
    __syncthreads();
    const cd *z = block_irfft<false>([&](int k) { return wt[k]; }, buf, nft, logn, tw);
    // trace, residual, weighted residual (:404-407 and the adjoint source; the real sequence is kept in
    // the .x of wt[0..nt), the rest of the padded sequence is zero)
    double lsum = 0.0;
    double *rsd = reinterpret_cast<double *>(wt);  // nt <= nft doubles fit in n2 complex entries
    const int o = ig * nt;                         // this width's trace in rf, dobs and the sample mask
    for (int it = tid; it < nft; it += nth) {
      double rt = 0.0;
      if (it < nt) {
        const double e = exp(sigma * (-t0 + it * dt));
        const double v = irfft_at(z, it) / nft / dt * e;
        rf[b * ldrf + o + it] = v;
        if (dobs) {
          const double r = obs.observed(set, o + it) ? v - dobs[o + it] : 0.0;
          lsum += r * r;
          rt = r * e / dt;
        }
      }
      rsd[it] = rt;
    }
    if (dobs == nullptr) continue;
    const double ss = block_reduce(lsum, red, false);
    if (tid == 0) U[b] = (accumulate || ig > 0) ? U[b] + 0.5 * ss : 0.5 * ss;
    if (grad == nullptr) continue;
    __syncthreads();
    const cd *zr = block_rfft<false>([&](int t) { return rsd[t]; }, buf, nft, logn, tw);
    // adjoint weights of this width
    for (int k = tid; k < n2; k += nth) {
      const double w = 1.0 / nft / dt * k * 2.0 * RFS_PI32;
      const double gx = w / 2 / f0;
      const double g = exp(-(gx * gx));
      const cd sq = s21[k] * s21[k];
      const double wa = norm2(sq);
      const double fai = fmax(wa, water * wmax2);
      const cd Mk = conj(sq) * g * cis(-w * t0) / fai;
      const double ck = (k == 0 || k == nft / 2) ? 1.0 : 2.0;
      cd rk = rfft_at<false>(zr, k, nft, tw);
      if (k == 0 || k == nft / 2) rk.y = 0.0;
      const cd wk = Mk * conj(rk) * (ck / nft);  // the residual sequence kept in wt has been consumed
      acc[k] = ig > 0 ? acc[k] + wk : wk;
    }
  }
  if (dobs == nullptr || grad == nullptr) return;
  __syncthreads();
  // grad_row = sum_k Re(acc_k D_row,k): one warp per row
  const int lane = tid & 31, wid = tid >> 5, nw = nth >> 5;
  for (int rr = wid; rr < nrow; rr += nw) {
    const double2 *dp = dspec + (b * (long long)nrow + rr) * n2;
    double acc_r = 0.0;
    for (int k = lane; k < n2; k += 32) {
      const double2 d = dp[k];
      acc_r += acc[k].x * d.x - acc[k].y * d.y;
    }
    for (int o = 16; o > 0; o >>= 1) acc_r += __shfl_down_sync(0xffffffffu, acc_r, o);
    if (lane == 0) grad[b * nrow + rr] = accumulate ? grad[b * nrow + rr] + acc_r : acc_r;
  }
}

// ---- Jacobian traces for the librf.kernel / kernel_all drop-ins: one block per (model, row)
//   out: [B][nrow][nt]
__global__ void rf_trace_kernel(const double2 *__restrict__ spec, const double2 *__restrict__ dspec,
                                long long B, int nrow, int nt, int nft, int logn, double dt,
                                double f0, double t0, double water, double sigma,
                                double *__restrict__ out, const double2 *__restrict__ tw) {
  extern __shared__ double smem[];
  const int n2 = nft / 2 + 1;
  cd *buf = reinterpret_cast<cd *>(smem);
  cd *s21 = buf + nft;
  double *red = reinterpret_cast<double *>(s21 + n2);
  const long long b = blockIdx.x / nrow;
  const int rr = (int)(blockIdx.x % nrow);
  const int tid = threadIdx.x, nth = blockDim.x;
  double lmax2 = 0.0;
  for (int k = tid; k < n2; k += nth) {
    const double2 a = spec[(b * 2 + 0) * n2 + k];
    s21[k] = cd(a.x, a.y);
    const double wa = a.x * a.x + a.y * a.y;
    lmax2 = fmax(lmax2, wa * wa);
  }
  const double wmax2 = block_reduce(lmax2, red, true);
  const double2 *dp = dspec + (b * (long long)nrow + rr) * n2;
  for (int k = tid; k < n2; k += nth) {
    const double w = 1.0 / nft / dt * k * 2.0 * RFS_PI32;
    const double gx = w / 2 / f0;
    const double g = exp(-(gx * gx));
    const cd sq = s21[k] * s21[k];
    const double fai = fmax(norm2(sq), water * wmax2);
    const double2 d = dp[k];
    s21[k] = conj(sq) * cd(d.x, d.y) * g * cis(-w * t0) / fai;  // in place: s21[k] is read by this thread only
  }
  __syncthreads();
  const cd *z = block_irfft<false>([&](int k) { return s21[k]; }, buf, nft, logn, tw);
  for (int it = tid; it < nt; it += nth)
    out[(b * nrow + rr) * (long long)nt + it] = irfft_at(z, it) / nft / dt * exp(sigma * (-t0 + it * dt));
}

}  // namespace rfs
