// K1 — batched phase-velocity root search (one thread per (model, period-sequence)).
//
// Replaces /root/reference/src/SWD/surfdisp96.f (surfdisp96 :54-368, getsol :398-491,
// nevill :568-687, half :689-701, dltar1 :727-787, dltar4 :791-891, var :894-1011,
// dnka :1044-1088) and the retry loop of /root/reference/src/SWD/surfdisp.cpp:93-100.
//
// B200 design: the reference's recursion getsol -> nevill -> dltar is flattened into ONE
// per-thread state machine whose loop body contains exactly one secular-function evaluation, so
// the 32 lanes of a warp (32 different models, same sequence) stay converged on the expensive
// Dunkin/Haskell layer sweep no matter where each lane is in its own scan / bisection / Neville
// step.  The scan grid (dc = float32 0.005), the period-to-period and mode-to-mode chaining, the
// `del1st` sign memory and the hybrid `nevill` refinement are reproduced exactly, because the
// returned root depends on them at the 1e-6 level (SURVEY.md §7 hard part 1).
// Model arrays live in HBM as [field][layer][model] (model fastest => coalesced, L1-resident).
#pragma once
#include "common.cuh"

namespace rfs {

// field indices of the SWD model block (all values are float32-rounded, stored as double)
// F_VTP/F_DTP/F_RTP: earth-flattening factors of bldsph (velocity, boundary, density); 1 when flat
enum { F_D = 0, F_A = 1, F_B = 2, F_RHO = 3, F_IA = 4, F_IB = 5, F_IRHO = 6, F_VTP = 7, F_DTP = 8,
       F_RTP = 9, SWD_NF = 10 };

// Model blocks of one batch.  Flat earth: all four pointers alias one block.  Spherical earth:
// root[f] is the model flattened by surfdisp96's `sphere` (float32, radius 6370), eig[f] the one
// flattened by sregn96/slegn96's `bldsph` (float64, radius 6371); f = 0 Rayleigh, 1 Love.
struct SwdBlocks {
  const double *root[2];
  const double *eig[2];
  int sphere;
};

struct SwdModel {
  const double *p;  // [SWD_NF][n][stride]
  int stride;       // models in the batch (B)
  int n;            // layers (last = half-space)
  int fs;           // field stride n*B
  // 32-bit element indices (the host keeps SWD_NF*n*B below 2^31, see run_swd): one IMAD per field
  // on top of the shared m*B+b term instead of a 64-bit multiply chain per load
  RFS_DEVINL SwdModel(const double *blk, long long B, int nl)
      : p(blk), stride((int)B), n(nl), fs(nl * (int)B) {}
  RFS_DEVINL double ld(int f, int m, long long b) const {
    return __ldg(p + (f * fs + (m * stride + (int)b)));
  }
};

// The same seven root-search fields of the NT threads of a block staged in shared memory,
// [layer][field][thread]: thread-constant base, one multiply per layer, immediate field offsets.
#define RFS_ROOT_NF 7  // F_D .. F_IRHO
template <int NT>
struct SmemColModel {
  const double *p;  // [n][RFS_ROOT_NF][NT]
  int n;
  RFS_DEVINL double ld(int f, int m, long long col) const {
    return p[(m * RFS_ROOT_NF + f) * NT + (int)col];
  }
};

// ---- Love secular function: Haskell 2-vector from the half-space up (surfdisp96.f:727-787)
// love_layer builds the layer terms, love_apply propagates + normalises the 2-vector; the split
// lets the team kernel (swd_roots_team.cuh) build layers in parallel with the same operations.
struct LoveL {
  double xmu, cosq, y, z;
};
template <class MT>
RFS_DEVINL LoveL love_layer(const MT &M, long long b, int m, double wvno, double omega) {
  LoveL L;
  const double beta1 = M.ld(F_B, m, b);
  const double rho1 = M.ld(F_RHO, m, b);
  const double dm = M.ld(F_D, m, b);
  L.xmu = rho1 * beta1 * beta1;
  const double xkb = omega / beta1;
  const double rb = sqrt((wvno + xkb) * fabs(wvno - xkb));
  const double q = dm * rb;
  if (wvno < xkb) {
    double sinq;
    sincos_cb(q, &sinq, &L.cosq);
    L.y = sinq / rb;
    L.z = -rb * sinq;
  } else if (wvno == xkb) {
    L.cosq = 1.0;
    L.y = dm;
    L.z = 0.0;
  } else {
    double fac = 0.0;
    if (q < 16.0) fac = exp_neg(2.0 * q);
    L.cosq = (1.0 + fac) * 0.5;
    const double sinq = (1.0 - fac) * 0.5;
    L.y = sinq / rb;
    L.z = rb * sinq;
  }
  return L;
}
// 2^-k for the vector whose largest |component| has the (31-bit, sign stripped) high word h:
// 2^k <= max < 2^(k+1).  Multiplying by it is exact, so the renormalisation below never rounds.
RFS_DEVINL double pow2_unscale(int h) {
  // biased exponent of 2^-(be-1023) for the maximum's biased exponent be = h >> 20, kept >= 1: a zero
  // or denormal maximum is scaled by 2^1023 (exact, still below 2), inf / NaN stay what they are
  const int sb = max(2046 - (h >> 20), 1);
  return __hiloint2double(sb << 20, 0);
}
#define RFS_HIABS(v) (__double2hiint(v) & 0x7fffffff)
// One layer of the Love recursion.  The reference divides the 2-vector by its max-norm after every
// layer (surfdisp96.f:778-784); those factors cancel in the final ratio e1/max(|e1|,|e2|), so the vector
// is only kept in range here by an exact power of two and normalised ONCE at the top (love_finish):
// same value in exact arithmetic, fewer roundings, and no division on the layer-to-layer critical path.
RFS_DEVINL void love_apply(const LoveL &L, double &e1, double &e2) {
  // explicit rounding (see RFS_FMA in common.cuh): the same bits from every kernel
  const double e10 = RFS_FMA(e1, L.cosq, RFS_MUL(RFS_MUL(e2, L.xmu), L.z));
  const double e20 = RFS_FMA(e2, L.cosq, RFS_MUL(e1, L.y) / L.xmu);
  const double sc = pow2_unscale(max(RFS_HIABS(e10), RFS_HIABS(e20)));
  e1 = e10 * sc;
  e2 = e20 * sc;
}
// the normalisation of the last layer step (normc): e1 / max(|e1|, |e2|)
RFS_DEVINL double love_finish(double e1, double e2) {
  double xnor = fmax(fabs(e1), fabs(e2));
  if (xnor < 1.e-40) xnor = 1.0;
  return e1 / xnor;
}
template <class MT>
RFS_DEVINL void love_halfspace(const MT &M, long long b, double wvno, double omega, double &e1,
                               double &e2) {
  const int mmax = M.n;
  const double beta1 = M.ld(F_B, mmax - 1, b);
  const double rho1 = M.ld(F_RHO, mmax - 1, b);
  const double xkb = omega / beta1;
  const double rb = sqrt((wvno + xkb) * fabs(wvno - xkb));
  e1 = rho1 * rb;
  e2 = 1.0 / (beta1 * beta1);
}
template <class MT>
RFS_DEVINL double dltar1_dev(double wvno, double omega, const MT &M, long long b, int llw) {
  const int mmax = M.n;
  double e1, e2;
  love_halfspace(M, b, wvno, omega, e1, e2);
  for (int m = mmax - 2; m >= llw - 1; m--) {
    const LoveL L = love_layer(M, b, m, wvno, omega);
    love_apply(L, e1, e2);
  }
  if (mmax - 2 >= llw - 1) return love_finish(e1, e2);
  return e1;
}

// hyperbolic / circular layer functions of surfdisp96.f `var` (:894-1011) for one wave type.
// x2 = (wvno+xk)*|wvno-xk| = r^2.  Division-free: r = x2*rsqrt(x2), 1/r = rsqrt(x2); the
// evanescent branch returns e = exp(-r d) so that exp(-2 r d) = e*e and a0 = e_p*e_q need no
// further exponentials (<= 2 ulp away from the reference's expressions).
struct VarHalf {
  double c, w, x, ex, e;  // cos-like, sin/r, (+-)r*sin, exponent, exp(-ex)
};
// P and S halves evaluated together: the two rsqrt / exp chains are independent straight-line
// code (no branch between them), which doubles the ILP of the latency-bound inner loop; the
// oscillatory (c > v) and grazing (c == v) cases are patched afterwards.
RFS_DEVINL void var_pair(double wvno, double xka, double xkb, double dpth, VarHalf &P, VarHalf &S) {
  const double x2a = (wvno + xka) * fabs(wvno - xka), x2b = (wvno + xkb) * fabs(wvno - xkb);
  const double ria = (x2a > 0.0) ? rsqrt_pos(x2a) : 0.0, rib = (x2b > 0.0) ? rsqrt_pos(x2b) : 0.0;
  const double ra = x2a * ria, rb = x2b * rib;
  const double pa = ra * dpth, pb = rb * dpth;
  const double ea = exp_neg(pa), eb = exp_neg(pb);
  const double fa = (pa < 16.0) ? ea * ea : 0.0, fb = (pb < 16.0) ? eb * eb : 0.0;
  const double sa = (1.0 - fa) * 0.5, sb = (1.0 - fb) * 0.5;
  P.c = (1.0 + fa) * 0.5;
  P.w = sa * ria;
  P.x = ra * sa;
  P.ex = pa;
  P.e = ea;
  S.c = (1.0 + fb) * 0.5;
  S.w = sb * rib;
  S.x = rb * sb;
  S.ex = pb;
  S.e = eb;
  if (!(wvno > xka)) {
    P.ex = 0.0;
    P.e = 1.0;
    if (wvno < xka) {
      double s;
      sincos_cb(pa, &s, &P.c);
      P.w = s * ria;
      P.x = -ra * s;
    } else {
      P.c = 1.0;
      P.w = dpth;
      P.x = 0.0;
    }
  }
  if (!(wvno > xkb)) {
    S.ex = 0.0;
    S.e = 1.0;
    if (wvno < xkb) {
      double s;
      sincos_cb(pb, &s, &S.c);
      S.w = s * rib;
      S.x = -rb * s;
    } else {
      S.c = 1.0;
      S.w = dpth;
      S.x = 0.0;
    }
  }
}
RFS_DEVINL VarHalf var_half(double wvno, double xk, double x2, double dpth) {
  VarHalf o;
  const double ri = (x2 > 0.0) ? rsqrt(x2) : 0.0;
  const double r = x2 * ri;
  const double pq = r * dpth;
  o.ex = 0.0;
  o.e = 1.0;
  if (wvno < xk) {
    double s;
    sincos_cb(pq, &s, &o.c);
    o.w = s * ri;
    o.x = -r * s;
  } else if (wvno == xk) {
    o.c = 1.0;
    o.w = dpth;
    o.x = 0.0;
  } else {
    o.ex = pq;
    o.e = exp_neg(pq);
    const double fac = (pq < 16.0) ? o.e * o.e : 0.0;
    o.c = (1.0 + fac) * 0.5;
    const double s = (1.0 - fac) * 0.5;
    o.w = s * ri;
    o.x = r * s;
  }
  return o;
}

// ---- Rayleigh secular function: Dunkin 5-vector compound matrix (surfdisp96.f:791-891).
// iom = 1/omega (hoisted per period); per-layer reciprocals 1/a, 1/b, 1/rho come from the model
// block.  Same formulas as dltar4/var/dnka/normc; divisions replaced by reciprocal multiplies.
struct Dunkin {
  double c11, c12, c13, c14, c15, c21, c22, c23, c24, c31, c32, c33, c34, c35, c41, c42, c43, c51,
      c53;
};
template <class MT>
RFS_DEVINL Dunkin dunkin_layer(const MT &M, long long b, int m, double wvno, double wvno2,
                               double omega, double iom) {
  const double bm = M.ld(F_B, m, b);
  const double dpth = M.ld(F_D, m, b), rho = M.ld(F_RHO, m, b), irho = M.ld(F_IRHO, m, b);
  const double xka = omega * M.ld(F_IA, m, b), xkb = omega * M.ld(F_IB, m, b);
  const double t = bm * iom;
  const double gammk = 2.0 * t * t;
  const double gam = gammk * wvno2;
  VarHalf P, S;
  var_pair(wvno, xka, xkb, dpth, P, S);
  const double exa = P.ex + S.ex;
  const double a0 = (exa < 60.0) ? P.e * S.e : 0.0;
  const double cpcq = P.c * S.c, cpy = P.c * S.w, cpz = P.c * S.x, cqw = S.c * P.w,
               cqx = S.c * P.x, xy = P.x * S.w, xz = P.x * S.x, wy = P.w * S.w, wz = P.w * S.x;
  // Dunkin matrix (dnka :1044-1088), unique entries only.  Every a*b+c below is an explicit FMA
  // (RFS_FMA: fixed rounding in every kernel that inlines this function).
  const double gamm1 = gam - 1.0, twgm1 = gam + gamm1, gmgmk = gam * gammk, gmgm1 = gam * gamm1,
               gm1sq = gamm1 * gamm1, rho2 = rho * rho, irho2 = irho * irho, a0pq = a0 - cpcq;
  Dunkin C;
  // c11 = cpcq - 2 gmgm1 a0pq - gmgmk xz - wvno2 gm1sq wy
  C.c11 = RFS_FMA(-RFS_MUL(wvno2, gm1sq), wy,
                  RFS_FMA(-gmgmk, xz, RFS_FMA(-RFS_MUL(2.0, gmgm1), a0pq, cpcq)));
  C.c12 = RFS_MUL(RFS_FMA(wvno2, cpy, -cqx), irho);
  // c13 = -(twgm1 a0pq + gammk xz + wvno2 gamm1 wy) / rho
  C.c13 = -RFS_MUL(RFS_FMA(RFS_MUL(wvno2, gamm1), wy, RFS_FMA(gammk, xz, RFS_MUL(twgm1, a0pq))), irho);
  C.c14 = RFS_MUL(RFS_FMA(-wvno2, cqw, cpz), irho);
  // c15 = -(2 wvno2 a0pq + xz + wvno2^2 wy) / rho^2
  C.c15 = -RFS_MUL(RFS_FMA(RFS_MUL(wvno2, wvno2), wy, RFS_FMA(RFS_MUL(2.0, wvno2), a0pq, xz)), irho2);
  C.c21 = RFS_MUL(RFS_FMA(gmgmk, cpz, -RFS_MUL(gm1sq, cqw)), rho);
  C.c22 = cpcq;
  C.c23 = RFS_FMA(gammk, cpz, -RFS_MUL(gamm1, cqw));
  C.c24 = -wz;
  C.c41 = RFS_MUL(RFS_FMA(gm1sq, cpy, -RFS_MUL(gmgmk, cqx)), rho);
  C.c42 = -xy;
  C.c43 = RFS_FMA(gamm1, cpy, -RFS_MUL(gammk, cqx));
  // c51 = -(2 gmgmk gm1sq a0pq + gmgmk^2 xz + gm1sq^2 wy) rho^2
  C.c51 = -RFS_MUL(RFS_FMA(RFS_MUL(gm1sq, gm1sq), wy,
                           RFS_FMA(RFS_MUL(gmgmk, gmgmk), xz,
                                   RFS_MUL(RFS_MUL(RFS_MUL(2.0, gmgmk), gm1sq), a0pq))),
                   rho2);
  // c53 = -(gammk gamm1 twgm1 a0pq + gam gammk^2 xz + gamm1 gm1sq wy) rho
  C.c53 = -RFS_MUL(RFS_FMA(RFS_MUL(gamm1, gm1sq), wy,
                           RFS_FMA(RFS_MUL(gmgmk, gammk), xz,
                                   RFS_MUL(RFS_MUL(RFS_MUL(gammk, gamm1), twgm1), a0pq))),
                   rho);
  const double tt = -2.0 * wvno2;
  C.c31 = tt * C.c53;
  C.c32 = tt * C.c43;
  C.c33 = a0 + 2.0 * (cpcq - C.c11);
  C.c34 = tt * C.c23;
  C.c35 = tt * C.c13;
  return C;
}
// e <- e * ca: ee(i) = sum_j e(j) ca(j,i), with ca(2,5)=c14 ca(4,4)=c22 ca(4,5)=c12
// ca(5,2)=c41 ca(5,4)=c21 ca(5,5)=c11; two partial sums per component shorten the chain.
// The reference divides the 5-vector by its max-norm after every layer (normc, surfdisp96.f:1013-1040).
// Those factors cancel: after the last layer the normalised vector is u / max|u| whatever positive
// scalings were applied on the way.  So the vector is kept in range by an EXACT power of two per layer
// (integer pipe, no rounding) and normalised once at the top (dunkin_finish): the same value in exact
// arithmetic, one division per evaluation instead of one per layer, and a layer-to-layer critical path
// of 4 dependent FP64 operations instead of ~25.
// rescale = false skips the power-of-two step for this layer: the scalings are exact and cancel in
// dunkin_finish, so they are only needed often enough to stay far from overflow (every second layer)
RFS_DEVINL void dunkin_apply(const Dunkin &C, double &e0, double &e1, double &e2, double &e3,
                             double &e4, bool rescale) {
#define RFS_ROW(a0_, a1_, a2_, a3_, a4_)                                                      \
  RFS_FMA(e4, a4_, RFS_ADD(RFS_FMA(e0, a0_, RFS_MUL(e1, a1_)), RFS_FMA(e2, a2_, RFS_MUL(e3, a3_))))
  const double n0 = RFS_ROW(C.c11, C.c21, C.c31, C.c41, C.c51);
  const double n1 = RFS_ROW(C.c12, C.c22, C.c32, C.c42, C.c41);
  const double n2 = RFS_ROW(C.c13, C.c23, C.c33, C.c43, C.c53);
  const double n3 = RFS_ROW(C.c14, C.c24, C.c34, C.c22, C.c21);
  const double n4 = RFS_ROW(C.c15, C.c14, C.c35, C.c12, C.c11);
#undef RFS_ROW
  if (!rescale) {
    e0 = n0;
    e1 = n1;
    e2 = n2;
    e3 = n3;
    e4 = n4;
    return;
  }
  const double sc = pow2_unscale(
      max(max(max(RFS_HIABS(n0), RFS_HIABS(n1)), max(RFS_HIABS(n2), RFS_HIABS(n3))), RFS_HIABS(n4)));
  e0 = n0 * sc;
  e1 = n1 * sc;
  e2 = n2 * sc;
  e3 = n3 * sc;
  e4 = n4 * sc;
}
// normc of the last layer step: e0, e1 <- e0 / max|e|, e1 / max|e| (only these two are used afterwards).
// max |e_i| on the integer pipe: the bit patterns of non-negative doubles order like unsigned integers
// (a NaN wins and poisons the result).
RFS_DEVINL void dunkin_finish(double &e0, double &e1, double e2, double e3, double e4) {
#define RFS_ABSBITS(v) \
  (((unsigned long long)((unsigned)__double2hiint(v) & 0x7fffffffu) << 32) | (unsigned)__double2loint(v))
  const unsigned long long u0 = RFS_ABSBITS(e0), u1 = RFS_ABSBITS(e1), u2 = RFS_ABSBITS(e2),
                           u3 = RFS_ABSBITS(e3), u4 = RFS_ABSBITS(e4);
#undef RFS_ABSBITS
  double t1 = __longlong_as_double((long long)max(max(max(u0, u1), max(u2, u3)), u4));
  if (t1 < 1.e-40) t1 = 1.0;
  const double it1 = 1.0 / t1;
  e0 = e0 * it1;
  e1 = e1 * it1;
}
// half-space start vector of dltar4 (surfdisp96.f:815-835)
template <class MT>
RFS_DEVINL void dunkin_halfspace(const MT &M, long long b, double wvno, double wvno2, double omega,
                                 double iom, double &e0, double &e1, double &e2, double &e3,
                                 double &e4) {
  const int mmax = M.n;
  const double bm = M.ld(F_B, mmax - 1, b);
  const double rho1 = M.ld(F_RHO, mmax - 1, b);
  const double xka = omega * M.ld(F_IA, mmax - 1, b), xkb = omega * M.ld(F_IB, mmax - 1, b);
  const double ra = sqrt((wvno + xka) * fabs(wvno - xka));
  const double rb = sqrt((wvno + xkb) * fabs(wvno - xkb));
  const double t = bm * iom;
  const double gammk = 2.0 * t * t;
  const double gam = gammk * wvno2;
  const double gamm1 = gam - 1.0;
  const double rarb = RFS_MUL(ra, rb);
  e0 = RFS_MUL(RFS_MUL(rho1, rho1), RFS_FMA(-RFS_MUL(gam, gammk), rarb, RFS_MUL(gamm1, gamm1)));
  e1 = -rho1 * ra;
  e2 = RFS_MUL(rho1, RFS_FMA(-gammk, rarb, gamm1));
  e3 = rho1 * rb;
  e4 = RFS_SUB(wvno2, rarb);
}
// water layer on top (surfdisp96.f:870-886)
template <class MT>
RFS_DEVINL double dunkin_water_top(const MT &M, long long b, double wvno, double omega, double e0,
                                   double e1) {
  const double dpth = M.ld(F_D, 0, b), rho1 = M.ld(F_RHO, 0, b);
  const double xka = omega * M.ld(F_IA, 0, b);
  const VarHalf P = var_half(wvno, xka, (wvno + xka) * fabs(wvno - xka), dpth);
  const double w0 = -rho1 * P.w;
  return RFS_FMA(P.c, e0, RFS_MUL(w0, e1));
}
// PAIRED: two layer matrices are formed per trip (independent dependency chains: twice the ILP) and
// applied in order -- the same operations and bits.  It costs ~40 registers: slower in the thread-mapped
// kernel, where occupancy hides latency (measured in round 1), faster where a warp is alone on its
// scheduler (team kernels whose lanes each evaluate a whole secular function, GL = 1).
template <class MT, bool PAIRED = false>
RFS_DEVINL double dltar4_dev(double wvno, double omga, double iomga, const MT &M, long long b,
                             int llw) {
  const int mmax = M.n;
  double omega = omga, iom = iomga;
  if (omega < 1.0e-4) {
    omega = 1.0e-4;
    iom = 1.0e4;
  }
  const double wvno2 = wvno * wvno;
  double e0, e1, e2, e3, e4;
  dunkin_halfspace(M, b, wvno, wvno2, omega, iom, e0, e1, e2, e3, e4);
  int m = mmax - 2;
  if (PAIRED) {
    for (; m - 1 >= llw - 1; m -= 2) {
      const Dunkin Ca = dunkin_layer(M, b, m, wvno, wvno2, omega, iom);
      const Dunkin Cb = dunkin_layer(M, b, m - 1, wvno, wvno2, omega, iom);
      dunkin_apply(Ca, e0, e1, e2, e3, e4, false);
      dunkin_apply(Cb, e0, e1, e2, e3, e4, true);
    }
  }
  for (; m >= llw - 1; m--) {
    const Dunkin C = dunkin_layer(M, b, m, wvno, wvno2, omega, iom);
    dunkin_apply(C, e0, e1, e2, e3, e4, (m & 3) == 3);
  }
  if (mmax - 2 >= llw - 1) dunkin_finish(e0, e1, e2, e3, e4);
  if (llw != 1) return dunkin_water_top(M, b, wvno, omega, e0, e1);
  return e0;
}

// One sequence = one wave family on one period list (optionally scaled: 1.05 T / 0.95 T for the
// group-velocity kernels, surfdisp.cpp:234-241).
struct SwdSeq {
  int ifunc;      // 1 Love, 2 Rayleigh
  int per_off;    // offset into the period table
  int nper;       // periods in this sequence (ascending)
  int out_off;    // offset (in periods) of this sequence in the output block
  double scale;   // period multiplier
};

// float32 Newton start value (gtsolh, surfdisp96.f:375-396) — all REAL*4
RFS_DEVINL float gtsolh_dev(float a, float b) {
  float c = __fmul_rn(0.95f, b);
  for (int i = 0; i < 5; i++) {
    float gamma = __fdiv_rn(b, a);
    float kappa = __fdiv_rn(c, b);
    float k2 = __fmul_rn(kappa, kappa);
    float gk = __fmul_rn(gamma, kappa);
    float gk2 = __fmul_rn(gk, gk);
    float fac1 = __fsqrt_rn(__fsub_rn(1.0f, gk2));
    float fac2 = __fsqrt_rn(__fsub_rn(1.0f, k2));
    float tk = __fsub_rn(2.0f, k2);
    float fr = __fsub_rn(__fmul_rn(tk, tk), __fmul_rn(__fmul_rn(4.0f, fac1), fac2));
    float t1 = __fmul_rn(__fmul_rn(-4.0f, tk), kappa);
    float t2 = __fdiv_rn(__fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(4.0f, fac2), gamma), gamma), kappa), fac1);
    float t3 = __fdiv_rn(__fmul_rn(__fmul_rn(4.0f, fac1), kappa), fac2);
    float frp = __fadd_rn(__fadd_rn(t1, t2), t3);
    frp = __fdiv_rn(frp, b);
    c = __fsub_rn(c, __fdiv_rn(fr, frp));
  }
  return c;
}

// prologue of surfdisp96 (:128-220): water-layer flag, largest S velocity and the float32 start
// value cc1 = 0.90 * 0.95 * (Rayleigh velocity of the slowest layer as a half space) -- all REAL*4
template <class MT>
RFS_DEVINL void swd_start_values(const MT &M, long long mb, int &llw, float &betmx, float &cc1) {
  const int mmax = M.n;
  llw = (M.ld(F_B, 0, mb) <= 0.0) ? 2 : 1;
  int jmn = 0, jsol = 1;
  float betmn = 1.e20f;
  betmx = -1.e20f;
  for (int i = 0; i < mmax; i++) {
    const float bi = (float)M.ld(F_B, i, mb), ai = (float)M.ld(F_A, i, mb);
    if (bi > 0.01f && bi < betmn) {
      betmn = bi;
      jmn = i;
      jsol = 1;
    } else if (bi <= 0.01f && ai < betmn) {
      betmn = ai;
      jmn = i;
      jsol = 0;
    }
    if (bi > betmx) betmx = bi;
  }
  if (jsol == 0)
    cc1 = betmn;
  else
    cc1 = gtsolh_dev((float)M.ld(F_A, jmn, mb), (float)M.ld(F_B, jmn, mb));
  cc1 = __fmul_rn(0.95f, cc1);
  cc1 = __fmul_rn(0.90f, cc1);
}

// phases of the flattened getsol/nevill state machine
enum { PH_SETUP = 0, PH_G_FIRST, PH_G_SCAN, PH_N_TOP, PH_N_OUTSIDE, PH_DONE };

// One column of Neville's table (nevill's x or y).  The caller owns the two columns as objects of their
// own: they are indexed at run time, so as members they would keep the whole state in local memory
// instead of registers, and as one object they change the register allocation of the team kernels.
struct alignas(16) SwdNevCol {
  double v[12];
};

// The mode and period loops of surfdisp96, getsol and nevill, flattened into one state machine that
// solves all modes 1..nmode of sequence `sq` for model b.  It asks for one secular value at a time,
// Delta(ceval), and never evaluates it itself:
//   start    once: prologue of surfdisp96 and the job's period range;
//   advance  while phase == PH_SETUP: next (mode, period) and its start values (PH_G_FIRST), or PH_DONE;
//   consume  one getsol/nevill step with Delta(ceval); stores an accepted root, cuts a failed mode off.
// The thread-mapped (swd_solve_sequence) and the team-mapped (swd_solve_team) searches both drive
// this one machine; they differ only in where and when the secular values are computed, so every
// mapping returns the same roots and counts the same evaluations.
//  cout  : [nmode_out][nper][stride] float32-rounded roots (0 where a mode does not exist)
//  cwork : [nper][stride] unrounded roots of the running mode (chain state), used when nmode > 1
// Neville's table xs/ys is most of the kernels' stack frame: the state is only passed by reference.
struct SwdRootSearch {
  static constexpr double dc = (double)0.005f;  // scan step
  // ---- job and output addressing
  const SwdSeq &sq;
  const double *periods;
  int nmode, all_modes;
  double *cout;
  long long cout_mode_stride;
  double *cwork;
  long long stride, b;
  unsigned int &n_evals;  // consumed secular values
  // ---- prologue of surfdisp96
  int llw;
  double cc, betmxd;
  // ---- loop-nest state (job / mode / period)
  int kb, jk;  // job = periods [kb, kb+jk)
  int iq = 1, k = 0, ift = 999, job_ierr = 0;
  double cprev = 0.0, del1st = 0.0;
  // ---- root-search state (getsol / nevill)
  double c1 = 0.0, c2 = 0.0, clow = 0.0, del1 = 0.0, del2 = 0.0, c3 = 0.0, del3 = 0.0, omega = 0.0,
         iomega = 0.0;
  double *xs, *ys;  // Neville's table, SwdNevCol::v of the caller
  int idir = 1, nev = 1, nctrl = 1, mm = 1, ifirst = 0;
  int phase = PH_SETUP;
  double ceval = 0.0;

  RFS_DEVINL SwdRootSearch(SwdNevCol &xs_, SwdNevCol &ys_, const SwdSeq &sq_, const double *periods_,
                           int nmode_, int all_modes_, double *cout_, long long cout_mode_stride_,
                           double *cwork_, long long stride_, long long b_, unsigned int &n_evals_)
      : sq(sq_), periods(periods_), nmode(nmode_), all_modes(all_modes_), cout(cout_),
        cout_mode_stride(cout_mode_stride_), cwork(cwork_), stride(stride_), b(b_),
        n_evals(n_evals_), xs(xs_.v), ys(ys_.v) {}

  // mb = the model's index for M.ld.  only_k < 0: the main pass over all periods; only_k >= 0: the
  // single-period job with which _surfdisp retries a period whose result was zero
  // (surfdisp.cpp:93-100, run by swd_retry_kernel)
  template <class MT>
  RFS_DEVINL void start(const MT &M, long long mb, int only_k) {
    float betmx, cc1;
    swd_start_values(M, mb, llw, betmx, cc1);
    cc = (double)cc1;
    betmxd = (double)betmx;
    kb = (only_k < 0) ? 0 : only_k;
    jk = (only_k < 0) ? sq.nper : 1;
  }

  // output index of period i of the job; the output block of mode iq
  RFS_DEVINL long long at(int i) const { return (long long)(sq.out_off + kb + i) * stride + b; }
  RFS_DEVINL double *mode_out() const {
    return cout + (all_modes ? (long long)(iq - 1) * cout_mode_stride : 0);
  }

  // label 1700/1750: mode iq is cut off from period k on (its results are 0), next mode
  RFS_DEVINL void cut_mode() {
    double *cq = mode_out();
    if (iq <= 1) job_ierr = 1;
    ift = k + 1;
    for (int i = k; i < jk; i++) cq[at(i)] = 0.0;
    iq++;
    k = 0;
  }

  // advance the (job, mode, period) nest until a root search starts or all is done
  RFS_DEVINL void advance() {
    for (;;) {
      if (iq <= nmode && k < jk && (k + 1 >= ift)) {  // reached through `if(k.ge.ift)`
        cut_mode();
        continue;
      }
      if (iq <= nmode && k >= jk) {  // mode finished normally
        iq++;
        k = 0;
        continue;
      }
      if (iq > nmode) {  // job finished
        phase = PH_DONE;
        return;
      }
      // ---- start values of (iq, k) (surfdisp96.f:257-276); surfdisp96's cm is cc
      const double one = 1.0e-2, onea = 1.5;
      const double twopi = 2.0 * RFS_PI64;
      const double t1 = __ldg(periods + sq.per_off + kb + k) * sq.scale;
      omega = twopi / t1;
      iomega = 1.0 / omega;
      if (k == 0 && iq == 1) {
        c1 = cc;
        clow = cc;
        ifirst = 1;
      } else if (k == 0 && iq > 1) {
        c1 = RFS_ADD(cwork[at(0)], RFS_MUL(one, dc));
        clow = c1;
        ifirst = 1;
      } else if (k > 0 && iq > 1) {
        ifirst = 0;
        clow = RFS_ADD(cwork[at(k)], RFS_MUL(one, dc));
        c1 = cprev;
        if (c1 < clow) c1 = clow;
      } else {
        ifirst = 0;
        c1 = RFS_SUB(cprev, RFS_MUL(onea, dc));
        clow = cc;
      }
      ceval = c1;
      phase = PH_G_FIRST;
      return;
    }
  }

  // label 1000 (getsol :457-470): the next scan point c2 = c1 +- dc, turned upward at clow
  RFS_DEVINL void next_scan_point() {
    for (;;) {
      c2 = (idir > 0) ? c1 + dc : c1 - dc;
      if (c2 <= clow) {
        idir = +1;
        c1 = clow;
        continue;
      }
      break;
    }
    ceval = c2;
  }

  // one step of getsol / nevill with val = Delta(ceval)
  RFS_DEVINL void consume(double val) {
    n_evals++;
    int iret = 0;  // 0 running, 1 root accepted, -1 failed, 2 nevill done
    bool body = false;
    if (phase == PH_G_FIRST) {
      del1 = val;
      if (ifirst == 1) del1st = del1;
      // plmn = dsign(1, del1st) * dsign(1, del1) >= 0 (:452-456)
      idir = (ifirst == 1 || neg1(del1st) == neg1(del1)) ? +1 : -1;
      next_scan_point();
      phase = PH_G_SCAN;
    } else if (phase == PH_G_SCAN) {  // one upward/downward scan step (getsol :457-479)
      del2 = val;
      if (neg1(del1) != neg1(del2)) {
        c3 = 0.5 * (c1 + c2);  // bracketed -> nevill: initial half
        ceval = c3;
        nev = 1;
        nctrl = 1;
        phase = PH_N_TOP;
      } else {
        c1 = c2;
        del1 = del2;
        if (c1 < cc || c1 >= (betmxd + dc)) {
          iret = -1;
        } else {
          next_scan_point();
        }
      }
    } else if (phase == PH_N_TOP) {
      del3 = val;
      nctrl = nctrl + 1;
      if (nctrl >= 100) {
        iret = 2;  // nevill exit by iteration cap -> cc = c3
      } else if (c3 < fmin(c1, c2) || c3 > fmax(c1, c2)) {
        nev = 0;
        c3 = 0.5 * (c1 + c2);
        ceval = c3;
        phase = PH_N_OUTSIDE;
      } else {
        body = true;
      }
    } else {  // PH_N_OUTSIDE
      del3 = val;
      body = true;
    }
    if (body) {
      const double s13 = del1 - del3;
      const double s32 = del3 - del2;
      if (neg1(del3) != neg1(del1)) {
        c2 = c3;
        del2 = del3;
      } else {
        c1 = c3;
        del1 = del3;
      }
      if (fabs(c1 - c2) <= 1.e-6 * c1) {
        iret = 2;
      } else {
        if (neg1(s13) != neg1(s32)) nev = 0;
        const double ss1 = fabs(del1), ss2 = fabs(del2);
        const double s1 = (double)0.01f * ss1, s2 = (double)0.01f * ss2;
        bool do_half = (s1 > ss2 || s2 > ss1 || nev == 0);
        if (!do_half) {
          if (nev == 2) {
            xs[mm] = c3;
            ys[mm] = del3;
          } else {
            xs[0] = c1;
            ys[0] = del1;
            xs[1] = c2;
            ys[1] = del2;
            mm = 1;
          }
          bool bad = false;
          for (int kk = 1; kk <= mm; kk++) {
            const int j = mm - kk;  // 0-based index of x(j)
            const double denom = ys[mm] - ys[j];
            if (fabs(denom) < 1.0e-10 * fabs(ys[mm])) {
              bad = true;
              break;
            }
            xs[j] = RFS_FMA(ys[mm], xs[j], RFS_MUL(-ys[j], xs[j + 1])) / denom;
          }
          if (!bad) {
            c3 = xs[0];
            nev = 2;
            mm = mm + 1;
            if (mm > 10) mm = 10;
          } else {
            do_half = true;
          }
        }
        if (do_half) {
          c3 = 0.5 * (c1 + c2);
          nev = 1;
          mm = 1;
        }
        ceval = c3;
        phase = PH_N_TOP;
      }
    }
    if (iret == 2) {
      c1 = c3;  // back in getsol (:483-487)
      iret = (c1 > betmxd) ? -1 : 1;
    }
    if (iret == 1) {
      cprev = c1;
      if (nmode > 1) cwork[at(k)] = c1;
      mode_out()[at(k)] = (double)(float)c1;  // cg(k)=sngl(c(k))
      k++;
      phase = PH_SETUP;
    } else if (iret == -1) {
      cut_mode();
      phase = PH_SETUP;
    }
  }
};

// K1: one thread per (model, sequence) drives SwdRootSearch; returns ierr of this job (1 =
// fundamental mode not found).
//
// The mode loop, the period loop, getsol and nevill are ONE loop whose body performs exactly one
// secular evaluation: lanes never wait for each other at period or mode boundaries.  The per-period
// retries of _surfdisp (surfdisp.cpp:93-100) are separate single-period jobs (swd_retry_kernel).
//
// Warp-cooperative tail: rare models need 5-10x more evaluations than the rest (upward scans from
// the floor velocity in the per-period retries).  All 32 lanes of a warp stay in the loop until
// the last one is done; lanes that are finished evaluate look-ahead scan points c2+j*dc for one
// scanning lane (same repeated additions, hence bit-identical grid) and hand the values over
// through shared memory (`wsm`, 32 doubles per warp).  `valid` = this lane owns a sequence.
// MT: model accessor; mb = this lane's model index for M.ld (the batch index b for the global block,
// the thread's column for a block staged in shared memory); b always indexes the outputs.
template <class MT>
RFS_DEVINL int swd_solve_sequence(const MT &M, long long b, long long mb, const SwdSeq &sq,
                                  const double *__restrict__ periods, int nmode, int all_modes,
                                  double *__restrict__ cout, long long cout_mode_stride,
                                  double *__restrict__ cwork, long long stride,
                                  unsigned int &n_evals, bool valid, double *wsm, int only_k) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int ifunc = sq.ifunc;
  SwdNevCol xs, ys;
  SwdRootSearch rs(xs, ys, sq, periods, nmode, all_modes, cout, cout_mode_stride, cwork, stride, b,
                   n_evals);
  rs.start(M, mb, only_k);
  if (!valid) rs.phase = PH_DONE;

  for (;;) {
    if (rs.phase == PH_SETUP) rs.advance();
    // ---- warp bookkeeping: who is finished, who is scanning upward
    const unsigned done_mask = __ballot_sync(FULL, rs.phase == PH_DONE);
    if (done_mask == FULL) break;
    const unsigned want_mask = __ballot_sync(FULL, rs.phase == PH_G_SCAN && rs.idir > 0);
    int nhelp = 0, hsrc = 0, hj = 0;
    bool helper = false;
    double e_c = rs.ceval, e_om = rs.omega, e_iom = rs.iomega;
    long long e_b = mb;
    int e_llw = rs.llw, e_if = ifunc;
    if (done_mask != 0u && want_mask != 0u) {
      hsrc = __ffs(want_mask) - 1;
      nhelp = __popc(done_mask);
      const double c_h = __shfl_sync(FULL, rs.ceval, hsrc);
      const double om_h = __shfl_sync(FULL, rs.omega, hsrc);
      const double iom_h = __shfl_sync(FULL, rs.iomega, hsrc);
      const long long b_h = __shfl_sync(FULL, mb, hsrc);
      const int llw_h = __shfl_sync(FULL, rs.llw, hsrc);
      const int if_h = __shfl_sync(FULL, ifunc, hsrc);
      if (rs.phase == PH_DONE) {
        helper = true;
        hj = __popc(done_mask & ((1u << lane) - 1u)) + 1;  // look-ahead index 1..nhelp
        double c = c_h;
        for (int t = 0; t < hj; t++) c = c + SwdRootSearch::dc;  // same additions as the scanning lane
        e_c = c;
        e_om = om_h;
        e_iom = iom_h;
        e_b = b_h;
        e_llw = llw_h;
        e_if = if_h;
      }
    }

    // ---- the single secular-function evaluation site
    double val = 0.0;
    if (rs.phase != PH_DONE || helper) {
      const double wv = e_om / e_c;
      val = (e_if == 1) ? dltar1_dev(wv, e_om, M, e_b, e_llw)
                        : dltar4_dev(wv, e_om, e_iom, M, e_b, e_llw);
    }
    if (nhelp) {
      if (helper) wsm[hj] = val;
      __syncwarp();
    }
    if (rs.phase == PH_DONE) {
      if (nhelp) __syncwarp();
      continue;
    }
    rs.consume(val);
    // the lane being helped consumes the look-ahead values while its scan simply slides upward (a
    // bracket or a failed scan leaves PH_G_SCAN).  A call site of its own keeps the common path
    // straight-line: one shared loop over val, wsm[1..] is 2 % slower (B200 at 1000 W).
    if (nhelp && lane == hsrc)
      for (int j = 1; j <= nhelp && rs.phase == PH_G_SCAN && rs.idir > 0; j++) rs.consume(wsm[j]);
    if (nhelp) __syncwarp();  // wsm may be rewritten in the next trip
  }
  return rs.job_ierr;
}

}  // namespace rfs
