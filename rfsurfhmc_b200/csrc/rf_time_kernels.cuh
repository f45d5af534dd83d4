// K5 — time-domain receiver functions: Ligorria-Ammon iterative deconvolution.
//
// Replaces /root/reference/src/RF/deconit.f90 (gauss_filter :15-32, apply_gaussian :34-52,
// shift_data :54-72, mycorrelate :99-115, myconvolve :117-133, deconit :135-198) and its callers
// cal_rf_time / cal_rf_par_time[_all] (/root/reference/src/RF/RFModule.f90:11-191).
//
// Re-design: the reference spends 8 FFTW transforms per iteration (each with plan create/destroy)
// on quantities that are linear in the spike train p.  Here everything except the argmax stays in
// the frequency domain: P = rfft(p) is updated analytically when a spike is added
// (P_k += a e^{-2 pi i k idx/N}), the residual spectrum is R = U_f - dt P G W and its power follows
// from Parseval, so ONE inverse FFT per iteration (the cross-correlation whose argmax picks the
// next spike) remains.  Same mathematics; values differ from the 8-FFT form at rounding level.
// One block per (model, row): row 0 = the receiver function itself (u = irfft(R22), w = irfft(R21)),
// row r>0 = Frechet trace r-1 (u = irfft(D_r), w = irfft(R21^2)).
#pragma once
#include "rf_kernels.cuh"

namespace rfs {

// Everything the iteration needs of u and w are two products: UW = U conj(W) and W2 = |W|^2:
//   cross-correlation spectrum   R conj(W) = UW - dt W2 P              (R = U - dt P W)
//   residual power (Parseval)    sum |R|^2 = sum |U|^2 - 2 dt Re(P conj(UW)) + dt^2 |P|^2 W2
// dynamic smem: cd buf[nft] + cd UW[n2] + cd P[n2] + double W2[n2] + 64 doubles   (74 KB at nft = 2048:
// three blocks per SM; the twiddle table stays in global memory / L1)
// Gaussian width: width ig of the block's row's set (GaussView, rfs_config_obs_gauss) or `shared`; a row of
// an out-of-range set computes with `shared` and is failed by rf_trace_grad_kernel.
__global__ void __launch_bounds__(256, 3) rf_time_kernel(const double2 *__restrict__ spec, const double2 *__restrict__ dspec,
                               long long B, int nrow, int nt, int nft, int logn, double dt,
                               GaussView gauss, int ig, double shared, double tshift, double *__restrict__ rf,
                               long long ldrf, double *__restrict__ traces, const double2 *__restrict__ tw) {
  extern __shared__ double smem[];
  const int n2 = nft / 2 + 1;
  cd *buf = reinterpret_cast<cd *>(smem);
  cd *UW = buf + nft;
  cd *P = UW + n2;
  double *W2 = reinterpret_cast<double *>(P + n2);
  double *red = W2 + n2;
  const int nrow1 = nrow + 1;
  const long long b = blockIdx.x / nrow1;
  const int r = (int)(blockIdx.x % nrow1);
  const int tid = threadIdx.x, nth = blockDim.x;
  const double minderr = (double)0.001f;
  const double f0 = gauss.row_a(b, ig, shared);

  // ---- spectra of u and w (the reference goes through the time domain: c2r drops Im of bins 0, N/2)
  double lpu = 0.0, lpw = 0.0;
  for (int k = tid; k < n2; k += nth) {
    const double2 a21 = spec[(b * 2 + 0) * n2 + k], a22 = spec[(b * 2 + 1) * n2 + k];
    cd su, sw;
    if (r == 0) {
      su = cd(a22.x, a22.y);
      sw = cd(a21.x, a21.y);
    } else {
      const double2 d = dspec[(b * (long long)nrow + (r - 1)) * n2 + k];
      su = cd(d.x, d.y);
      const cd s21(a21.x, a21.y);
      sw = s21 * s21;
    }
    if (k == 0 || k == nft / 2) {
      su.y = 0.0;
      sw.y = 0.0;
    }
    const double freq = (double)k / (nft * dt);
    const double gx = 2 * RFS_PI32 * freq / f0;
    const double g = exp(-0.25 * (gx * gx));
    const cd Uf = su * g;
    const cd Wf = sw * g;  // also G * rfft(wcopy): the factor G of apply_gaussian(temp1) is the same g
    const double wgt = (k == 0 || k == nft / 2) ? 1.0 : 2.0;
    lpu += wgt * norm2(Uf);
    lpw += wgt * norm2(Wf);
    UW[k] = Uf * conj(Wf);
    W2[k] = norm2(Wf);
    P[k] = cd(0.0, 0.0);
  }
  const double su2 = block_reduce(lpu, red, false);  // sum_k w_k |U_k|^2 = N * sum_t u_t^2
  const double pw = block_reduce(lpw, red, false) / (double)nft;
  const double pu = su2 / (double)nft;
  const double invpw = 1. / pw / dt;
  const double invpu = 1. / pu / dt;
  double sumsq_i = 1.0;
  double d_error = 100 * invpw + minderr;
  for (int it = 1; it <= 200; it++) {
    if (fabs(d_error) <= minderr) break;
    // cuw = irfft( rfft(rflt) conj(rfft(wflt)) ) dt ,  rfft(rflt) = Uf - dt P Wc
    const cd *z = block_irfft<false>([&](int k) { return UW[k] - (dt * W2[k]) * P[k]; }, buf, nft, logn, tw);
    // first maximum of |cuw| over the first nft/2 lags (maxloc, deconit.f90:178)
    double best = -1.0;
    int bi = 0x7fffffff;
    for (int t = tid; t < nft / 2; t += nth) {
      const double v = fabs(irfft_at(z, t));
      if (v > best) {
        best = v;
        bi = t;
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_down_sync(0xffffffffu, best, o);
      const int oi = __shfl_down_sync(0xffffffffu, bi, o);
      if (ob > best || (ob == best && oi < bi)) {
        best = ob;
        bi = oi;
      }
    }
    __syncthreads();
    if ((tid & 31) == 0) {
      red[tid >> 5] = best;
      red[32 + (tid >> 5)] = (double)bi;
    }
    __syncthreads();
    if (tid == 0) {
      const int nw = (nth + 31) >> 5;
      double bb = red[0];
      int ii = (int)red[32];
      for (int w = 1; w < nw; w++) {
        const double ob = red[w];
        const int oi = (int)red[32 + w];
        if (ob > bb || (ob == bb && oi < ii)) {
          bb = ob;
          ii = oi;
        }
      }
      red[0] = (double)ii;
      red[1] = irfft_at(z, ii) / nft * dt;  // cuw(idx) = irfft(..)*dt
    }
    __syncthreads();
    const int idx = (int)red[0];
    const double amp = red[1] * invpw / dt;
    __syncthreads();
    // P += amp * rfft(delta_idx);  new residual power by Parseval
    double l = 0.0;
    for (int k = tid; k < n2; k += nth) {
      // exp(-2 pi i k idx / nft) from the twiddle table
      const int kk = (k * idx) & (nft - 1);  // nft is a power of two, k*idx < 2^24
      const cd ph = tw_lookup<false>(tw, kk, nft, -1);
      const cd pk = P[k] + amp * ph;
      P[k] = pk;
      const cd uw = UW[k];
      const double w = (k == 0 || k == nft / 2) ? 1.0 : 2.0;
      l += w * (dt * W2[k] * norm2(pk) - 2.0 * (pk.x * uw.x + pk.y * uw.y));
    }
    const double sumsq = (su2 + dt * block_reduce(l, red, false)) / (double)nft * dt * invpu;
    d_error = 100. * (sumsq_i - sumsq);
    sumsq_i = sumsq;
  }
  // ---- p <- gaussian(p), shift by tshift, back to time (deconit.f90:191-194)
  for (int k = tid; k < n2; k += nth) {
    const double freq = (double)k / (nft * dt);
    const double gx = 2 * RFS_PI32 * freq / f0;
    const double g = exp(-0.25 * (gx * gx));
    cd pk = P[k] * g;
    if (k == 0 || k == nft / 2) pk.y = 0.0;  // irfft/rfft round trip inside apply_gaussian
    P[k] = pk * cis(-((double)k / (nft * dt) * RFS_PI32 * 2 * tshift));
  }
  __syncthreads();
  const cd *z = block_irfft<false>([&](int k) { return P[k]; }, buf, nft, logn, tw);
  double *dst = (r == 0) ? rf + b * ldrf : traces + (b * (long long)nrow + (r - 1)) * nt;
  for (int t = tid; t < nt; t += nth) dst[t] = irfft_at(z, t) / nft;
}

// misfit and gradient from materialised Frechet traces (time-domain method, where the adjoint
// shortcut does not apply because deconit is nonlinear).  One thread per (model, layer).
//   traces [B][4][n][nt] (rho, vp, vs, h);  chain [P][n][B];  rf [B][ldrf];  grad [B][P n]
//   P = 3: the third block is the Vp/Vs gradient dadk*kvp + drda*dadk*krho (dadk = vs)
//   flag [B] or NULL: only written (0) for a row whose observation-set index is out of range; such a
//   row gets U 0, grad 0 and a NaN trace.  The residual is 0 at the samples the row's set does not fit
//   (ObsSets::observed).
template <int P>
__global__ void rf_trace_grad_kernel(const double *__restrict__ traces, const double *__restrict__ chain,
                                     double *__restrict__ rf, long long ldrf, ObsSets obs, long long B,
                                     int n, int nt, double *__restrict__ U, double *__restrict__ grad,
                                     unsigned char *__restrict__ flag, int accumulate) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * n) return;
  const long long b = i % B;
  const int m = (int)(i / B);
  const int set = obs.row_set(b);
  if (set < 0) {
    grad[b * P * n + m] = 0.0;
    grad[b * P * n + n + m] = 0.0;
    if (P == 3) grad[b * P * n + 2 * n + m] = 0.0;
    if (m == 0) {
      for (int t = 0; t < nt; t++) rf[b * ldrf + t] = nan("");
      U[b] = 0.0;
      if (flag) flag[b] = 0;
    }
    return;
  }
  const double *dobs = obs.row(set);
  const long long nB = (long long)n * B;
  const double dadb = chain[0 * nB + m * B + b], drda = chain[1 * nB + m * B + b];
  const double dadk = P == 3 ? chain[2 * nB + m * B + b] : 0.0;
  const double *kr = traces + ((b * 4 + 0) * n + m) * (long long)nt;
  const double *ka = traces + ((b * 4 + 1) * n + m) * (long long)nt;
  const double *kb = traces + ((b * 4 + 2) * n + m) * (long long)nt;
  const double *kh = traces + ((b * 4 + 3) * n + m) * (long long)nt;
  double g0 = 0.0, g1 = 0.0, g2 = 0.0, us = 0.0;
  for (int t = 0; t < nt; t++) {
    const double res = obs.observed(set, t) ? rf[b * ldrf + t] - dobs[t] : 0.0;
    g0 += (kb[t] + dadb * ka[t] + drda * dadb * kr[t]) * res;
    g1 += kh[t] * res;
    if (P == 3) g2 += (dadk * ka[t] + drda * dadk * kr[t]) * res;
    us += res * res;
  }
  if (accumulate) {
    g0 += grad[b * P * n + m];
    g1 += grad[b * P * n + n + m];
    if (P == 3) g2 += grad[b * P * n + 2 * n + m];
  }
  grad[b * P * n + m] = g0;
  grad[b * P * n + n + m] = g1;
  if (P == 3) grad[b * P * n + 2 * n + m] = g2;
  if (m == 0) U[b] = accumulate ? U[b] + 0.5 * us : 0.5 * us;
}

}  // namespace rfs
