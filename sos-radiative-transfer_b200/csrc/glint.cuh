// Cox-Munk ocean glint (include/sos_b200.h: SOS_SURFACE_OCEAN, sos_build_glint_modes, sos_glint_correction).
//
// rho_glint(mu_i, mu_v, phi) = r(omega) exp(-tan^2 theta_n / sigma^2) S / (4 sigma^2 mu_i mu_v mu_n^4), reflectance-factor
// units: the isotropic slope distribution of Cox & Munk (1954) with variance sigma^2 = 0.003 + 0.00512 W (computed by the
// host), the unpolarised Fresnel reflectance r at the local incidence angle omega, cos 2 omega = mu_i mu_v - sin_i sin_v cos phi,
// the facet tilt mu_n = (mu_i + mu_v) / (2 cos omega) and Smith shadowing S = 1 / (1 + Lambda(mu_i) + Lambda(mu_v)).  phi is
// the engine's propagation azimuth relative to the incident light's (DESIGN §10), so the glint sits at phi = 0.  Every
// operation is written symmetric in (mu_i, mu_v): the reflectance is exactly reciprocal.
//
// Mode matrices: R_m(mu_i, mu_c) = (1/pi) int_0^pi rho_glint cos(m phi) dphi (trapezoid on the host's nodes), stored in the
// transposed layout of brdf.cuh ([c][i]); the entries of the downward column mu = 0- are 0 (quadrature weight 0).  The
// coupling is the one-matrix form of sosbrdf::coupling.
#pragma once
#include "brdf.cuh"

namespace sosglint {

// Smith's Lambda(mu) = (e^{-nu^2} / (nu sqrt(pi)) - erfc(nu)) / 2, nu = mu / (sigma sqrt(1 - mu^2)); Lambda(1) = 0 exactly
__device__ __forceinline__ double smith_lambda(double mu, double sigma) {
  if (mu >= 1.0) return 0.0;
  const double nu = mu / (sigma * sqrt((1.0 - mu) * (1.0 + mu)));
  return 0.5 * (exp(-nu * nu) / (nu * 1.7724538509055160273) - erfc(nu));
}

__device__ __forceinline__ double shadowing(double mi, double mv, double sigma) {
  return 1.0 / (1.0 + (smith_lambda(mi, sigma) + smith_lambda(mv, sigma)));
}

// unpolarised Fresnel reflectance at incidence cosine ci, relative refractive index n > 1
__device__ __forceinline__ double fresnel(double ci, double n) {
  const double ct = sqrt(1.0 - (1.0 - ci * ci) / (n * n));
  const double rs = (ci - n * ct) / (ci + n * ct), rp = (n * ci - ct) / (n * ci + ct);
  return 0.5 * (rs * rs + rp * rp);
}

// rho_glint at cos phi = cphi with the shadowing factor S (independent of phi) given: mi, mv in (0, 1].  With
// D = 4 cos^2 omega - (mi + mv)^2 = (s_i - s_v)^2 + 2 s_i s_v (1 - cos phi), a sum of two terms >= 0 (no cancellation near the
// specular direction, where the grazing columns would lose digits to it): mu_n^2 = (mi + mv)^2 / ((mi + mv)^2 + D) and
// tan^2 theta_n = D / (mi + mv)^2; at the specular point D = 0 exactly.
__device__ __forceinline__ double glint(double mi, double mv, double cphi, double sigma2, double n, double S) {
  const double si = sqrt((1.0 - mi) * (1.0 + mi)), sv = sqrt((1.0 - mv) * (1.0 + mv));
  const double D = (si - sv) * (si - sv) + 2.0 * (si * sv) * (1.0 - cphi);
  const double sum2 = (mi + mv) * (mi + mv);
  const double q = sum2 + D;                                           // 4 cos^2 omega
  const double mn2 = sum2 / q;                                         // mu_n^2
  return fresnel(0.5 * sqrt(q), n) * exp(-(D / sum2) / sigma2) * S / (4.0 * sigma2 * (mi * mv) * (mn2 * mn2));
}

// One thread per element (c, i): rho_glint once per azimuth node, every mode accumulated in shared memory
// ([n_modes][BUILD_THREADS], one column per thread).  wcos[k][m] = trapezoid weight of node k * cos(m phi_k) / pi, cphi[k] =
// cos(phi_k).
__global__ void __launch_bounds__(sosbrdf::BUILD_THREADS)
glint_modes_kernel(const double* __restrict__ mu, int M, double sigma2, double n, const double* __restrict__ cphi,
                   const double* __restrict__ wcos, int n_nodes, int n_modes, double* __restrict__ R, int ldr, size_t stride) {
  constexpr int T = sosbrdf::BUILD_THREADS;
  extern __shared__ double acc[];
  const long long e = static_cast<long long>(blockIdx.x) * T + threadIdx.x;
  if (e >= static_cast<long long>(M) * (M - 1)) return;
  const int c = static_cast<int>(e / (M - 1)), i = static_cast<int>(e % (M - 1));
  const double mc = fabs(mu[c]), mi = mu[M + 1 + i];
  const int K = n_modes;
  double* my = acc + threadIdx.x;
  for (int j = 0; j < K; ++j) my[j * T] = 0.0;
  if (mc > 0.0) {
    const double S = shadowing(mc, mi, sqrt(sigma2));
    for (int k = 0; k < n_nodes; ++k) {
      const double r = glint(mc, mi, cphi[k], sigma2, n, S);
      const double* __restrict__ w = wcos + static_cast<size_t>(k) * K;
      for (int j = 0; j < K; ++j) my[j * T] += w[j] * r;
    }
  }
  const size_t off = static_cast<size_t>(c) * ldr + i;
  for (int j = 0; j < K; ++j) R[off + j * stride] = my[j * T];
}

}  // namespace sosglint
