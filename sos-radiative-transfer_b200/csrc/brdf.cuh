// Ross-Li bidirectional ground reflectance (include/sos_b200.h: SOS_SURFACE_ROSSLI, sos_build_brdf_modes).
//
// rho(mu_i, mu_v, psi) = f_iso + f_vol K_vol + f_geo K_geo with the RossThick and LiSparse-Reciprocal kernels of Lucht,
// Schaaf & Strahler (2000), h/b = 2, b/r = 1; psi is the Ross-Li relative azimuth (hot spot at psi = 0).  Both zenith
// arguments are clamped to mu >= mu_min (the caller's constant, brdf.BRDF_MU_MIN): K_geo grows like sec(theta) towards the
// horizon.  The kernels are linear in the weights, so the surface coupling of every scenario is made of two grid-only
// matrices per azimuthal mode; the isotropic weight is the lambert_diffuse coupling itself.
//
// Mode matrices, engine convention (phi = propagation azimuth relative to the incident light's, psi = phi - pi):
//   R^k_m(mu_i, mu_c) = (1/pi) int_0^pi K_k(mu_i, mu_c, phi - pi) cos(m phi) dphi   (trapezoid on the host's nodes)
// stored TRANSPOSED for the coupling mat-vec: element (c, i) at R + m * mode_stride + c * ldr + i, c = 0 .. M-1 the
// downward columns (|mu_c|), i = 0 .. M-2 the upward columns M+1 .. N-1, so that the threads of a CTA, one per upward
// column, read consecutive addresses.
#pragma once
#include "common.cuh"

namespace sosbrdf {

constexpr int MAX_MODES = 64;
constexpr int MAX_NODES = 1024;
constexpr int MAX_SETS = 64;      // mode matrix pairs one plan can index (sos_plan_set_brdf)
constexpr int BUILD_THREADS = 64;

// What the coupling kernels read (plan-owned buffers; all nullptr on other surfaces).  The Cox-Munk ocean (glint.cuh) uses
// the same buffers with one matrix per set: R[2 j] = glint, R[2 j + 1] = nullptr, f = (f_glint, 0), the second beam unread.
struct BrdfDev {
  const double* const* R;  // [n_sets][2] device pointers: R[2 j] = vol, R[2 j + 1] = geo, [M][ldr] each (transposed, above)
  const int* set;          // [S] mode matrix pair of each scenario
  const double* f;         // [S][2] (f_vol, f_geo)
  const double* beam;      // [S][2][M-1] beta_{k,m}(mu_i) = R^k_m(mu_i, mu0): the direct-beam reflection per unit e^{-T/mu0}
  int ldr;
};

__device__ __forceinline__ void rossli_kernels(double mi, double mv, double cpsi, double& kvol, double& kgeo) {
  const double PI = 3.14159265358979323846;
  const double si = sqrt((1.0 - mi) * (1.0 + mi)), sv = sqrt((1.0 - mv) * (1.0 + mv));
  const double cx = fmin(fmax(mi * mv + si * sv * cpsi, -1.0), 1.0);
  const double xi = acos(cx);
  kvol = ((0.5 * PI - xi) * cx + sin(xi)) / (mi + mv) - 0.25 * PI;
  const double ti = si / mi, tv = sv / mv, seci = 1.0 / mi, secv = 1.0 / mv;
  const double d2 = (ti - tv) * (ti - tv) + 2.0 * ti * tv * (1.0 - cpsi);   // D^2 without cancellation at the hot spot
  const double tts = ti * tv, s2 = (1.0 - cpsi) * (1.0 + cpsi);   // sin^2 psi
  const double ct = fmin(fmax(2.0 * sqrt(d2 + tts * tts * s2) / (seci + secv), -1.0), 1.0);
  const double t = acos(ct);
  const double O = (t - sin(t) * ct) * (seci + secv) / PI;
  kgeo = O - (seci + secv) + 0.5 * (1.0 + cx) * (seci * secv);
}

// One thread per element (c, i): both kernels once per azimuth node, every mode accumulated.  The mode accumulators live
// in shared memory, one column per thread: [2 n_modes][BUILD_THREADS].  wcos[k][m] = trapezoid weight of node k * cos(m phi_k)
// / pi, cpsi[k] = cos(phi_k - pi).
__global__ void __launch_bounds__(BUILD_THREADS)
brdf_modes_kernel(const double* __restrict__ mu, int M, double mu_min, const double* __restrict__ cpsi,
                  const double* __restrict__ wcos, int n_nodes, int n_modes, double* __restrict__ Rvol,
                  double* __restrict__ Rgeo, int ldr, size_t stride) {
  extern __shared__ double acc[];
  const long long e = static_cast<long long>(blockIdx.x) * BUILD_THREADS + threadIdx.x;
  if (e >= static_cast<long long>(M) * (M - 1)) return;
  const int c = static_cast<int>(e / (M - 1)), i = static_cast<int>(e % (M - 1));
  const double mc = fmax(fabs(mu[c]), mu_min), mi = fmax(mu[M + 1 + i], mu_min);
  const int K = n_modes;
  double* my = acc + threadIdx.x;
  for (int j = 0; j < 2 * K; ++j) my[j * BUILD_THREADS] = 0.0;
  for (int k = 0; k < n_nodes; ++k) {
    double kv, kg;
    rossli_kernels(mc, mi, cpsi[k], kv, kg);
    const double* __restrict__ w = wcos + static_cast<size_t>(k) * K;
    for (int j = 0; j < K; ++j) {
      my[j * BUILD_THREADS] += w[j] * kv;
      my[(K + j) * BUILD_THREADS] += w[j] * kg;
    }
  }
  const size_t off = static_cast<size_t>(c) * ldr + i;
  for (int j = 0; j < K; ++j) {
    Rvol[off + j * stride] = my[j * BUILD_THREADS];
    Rgeo[off + j * stride] = my[(K + j) * BUILD_THREADS];
  }
}

// The two kernel mat-vecs of one upward column i: sum_c u_c R^k[c][i] in ascending c (a fixed order: deterministic).
__device__ __forceinline__ void coupling(const BrdfDev& b, int s, const double* __restrict__ u, int M, int i, double& sv,
                                         double& sg) {
  const int j = b.set[s];
  const double* __restrict__ Rv = b.R[2 * j] + i;
  const double* __restrict__ Rg = b.R[2 * j + 1] + i;
  const size_t ld = static_cast<size_t>(b.ldr);
  double av = 0.0, ag = 0.0;
#pragma unroll 4
  for (int c = 0; c < M; ++c) {
    av += u[c] * Rv[c * ld];
    ag += u[c] * Rg[c * ld];
  }
  sv = av;
  sg = ag;
}

// The one-matrix form (the ocean's glint): sum_c u_c R[c][i] in ascending c.
__device__ __forceinline__ double coupling(const BrdfDev& b, int s, const double* __restrict__ u, int M, int i) {
  const double* __restrict__ R = b.R[2 * b.set[s]] + i;
  const size_t ld = static_cast<size_t>(b.ldr);
  double a = 0.0;
#pragma unroll 4
  for (int c = 0; c < M; ++c) a += u[c] * R[c * ld];
  return a;
}

// u_c = -2 w_c mu_c I[L-1, c], c = 0 .. M-1, with w the trapezoid weights of the ascending downward half (the abscissae of
// the lambert_readme coupling): the reflected radiance of mode m is 2 int_0^1 rho_m(mu, mu') I_m(-mu') mu' dmu' = sum_c u_c R[c][i]
__device__ __forceinline__ double coupling_weight(const double* __restrict__ mu, int M, int c) {
  const double hi = (c + 1 < M) ? mu[c + 1] : mu[c], lo = (c > 0) ? mu[c - 1] : mu[c];
  return -2.0 * (0.5 * (hi - lo)) * mu[c];
}

}  // namespace sosbrdf
