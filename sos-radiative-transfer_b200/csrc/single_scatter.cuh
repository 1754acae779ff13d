// Exact single scattering of azimuth-resolved radiance (include/sos_b200.h: sos_single_scatter_correction).
//
// The first order is linear in its coefficient vectors C_atm = alb_atm P0_atm and C_mix = C_atm f_atm + alb_aer P0_aer f_aer
// (first_order.cuh), so its K-term Fourier series is replaced by the exact value at an azimuth phi by adding the closed form
// of the difference
//     dP0(mu, phi) = p(cos Theta(mu, mu0, phi)) / T - sum_{m < K} (2 - delta_m0) P0_m(mu) cos(m phi)
// (cos Theta = -mu0 mu + sqrt(1 - mu0^2) sqrt(1 - mu^2) cos phi; T the mode-0 normalisation of the series).  The closed form
// reads C at the column (direct beam) and at its mirror (mirror-reflected beam), so one thread evaluates dP0 at those two
// columns for both phase functions and then walks the requested rows with the calls of first_order_regions_kernel.
// A specular ground keeps the mirror term and the upward carry rho I1[L-1, mirror]; a diffuse ground (Lambert, Ross-Li,
// ocean) has neither: its order-1 surface terms are not single scattering by the phase function and stay the series.
#pragma once
#include "common.cuh"
#include "first_order.cuh"
#include "phase.cuh"

namespace sosss {

constexpr int THREADS = 128;

// one entry = one geometry of a mode-0 batch (mirrors sos_ss_entry of include/sos_b200.h)
struct Entry {
  int scenario, geo;
  int family[2], series[2], tab_off[2], tab_n[2];
  double g[2], norm[2], w[4];
};

struct Tables {
  const Entry* ent;     // [n]
  const double* P0m;    // [n_vec][K][N] the mode vectors the radiance was summed with
  const double* tab;    // tabulated phase functions: abscissae at tab_off, values at tab_off + tab_n
  const double* wcos;   // [n_az][K]: 1 (m = 0), 2 cos(m phi_p)
  const double* cphi;   // [n_az]
  const int* rows;      // [n_rows]
};

// dP0 of part j (0 atmosphere, 1 aerosol) at column col and azimuth p
__device__ __forceinline__ double delta_p0(const Entry& e, int j, const Tables& t, int K, int N, int p, int col, double mu,
                                           double mu0) {
  if (e.family[j] < 0) return 0.0;   // isotropic: the series is exact
  sosphase::PhaseArgs a;
  a.family = e.family[j]; a.g = e.g[j];
  a.tab_x = t.tab + e.tab_off[j]; a.tab_y = a.tab_x + e.tab_n[j]; a.tab_n = e.tab_n[j];
  const double c = -mu0 * mu + sqrt(1.0 - mu0 * mu0) * sqrt(1.0 - mu * mu) * t.cphi[p];
  const double* __restrict__ v = t.P0m + static_cast<size_t>(e.series[j]) * K * N + col;
  const double* __restrict__ w = t.wcos + static_cast<size_t>(p) * K;
  double series = 0.0;
  for (int m = 0; m < K; ++m) series = fma(w[m], v[static_cast<size_t>(m) * N], series);
  return sosphase::phase_value(a, c) / e.norm[j] - series;
}

// thread = (entry k, azimuth p, column m); out[geo][r][p][m] += first order of dC at every requested row r
__global__ void __launch_bounds__(THREADS)
single_scatter_kernel(const GridDev g, const Tables t, int n, int K, int n_rows, int n_az, double* __restrict__ out) {
  const long long e_id = static_cast<long long>(blockIdx.x) * THREADS + threadIdx.x;
  const int L = g.L, M = g.M, N = g.N;
  if (e_id >= static_cast<long long>(n) * n_az * N) return;
  const int m = static_cast<int>(e_id % N);
  const int p = static_cast<int>((e_id / N) % n_az);
  const int k = static_cast<int>(e_id / (static_cast<long long>(N) * n_az));
  const Entry e = t.ent[k];
  const int s = e.scenario;
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const sos_scenario sc = g.scen[s];
  const double PI = 3.14159265358979323846;
  const double mu0 = sc.mu0;
  const double F0 = PI / mu0;
  const double T = sc.tauStar_tot;
  const double q = 1.0 / (4.0 * PI);
  const bool diffuse = g.surface == SOS_SURFACE_LAMBERT_DIFFUSE || g.surface == SOS_SURFACE_ROSSLI || g.surface == SOS_SURFACE_OCEAN;
  const double S = diffuse ? 0.0 : F0 * sc.grd_alb * exp(-T / mu0);
  const int mir = N - 1 - m;

  // dC at the column and at its mirror
  double Catm[2], Cmix[2];
  for (int h = 0; h < 2; ++h) {
    const int col = h ? mir : m;
    const double mu = g.mu[col];
    const double ca = delta_p0(e, 0, t, K, N, p, col, mu, mu0) * e.w[0];
    Catm[h] = ca;
    Cmix[h] = ca * e.w[1] + (delta_p0(e, 1, t, K, N, p, col, mu, mu0) * e.w[2]) * e.w[3];
  }
  double* __restrict__ o = out + (static_cast<size_t>(e.geo) * n_rows * n_az + p) * N + m;
  const size_t row_step = static_cast<size_t>(n_az) * N;

  if (m == M - 1 || m == M) {
    for (int r = 0; r < n_rows; ++r) {
      const int row = t.rows[r];
      const double tt = tau[row];
      const bool mix = sosfirst::region_of(g, row) == 1;
      const double Cm = mix ? Cmix[0] : Catm[0], Cr = mix ? Cmix[1] : Catm[1];
      o[r * row_step] += (mu0 / (mu0 + g.mu[m])) * Cm * (F0 * q) * exp(-tt / mu0) +
                         (mu0 / (mu0 - g.mu[m])) * Cr * (S * q) * exp(-(T - tt) / mu0);
    }
    return;
  }

  sosfirst::Col c;
  c.mu0 = mu0; c.F0q = F0 * q; c.Sq = S * q; c.T = T;
  c.mu = g.mu[m];
  c.inv_mu = 1.0 / c.mu;
  c.Cm_atm = Catm[0]; c.Cmir_atm = Catm[1];
  c.Cm_mix = Cmix[0]; c.Cmir_mix = Cmix[1];
  if (m < M - 1) {
    c.down = true;
    c.special = fabs(c.mu + mu0) < SOS_MU0_TOLERANCE;
    for (int r = 0; r < n_rows; ++r) {
      const int row = t.rows[r];
      const int kr = sosfirst::region_of(g, row);
      const double tt = tau[row];
      o[r * row_step] += sosfirst::i1_value(c, kr == 1, tt, exp(-tt / mu0), exp(-(T - tt) / mu0),
                                            sosfirst::down_carry(g, c, tau, kr, T), sosfirst::down_region(g, tau, kr, T, mu0));
    }
    return;
  }

  // upward column: carry at the surface row = rho * (mirror downward column at row L-1), 0 over a diffuse ground
  const int R = g.nreg;
  double surf_carry = 0.0;
  if (!diffuse) {
    sosfirst::Col d = c;
    d.mu = g.mu[mir];
    d.inv_mu = 1.0 / d.mu;
    d.down = true;
    d.special = fabs(d.mu + mu0) < SOS_MU0_TOLERANCE;
    d.Cm_atm = Catm[1]; d.Cmir_atm = Catm[0];
    d.Cm_mix = Cmix[1]; d.Cmir_mix = Cmix[0];
    const double tt = tau[L - 1];
    surf_carry = sc.grd_alb * sosfirst::i1_value(d, (R - 1) == 1, tt, exp(-tt / mu0), exp(-(T - tt) / mu0),
                                                 sosfirst::down_carry(g, d, tau, R - 1, T),
                                                 sosfirst::down_region(g, tau, R - 1, T, mu0));
  }
  c.down = false;
  c.special = fabs(c.mu - mu0) < SOS_MU0_TOLERANCE;
  sosfirst::RegionK rks[3];
  double carry_k[3];
  for (int kk = 0; kk < R; ++kk)
    rks[kk] = (kk == R - 1) ? sosfirst::region_consts(tau[L - 1], T, T, mu0)
                            : sosfirst::region_consts(tau[g.rstart[kk + 1]], tau[g.rstart[kk + 1] - 1], T, mu0);
  carry_k[R - 1] = surf_carry;
  for (int kk = R - 2; kk >= 0; --kk) {
    const double tt = tau[g.rstart[kk + 1]];
    carry_k[kk] = sosfirst::i1_value(c, (kk + 1) == 1, tt, exp(-tt / mu0), exp(-(T - tt) / mu0), carry_k[kk + 1], rks[kk + 1]);
  }
  for (int r = 0; r < n_rows; ++r) {
    const int row = t.rows[r];
    const int kr = sosfirst::region_of(g, row);
    const double tt = tau[row];
    o[r * row_step] += sosfirst::i1_value(c, kr == 1, tt, exp(-tt / mu0), exp(-(T - tt) / mu0), carry_k[kr], rks[kr]);
  }
}

}  // namespace sosss
