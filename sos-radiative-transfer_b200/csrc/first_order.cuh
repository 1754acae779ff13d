// Closed-form first order of scattering.
//   three regions : SOS_Aer_main_specular.py:104-292 (the Lambertian driver shares it after "repair A",
//                   SURVEY.md 8c)
//   single layer  : I1_NumInt, SOS_Aer_I1_In.py:13-58
//
// Every general column is   carry * e^{(tau_t - tau_b)/mu}
//                         + mu0/(mu0+mu) C[m]      F0/(4pi) (e^{-tau_t/mu0} - e^{-tau_d/mu0} e^{(tau_t-tau_d)/mu})
//                         + mu0/(mu0-mu) C[mirror] S /(4pi) (e^{-(T-tau_t)/mu0} - e^{-(T-tau_s)/mu0} e^{(tau_t-tau_s)/mu})
// with region-dependent (tau_b, tau_d, tau_s) -- the same expression for both hemispheres because
// -(tau_b - tau_t)/mu == (tau_t - tau_b)/mu.  The carries are the values of the same closed form at the
// region boundary rows, so each thread first re-evaluates its column's short carry chain (<= 5 values)
// and then fills its rows; no inter-thread dependency, one launch.
//
// A diffuse Lambert ground (SOS_SURFACE_LAMBERT_DIFFUSE) has no mirror term (S = 0); the carry of every upward column at
// the surface row is the isotropic b_s of first_order_surface_kernel, a pre-pass with one CTA per scenario.  A Ross-Li
// ground (SOS_SURFACE_ROSSLI) has one such carry per upward column: b_s plus the reflection of the beam and of order 1's
// downward light by the two kernels (brdf.cuh); so has the ocean (SOS_SURFACE_OCEAN), with the one glint matrix (glint.cuh).
#pragma once
#include "common.cuh"
#include "sweep.cuh"  // sossweep::block_sum

namespace sosfirst {

struct Col {
  double mu, inv_mu, mu0, F0q, Sq, T;  // inv_mu = 1/mu: the two column-dependent exponents per element use a multiply, not a division
  double Cm_atm, Cmir_atm, Cm_mix, Cmir_mix;
  bool down, special;
};

// Region-dependent constants of the closed form (column independent).
struct RegionK {
  double tau_d, tau_s;  // tau_b == tau_d for every region
  double ed;            // exp(-tau_d / mu0)
  double esr;           // exp(-(T - tau_s) / mu0)
};
__device__ __forceinline__ RegionK region_consts(double tau_d, double tau_s, double T, double mu0) {
  RegionK r;
  r.tau_d = tau_d; r.tau_s = tau_s;
  r.ed = exp(-tau_d / mu0);
  r.esr = exp(-(T - tau_s) / mu0);
  return r;
}

// value of the closed form at optical depth tt; e0 = exp(-tt/mu0) and es = exp(-(T-tt)/mu0) depend on
// the row only and are shared by all columns (2 column-dependent exps per element instead of 7)
__device__ __forceinline__ double i1_value(const Col& c, bool mix, double tt, double e0, double es, double carry,
                                           const RegionK& rk) {
  const double Cm = mix ? c.Cm_mix : c.Cm_atm;
  const double Cr = mix ? c.Cmir_mix : c.Cmir_atm;
  double direct, surf;
  double xd = 0.0;
  bool have_xd = false;
  if (c.down && c.special) {  // |mu + mu0| < 1e-4 (:133-140)
    direct = Cm * c.F0q * e0 * (tt - rk.tau_d) / c.mu0;
  } else {
    xd = exp((tt - rk.tau_d) * c.inv_mu);
    have_xd = true;
    direct = (c.mu0 / (c.mu0 + c.mu)) * Cm * c.F0q * (e0 - rk.ed * xd);
  }
  if (!c.down && c.special) {  // |mu - mu0| < 1e-4 (:225-233)
    surf = Cr * c.Sq * es * (rk.tau_s - tt) / c.mu0;
  } else {
    surf = (c.mu0 / (c.mu0 - c.mu)) * Cr * c.Sq * (es - rk.esr * exp((tt - rk.tau_s) * c.inv_mu));
  }
  double v = direct + surf;
  if (carry != 0.0) {
    if (!have_xd) xd = exp((tt - rk.tau_d) * c.inv_mu);
    v = carry * xd + v;
  }
  return v;
}

__device__ __forceinline__ int region_of(const GridDev& g, int t) {
  int k = 0;
  while (k + 1 < g.nreg && t >= g.rstart[k + 1]) ++k;
  return k;
}

// downward regions: region 0 starts at the top (tau_d = tau_s = 0, no carry); region k >= 1 carries row
// rstart[k]-1 with tau_d = tau[rstart[k]-1], tau_s = tau[rstart[k]]   (:113-198)
__device__ __forceinline__ RegionK down_region(const GridDev& g, const double* __restrict__ tau, int k, double T, double mu0) {
  if (k == 0) return region_consts(0.0, 0.0, T, mu0);
  return region_consts(tau[g.rstart[k] - 1], tau[g.rstart[k]], T, mu0);
}

// carry into region k of a downward column = value at row rstart[k]-1, chained from the top
__device__ double down_carry(const GridDev& g, const Col& c, const double* __restrict__ tau, int k, double T) {
  double carry = 0.0;
  for (int r = 1; r <= k; ++r) {
    const int cb = g.rstart[r] - 1;  // carry row of region r, lies in region r-1
    const RegionK rk = down_region(g, tau, r - 1, T, c.mu0);
    const double tt = tau[cb];
    carry = i1_value(c, (r - 1) == 1, tt, exp(-tt / c.mu0), exp(-(T - tt) / c.mu0), carry, rk);
  }
  return carry;
}

// PER_COLUMN: bs holds one surface carry per upward column, [S][M-1] (Ross-Li ground); otherwise one per scenario, [S]
// (diffuse Lambert ground), or bs is nullptr (mirror coupling).  Separate instantiations: the others compile as without it.
template <bool PER_COLUMN>
__global__ void __launch_bounds__(128)
first_order_regions_kernel(const GridDev g, const double* __restrict__ Cs /*[S][2][N]*/, double* __restrict__ I1,
                           double* __restrict__ I1_copy /*second destination (the accumulator I of the order loop) or nullptr*/,
                           int rows_per_block, const double* __restrict__ bs /*diffuse ground, or nullptr*/) {
  const int s = blockIdx.z;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  const int L = g.L, M = g.M, N = g.N, ld = g.ld;
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const sos_scenario sc = g.scen[s];
  const double* __restrict__ Catm = Cs + static_cast<size_t>(s) * 2 * N;
  const double* __restrict__ Cmix = Catm + N;
  double* __restrict__ out = I1 + static_cast<size_t>(s) * L * ld;
  double* __restrict__ out2 = I1_copy ? I1_copy + static_cast<size_t>(s) * L * ld : nullptr;
  auto put = [&](int t, int col, double v) {
    const size_t at = static_cast<size_t>(t) * ld + col;
    out[at] = v;
    if (out2) out2[at] = v;
  };
  const int ta = blockIdx.y * rows_per_block;
  const int tb = min(L, ta + rows_per_block);
  const double PI = 3.14159265358979323846;
  const double mu0 = sc.mu0;
  const double F0 = PI / mu0;
  const double T = sc.tauStar_tot;
  const double q = 1.0 / (4.0 * PI);
  const double S = bs ? 0.0 : F0 * sc.grd_alb * exp(-T / mu0);  // the mirror-reflected beam

  // row-only exponentials, shared by the 128 columns of the block
  __shared__ double sh_e0[64], sh_es[64];
  if (threadIdx.x < tb - ta) {
    const double tt = tau[ta + threadIdx.x];
    sh_e0[threadIdx.x] = exp(-tt / mu0);
    sh_es[threadIdx.x] = exp(-(T - tt) / mu0);
  }
  __syncthreads();
  if (m >= g.N) return;

  if (m == M - 1 || m == M) {
    // mu = 0-: C[M-1] F0/(4pi) e^{-tau/mu0} + C[M] S/(4pi) e^{-(T-tau)/mu0}   (:124-131); mu = 0+ mirrored (:217-224)
    const int mir = N - 1 - m;
    for (int t = ta; t < tb; ++t) {
      int k = 0;
      while (k + 1 < g.nreg && t >= g.rstart[k + 1]) ++k;
      const double* C = (k == 1) ? Cmix : Catm;
      put(t, m, (mu0 / (mu0 + g.mu[m])) * C[m] * (F0 * q) * sh_e0[t - ta] + (mu0 / (mu0 - g.mu[m])) * C[mir] * (S * q) * sh_es[t - ta]);
    }
    return;
  }

  Col c;
  c.mu0 = mu0; c.F0q = F0 * q; c.Sq = S * q; c.T = T;
  if (m < M - 1) {
    c.mu = g.mu[m];
    c.inv_mu = 1.0 / c.mu;
    c.down = true;
    c.special = fabs(c.mu + mu0) < SOS_MU0_TOLERANCE;
    c.Cm_atm = Catm[m]; c.Cmir_atm = Catm[N - 1 - m];
    c.Cm_mix = Cmix[m]; c.Cmir_mix = Cmix[N - 1 - m];
    int kcur = -1;
    double carry = 0.0;
    RegionK rk;
    for (int t = ta; t < tb; ++t) {
      const int k = region_of(g, t);
      if (k != kcur) { kcur = k; carry = down_carry(g, c, tau, k, T); rk = down_region(g, tau, k, T, mu0); }
      put(t, m, i1_value(c, k == 1, tau[t], sh_e0[t - ta], sh_es[t - ta], carry, rk));
    }
    return;
  }

  // ---- upward column: needs the mirror downward column at the surface row first (a diffuse ground: b_s) ----
  const int mir = N - 1 - m;
  const int R = g.nreg;
  double surf_carry;
  if (bs) {
    surf_carry = PER_COLUMN ? bs[static_cast<size_t>(s) * (M - 1) + (m - M - 1)] : bs[s];
  } else {
    Col d;
    d.mu0 = mu0; d.F0q = c.F0q; d.Sq = c.Sq; d.T = T;
    d.mu = g.mu[mir];
    d.inv_mu = 1.0 / d.mu;
    d.down = true;
    d.special = fabs(d.mu + mu0) < SOS_MU0_TOLERANCE;
    d.Cm_atm = Catm[mir]; d.Cmir_atm = Catm[m];
    d.Cm_mix = Cmix[mir]; d.Cmir_mix = Cmix[m];
    const double tt = tau[L - 1];
    const double surf_down = i1_value(d, (R - 1) == 1, tt, exp(-tt / mu0), exp(-(T - tt) / mu0), down_carry(g, d, tau, R - 1, T),
                                      down_region(g, tau, R - 1, T, mu0));
    surf_carry = sc.grd_alb * surf_down;
  }

  c.mu = g.mu[m];
  c.inv_mu = 1.0 / c.mu;
  c.down = false;
  c.special = fabs(c.mu - mu0) < SOS_MU0_TOLERANCE;
  c.Cm_atm = Catm[m]; c.Cmir_atm = Catm[mir];
  c.Cm_mix = Cmix[m]; c.Cmir_mix = Cmix[mir];

  // upward regions, bottom first:
  //   last region : carry = rho * I1[L-1, mirror] (diffuse ground: b_s), tau_d = tau[L-1], tau_s = T  (:206-216)
  //   region k    : carry = I1[rstart[k+1], m],    tau_d = tau[rstart[k+1]], tau_s = tau[rstart[k+1]-1]
  RegionK rks[3];
  double carry_k[3];
  for (int k = 0; k < R; ++k)
    rks[k] = (k == R - 1) ? region_consts(tau[L - 1], T, T, mu0) : region_consts(tau[g.rstart[k + 1]], tau[g.rstart[k + 1] - 1], T, mu0);
  carry_k[R - 1] = surf_carry;
  for (int k = R - 2; k >= 0; --k) {
    const double tt = tau[g.rstart[k + 1]];  // first row of the region below = carry row
    carry_k[k] = i1_value(c, (k + 1) == 1, tt, exp(-tt / mu0), exp(-(T - tt) / mu0), carry_k[k + 1], rks[k + 1]);
  }
  for (int t = ta; t < tb; ++t) {
    const int k = region_of(g, t);
    put(t, m, i1_value(c, k == 1, tau[t], sh_e0[t - ta], sh_es[t - ta], carry_k[k], rks[k]));
  }
}

// Diffuse Lambert ground: b_s[s] = rho (e^{-T/mu0} - 2 trapz(I1[L-1, 0..M-1] mu, mu)), the upward radiance the ground
// reflects of the direct beam (irradiance pi e^{-T/mu0} with F0 = pi/mu0) and of order 1's own downward light.  One CTA
// per scenario evaluates row L-1 of the downward columns with the calls and row factors of first_order_regions_kernel
// (S = 0), so these are the values it stores; the trapezoid is the one of the lambert_readme coupling (sweep.cuh: ascending
// abscissa, the interval next to mu = 0- included) and is summed by the deterministic block sum.
// NK kernel matrices (Ross-Li ground: 2, ocean: 1; 0 = the diffuse Lambert ground above): bs[s][i] = b_s + sum_k f_k
// (e^{-T/mu0} beam_k[i] + sum_c u_c R^k[c][i]) for the upward columns i = 0 .. M-2, u_c = -2 w_c mu_c I1[L-1, c]
// (sosbrdf::coupling_weight); with grd_alb = the isotropic part, b_s is the term above.
// Dynamic shared memory: (M + 32) doubles.
template <int NK>
__global__ void __launch_bounds__(128)
first_order_surface_kernel(const GridDev g, const double* __restrict__ Cs /*[S][2][N]*/, double* __restrict__ bs,
                           const sosbrdf::BrdfDev brdf) {
  extern __shared__ double fo_row[];  // [M] row L-1 of the downward half, then [32] block_sum scratch
  const int s = blockIdx.x;
  const int L = g.L, M = g.M, N = g.N, R = g.nreg;
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const sos_scenario sc = g.scen[s];
  const double* __restrict__ Catm = Cs + static_cast<size_t>(s) * 2 * N;
  const double* __restrict__ Cmix = Catm + N;
  const double PI = 3.14159265358979323846;
  const double mu0 = sc.mu0;
  const double F0 = PI / mu0;
  const double T = sc.tauStar_tot;
  const double q = 1.0 / (4.0 * PI);
  const double S = 0.0;
  const double tt = tau[L - 1];
  const double e0 = exp(-tt / mu0), es = exp(-(T - tt) / mu0);
  const int k = R - 1;  // region of the surface row
  const RegionK rk = down_region(g, tau, k, T, mu0);
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    if (m == M - 1) {
      const double* C = (k == 1) ? Cmix : Catm;
      fo_row[m] = (mu0 / (mu0 + g.mu[m])) * C[m] * (F0 * q) * e0 + (mu0 / (mu0 - g.mu[m])) * C[N - 1 - m] * (S * q) * es;
      continue;
    }
    Col c;
    c.mu0 = mu0; c.F0q = F0 * q; c.Sq = S * q; c.T = T;
    c.mu = g.mu[m];
    c.inv_mu = 1.0 / c.mu;
    c.down = true;
    c.special = fabs(c.mu + mu0) < SOS_MU0_TOLERANCE;
    c.Cm_atm = Catm[m]; c.Cmir_atm = Catm[N - 1 - m];
    c.Cm_mix = Cmix[m]; c.Cmir_mix = Cmix[N - 1 - m];
    fo_row[m] = i1_value(c, k == 1, tt, e0, es, down_carry(g, c, tau, k, T), rk);
  }
  __syncthreads();
  double part = 0.0;
  for (int c0 = threadIdx.x; c0 < M - 1; c0 += blockDim.x) {
    const int c1 = c0 + 1;
    part += (g.mu[c1] - g.mu[c0]) * (fo_row[c1] * g.mu[c1] + fo_row[c0] * g.mu[c0]) * 0.5;
  }
  const double down = -2.0 * sossweep::block_sum(part, fo_row + M);
  const double b_s = sc.grd_alb * (exp(-T / mu0) + down);
  if constexpr (NK == 0) {
    if (threadIdx.x == 0) bs[s] = b_s;
  } else {
    for (int c = threadIdx.x; c < M; c += blockDim.x) fo_row[c] *= sosbrdf::coupling_weight(g.mu, M, c);   // (block_sum synced)
    __syncthreads();
    const double E = exp(-T / mu0), fv = brdf.f[2 * s], fg = brdf.f[2 * s + 1];
    const double* __restrict__ bv = brdf.beam + static_cast<size_t>(s) * 2 * (M - 1);
    const double* __restrict__ bg = bv + (M - 1);
    for (int i = threadIdx.x; i < M - 1; i += blockDim.x) {
      if constexpr (NK == 2) {
        double sv, sgeo;
        sosbrdf::coupling(brdf, s, fo_row, M, i, sv, sgeo);
        bs[static_cast<size_t>(s) * (M - 1) + i] = b_s + (fv * (E * bv[i] + sv) + fg * (E * bg[i] + sgeo));
      } else {
        bs[static_cast<size_t>(s) * (M - 1) + i] = b_s + fv * (E * bv[i] + sosbrdf::coupling(brdf, s, fo_row, M, i));
      }
    }
  }
}

// I1_NumInt (SOS_Aer_I1_In.py:13-58): one homogeneous layer above a black surface
__global__ void __launch_bounds__(128)
first_order_single_kernel(const GridDev g, const double* __restrict__ Cs /*[S][2][N], plane 0 = alb*P0*/,
                          double* __restrict__ I1, double* __restrict__ I1_copy, int rows_per_block) {
  const int s = blockIdx.z;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= g.N) return;
  const int L = g.L, M = g.M, N = g.N, ld = g.ld;
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const sos_scenario sc = g.scen[s];
  const double C = Cs[static_cast<size_t>(s) * 2 * N + m];
  double* __restrict__ out = I1 + static_cast<size_t>(s) * L * ld;
  double* __restrict__ out2 = I1_copy ? I1_copy + static_cast<size_t>(s) * L * ld : nullptr;
  const int ta = blockIdx.y * rows_per_block;
  const int tb = min(L, ta + rows_per_block);
  const double PI = 3.14159265358979323846;
  const double mu0 = sc.mu0, mu = g.mu[m], T = sc.tauStar_tot;
  const double k = C / (4.0 * PI);
  const double norm = PI / mu0;  // (:58)
  const double eS = exp(-T / mu0);
  const double inv_mu = 1.0 / mu, w0 = mu0 / (mu0 + mu);
  for (int t = ta; t < tb; ++t) {
    const double tt = tau[t];
    const double e0 = exp(-tt / mu0);
    double v;
    if (m == M - 1 || m == M) {
      v = k * w0 * e0;                                                  // (:39,:50)
    } else if (m < M - 1) {
      if (fabs(mu + mu0) < SOS_MU0_TOLERANCE) v = k * e0 * tt / mu0;    // (:41-43)
      else v = w0 * k * (e0 - exp(tt * inv_mu));                        // (:34-37)
    } else {
      v = w0 * k * (e0 - eS * exp(-(T - tt) * inv_mu));                 // (:54-55)
    }
    out[static_cast<size_t>(t) * ld + m] = v * norm;
    if (out2) out2[static_cast<size_t>(t) * ld + m] = v * norm;
  }
}

}  // namespace sosfirst
