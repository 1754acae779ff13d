// Flux / mean-diffusivity / heating-rate quadratures (SOS_Aer_graphe.py:8-10,39-41,70-91,154-158;
// SOS_Aer_critical_albedo.py:377-382) and the contraction-operand builder.
#pragma once
#include "common.cuh"
#include "glint.cuh"

namespace sosquad {

// one CTA per (layer, scenario): sums[s][t][0..2] = trapz(I mu)|down, trapz(I mu)|up, trapz(I)|all
__global__ void __launch_bounds__(256)
row_sums_kernel(const GridDev g, const double* __restrict__ I, double* __restrict__ sums) {
  __shared__ double sc[3][8];
  const int s = blockIdx.y, t = blockIdx.x;
  const int M = g.M, N = g.N;
  const double* __restrict__ row = I + (static_cast<size_t>(s) * g.L + t) * g.ld;
  double a = 0.0, b = 0.0, c = 0.0;
  // interval k..k+1, k != M-1 (zero width between the two mu=0 nodes)
  for (int k = threadIdx.x; k < N - 1; k += blockDim.x) {
    const double m0 = g.mu[k], m1 = g.mu[k + 1];
    const double d = m1 - m0;
    const double y0 = row[k], y1 = row[k + 1];
    const double f = d * (y1 * m1 + y0 * m0) * 0.5;
    if (k < M - 1) a += f; else if (k >= M) b += f;
    c += d * (y1 + y0) * 0.5;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  if (lane == 0) { sc[0][warp] = a; sc[1][warp] = b; sc[2][warp] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0, tb = 0, tc = 0;
    for (int w = 0; w < 8; ++w) { ta += sc[0][w]; tb += sc[1][w]; tc += sc[2][w]; }
    double* o = sums + (static_cast<size_t>(s) * g.L + t) * 3;
    o[0] = ta; o[1] = tb; o[2] = tc;
  }
}

__global__ void __launch_bounds__(128)
quadrature_outputs_kernel(const GridDev g, const double* __restrict__ sums, const double* __restrict__ z,
                          double direct_scale, double* __restrict__ flux_up, double* __restrict__ flux_down,
                          double* __restrict__ net_flux, double* __restrict__ diffusivity, double* __restrict__ heating) {
  const int s = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int L = g.L;
  if (t >= L) return;
  const double PI = 3.14159265358979323846;
  const sos_scenario sc = g.scen[s];
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const double F0 = PI / sc.mu0;
  const double tl = tau[L - 1];
  const double* q = sums + (static_cast<size_t>(s) * L + t) * 3;
  const size_t o = static_cast<size_t>(s) * L + t;
  const double dn = exp(-tau[t] / sc.mu0);
  // the collimated beam reflected by a mirror ground; a diffuse Lambert, Ross-Li or ocean ground puts it into the field itself
  const double alb_dir =
      (g.surface == SOS_SURFACE_LAMBERT_DIFFUSE || g.surface == SOS_SURFACE_ROSSLI || g.surface == SOS_SURFACE_OCEAN) ? 0.0 : sc.grd_alb;
  const double up = alb_dir * exp(-(2.0 * tl - tau[t]) / sc.mu0);
  if (flux_down) flux_down[o] = q[0] - (F0 * direct_scale) * dn;                 // graphe.py:157 / :77
  if (flux_up) flux_up[o] = q[1] + (F0 * direct_scale) * up;                     // graphe.py:158 / :78
  if (net_flux) net_flux[o] = (q[0] + q[1]) - F0 * dn + F0 * up;                 // graphe.py:41
  if (diffusivity) diffusivity[o] = -(q[0] + q[1]) / q[2];                       // graphe.py:10
  if (heating) {
    // heating rate always uses the F0/(4 pi) direct terms (graphe.py:77-78)
    const double ds = 1.0 / (4.0 * PI);
    auto total = [&](int i) {
      const double* qi = sums + (static_cast<size_t>(s) * L + i) * 3;
      return (qi[0] - (F0 * ds) * exp(-tau[i] / sc.mu0)) + (qi[1] + (F0 * ds) * alb_dir * exp(-(2.0 * tl - tau[i]) / sc.mu0));
    };
    auto hr = [&](int i) {  // i in [0, L-2]
      return -(1.0 / (1.225 * 1004.0)) * (total(i + 1) - total(i)) / (z[i + 1] - z[i]);
    };
    // sequential semantics of graphe.py:85,89,90: hr[L-1] = hr[L-2]; hr[idx_up-1] = hr[idx_up-2];
    // hr[idx_down] = hr[idx_down-1] (which may itself be the replaced idx_up-1 entry)
    int i = t;
    if (i == L - 1) i = L - 2;
    if (g.nreg == 3) {
      const int idx_up = g.rstart[1], idx_down = g.rstart[2] - 1;
      if (t == idx_down) i = idx_down - 1;
      if (i == idx_up - 1 && (t == idx_up - 1 || t == idx_down)) i = idx_up - 2;
    }
    if (i < 0) i = 0;
    heating[o] = hr(i);
  }
}

// A[k][m] = 0.25 * w_k * P[m][N-1-k]   (SOS_Aer_I1_In.py:73 as a GEMM operand; SURVEY.md A.4)
__global__ void __launch_bounds__(256)
build_contraction_kernel(const double* __restrict__ P, int ldp, double* __restrict__ A, int lda, int N,
                         const double* __restrict__ wmu) {
  __shared__ double tile[32][33];
  const int k0 = blockIdx.y * 32, m0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  // read P[m0+r][N-1-(k0+c)] with c fastest (reversed but contiguous)
  for (int r = ty; r < 32; r += 8) {
    const int m = m0 + r, k = k0 + tx;
    tile[r][tx] = (m < N && k < N) ? P[static_cast<size_t>(m) * ldp + (N - 1 - k)] : 0.0;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, m = m0 + tx;
    if (k < N && m < N) A[static_cast<size_t>(k) * lda + m] = 0.25 * wmu[k] * tile[tx][r];
  }
}


// Azimuth synthesis (include/sos_b200.h: sos_azimuth_synthesis).  Thread = one mu column of one (geometry, row) and AZ_CHUNK
// azimuths; the members of the geometry are summed in ascending order (no atomics: deterministic).  HBM bound: every
// member row is read once per azimuth chunk (the chunks of one row hit L2), every output element written once.
constexpr int AZ_THREADS = 128;
constexpr int AZ_CHUNK = 8;

struct SynthTables {
  const int* geo;       // [n_present] geometry of each present group
  const int* mem_off;   // [n_present + 1]
  const int* members;   // member scenarios of the groups, ascending within a group
  const double* w;      // [S][n_az]
  const int* rows;      // [n_rows]
};

__global__ void __launch_bounds__(AZ_THREADS)
azimuth_synthesis_kernel(const double* __restrict__ I, int L, int ld, int N, const SynthTables t, int n_rows, int n_az,
                         double* __restrict__ out, int accumulate) {
  const int col = blockIdx.x * AZ_THREADS + threadIdx.x;
  if (col >= N) return;
  const int gi = blockIdx.y / n_rows, r = blockIdx.y % n_rows;
  const int p0 = blockIdx.z * AZ_CHUNK;
  const int np = min(AZ_CHUNK, n_az - p0);
  const int row = t.rows[r];
  double acc[AZ_CHUNK];
#pragma unroll
  for (int q = 0; q < AZ_CHUNK; ++q) acc[q] = 0.0;
  for (int j = t.mem_off[gi]; j < t.mem_off[gi + 1]; ++j) {
    const int s = t.members[j];
    const double v = __ldg(&I[(static_cast<size_t>(s) * L + row) * ld + col]);
    const double* __restrict__ w = t.w + static_cast<size_t>(s) * n_az + p0;
#pragma unroll
    for (int q = 0; q < AZ_CHUNK; ++q)
      if (q < np) acc[q] = fma(__ldg(&w[q]), v, acc[q]);
  }
  double* o = out + ((static_cast<size_t>(t.geo[gi]) * n_rows + r) * n_az + p0) * N + col;
#pragma unroll
  for (int q = 0; q < AZ_CHUNK; ++q)
    if (q < np) o[static_cast<size_t>(q) * N] = accumulate ? o[static_cast<size_t>(q) * N] + acc[q] : acc[q];
}

// Exact direct glint of azimuth-resolved radiance (sos_glint_correction).  One thread per output element (entry k,
// requested row r, azimuth p, upward column i): out[geo[k]][r][p][M+1+i] += E (rho_glint(mu_i, mu0, phi_p) - sum_{m<K} w[p][m]
// beam[k][m][i]) e^{-(T - tau[k][r]) / mu_i}, E = e^{-T/mu0}, w[p][m] = 1 (m = 0) or 2 cos(m phi_p): the once-reflected direct
// beam, transmitted without scattering to the row, with its truncated Fourier series replaced by the exact value.
struct GlintCorrection {
  const int* geo;       // [n] geometry (first index of out) of each entry
  const double* par;    // [n][4] mu0, tauStar_tot, sigma^2, n_ref
  const double* tau;    // [n][n_rows] tau at the requested rows
  const double* beam;   // [n][K][M-1]
  const double* w;      // [n_az][K]
  const double* cphi;   // [n_az]
};

__global__ void __launch_bounds__(128)
glint_correction_kernel(const double* __restrict__ mu, int M, int N, const GlintCorrection t, int n, int K, int n_rows,
                        int n_az, double* __restrict__ out) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long per_k = static_cast<long long>(n_rows) * n_az * (M - 1);
  if (e >= per_k * n) return;
  const int k = static_cast<int>(e / per_k);
  long long rest = e % per_k;
  const int i = static_cast<int>(rest % (M - 1));
  rest /= (M - 1);
  const int p = static_cast<int>(rest % n_az), r = static_cast<int>(rest / n_az);
  const double* __restrict__ par = t.par + 4 * static_cast<size_t>(k);
  const double mu0 = par[0], T = par[1], sigma2 = par[2], nref = par[3];
  const double mi = mu[M + 1 + i];
  const double rho = sosglint::glint(mi, mu0, t.cphi[p], sigma2, nref, sosglint::shadowing(mi, mu0, sqrt(sigma2)));
  const double* __restrict__ b = t.beam + static_cast<size_t>(k) * K * (M - 1) + i;
  const double* __restrict__ w = t.w + static_cast<size_t>(p) * K;
  double series = 0.0;
  for (int m = 0; m < K; ++m) series += w[m] * b[static_cast<size_t>(m) * (M - 1)];
  const double tr = exp(-(T - t.tau[static_cast<size_t>(k) * n_rows + r]) / mi);
  double* o = out + ((static_cast<size_t>(t.geo[k]) * n_rows + r) * n_az + p) * N + (M + 1 + i);
  *o += exp(-T / mu0) * (rho - series) * tr;
}

}  // namespace sosquad
