// Azimuth-averaged phase functions on the device (SURVEY.md 8f rank 1): P0(mu, mu0) and P(mu, mu') of the
// analytic / tabulated families of SOS_Aer_phase_func.py:68-292 -- Rayleigh (:97), Henyey-Greenstein
// (:158), tabulated FWC with the reference's searchsorted + linear interpolation (:202-236).  Same
// quadrature as the reference: 25 azimuth nodes on [0, pi], both half-rings, composite trapezoid; the raw
// matrix is symmetric and every COLUMN is then normalised to trapz(P[:, n], mu) = 4 (:131).
// The reference spends 89-112 s per matrix at N = 1002 in a triple Python loop; this is two launches.
#pragma once
#include "common.cuh"

namespace sosphase {

constexpr int NPHI = 25;
enum Family { RAYLEIGH = 0, HG = 1, TABLE = 2 };

struct PhaseArgs {
  int family;
  double g;
  const double* tab_x;  // TABLE: abscissae (ascending), device
  const double* tab_y;
  int tab_n;
  double phi[NPHI];     // linspace(0, pi, 25) as computed by the host (NumPy), so that nodes are identical
  double cphi[NPHI];    // cos(0 - phi)
};

__device__ __forceinline__ double phase_value(const PhaseArgs& a, double c) {
  if (a.family == RAYLEIGH) return 0.75 * (1.0 + c * c);
  if (a.family == HG) {
    const double g = a.g;
    return (1.0 - g * g) / pow(1.0 + g * g - 2.0 * g * c, 1.5);
  }
  // np.clip + np.searchsorted(side='left') + linear interpolation (:214-236)
  c = fmin(fmax(c, -1.0), 1.0);
  int lo = 0, hi = a.tab_n;  // first index with tab_x[idx] >= c
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a.tab_x[mid] < c) lo = mid + 1; else hi = mid;
  }
  if (lo == 0) return a.tab_y[0];
  if (lo >= a.tab_n) return a.tab_y[a.tab_n - 1];
  const double x0 = a.tab_x[lo - 1], x1 = a.tab_x[lo];
  const double w = (c - x0) / (x1 - x0);
  return a.tab_y[lo - 1] + w * (a.tab_y[lo] - a.tab_y[lo - 1]);
}

// trapz over phi of f(-(cc + ss cos phi)) + f(-(cc - ss cos phi))
__device__ __forceinline__ double ring_integral(const PhaseArgs& a, double cc, double ss) {
  double sum = 0.0;
  double prev = 0.0;
#pragma unroll 5
  for (int k = 0; k < NPHI; ++k) {
    const double x = ss * a.cphi[k];
    const double y = phase_value(a, -(cc + x)) + phase_value(a, -(cc - x));
    if (k > 0) sum += (a.phi[k] - a.phi[k - 1]) * (y + prev) / 2.0;
    prev = y;
  }
  return sum;
}

// raw symmetric matrix R[m][n] (only m >= n is computed by the reference and mirrored; cc and ss are
// symmetric in (m, n) bit for bit, so computing every entry gives the same matrix)
__global__ void __launch_bounds__(256)
phase_raw_kernel(const PhaseArgs a, const double* __restrict__ mu, int N, double* __restrict__ P, int ldp) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int m = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (m >= N || n >= N) return;
  const double um = mu[m], un = mu[n];
  const double cc = um * un;
  const double ss = sqrt(1.0 - un * un) * sqrt(1.0 - um * um);
  const double PI = 3.14159265358979323846;
  P[static_cast<size_t>(m) * ldp + n] = ring_integral(a, cc, ss) / (2.0 * PI);
}

// column integrals trapz(R[:, n], mu): one thread per column, coalesced over n
__global__ void __launch_bounds__(128)
phase_colint_kernel(const double* __restrict__ mu, int N, const double* __restrict__ P, int ldp, double* __restrict__ colint) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double s = 0.0;
  double prev = P[n];
  for (int m = 1; m < N; ++m) {
    const double cur = P[static_cast<size_t>(m) * ldp + n];
    s += (mu[m] - mu[m - 1]) * (cur + prev) / 2.0;
    prev = cur;
  }
  colint[n] = s;
}

__global__ void __launch_bounds__(256)
phase_normalise_kernel(int N, double* __restrict__ P, int ldp, const double* __restrict__ colint) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int m = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (m >= N || n >= N) return;
  const size_t i = static_cast<size_t>(m) * ldp + n;
  P[i] = 4.0 * P[i] / colint[n];
}

// trapz(P0, mu) by one CTA of 256 threads (fixed partition and tree: every caller gets the same bits); P0 must be complete
__device__ __forceinline__ double p0_total(const double* __restrict__ mu, int N, const double* P0, double* part) {
  double s = 0.0;
  for (int m = 1 + threadIdx.x; m < N; m += blockDim.x) s += (mu[m] - mu[m - 1]) * (P0[m] + P0[m - 1]) / 2.0;
  part[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
    __syncthreads();
  }
  const double tot = part[0];
  __syncthreads();
  return tot;
}

// P0(mu, mu0): one CTA; (:92-105)
__global__ void __launch_bounds__(256)
phase_p0_kernel(const PhaseArgs a, const double* __restrict__ mu, int N, double mu0, double* __restrict__ P0) {
  __shared__ double part[256];
  const double PI = 3.14159265358979323846;
  const double s0 = sqrt(1.0 - mu0 * mu0);
  for (int m = threadIdx.x; m < N; m += blockDim.x) {
    const double um = mu[m];
    P0[m] = ring_integral(a, um * mu0, s0 * sqrt(1.0 - um * um)) / (4.0 * PI);
  }
  __syncthreads();
  const double tot = p0_total(mu, N, P0, part);
  for (int m = threadIdx.x; m < N; m += blockDim.x) P0[m] = P0[m] / tot * 2.0;
}

// ------------------------------------------------------------------------------------------
// Azimuthal Fourier modes m = 0 .. n_modes-1 (include/sos_b200.h: sos_build_phase_modes).  The azimuth of the scattered
// direction relative to the incident one is integrated with the cos(m phi) weight instead of averaged out; the m = 0
// accumulator repeats ring_integral's operations in its order (bit-identical at the same nodes), the m >= 1 ones use the
// trapezoid as a weighted sum (weights * cos(m phi_k) precomputed by the host).
constexpr int MAX_MODES = 64;
constexpr int MAX_NPHI = 1024;
constexpr int MODE_THREADS = 128;

struct ModeArgs {
  PhaseArgs pa;          // family and table (its 25-node arrays are unused)
  int n_phi, n_modes;
  const double* phi;     // [n_phi] nodes, device
  const double* cphi;    // [n_phi] cos(0 - phi_k)
  const double* wcos;    // [n_phi][n_modes] trapezoid weight of node k * cos(m phi_k) (column 0 unused)
};

// one thread per element: P0 = false -> element (m, n) of the raw matrix R_m / (2 pi) (mode m at P + m*stride, [N][ldp]);
// P0 = true -> element m of the raw solar vector / (4 pi) (mode m at P + m*N).  Mode-m >= 1 accumulators live in shared
// memory, one column per thread: [n_modes - 1][MODE_THREADS].
template <bool P0>
__global__ void __launch_bounds__(MODE_THREADS)
phase_modes_raw_kernel(const ModeArgs a, const double* __restrict__ mu, int N, double mu0, double* __restrict__ P, int ldp,
                       size_t stride) {
  extern __shared__ double acc[];
  const long long e = static_cast<long long>(blockIdx.x) * MODE_THREADS + threadIdx.x;
  const long long n_el = P0 ? N : static_cast<long long>(N) * N;
  if (e >= n_el) return;
  const int m = P0 ? static_cast<int>(e) : static_cast<int>(e / N);
  const int n = P0 ? 0 : static_cast<int>(e % N);
  const double PI = 3.14159265358979323846;
  double cc, ss;
  const double um = mu[m];
  if (P0) {
    cc = um * mu0;
    ss = sqrt(1.0 - mu0 * mu0) * sqrt(1.0 - um * um);
  } else {
    const double un = mu[n];
    cc = um * un;
    ss = sqrt(1.0 - un * un) * sqrt(1.0 - um * um);
  }
  const int K = a.n_modes;
  double* my = acc + threadIdx.x;
  for (int j = 1; j < K; ++j) my[(j - 1) * MODE_THREADS] = 0.0;
  double sum = 0.0, prev = 0.0;
  for (int k = 0; k < a.n_phi; ++k) {
    const double x = ss * a.cphi[k];
    const double fb = phase_value(a.pa, -(cc + x)), fa = phase_value(a.pa, -(cc - x));
    const double y = fb + fa;
    if (k > 0) sum += (a.phi[k] - a.phi[k - 1]) * (y + prev) / 2.0;
    prev = y;
    const double odd = fa - fb;
    const double* __restrict__ w = a.wcos + static_cast<size_t>(k) * K;
    for (int j = 1; j < K; ++j) my[(j - 1) * MODE_THREADS] += w[j] * ((j & 1) ? odd : y);
  }
  const double scale = P0 ? 4.0 * PI : 2.0 * PI;
  const size_t off = P0 ? static_cast<size_t>(m) : static_cast<size_t>(m) * ldp + n;
  const size_t step = P0 ? static_cast<size_t>(N) : stride;
  P[off] = sum / scale;
  for (int j = 1; j < K; ++j) P[off + j * step] = my[(j - 1) * MODE_THREADS] / scale;
}

// every mode of the raw solar vector divided by the trapz of MODE 0, as phase_p0_kernel does for one vector; one CTA
__global__ void __launch_bounds__(256)
phase_p0_modes_norm_kernel(const double* __restrict__ mu, int N, int n_modes, double* __restrict__ P0) {
  __shared__ double part[256];
  const double tot = p0_total(mu, N, P0, part);
  for (int i = threadIdx.x; i < n_modes * N; i += blockDim.x) P0[i] = P0[i] / tot * 2.0;
}

}  // namespace sosphase
