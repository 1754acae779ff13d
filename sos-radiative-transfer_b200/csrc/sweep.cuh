// Layer integration of one scattering order: In_NumInt (SOS_Aer_I1_In.py:77-130) and its inlined
// three-region form (SOS_Aer_main_specular.py:327-449; Lambert surface SOS_Aer_main_lambertian.py:399,401).
//
// The reference evaluates every (layer, mu) value as a trapezoid over the whole slice above/below it
// (O(L^2 N)).  With a_t = exp(-dtau_t/|mu|) this is the linear recurrence
//     down:  D_t = D_{t-1} a_t - dtau_t/(2 mu) (J_{t-1} a_t + J_t)
//     up:    U_t = U_{t+1} a_t + s_t dtau_t/(2 mu) (J_t + J_{t+1} a_t)      (s_t = 0 on carry gaps)
// which is evaluated here as a chunked scan in three launches:
//   1. sweep_local   every (scenario, chunk, mu column) runs its chunk from a zero carry and keeps only
//                    the chunk aggregate = the last local value (the products of a_t telescope to
//                    exp((tau_t - tau_start)/mu), so no separate "a" aggregate is needed); reads J once.
//   2. sweep_carry   one CTA per scenario chains the chunk carries (down), finishes the surface row
//                    (mu->0 columns + extrapolation), applies the specular/Lambert coupling, chains the
//                    up carries and re-seeds them from the *blended* boundary rows (SURVEY.md A.7).
//   3. sweep_apply   the same (scenario, chunk, column) threads rerun the recurrence from the TRUE carry,
//                    write I_n and accumulate I += I_n (SOS_Aer_main_specular.py:454-456) in one pass;
//      sweep_zone    one small CTA per (scenario, layer) finishes the ~160 columns next to mu = 0:
//                    windowed / Taylor columns (SOS_Aer_In_limit.py:70-109), the polynomial
//                    extrapolation (:113-141, a fixed linear map W), the find-first second-difference
//                    blend (SOS_Aer_I1_In.py:101-108) and the convergence ratios of :309.
//   Traffic: J 8 (pass 1) + J 8 + I_n 8 + I 16 (pass 3) = 40 B per element (32 B is the algorithmic minimum).
//
// Generated source.  On rows that use the molecular operand alone (every row outside the aerosol layer,
// SOS_Aer_main_specular.py:323) the contraction operand is A = Us Vt with Vt = [1; mu^2] (gemm_lowrank.cuh), so
//     J[t, m] = c0[t] + c1[t] mu_m^2,     c_r[t] = coef * sum_k I_{n-1}[t, k] Us[k][r]
// and the two numbers c_r[t] per row are all the next order needs from this one.  Inside sos_solve the sweeps therefore
// REBUILD J from c on those rows instead of reading it (SrcGen / SrcAt below), sweep_apply_kernel emits the partial
// projections of the I_n it produces (one slot per warp and row; butterfly transpose-reduce, a fixed tree: deterministic)
// and sweep_zone_kernel adds the columns it finishes, sums the slots and writes the next order's c.  On those rows
// neither J nor I_n touches memory (I_n is kept only where something reads it: the aerosol rows for the dense
// contraction, the columns next to mu = 0 for the zone kernel, the TOA / surface rows for the ratios and the surface
// coupling): per element and order that leaves the read-modify-write of I, 16 B, on 746 of the 800 default rows; the
// local pass of those rows reads nothing at all.
#pragma once
#include <type_traits>
#include "brdf.cuh"
#include "common.cuh"
#include "layer_shard.cuh"

namespace sossweep {

struct SrcGen {
  const double* cj;        // [S][Lp][2] source coefficients of this order; nullptr: every J row is read from memory
  double* cj_out;          // ... of the next order (written by sweep_zone_kernel)
  int Lp;
  double* proj;            // [S][L][nslots][2] partial projections of I_n (one slot per warp of sweep_apply_kernel)
  int nslots;
  int zlo, zu_end;         // columns the zone kernel may read raw: downward m >= zlo, upward m < zu_end (I_n stored there on every row)
  int zu_proj;             // ... upward m < zu_proj (<= zu_end) and downward m >= zlo are left out of the apply pass's projections
                           // and projected by the zone kernel with their final values; a blend that reaches past zu_proj corrects
                           // the raw projection of the apply pass by (final - raw)
  int store_all;           // store I_n everywhere (debugging aid)
  int ldr;
  int rank[SOS_MAX_PHASE];
  const double* Ut[SOS_MAX_PHASE];
};

// J[t, m] of one scenario: read, or rebuilt on the molecular rows
struct SrcAt {
  const double* Js;
  const double2* cj2;
  int ld, a0, a1;
  bool gen;
  __device__ __forceinline__ SrcAt(const GridDev& g, const SrcGen& sg, const double* J, int s)
      : Js(J + static_cast<size_t>(s) * g.L * g.ld), cj2(nullptr), ld(g.ld), a0(g.nreg == 3 ? g.rstart[1] : g.L),
        a1(g.nreg == 3 ? g.rstart[2] : g.L), gen(sg.cj != nullptr && sg.rank[g.scen[s].phase_atm] > 0) {
    if (gen) cj2 = reinterpret_cast<const double2*>(sg.cj) + static_cast<size_t>(s) * sg.Lp;
  }
  __device__ __forceinline__ bool gen_row(int t) const { return gen && (t < a0 || t >= a1); }
  __device__ __forceinline__ double operator()(int t, int m, double mu) const {
    if (gen_row(t)) {
      const double2 c = cj2[t];
      return fma(c.y, mu * mu, c.x);
    }
    return Js[static_cast<size_t>(t) * ld + m];
  }
};

__device__ __forceinline__ double shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }

// v[0..7] of every lane -> the sum over the warp of v[lane >> 2], in every lane (fixed tree: deterministic)
__device__ __forceinline__ double transpose_reduce8(double (&v)[8], int lane) {
  const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double keep = h16 ? v[i + 4] : v[i], send = h16 ? v[i] : v[i + 4];
    v[i] = keep + shfl_xor_d(send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const double keep = h8 ? v[i + 2] : v[i], send = h8 ? v[i] : v[i + 2];
    v[i] = keep + shfl_xor_d(send, 8);
  }
  {
    const double keep = h4 ? v[1] : v[0], send = h4 ? v[0] : v[1];
    v[0] = keep + shfl_xor_d(send, 4);
  }
  v[0] += shfl_xor_d(v[0], 2);
  v[0] += shfl_xor_d(v[0], 1);
  return v[0];
}

// column of a (block, thread) of the two scan passes: blocks [0, nbd) hold the downward columns 0 .. M-2, the others
// the upward columns M+1 .. N-1, so that no warp mixes the two directions (its rows run together: warp collectives)
__device__ __forceinline__ int scan_blocks_down(int M, int threads) { return (M - 1 + threads - 1) / threads; }

// exp(x) for the attenuation factors a_t = exp(-dtau/|mu|): almost every argument is tiny (dtau ~ 1e-4 ..
// 3e-3 per layer), where a degree-8 Taylor polynomial is exact to < 1e-19 relative (|x| <= 2^-5:
// x^9/9! < 1e-19) and costs 8 DFMA instead of the ~30 instructions of the general routine.  The two
// scan passes are FP64-pipe bound, not HBM bound, without this.
// (the coefficients sit in constant memory so that every DFMA takes its constant-bank operand directly: as 64-bit
// immediates they cost two UMOVs per DFMA, a third of all instructions of the issue-bound local pass)
__constant__ double kExpTaylor[8] = {1.0 / 40320.0, 1.0 / 5040.0, 1.0 / 720.0, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5, 1.0};
__device__ __forceinline__ double exp_small(double x) {
  if (fabs(x) <= 0.03125) {
    double p = kExpTaylor[0];
    p = fma(p, x, kExpTaylor[1]);
    p = fma(p, x, kExpTaylor[2]);
    p = fma(p, x, kExpTaylor[3]);
    p = fma(p, x, kExpTaylor[4]);
    p = fma(p, x, kExpTaylor[5]);
    p = fma(p, x, kExpTaylor[6]);
    p = fma(p, x, kExpTaylor[7]);
    return fma(p, x, kExpTaylor[7]);
  }
  return exp(x);
}

// exp(x) for |x| <= 2^-10 (x^5/5! < 7e-18 relative): what almost every scan step of a thin atmosphere needs
constexpr double kTinyArg = 0.0009765625;
__device__ __forceinline__ double exp_tiny(double x) {
  double p = kExpTaylor[4];
  p = fma(p, x, kExpTaylor[5]);
  p = fma(p, x, kExpTaylor[6]);
  p = fma(p, x, kExpTaylor[7]);
  return fma(p, x, kExpTaylor[7]);
}
// the polynomial branch of exp_small alone (|x| <= 2^-5 guaranteed by the caller)
__device__ __forceinline__ double exp_poly8(double x) {
  double p = kExpTaylor[0];
  p = fma(p, x, kExpTaylor[1]);
  p = fma(p, x, kExpTaylor[2]);
  p = fma(p, x, kExpTaylor[3]);
  p = fma(p, x, kExpTaylor[4]);
  p = fma(p, x, kExpTaylor[5]);
  p = fma(p, x, kExpTaylor[6]);
  p = fma(p, x, kExpTaylor[7]);
  return fma(p, x, kExpTaylor[7]);
}
__device__ __forceinline__ double warp_max_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

constexpr int LOCAL_THREADS = 128;
constexpr int LOCAL_UNROLL = 4;  // (8 rows in flight was measured: lower occupancy, 0.756 vs 0.744 ms per order at S = 96)
constexpr int ROW_THREADS = 256;
constexpr int CARRY_THREADS = 1024;

// ------------------------------------------------------------------------------------------
// 1. chunk-local recurrences
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LOCAL_THREADS)
sweep_local_kernel(const GridDev g, const SrcGen sg, const double* __restrict__ J, double* __restrict__ aggD, double* __restrict__ aggU) {
  const int s = blockIdx.z;
  if (!g.state[s].active) return;
  const int c = g.c_lo + blockIdx.y;  // (layer-sharded plans own the chunks [c_lo, c_hi))
  const int L = g.L, M = g.M, ld = g.ld;
  const int nbd = scan_blocks_down(M, LOCAL_THREADS);
  const bool up = static_cast<int>(blockIdx.x) >= nbd;
  const int m = up ? M + 1 + (blockIdx.x - nbd) * LOCAL_THREADS + threadIdx.x : blockIdx.x * LOCAL_THREADS + threadIdx.x;
  if (up ? (m >= g.N) : (m >= M - 1)) return;
  if (m < g.col0 || m >= g.col1) return;
  const int t0 = g.chunk_start[c], t1 = g.chunk_start[c + 1];
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const SrcAt src(g, sg, J, s);
  const double* __restrict__ Js = src.Js;
  const double mu = g.mu[m];
  const double imu = 1.0 / mu;  // one division per thread; the scan steps multiply
  const double q = mu * mu;
  const size_t agg = (static_cast<size_t>(s) * g.nchunks + c) * g.N + m;
  const bool cg = src.gen_row(t0);  // chunks never straddle a region: the whole chunk is rebuilt, or read
  // J of a row of THIS chunk (one kind of row); rows outside go through src()
  auto jrow = [&](auto gen_tag, int t) -> double {
    if (decltype(gen_tag)::value) {
      const double2 cc = src.cj2[t];
      return fma(cc.y, q, cc.x);
    }
    return Js[static_cast<size_t>(t) * ld + m];
  };

  if (!up) {
    if (fabs(mu) < SOS_MU_THRESHOLD) return;  // windowed / Taylor columns are row-local (sweep_zone_kernel)
    double D = 0.0;
    int t = t0;
    double Jp;
    if (t == 0) {
      Jp = src(0, m, mu);
      t = 1;
    } else {
      Jp = src(t - 1, m, mu);
    }
    double tp = tau[t - 1 < 0 ? 0 : t - 1];
    auto body = [&](auto gen_tag) {
      // LOCAL_UNROLL independent loads / exps in flight, one dependent DFMA chain
      for (; t + LOCAL_UNROLL - 1 < t1; t += LOCAL_UNROLL) {
        double tc[LOCAL_UNROLL], jv[LOCAL_UNROLL], a[LOCAL_UNROLL], b[LOCAL_UNROLL];
#pragma unroll
        for (int u = 0; u < LOCAL_UNROLL; ++u) {
          tc[u] = tau[t + u];
          jv[u] = jrow(gen_tag, t + u);
        }
#pragma unroll
        for (int u = 0; u < LOCAL_UNROLL; ++u) {
          const double d = tc[u] - (u ? tc[u - 1] : tp);
          a[u] = exp_small(d * imu);
          b[u] = (d * 0.5) * ((u ? jv[u - 1] : Jp) * a[u] + jv[u]) * imu;
        }
#pragma unroll
        for (int u = 0; u < LOCAL_UNROLL; ++u) D = D * a[u] - b[u];
        Jp = jv[LOCAL_UNROLL - 1];
        tp = tc[LOCAL_UNROLL - 1];
      }
      for (; t < t1; ++t) {
        const double tc = tau[t];
        const double jc = jrow(gen_tag, t);
        const double d = tc - tp;
        const double a = exp_small(d * imu);
        D = D * a - (d * 0.5) * (Jp * a + jc) * imu;
        Jp = jc;
        tp = tc;
      }
    };
    if (cg) {
      // rebuilt source: nothing is read but tau and the two coefficients of each row; 4 rows per step, the short
      // polynomial where every step of the group is tiny (x = dtau / mu is the same sign-definite exponent everywhere)
      const double2* __restrict__ pc = src.cj2 + t;
      const double* __restrict__ pt = tau + t;
      const double ximax = fabs(imu);
      for (; t + 3 < t1; t += 4, pc += 4, pt += 4) {
        double tc[4], jv[4], x[4], a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          tc[u] = pt[u];
          const double2 cc = pc[u];
          jv[u] = fma(cc.y, q, cc.x);
        }
        double dmax = 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const double d = tc[u] - (u ? tc[u - 1] : tp);
          dmax = fmax(dmax, d);
          x[u] = d * imu;
        }
        if (dmax * ximax <= kTinyArg) {
#pragma unroll
          for (int u = 0; u < 4; ++u) a[u] = exp_tiny(x[u]);
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) a[u] = exp_small(x[u]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) D = fma(D, a[u], -(0.5 * x[u]) * fma(u ? jv[u - 1] : Jp, a[u], jv[u]));
        Jp = jv[3];
        tp = tc[3];
      }
      body(std::true_type{});
    } else {
      body(std::false_type{});
    }
    aggD[agg] = D;
  } else {
    double U = 0.0;
    int t = t1 - 1;
    double Jn, tn;
    if (t == L - 1) {
      Jn = src(t, m, mu);
      tn = tau[t];
      --t;
    } else {
      Jn = src(t + 1, m, mu);
      tn = tau[t + 1];
      // chunk ends at a region boundary: the slice stops one row short of the carry row
      // (SOS_Aer_main_specular.py:413,433) -> pure attenuation, no source on this step
      if (g.chunk_region[c + 1] != g.chunk_region[c]) {
        Jn = src(t, m, mu);
        tn = tau[t];
        --t;
      }
    }
    auto body = [&](auto gen_tag) {
      for (; t - (LOCAL_UNROLL - 1) >= t0; t -= LOCAL_UNROLL) {
        double tc[LOCAL_UNROLL], jv[LOCAL_UNROLL], a[LOCAL_UNROLL], b[LOCAL_UNROLL];
#pragma unroll
        for (int u = 0; u < LOCAL_UNROLL; ++u) {
          tc[u] = tau[t - u];
          jv[u] = jrow(gen_tag, t - u);
        }
#pragma unroll
        for (int u = 0; u < LOCAL_UNROLL; ++u) {
          const double d = (u ? tc[u - 1] : tn) - tc[u];
          a[u] = exp_small(-d * imu);
          b[u] = (d * 0.5) * (jv[u] + (u ? jv[u - 1] : Jn) * a[u]) * imu;
        }
#pragma unroll
        for (int u = 0; u < LOCAL_UNROLL; ++u) U = U * a[u] + b[u];
        Jn = jv[LOCAL_UNROLL - 1];
        tn = tc[LOCAL_UNROLL - 1];
      }
      for (; t >= t0; --t) {
        const double tc = tau[t];
        const double jc = jrow(gen_tag, t);
        const double d = tn - tc;
        const double a = exp_small(-d * imu);
        U = U * a + (d * 0.5) * (jc + Jn * a) * imu;
        Jn = jc;
        tn = tc;
      }
    };
    if (cg) {
      const double2* __restrict__ pc = src.cj2 + t;
      const double* __restrict__ pt = tau + t;
      const double ximax = fabs(imu);
      for (; t - 3 >= t0; t -= 4, pc -= 4, pt -= 4) {
        double tc[4], jv[4], x[4], a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          tc[u] = pt[-u];
          const double2 cc = pc[-u];
          jv[u] = fma(cc.y, q, cc.x);
        }
        double dmax = 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const double d = (u ? tc[u - 1] : tn) - tc[u];
          dmax = fmax(dmax, d);
          x[u] = -d * imu;
        }
        if (dmax * ximax <= kTinyArg) {
#pragma unroll
          for (int u = 0; u < 4; ++u) a[u] = exp_tiny(x[u]);
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) a[u] = exp_small(x[u]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) U = fma(U, a[u], -(0.5 * x[u]) * fma(u ? jv[u - 1] : Jn, a[u], jv[u]));
        Jn = jv[3];
        tn = tc[3];
      }
      body(std::true_type{});
    } else {
      body(std::false_type{});
    }
    aggU[agg] = U;
  }
}

// ------------------------------------------------------------------------------------------
// row-level helpers of sweep_carry_kernel (one CTA works on one row in smem)
// ------------------------------------------------------------------------------------------

// |mu| < MU_THRESHOLD downward column m at layer t (improved_asymptotic_downward_radiance,
// SOS_Aer_In_limit.py:70-109).  One warp per call; every lane returns the value.
__device__ __forceinline__ double asymptotic_column(const GridDev& g, const SrcAt& src,
                                                    const double* __restrict__ tau, int t, int r0, int m) {
  const int lane = threadIdx.x & 31;
  const double mu = g.mu[m];
  const double jt = src(t, m, mu);
  if (fabs(mu) < SOS_MU_VERY_SMALL) {  // Taylor: -J + mu dJ/dtau (:79-93)
    double slope = 0.0;
    if (t > r0) slope = (jt - src(t - 1, m, mu)) / (tau[t] - tau[t - 1]);
    return -jt + mu * slope;
  }
  // windowed trapezoid over tau' >= tau_t - 5|mu| inside the region slice (:96-107)
  const double tt = tau[t];
  const double lim = tt - 5.0 * fabs(mu);
  int lo = r0, hi = t;  // first k in [r0, t] with tau[k] >= lim (tau is non-decreasing)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (tau[mid] >= lim) hi = mid; else lo = mid + 1;
  }
  const int k0 = lo;
  double sum = 0.0;
  bool bad = false;
  // interval k..k+1 handled by lane (k-k0)%32; fixed order -> deterministic
  for (int k = k0 + lane; k < t; k += 32) {
    const double f0 = src(k, m, mu) * exp((tt - tau[k]) / mu);
    const double f1 = src(k + 1, m, mu) * exp((tt - tau[k + 1]) / mu);
    bad |= !isfinite(f0) || !isfinite(f1);
    sum += (tau[k + 1] - tau[k]) * (f1 + f0) * 0.5;
  }
  if (t == k0) bad |= !isfinite(jt);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  bad = __any_sync(0xffffffffu, bad);
  if (bad) return -jt;  // (:104-105)
  return -sum / mu;
}

// Complete the downward half of a row held in smem `row[0..M-1]`:
// windowed/Taylor columns that survive the extrapolation, then the extrapolation itself.
// Must be called by all threads of the CTA; contains __syncthreads.
__device__ __forceinline__ void finish_down_row(const GridDev& g, double* row, const SrcAt& src,
                                                const double* __restrict__ tau, int t, int region, int idx_width,
                                                int wclass) {
  const int M = g.M;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int r0 = g.rstart[region];
  // columns first_small .. M-2 are non-standard; those >= M - idx are overwritten below -> skip them
  const int hi = min(M - 1, M - idx_width);
  for (int m = g.first_small + warp; m < hi; m += nwarps) {
    const double v = asymptotic_column(g, src, tau, t, r0, m);
    if (lane == 0) row[m] = v;
  }
  __syncthreads();
  if (idx_width > 0) {
    // sources (columns < M - idx) and targets (columns >= M - idx) never overlap
    const int ns = g.wns[wclass];
    const int src0 = (idx_width < 2) ? (M - idx_width - 2) : (M - idx_width - ns);
    const double* __restrict__ W = g.W + g.woff[wclass];
    for (int i = threadIdx.x; i < idx_width; i += blockDim.x) {
      double v = 0.0;
      for (int j = 0; j < ns; ++j) v += W[i * ns + j] * row[src0 + j];
      row[M - 1 - i] = v;
    }
  }
  __syncthreads();
}

// Blend of the upward half towards mu = 0+ (SOS_Aer_I1_In.py:101-108).  row[M] must already hold J[t,M].
// `found` is a shared int.  All threads of the CTA must call; returns false on search overrun (Q11).
__device__ __forceinline__ bool blend_up_row(const GridDev& g, double* row, int* found) {
  const int M = g.M, N = g.col1;  // the search never leaves the owned columns
  if (threadIdx.x == 0) *found = 0x7fffffff;
  __syncthreads();
  for (int base = M + 1; base + 2 <= N - 1; base += blockDim.x) {
    const int i = base + threadIdx.x;
    if (i + 2 <= N - 1) {
      const double d = fabs((row[i] - row[i + 1]) - (row[i + 1] - row[i + 2]));
      if (!(d > SOS_BLEND_THRESHOLD)) atomicMin(found, i);
    }
    __syncthreads();
    const int f = *found;
    __syncthreads();
    if (f != 0x7fffffff) break;
  }
  const int f = *found;
  if (f == 0x7fffffff) return false;
  const int istar = f + 1;
  const double v0 = row[M], v1 = row[istar], mus = g.mu[istar];
  __syncthreads();
  for (int m = M + 1 + threadIdx.x; m < istar; m += blockDim.x) {
    const double w = g.mu[m] / mus;
    row[m] = (1.0 - w) * v0 + w * v1;
  }
  __syncthreads();
  return true;
}

__device__ __forceinline__ int width_class(const GridDev& g, int idx_width) {
  // widths are one of the four classes of sos_extrap_layout (or 0)
  int c = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (g.widx[k] == idx_width) c = k;
  return c;
}

// deterministic block sum (blockDim.x multiple of 32, <= 1024); result valid in all threads
__device__ __forceinline__ double block_sum(double v, double* scratch /*[32]*/) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  double tot = 0.0;
  for (int w = 0; w < nwarps; ++w) tot += scratch[w];
  __syncthreads();
  return tot;
}

// ------------------------------------------------------------------------------------------
// 2. carry chain (one CTA per scenario)
// ------------------------------------------------------------------------------------------
// NK = number of kernel matrices of a bidirectional ground (brdf.cuh): 2 for the Ross-Li ground (SOS_SURFACE_ROSSLI), 1 for
// the ocean's glint (SOS_SURFACE_OCEAN), each the lambert_readme term with grd_alb as the isotropic part plus NK mat-vecs;
// 0 for every other surface.  Separate instantiations, so that the kernel of the other surfaces is compiled as without them.
template <int NK>
__global__ void __launch_bounds__(CARRY_THREADS)
sweep_carry_kernel(const GridDev g, const SrcGen sg, const double* __restrict__ J, const double* __restrict__ aggD,
                   const double* __restrict__ aggU, double* __restrict__ carryD, double* __restrict__ carryU,
                   const sosbrdf::BrdfDev brdf) {
  extern __shared__ double sm_row[];  // [N] + scratch[32] + tau at the chunk boundaries: [nch + 1] (down), [nch + 1] (up)
  __shared__ int found;
  const int s = blockIdx.x;
  if (!g.state[s].active) return;
  const int L = g.L, M = g.M, N = g.N, nch = g.nchunks;
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const SrcAt src(g, sg, J, s);
  const sos_scenario sc = g.scen[s];
  double* row = sm_row;
  double* scratch = sm_row + N;
  // the decay of a carry across chunk c needs tau at the chunk boundaries: staged once (read through chunk_start -> tau inside
  // the chains they are two dependent loads in front of every batch of exps)
  double* td = scratch + 32;      // td[c] = tau at the last row before chunk c
  double* tu = td + nch + 1;      // tu[c] = tau at the first row of chunk c (tu[nch] = tau at the surface row)
  for (int c = threadIdx.x; c <= nch; c += blockDim.x) {
    const int t0 = g.chunk_start[c];
    td[c] = tau[t0 > 0 ? t0 - 1 : 0];
    tu[c] = tau[t0 < L ? t0 : L - 1];
  }
  __syncthreads();
  const size_t base = static_cast<size_t>(s) * nch * N;

  // ---- down: chain the standard columns through the chunks ----
  // (the loads of the chunk aggregates and the decay factors do not depend on the carry: fetch them
  //  eight chunks at a time so that only the FMA chain is serial)
  for (int m = threadIdx.x; m < M - 1; m += blockDim.x) {
    const double mu = g.mu[m];
    double cd = 0.0;
    if (fabs(mu) >= SOS_MU_THRESHOLD && m >= g.col0 && m < g.col1) {
      for (int c0 = 0; c0 < nch; c0 += 8) {
        double ag[8], ex[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int c = c0 + u;
          ag[u] = 0.0;
          ex[u] = 0.0;
          if (c < nch) {
            ag[u] = aggD[base + static_cast<size_t>(c) * N + m];
            if (c > 0) ex[u] = exp((td[c + 1] - td[c]) / mu);
          }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int c = c0 + u;
          if (c < nch) {
            carryD[base + static_cast<size_t>(c) * N + m] = cd;
            cd = ag[u] + cd * ex[u];
          }
        }
      }
    }
    row[m] = cd;  // true D at the surface row for standard columns
  }
  if (threadIdx.x == 0) row[M - 1] = 0.0;
  __syncthreads();

  // ---- surface row: finish the downward half, then couple ----
  const int last_region = g.nreg - 1;
  if (g.surface != SOS_SURFACE_NONE) {
    const int idxw = sc.extrap_width[last_region];
    finish_down_row(g, row, src, tau, L - 1, last_region, idxw, width_class(g, idxw));
  }
  double lambert = 0.0;
  if (g.surface == SOS_SURFACE_LAMBERT) {
    // -2 rho trapz(I[L-1,c] mu[c], mu[c]) over c = M-2 .. 0 (descending abscissa, column M-1 excluded)
    double part = 0.0;
    for (int j = threadIdx.x; j < M - 2; j += blockDim.x) {
      const int c0 = M - 2 - j, c1 = c0 - 1;
      part += (g.mu[c1] - g.mu[c0]) * (row[c1] * g.mu[c1] + row[c0] * g.mu[c0]) * 0.5;
    }
    lambert = -2.0 * sc.grd_alb * block_sum(part, scratch);
  } else if (NK > 0 || g.surface == SOS_SURFACE_LAMBERT_README || g.surface == SOS_SURFACE_LAMBERT_DIFFUSE) {
    // README.md:215: -2 rho int_{-1}^{0} I mu dmu with the abscissa ascending and the interval next to mu = 0 included
    double part = 0.0;
    for (int c0 = threadIdx.x; c0 < M - 1; c0 += blockDim.x) {
      const int c1 = c0 + 1;
      part += (g.mu[c1] - g.mu[c0]) * (row[c1] * g.mu[c1] + row[c0] * g.mu[c0]) * 0.5;
    }
    lambert = -2.0 * sc.grd_alb * block_sum(part, scratch);
  }
  // seeds into the upper half of the row buffer
  if constexpr (NK > 0) {
    // the downward half becomes u_c = -2 w_c mu_c I[L-1, c] in place (the up chain reads row[M ..] only); every upward
    // column adds f_vol sum_c u_c R^vol[c][i] + f_geo sum_c u_c R^geo[c][i] (Ross-Li) or f_glint sum_c u_c R[c][i] (ocean)
    // to the isotropic term
    for (int c = threadIdx.x; c < M; c += blockDim.x) row[c] *= sosbrdf::coupling_weight(g.mu, M, c);
    __syncthreads();
    const double fv = brdf.f[2 * s], fg = brdf.f[2 * s + 1];
    for (int m = M + 1 + threadIdx.x; m < N; m += blockDim.x) {
      if constexpr (NK == 2) {
        double sv, sgeo;
        sosbrdf::coupling(brdf, s, row, M, m - M - 1, sv, sgeo);
        row[m] = lambert + (fv * sv + fg * sgeo);
      } else {
        row[m] = lambert + fv * sosbrdf::coupling(brdf, s, row, M, m - M - 1);
      }
    }
  } else {
    for (int m = M + 1 + threadIdx.x; m < N; m += blockDim.x) {
      double seed = 0.0;
      if (g.surface == SOS_SURFACE_SPECULAR) seed = sc.grd_alb * row[N - 1 - m];
      else if (g.surface == SOS_SURFACE_LAMBERT || g.surface == SOS_SURFACE_LAMBERT_README || g.surface == SOS_SURFACE_LAMBERT_DIFFUSE)
        seed = lambert;
      row[m] = seed;
    }
  }
  __syncthreads();

  // ---- up: chain from the surface, re-seeding from blended rows at region boundaries ----
  int c = nch - 1;
  while (c >= 0) {
    // batch [ce, c]: at most 8 chunks, ending at the first chunk that starts a region
    int ce = c, nb = 1;
    while (nb < 8 && ce > 0 && g.chunk_region[ce - 1] == g.chunk_region[ce]) { --ce; ++nb; }
    for (int m = M + 1 + threadIdx.x; m < N; m += blockDim.x) {
      if (m < g.col0 || m >= g.col1) continue;
      const double mu = g.mu[m];
      double ag[8], ex[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int cc = c - u;
        ag[u] = 0.0;
        ex[u] = 0.0;
        if (cc >= ce) {
          ag[u] = aggU[base + static_cast<size_t>(cc) * N + m];
          ex[u] = exp(-(tu[cc + 1] - tu[cc]) / mu);
        }
      }
      double cu = row[m];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int cc = c - u;
        if (cc >= ce) {
          carryU[base + static_cast<size_t>(cc) * N + m] = cu;
          cu = ag[u] + cu * ex[u];  // raw U at the first row of chunk cc
        }
      }
      row[m] = cu;
    }
    if (ce > 0 && g.chunk_region[ce - 1] != g.chunk_region[ce]) {
      // row chunk_start[ce] is the carry row of the region above and is read after its blend (A.7)
      if (threadIdx.x == 0) row[M] = src(g.chunk_start[ce], M, g.mu[M]);
      __syncthreads();
      if (!blend_up_row(g, row, &found) && threadIdx.x == 0) atomicOr(&g.state[s].status, SOS_STATUS_BLEND_OVERRUN);
    }
    c = ce - 1;
  }
}

// The carry chain of a single-region grid without surface coupling (the single-layer operator In_NumInt,
// SOS_Aer_I1_In.py:77-130): no row-level work couples the columns, so every column chains on its own.  With many chunks
// (one large grid: 10 000 layers = hundreds of chunks) a serial chain per column is the critical path of the sweeps, so the
// chain itself is a two-level scan: a CTA owns 16 columns, thread (g, col) owns a group of consecutive chunks of its
// column (in chain order: top-down for the downward half, bottom-up for the upward one).  It composes its group into one
// affine map carry_out = B + P carry_in (all loads of the group in flight at once), the 32 maps of a column are chained
// through shared memory by one thread (32 FMAs), and every thread re-chains its group from the true incoming carry.  A
// fixed order of operations: deterministic, and the same for sharded and unsharded plans.  Layer-sharded plans exchange
// their aggregates with the peers here, column group by column group (layer_shard.cuh: exchange_aggregates).
constexpr int CARRY_COLS = soslayer::COL_GROUP;  // columns per CTA (one 128-byte line of an aggregate row)
constexpr int CARRY_GROUPS = 32;   // chunk groups per column
__global__ void __launch_bounds__(CARRY_COLS * CARRY_GROUPS)
sweep_carry_cols_kernel(const GridDev g, const double* __restrict__ aggD, const double* __restrict__ aggU,
                        double* __restrict__ carryD, double* __restrict__ carryU, const soslayer::LayerPeers lp) {
  extern __shared__ double sm_tb[];  // [nch + 1] tau at the last row before each chunk (down), [nch + 1] at its first row (up)
  __shared__ double sP[CARRY_GROUPS][CARRY_COLS + 1], sB[CARRY_GROUPS][CARRY_COLS + 1];
  const int s = blockIdx.y;
  if (!g.state[s].active) return;
  const int L = g.L, M = g.M, N = g.N, nch = g.nchunks;
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  double* td = sm_tb;
  double* tu = sm_tb + nch + 1;
  for (int c = threadIdx.x; c <= nch; c += blockDim.x) {
    const int t0 = g.chunk_start[c];
    td[c] = tau[t0 > 0 ? t0 - 1 : 0];
    tu[c] = tau[t0 < L ? t0 : L - 1];
  }
  if (lp.n > 1) {
    // (aggD / aggU are this rank's tables inside its mailbox; the peers' CTAs of the same column group write theirs into them)
    if (soslayer::exchange_aggregates(g, lp, blockIdx.x) && threadIdx.x == 0) atomicOr(&g.state[s].status, SOS_STATUS_PEER_TIMEOUT | SOS_STATUS_NONFINITE);
  }
  __syncthreads();
  const int tx = threadIdx.x & (CARRY_COLS - 1), ty = threadIdx.x / CARRY_COLS;
  const int m = blockIdx.x * CARRY_COLS + tx;
  const bool up = m > M;
  // windowed / Taylor columns are row-local (sweep_zone_kernel); mu = 0 has no recurrence
  const bool live = m < N && m >= g.col0 && m < g.col1 && m != M - 1 && m != M && (up || fabs(g.mu[m]) >= SOS_MU_THRESHOLD);
  const double imu = live ? 1.0 / g.mu[m] : 0.0;
  const double* __restrict__ agg = up ? aggU : aggD;
  double* __restrict__ carry = up ? carryU : carryD;
  const size_t base = static_cast<size_t>(s) * nch * N + (live ? m : 0);
  const int k = (nch + CARRY_GROUPS - 1) / CARRY_GROUPS;
  const int j0 = ty * k, j1 = min(nch, j0 + k);   // this thread's positions in chain order
  // chunk at chain position j, and the attenuation of a carry across it
  auto chunk_of = [&](int j) { return up ? nch - 1 - j : j; };
  auto decay = [&](int c) -> double {
    if (up) return exp(-(tu[c + 1] - tu[c]) * imu);
    return c > 0 ? exp((td[c + 1] - td[c]) * imu) : 0.0;  // (nothing enters the first chunk from above)
  };
  // (groups of up to eight chunks keep their aggregates and decay factors in registers between the two passes)
  double P = 1.0, B = 0.0;
  double ag0[8], ex0[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) { ag0[u] = 0.0; ex0[u] = 1.0; }
  if (live) {
    for (int jb = j0; jb < j1; jb += 8) {
      double ag[8], ex[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int j = jb + u;
        ag[u] = j < j1 ? agg[base + static_cast<size_t>(chunk_of(j)) * N] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) ex[u] = (jb + u < j1) ? decay(chunk_of(jb + u)) : 1.0;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (jb + u < j1) {
          B = fma(B, ex[u], ag[u]);
          P *= ex[u];
        }
        if (jb == j0) { ag0[u] = ag[u]; ex0[u] = ex[u]; }
      }
    }
  }
  sP[ty][tx] = P;
  sB[ty][tx] = B;
  __syncthreads();
  if (ty == 0) {
    // incoming carry of every group of this column (nothing enters the chain: TOA above, no surface coupling below)
    double cin = 0.0;
#pragma unroll 8
    for (int q = 0; q < CARRY_GROUPS; ++q) {
      const double p = sP[q][tx], b = sB[q][tx];
      sB[q][tx] = cin;
      cin = fma(cin, p, b);
    }
  }
  __syncthreads();
  if (!live) return;
  double cc = sB[ty][tx];
  for (int jb = j0; jb < j1; jb += 8) {
    double ag[8], ex[8];
    if (jb == j0) {
#pragma unroll
      for (int u = 0; u < 8; ++u) { ag[u] = ag0[u]; ex[u] = ex0[u]; }
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int j = jb + u;
        ag[u] = j < j1 ? agg[base + static_cast<size_t>(chunk_of(j)) * N] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) ex[u] = (jb + u < j1) ? decay(chunk_of(jb + u)) : 1.0;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (jb + u < j1) {
        carry[base + static_cast<size_t>(chunk_of(jb + u)) * N] = cc;  // value entering the chunk (down: at the row above it, up: at the row below it)
        cc = fma(cc, ex[u], ag[u]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// 3. apply the carries (chunk x column threads) and finish the mu -> 0 zone (row CTAs)
// ------------------------------------------------------------------------------------------

// first downward column of the row-wise zone: all non-standard columns, the extrapolation targets and
// their sources (largest width of the scenario)
__device__ __forceinline__ int zone_lo(const GridDev& g, const sos_scenario& sc) {
  int w = 0;
  for (int k = 0; k < g.nreg; ++k) w = max(w, sc.extrap_width[k]);
  const int ns = (w <= 0) ? 0 : (w < 2 ? 2 : min(5, w));
  return max(0, min(g.first_small, g.M - w - ns));
}

// Second sweep pass: the same recurrences as sweep_local_kernel, now started from the TRUE carry of the
// chunk, writing the final I_n and accumulating I += I_n in the same pass (J 8 + I_n 8 + I 16 bytes per
// element; 16 where the source is rebuilt and I_n is not kept).  The few columns next to mu = 0 that the reference
// post-processes are corrected afterwards by sweep_zone_kernel (it replaces the raw value in I_n and adds the
// difference to I).  Every lane of a warp runs the same rows (lanes without a column compute on zeros and store
// nothing), so the projections of a group of four rows are reduced with one butterfly.
__global__ void __launch_bounds__(LOCAL_THREADS)
sweep_apply_kernel(const GridDev g, const SrcGen sg, const double* __restrict__ J, double* __restrict__ In,
                   const double* __restrict__ carryD, const double* __restrict__ carryU,
                   double* __restrict__ I, double* __restrict__ saved) {
  const int s = blockIdx.z;
  if (!g.state[s].active) return;
  const int c = g.c_lo + blockIdx.y;  // (layer-sharded plans own the chunks [c_lo, c_hi))
  const int L = g.L, M = g.M, ld = g.ld;
  const int lane = threadIdx.x & 31;
  const int nbd = scan_blocks_down(M, LOCAL_THREADS);
  const bool up = static_cast<int>(blockIdx.x) >= nbd;
  const int m = up ? M + 1 + (blockIdx.x - nbd) * LOCAL_THREADS + threadIdx.x : blockIdx.x * LOCAL_THREADS + threadIdx.x;
  const bool in_range = up ? (m < g.N) : (m < M - 1);
  const double mu_raw = in_range ? g.mu[m] : (up ? 1.0 : -1.0);
  // windowed / Taylor columns are row-local (sweep_zone_kernel); mu-block plans own [col0, col1)
  const bool valid = in_range && (up || fabs(mu_raw) >= SOS_MU_THRESHOLD) && m >= g.col0 && m < g.col1;
  if (!__any_sync(0xffffffffu, valid)) return;
  const int t0 = g.chunk_start[c], t1 = g.chunk_start[c + 1];
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const size_t fbase = static_cast<size_t>(s) * L * ld;
  const SrcAt src(g, sg, J, s);
  const double* __restrict__ Js = src.Js;
  double* __restrict__ Is = In + fbase;
  double* __restrict__ Ia = I ? I + fbase : nullptr;
  double* __restrict__ Sv = saved ? saved + fbase : nullptr;
  const double mu = valid ? mu_raw : (up ? 1.0 : -1.0);
  const double imu = 1.0 / mu;  // one division per thread; the scan steps multiply
  const double q = mu * mu;
  const size_t agg = (static_cast<size_t>(s) * g.nchunks + c) * g.N + (valid ? m : 0);
  const bool cg = src.gen_row(t0);  // the whole chunk is rebuilt, or read
  const bool zonecol = up ? (m < sg.zu_end) : (m >= sg.zlo);
  const bool keep_in = !cg || zonecol || sg.store_all;  // I_n of this column is read by someone on every row
  const int op = g.scen[s].phase_atm;
  const bool zoneproj = up ? (m < sg.zu_proj) : (m >= sg.zlo);  // projected by the zone kernel (final values)
  const double us0 = (cg && valid && !zoneproj) ? sg.Ut[op][m] : 0.0;
  const double us1 = (cg && valid && !zoneproj) ? sg.Ut[op][sg.ldr + m] : 0.0;
  double* const projs = cg ? sg.proj + (static_cast<size_t>(s) * L * sg.nslots + blockIdx.x * (LOCAL_THREADS / 32) + (threadIdx.x >> 5)) * 2 : nullptr;
  const int forced = up ? 0 : L - 1;  // the row whose I_n everybody stores: ratios, surface coupling

  auto jrow = [&](auto gen_tag, int t) -> double {
    if (decltype(gen_tag)::value) {
      const double2 cc = src.cj2[t];
      return fma(cc.y, q, cc.x);
    }
    return valid ? Js[static_cast<size_t>(t) * ld + m] : 0.0;
  };
  auto jany = [&](int t) -> double { return (valid || src.gen_row(t)) ? src(t, valid ? m : 0, mu) : 0.0; };
  // store I_n (and I_saved); accumulate with the I value that was prefetched together with J
  auto emit = [&](int t, double v, double iold) {
    if (valid) {
      const size_t o = static_cast<size_t>(t) * ld + m;
      if (keep_in || t == forced) Is[o] = v;
      if (Sv) Sv[o] = v;
      if (Ia) Ia[o] = iold + v;
    }
  };
  auto iold = [&](int t) -> double { return (Ia && valid) ? Ia[static_cast<size_t>(t) * ld + m] : 0.0; };
  // projections of one row (tail rows and the rows outside the unrolled loop): plain butterfly
  auto project1 = [&](int t, double v) {
    if (!cg) return;
    double p0 = v * us0, p1 = v * us1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { p0 += shfl_xor_d(p0, o); p1 += shfl_xor_d(p1, o); }
    if (lane == 0) *reinterpret_cast<double2*>(projs + static_cast<size_t>(t) * sg.nslots * 2) = make_double2(p0, p1);
  };
  // ... of four rows t, t + step, ...: transpose-reduce
  auto project4 = [&](int t, int step, double v0, double v1, double v2, double v3) {
    if (!cg) return;
    double v[8] = {v0 * us0, v1 * us0, v2 * us0, v3 * us0, v0 * us1, v1 * us1, v2 * us1, v3 * us1};
    const double tot = transpose_reduce8(v, lane);
    const int idx = lane >> 2;
    if ((lane & 3) == 0) projs[static_cast<size_t>(t + step * (idx & 3)) * sg.nslots * 2 + (idx >> 2)] = tot;
  };

  if (!up) {
    double D = (t0 > 0 && valid) ? carryD[agg] : 0.0;
    int t = t0;
    double Jp;
    if (t == 0) {
      Jp = jany(0);
      emit(0, 0.0, iold(0));
      project1(0, 0.0);
      t = 1;
    } else {
      Jp = jany(t - 1);
    }
    double tp = tau[t - 1 < 0 ? 0 : t - 1];
    auto body = [&](auto gen_tag) {
      for (; t + 3 < t1; t += 4) {
        const double tc0 = tau[t], tc1 = tau[t + 1], tc2 = tau[t + 2], tc3 = tau[t + 3];
        const double j0 = jrow(gen_tag, t), j1 = jrow(gen_tag, t + 1), j2 = jrow(gen_tag, t + 2), j3 = jrow(gen_tag, t + 3);
        const double i0 = iold(t), i1 = iold(t + 1), i2 = iold(t + 2), i3 = iold(t + 3);
        const double d0 = tc0 - tp, d1 = tc1 - tc0, d2 = tc2 - tc1, d3 = tc3 - tc2;
        const double a0 = exp_small(d0 * imu), a1 = exp_small(d1 * imu), a2 = exp_small(d2 * imu), a3 = exp_small(d3 * imu);
        const double b0 = (d0 * 0.5) * (Jp * a0 + j0) * imu;
        const double b1 = (d1 * 0.5) * (j0 * a1 + j1) * imu;
        const double b2 = (d2 * 0.5) * (j1 * a2 + j2) * imu;
        const double b3 = (d3 * 0.5) * (j2 * a3 + j3) * imu;
        const double D0 = D * a0 - b0, D1 = D0 * a1 - b1, D2 = D1 * a2 - b2, D3 = D2 * a3 - b3;
        emit(t, D0, i0);
        emit(t + 1, D1, i1);
        emit(t + 2, D2, i2);
        emit(t + 3, D3, i3);
        project4(t, 1, D0, D1, D2, D3);
        D = D3;
        Jp = j3;
        tp = tc3;
      }
      for (; t < t1; ++t) {
        const double tc = tau[t];
        const double jc = jrow(gen_tag, t);
        const double io = iold(t);
        const double d = tc - tp;
        const double a = exp_small(d * imu);
        D = D * a - (d * 0.5) * (Jp * a + jc) * imu;
        emit(t, D, io);
        project1(t, D);
        Jp = jc;
        tp = tc;
      }
    };
    if (cg) body(std::true_type{}); else body(std::false_type{});
  } else {
    double U = valid ? carryU[agg] : 0.0;  // value at the carry row (t1, or the surface seed for the last chunk)
    int t = t1 - 1;
    double Jn, tn;
    if (t == L - 1) {
      Jn = jany(t);
      tn = tau[t];
      emit(t, U, iold(t));  // zero-length integral: the surface row is the seed itself
      project1(t, U);
      --t;
    } else {
      Jn = jany(t + 1);
      tn = tau[t + 1];
      if (g.chunk_region[c + 1] != g.chunk_region[c]) {  // carry gap: pure attenuation on this step
        const double tc = tau[t];
        U = U * exp(-(tn - tc) / mu);
        emit(t, U, iold(t));
        project1(t, U);
        Jn = jany(t);
        tn = tc;
        --t;
      }
    }
    auto body = [&](auto gen_tag) {
      for (; t - 3 >= t0; t -= 4) {
        const double tc0 = tau[t], tc1 = tau[t - 1], tc2 = tau[t - 2], tc3 = tau[t - 3];
        const double j0 = jrow(gen_tag, t), j1 = jrow(gen_tag, t - 1), j2 = jrow(gen_tag, t - 2), j3 = jrow(gen_tag, t - 3);
        const double i0 = iold(t), i1 = iold(t - 1), i2 = iold(t - 2), i3 = iold(t - 3);
        const double d0 = tn - tc0, d1 = tc0 - tc1, d2 = tc1 - tc2, d3 = tc2 - tc3;
        const double a0 = exp_small(-d0 * imu), a1 = exp_small(-d1 * imu), a2 = exp_small(-d2 * imu), a3 = exp_small(-d3 * imu);
        const double b0 = (d0 * 0.5) * (j0 + Jn * a0) * imu;
        const double b1 = (d1 * 0.5) * (j1 + j0 * a1) * imu;
        const double b2 = (d2 * 0.5) * (j2 + j1 * a2) * imu;
        const double b3 = (d3 * 0.5) * (j3 + j2 * a3) * imu;
        const double U0 = U * a0 + b0, U1 = U0 * a1 + b1, U2 = U1 * a2 + b2, U3 = U2 * a3 + b3;
        emit(t, U0, i0);
        emit(t - 1, U1, i1);
        emit(t - 2, U2, i2);
        emit(t - 3, U3, i3);
        project4(t, -1, U0, U1, U2, U3);
        U = U3;
        Jn = j3;
        tn = tc3;
      }
      for (; t >= t0; --t) {
        const double tc = tau[t];
        const double jc = jrow(gen_tag, t);
        const double io = iold(t);
        const double d = tn - tc;
        const double a = exp_small(-d * imu);
        U = U * a + (d * 0.5) * (jc + Jn * a) * imu;
        emit(t, U, io);
        project1(t, U);
        Jn = jc;
        tn = tc;
      }
    };
    if (cg) body(std::true_type{}); else body(std::false_type{});
  }
}

// The apply pass with TWO adjacent columns per thread (16-byte accesses: 2 KB per row and CTA, half the per-row
// overhead per element) for grids with an odd number of angles per half (the reference's: the first upward column
// M + 1 is then even, so every pair is 16-byte aligned and lies inside one half).  Same recurrences, same outputs;
// the projections of a group of four rows are reduced through a small per-warp buffer in shared memory.
constexpr int APPLY2_THREADS = 128;
#ifndef SOS_APPLY2_RING
#define SOS_APPLY2_RING 4
#endif
#ifndef SOS_APPLY2_MINB
#define SOS_APPLY2_MINB 4
#endif
constexpr int APPLY2_RING = SOS_APPLY2_RING;   // groups of four rows in the I ring: three in flight (12 rows, 24 KB per CTA) + the one consumed
constexpr int APPLY2_STAGE = 160;  // longest chunk whose per-row scalars are staged in shared memory
constexpr int PROJ_STRIDE = 34;  // doubles per row of the per-warp buffer (16-byte aligned rows, conflict-free 128-bit reads)

// v[0..7] of every lane -> the sum over the warp of v[lane >> 2], in the four lanes of quad lane >> 2 (fixed order)
__device__ __forceinline__ double quad_reduce8(double* buf, const double (&v)[8], int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) buf[i * PROJ_STRIDE + lane] = v[i];
  __syncwarp();
  const double2* row = reinterpret_cast<const double2*>(buf + (lane >> 2) * PROJ_STRIDE + (lane & 3) * 8);
  const double2 a = row[0], b = row[1], c = row[2], d = row[3];
  double sum = ((a.x + a.y) + (b.x + b.y)) + ((c.x + c.y) + (d.x + d.y));
  sum += shfl_xor_d(sum, 1);
  sum += shfl_xor_d(sum, 2);
  __syncwarp();
  return sum;
}

__global__ void __launch_bounds__(APPLY2_THREADS, SOS_APPLY2_MINB)
sweep_apply2_kernel(const GridDev g, const SrcGen sg, const double* __restrict__ J, double* __restrict__ In,
                    const double* __restrict__ carryD, const double* __restrict__ carryU,
                    double* __restrict__ I, double* __restrict__ saved) {
  __shared__ __align__(16) double s_proj[APPLY2_THREADS / 32][8 * PROJ_STRIDE];
  __shared__ __align__(16) double2 s_ring[APPLY2_RING * 4 * APPLY2_THREADS];
  __shared__ __align__(16) double2 s_cj[APPLY2_STAGE];
  __shared__ double s_tau[APPLY2_STAGE];
  const int s = blockIdx.z;
  if (!g.state[s].active) return;
  const int c = g.c_lo + blockIdx.y;  // (layer-sharded plans own the chunks [c_lo, c_hi))
  const int L = g.L, M = g.M, N = g.N, ld = g.ld;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nbd = ((M - 1) / 2 + APPLY2_THREADS - 1) / APPLY2_THREADS;
  const bool up = static_cast<int>(blockIdx.x) >= nbd;
  const int m0 = (up ? M + 1 : 0) + 2 * ((up ? blockIdx.x - nbd : blockIdx.x) * APPLY2_THREADS + threadIdx.x);
  const bool live = up ? (m0 < N) : (m0 < M - 1);
  const int t0 = g.chunk_start[c], t1 = g.chunk_start[c + 1];
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const size_t fbase = static_cast<size_t>(s) * L * ld;
  const SrcAt src(g, sg, J, s);
  const bool cg = src.gen_row(t0);  // the whole chunk is rebuilt, or read
  // the per-row scalars of the chunk (tau, source coefficients) go to shared memory once: read row by row from global
  // they cost an exposed L2 round trip per step of the main loop
  const bool staged = t1 - t0 <= APPLY2_STAGE;
  if (staged) {
    for (int i = threadIdx.x; i < t1 - t0; i += APPLY2_THREADS) {
      s_tau[i] = tau[t0 + i];
      if (cg) s_cj[i] = src.cj2[t0 + i];
    }
    __syncthreads();
  }
  const int op = g.scen[s].phase_atm;
  const size_t agg = (static_cast<size_t>(s) * g.nchunks + c) * N;
  bool stdc[2], anyzone = false;
  double mu[2], imu[2], q[2], us0[2], us1[2], X[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int m = m0 + k;
    mu[k] = live ? g.mu[m] : (up ? 1.0 : -1.0);
    stdc[k] = live && (up || fabs(mu[k]) >= SOS_MU_THRESHOLD);  // windowed / Taylor columns are row-local (sweep_zone_kernel)
    // columns without a recurrence get a zero exponent: a = 1, b = 0, their X stays 0 and I is written back unchanged
    imu[k] = stdc[k] ? 1.0 / mu[k] : 0.0;
    q[k] = mu[k] * mu[k];
    const bool zonecol = up ? (m < sg.zu_end) : (m >= sg.zlo);
    anyzone |= zonecol;
    const bool projected = cg && stdc[k] && !(up ? (m < sg.zu_proj) : (m >= sg.zlo));  // the others: zone kernel, final values
    us0[k] = projected ? sg.Ut[op][m] : 0.0;
    us1[k] = projected ? sg.Ut[op][sg.ldr + m] : 0.0;
    X[k] = 0.0;
    if (stdc[k]) X[k] = up ? carryU[agg + m] : (t0 > 0 ? carryD[agg + m] : 0.0);
  }
  const bool act = stdc[0] || stdc[1];                   // this thread stores
  if (!__any_sync(0xffffffffu, act)) return;
  const bool keep_in = !cg || anyzone || sg.store_all;   // I_n of this pair is read by someone on every row
  const int forced = up ? 0 : L - 1;                     // the row whose I_n everybody stores: ratios, surface coupling
  const double ximax = warp_max_d(fmax(fabs(imu[0]), fabs(imu[1])));  // the exp polynomial is chosen per warp
  const int ldv = ld / 2;
  double2* const Iv = reinterpret_cast<double2*>(I + fbase + (act ? m0 : 0));
  double2* const Nv = reinterpret_cast<double2*>(In + fbase + (act ? m0 : 0));
  double2* const Sv = saved ? reinterpret_cast<double2*>(saved + fbase + (act ? m0 : 0)) : nullptr;
  const double2* const Jv = reinterpret_cast<const double2*>(src.Js + (act ? m0 : 0));
  const size_t pstep = static_cast<size_t>(sg.nslots) * 2;
  double* const projs = cg ? sg.proj + (static_cast<size_t>(s) * L * sg.nslots + blockIdx.x * (APPLY2_THREADS / 32) + warp) * 2 : nullptr;
  double* const pbuf = s_proj[warp];
  const double sgn = up ? -1.0 : 1.0;  // x = sgn * dtau / mu is the (negative) exponent of the attenuation in either direction

  // J[t, m0 + k] of any row (rows of this chunk and the one next to it)
  auto jpair = [&](int t, double (&j)[2]) {
    if (src.gen_row(t)) {
      const double2 cc = src.cj2[t];
      j[0] = fma(cc.y, q[0], cc.x);
      j[1] = fma(cc.y, q[1], cc.x);
    } else if (act) {
      const double2 jv = Jv[static_cast<size_t>(t) * ldv];
      j[0] = jv.x;
      j[1] = jv.y;
    } else {
      j[0] = j[1] = 0.0;
    }
  };
  auto emit = [&](int t, const double (&v)[2]) {
    if (act) {
      const size_t o = static_cast<size_t>(t) * ldv;
      const double2 iv = Iv[o];
      Iv[o] = make_double2(iv.x + v[0], iv.y + v[1]);
      if (keep_in || t == forced) Nv[o] = make_double2(v[0], v[1]);
      if (Sv) Sv[o] = make_double2(v[0], v[1]);
    }
  };
  auto project1 = [&](int t, const double (&v)[2]) {
    if (!cg) return;
    double p0 = fma(v[1], us0[1], v[0] * us0[0]), p1 = fma(v[1], us1[1], v[0] * us1[0]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { p0 += shfl_xor_d(p0, o); p1 += shfl_xor_d(p1, o); }
    if (lane == 0) *reinterpret_cast<double2*>(projs + static_cast<size_t>(t) * pstep) = make_double2(p0, p1);
  };
  // one row of the recurrence: d = |tau step|, jn = J of the row processed before
  auto step1 = [&](int t, double d, double (&jn)[2]) {
    double j[2], v[2];
    jpair(t, j);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double x = sgn * d * imu[k];
      const double a = exp_small(x);
      X[k] = fma(X[k], a, -(0.5 * x) * fma(jn[k], a, j[k]));
      v[k] = stdc[k] ? X[k] : 0.0;
      jn[k] = j[k];
    }
    emit(t, v);
    project1(t, v);
  };

  double jn[2];
  int t;
  double tn;  // tau of the row processed before
  if (!up) {
    t = t0;
    if (t == 0) {
      jpair(0, jn);
      const double z[2] = {0.0, 0.0};
      emit(0, z);
      project1(0, z);
      t = 1;
    } else {
      jpair(t - 1, jn);
    }
    tn = tau[t - 1 < 0 ? 0 : t - 1];
  } else {
    t = t1 - 1;
    if (t == L - 1) {
      jpair(t, jn);
      tn = tau[t];
      const double v[2] = {stdc[0] ? X[0] : 0.0, stdc[1] ? X[1] : 0.0};
      emit(t, v);  // zero-length integral: the surface row is the seed itself
      project1(t, v);
      --t;
    } else {
      jpair(t + 1, jn);
      tn = tau[t + 1];
      if (g.chunk_region[c + 1] != g.chunk_region[c]) {  // carry gap: pure attenuation on this step
        const double tc = tau[t];
        double v[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          X[k] = X[k] * exp(-(tn - tc) / mu[k]);
          v[k] = stdc[k] ? X[k] : 0.0;
        }
        emit(t, v);
        project1(t, v);
        jpair(t, jn);
        tn = tc;
        --t;
      }
    }
  }

  // ---- four rows per step; the I rows of the next three steps are already on their way into this thread's private
  //      slots of a shared-memory ring (cp.async: no registers held, no barrier needed) ----
  const int dir = up ? -1 : 1;
  auto main_loop = [&](auto gen_tag) {
    constexpr bool GEN = decltype(gen_tag)::value;
    double2* const ring = s_ring + threadIdx.x;  // slot (g, u) of this thread: ring[(g * 4 + u) * APPLY2_THREADS]
    const ptrdiff_t rstep = static_cast<ptrdiff_t>(dir) * ldv;  // one row, in double2 units
    const double2* pf = Iv + static_cast<size_t>(t) * ldv;      // first row of the next group to prefetch
    int pf_t = t, pf_g = 0;
    auto prefetch = [&]() {
      if (up ? (pf_t - 3 >= t0) : (pf_t + 3 < t1)) {
#pragma unroll
        for (int u = 0; u < 4; ++u) cp_async16(ring + (pf_g * 4 + u) * APPLY2_THREADS, pf + u * rstep);
        pf += 4 * rstep;
        pf_t += 4 * dir;
      }
      cp_async_commit();
      pf_g = (pf_g + 1 == APPLY2_RING) ? 0 : pf_g + 1;
    };
#pragma unroll
    for (int i = 0; i < APPLY2_RING - 1; ++i) prefetch();
    int cg_slot = 0;
    double2* po = Iv + static_cast<size_t>(t) * ldv;            // row t of I (I_n / I_saved at fixed offsets from it)
    const ptrdiff_t dN = Nv - Iv, dS = Sv ? Sv - Iv : 0;
    const double2* pj = Jv + static_cast<size_t>(t) * ldv;
    const double2* pc = GEN ? (staged ? s_cj + (t - t0) : src.cj2 + t) : nullptr;
    const double* pt = staged ? s_tau + (t - t0) : tau + t;
    double* pp = GEN ? projs + static_cast<size_t>(t) * pstep + (lane >> 4) + static_cast<ptrdiff_t>(dir) * ((lane >> 2) & 3) * static_cast<ptrdiff_t>(pstep) : nullptr;
    while (up ? (t - 3 >= t0) : (t + 3 < t1)) {
      double tc[4], j[4][2], x[4][2], a[4][2], v[4][2];
      double2 iv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        tc[u] = pt[dir * u];
        if (GEN) {
          const double2 cc = pc[dir * u];
          j[u][0] = fma(cc.y, q[0], cc.x);
          j[u][1] = fma(cc.y, q[1], cc.x);
        } else {
          const double2 jv = pj[u * rstep];
          j[u][0] = jv.x;
          j[u][1] = jv.y;
        }
      }
      double dmax = 0.0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const double d = up ? ((u ? tc[u - 1] : tn) - tc[u]) : (tc[u] - (u ? tc[u - 1] : tn));
        dmax = fmax(dmax, d);
        x[u][0] = sgn * d * imu[0];
        x[u][1] = sgn * d * imu[1];
      }
      if (dmax * ximax <= kTinyArg) {
#pragma unroll
        for (int u = 0; u < 4; ++u) { a[u][0] = exp_tiny(x[u][0]); a[u][1] = exp_tiny(x[u][1]); }
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u) { a[u][0] = exp_small(x[u][0]); a[u][1] = exp_small(x[u][1]); }
      }
      // (columns without a recurrence have x = 0: a = 1, b = 0, X stays 0 -- no select needed)
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          X[k] = fma(X[k], a[u][k], -(0.5 * x[u][k]) * fma(u ? j[u - 1][k] : jn[k], a[u][k], j[u][k]));
          v[u][k] = X[k];
        }
      cp_async_wait<APPLY2_RING - 2>();  // this group's I rows have landed
#pragma unroll
      for (int u = 0; u < 4; ++u) iv[u] = ring[(cg_slot * 4 + u) * APPLY2_THREADS];
      prefetch();  // refills the slot consumed in the previous step
      if (act) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          double2* o = po + u * rstep;
          *o = make_double2(iv[u].x + v[u][0], iv[u].y + v[u][1]);
          if (!GEN || keep_in || t + dir * u == forced) o[dN] = make_double2(v[u][0], v[u][1]);
          if (Sv) o[dS] = make_double2(v[u][0], v[u][1]);
        }
      }
      if (GEN) {
        double pv[8];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          pv[u] = fma(v[u][1], us0[1], v[u][0] * us0[0]);
          pv[4 + u] = fma(v[u][1], us1[1], v[u][0] * us1[0]);
        }
        const double tot = quad_reduce8(pbuf, pv, lane);
        if ((lane & 3) == 0) *pp = tot;
        pp += 4 * static_cast<ptrdiff_t>(dir) * static_cast<ptrdiff_t>(pstep);
        pc += 4 * dir;
      }
      jn[0] = j[3][0];
      jn[1] = j[3][1];
      tn = tc[3];
      t += 4 * dir;
      po += 4 * rstep;
      pj += 4 * rstep;
      pt += 4 * dir;
      cg_slot = (cg_slot + 1 == APPLY2_RING) ? 0 : cg_slot + 1;
    }
    cp_async_wait<0>();
  };
  if (cg) main_loop(std::true_type{}); else main_loop(std::false_type{});
  // ---- tail rows ----
  for (; up ? (t >= t0) : (t < t1); t += dir) {
    const double tc = tau[t];
    step1(t, up ? tn - tc : tc - tn, jn);
    tn = tc;
  }
}

// Row-wise post-processing of the columns next to mu = 0: windowed / Taylor columns
// (SOS_Aer_In_limit.py:70-109), the extrapolation W (:113-141), I_n[t, mu=0+] = J (SOS_Aer_I1_In.py:100),
// the find-first second-difference blend (:101-108) and, on the TOA / surface rows, the convergence
// ratios of SOS_Aer_main_specular.py:309.  ONE WARP per (layer, scenario): it reads the ~40 raw values
// it needs, rewrites only the columns that change and corrects I by (new - raw) for those the apply
// pass had already accumulated.  With a generated source it also finishes the next order's coefficients of its row:
// projections of the zone columns (final values) + the apply pass's slots.
constexpr int ZONE_ROWS = 8;
#ifndef SOS_ZONE_UP
#define SOS_ZONE_UP 31
#endif
constexpr int ZONE_UP = SOS_ZONE_UP;  // upward columns next to mu = 0+ fetched eagerly for the blend search (and projected here): with
                                      // column M itself one warp-wide step of every loop over them

__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(dst))), "l"(src) : "memory");
}

// Two rounds of loads per row: (1) the active flag together with the scenario's words, (2) everything the row needs
// (raw values on both sides of mu = 0 as asynchronous copies into a per-warp shared-memory row, the projection slots)
// -- the addresses of round 2 depend on kernel parameters only.  The fix-ups run on shared memory, and I is corrected
// with fire-and-forget reductions (red.global.add: each element is touched by exactly one lane, so the result does not
// depend on timing) instead of read-modify-write round trips.  A blend that reaches past the eager window (a few per
// cent of the rows) continues from global memory.
__global__ void __launch_bounds__(32 * ZONE_ROWS, 4)
sweep_zone_kernel(const GridDev g, const SrcGen sg, const double* __restrict__ J, double* __restrict__ In,
                  double* __restrict__ I, double* __restrict__ saved, int zone_buf) {
  extern __shared__ double sm_zone[];  // per warp: zone_buf downward values of columns [zl, M), then ZONE_UP + 4 upward ones
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s = blockIdx.y, t = g.row0 + blockIdx.x * ZONE_ROWS + warp;  // (layer-sharded plans own the rows [row0, row1))
  const int L = g.L, M = g.M, ld = g.ld;
  if (t >= g.row1) return;
  // ---- round 1 ----
  const sos_scenario* __restrict__ scp = g.scen + s;
  const int active = g.state[s].active;
  const int op = scp->phase_atm;
  // (at most three regions: rstart[nreg] = L)
  const int region = (g.nreg > 1 && t >= g.rstart[1] ? 1 : 0) + (g.nreg > 2 && t >= g.rstart[2] ? 1 : 0);
  const int idxw = scp->extrap_width[region];
  const double coef_atm = scp->coef_atm;
  if (!active) return;
  const size_t fbase = static_cast<size_t>(s) * L * ld;
  double* __restrict__ Is = In + fbase;
  double* __restrict__ Ia = I ? I + fbase : nullptr;
  double* __restrict__ Sv = saved ? saved + fbase : nullptr;
  const size_t roff = static_cast<size_t>(t) * ld;
  const int c_lo = g.col0, c_hi = g.col1;
  const bool own_down_zone = (c_lo < M && c_hi >= M);
  const bool own_up_zone = (c_lo <= M && c_hi > M + 1);
  double* row_dn = sm_zone + static_cast<size_t>(warp) * (zone_buf + ZONE_UP + 4);
  double* row_up = row_dn + zone_buf;  // row_up[i] = I_n[t, M + i]
  // with a generated source the zone is the plan-wide one (the apply pass left those columns out of its projections); it
  // contains the zone of every scenario, also of those whose source is not rebuilt
  const bool plan_gen = sg.cj != nullptr;
  const int zl = plan_gen ? sg.zlo : zone_lo(g, *scp);
  const int eager = min(c_hi, M + 1 + ZONE_UP);  // (rows of a rebuilt source store I_n up to zu_end >= M + 1 + ZONE_UP)

  // ---- round 2: every load of the row in flight at once ----
  if (own_down_zone) {
    const int nstd = min(M - 1, g.first_small);  // standard columns: raw values stored and accumulated by the apply pass
    for (int m = zl + lane; m < M; m += 32) {
      if (m < nstd) cp_async8(&row_dn[m - zl], &Is[roff + m]);
      else row_dn[m - zl] = 0.0;
    }
  }
  if (own_up_zone)
    for (int m = M + 1 + lane; m < eager; m += 32) cp_async8(&row_up[m - M], &Is[roff + m]);
  cp_async_commit();
  const SrcAt src(g, sg, J, s);
  const double* __restrict__ tau = g.tau + static_cast<size_t>(s) * L;
  const bool project = src.gen_row(t);  // this row's I_n feeds a rebuilt source: finish its coefficients
  const double* __restrict__ Ut = sg.Ut[op];
  const int lim = src.gen ? min(c_hi, sg.zu_end) : c_hi;  // the blend search never leaves the owned / stored columns
  const int pend = min(sg.zu_proj, g.N);                  // upward columns < pend are projected here, the others by the apply pass
  double v0 = 0.0;
  if (own_up_zone) v0 = src(t, M, g.mu[M]);  // I_n[t, mu = 0+] = J[t, mu = 0+]
  double p0 = 0.0, p1 = 0.0;  // projections: the apply pass's slots first
  if (project) {
    const double2* __restrict__ pr = reinterpret_cast<const double2*>(sg.proj + (static_cast<size_t>(s) * L + t) * sg.nslots * 2);
    for (int j = lane; j < sg.nslots; j += 32) {
      const double2 v = pr[j];
      p0 += v.x;
      p1 += v.y;
    }
  }
  cp_async_wait<0>();
  __syncwarp();

  if (own_down_zone) {
    double* row = row_dn - zl;  // row[m] valid for m in [zl, M)
    const int r0 = g.rstart[region];
    // non-standard columns that survive the extrapolation: computed here, never touched by the apply pass
    const int hi = min(M - 1, M - idxw);
    for (int m = g.first_small; m < hi; ++m) {
      const double v = asymptotic_column(g, src, tau, t, r0, m);
      if (lane == 0) {
        row[m] = v;
        Is[roff + m] = v;
        if (Sv) Sv[roff + m] = v;
        if (Ia) atomicAdd(&Ia[roff + m], v);
      }
    }
    __syncwarp();
    if (idxw > 0) {
      const int wclass = width_class(g, idxw);
      const int ns = g.wns[wclass];
      const int src0 = (idxw < 2) ? (M - idxw - 2) : (M - idxw - ns);
      const double* __restrict__ W = g.W + g.woff[wclass];
      for (int i = lane; i < idxw; i += 32) {
        const int m = M - 1 - i;  // sources (< M - idx) and targets (>= M - idx) never overlap
        double v = 0.0;
        if (ns == 5) {  // (every width >= 5: the parabola through five columns; same operations in the same order)
          const double* __restrict__ w5 = W + i * 5;
          const double* r5 = row + src0;
          v = fma(w5[0], r5[0], v);
          v = fma(w5[1], r5[1], v);
          v = fma(w5[2], r5[2], v);
          v = fma(w5[3], r5[3], v);
          v = fma(w5[4], r5[4], v);
        } else {
          for (int k = 0; k < ns; ++k) v = fma(W[i * ns + k], row[src0 + k], v);
        }
        const bool std_col = m < min(M - 1, g.first_small);
        const double raw = row[m];
        row[m] = v;
        Is[roff + m] = v;
        if (Sv) Sv[roff + m] = v;
        if (Ia) atomicAdd(&Ia[roff + m], std_col ? (v - raw) : v);  // standard targets were accumulated raw
      }
    } else if (lane == 0) {
      row[M - 1] = 0.0;
      Is[roff + M - 1] = 0.0;  // mu = 0- stays 0 when nothing is extrapolated
      if (Sv) Sv[roff + M - 1] = 0.0;
    }
    __syncwarp();
    if (project) {
      for (int m = zl + lane; m < M; m += 32) {
        p0 = fma(row[m], Ut[m], p0);
        p1 = fma(row[m], Ut[sg.ldr + m], p1);
      }
    }
  }

  if (own_up_zone) {
    if (lane == 0) {
      row_up[0] = v0;
      Is[roff + M] = v0;
      if (Sv) Sv[roff + M] = v0;
      if (Ia) atomicAdd(&Ia[roff + M], v0);
    }
    __syncwarp();
    // find-first over the raw values written by the apply pass: the eager window in shared memory, then (rare) on
    int istar = -1;
    int base = M + 1;
    for (; base + 2 <= eager - 1 && istar < 0; base += 32) {
      const int i = base + lane;
      bool hit = false;
      if (i + 2 <= eager - 1) {
        const double a = row_up[i - M], b = row_up[i + 1 - M], cc = row_up[i + 2 - M];
        hit = !(fabs((a - b) - (b - cc)) > SOS_BLEND_THRESHOLD);
      }
      const unsigned mask = __ballot_sync(0xffffffffu, hit);
      if (mask) istar = base + __ffs(mask) - 1 + 1;
    }
    if (istar < 0 && eager < lim) {
      // (the triples that straddle the end of the eager window are examined again from global memory)
      for (base = max(M + 1, eager - 2 - 31); base + 2 <= lim - 1 && istar < 0; base += 32) {
        const int i = base + lane;
        bool hit = false;
        if (i + 2 <= lim - 1 && i + 2 >= eager) {
          const double a = Is[roff + i], b = Is[roff + i + 1], cc = Is[roff + i + 2];
          hit = !(fabs((a - b) - (b - cc)) > SOS_BLEND_THRESHOLD);
        }
        const unsigned mask = __ballot_sync(0xffffffffu, hit);
        if (mask) istar = base + __ffs(mask) - 1 + 1;
      }
    }
    if (istar < 0) {
      if (lane == 0) atomicOr(&g.state[s].status, (lim >= g.N) ? SOS_STATUS_BLEND_OVERRUN : SOS_STATUS_STRIP_FALLBACK);
    } else {
      const double v1 = (istar < eager) ? row_up[istar - M] : Is[roff + istar];
      const double mus = g.mu[istar];
      __syncwarp();  // every lane has read what it needs before anything is overwritten
      for (int m = M + 1 + lane; m < istar; m += 32) {
        const double w = g.mu[m] / mus;
        const double val = (1.0 - w) * v0 + w * v1;
        const double old = (m < eager) ? row_up[m - M] : Is[roff + m];
        if (m < eager) row_up[m - M] = val;
        Is[roff + m] = val;
        if (Sv) Sv[roff + m] = val;
        if (Ia) atomicAdd(&Ia[roff + m], val - old);
        if (project && m >= pend) {  // past the columns projected below: the apply pass projected the raw value
          p0 = fma(val - old, Ut[m], p0);
          p1 = fma(val - old, Ut[sg.ldr + m], p1);
        }
      }
    }
    __syncwarp();
  }

  if (project) {
    // the next order's source coefficients of this row: + the zone columns (final values: all inside the eager window)
    for (int m = M + lane; m < min(pend, eager); m += 32) {
      const double v = row_up[m - M];
      p0 = fma(v, Ut[m], p0);
      p1 = fma(v, Ut[sg.ldr + m], p1);
    }
    // both sums with one butterfly: the lower half warp finishes p0, the upper one p1 (fixed tree: deterministic)
    const bool upper = lane >= 16;
    double mine = upper ? p1 : p0;
    mine += shfl_xor_d(upper ? p0 : p1, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) mine += shfl_xor_d(mine, o);
    const double other = __shfl_sync(0xffffffffu, mine, 16);
    if (lane == 0)
      *reinterpret_cast<double2*>(sg.cj_out + (static_cast<size_t>(s) * sg.Lp + t) * 2) = make_double2(coef_atm * mine, coef_atm * other);
  }

  // ---- convergence ratios on the TOA / surface rows (whole half-row, read back from global) ----
  const bool toa = (t == 0), surf = (t == L - 1);
  if (Ia && (toa || surf)) {
    __threadfence();  // this warp's own reductions into I have landed before it reads the row back
    __syncwarp();
    double rmax = -INFINITY;
    bool nonfinite = false;
    const int a0 = toa ? max(M, c_lo) : c_lo;
    const int a1 = toa ? c_hi : min(M, c_hi);
    // an order-capped member (an azimuthal mode m >= 1) stops on its cap: its ratio is meaningless (0/0 on the mu = +-1
    // columns), only a non-finite I_n is an error
    const bool capped = g.scen[s].order_cap > 0;
    for (int m = a0 + lane; m < a1; m += 32) {
      const double v = Is[roff + m];
      const double r = v / __ldcg(&Ia[roff + m]);
      if (capped ? !isfinite(v) : isnan(r)) nonfinite = true; else rmax = fmax(rmax, r);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
    nonfinite = __any_sync(0xffffffffu, nonfinite);
    if (lane == 0) {
      if (toa) g.state[s].ratio_toa = rmax;
      if (surf) g.state[s].ratio_surf = rmax;
      if (nonfinite || (rmax == INFINITY && !capped)) atomicOr(&g.state[s].status, SOS_STATUS_NONFINITE);  // -inf: no owned column
    }
  }
}

// ------------------------------------------------------------------------------------------
// convergence bookkeeping
// ------------------------------------------------------------------------------------------
// ascending list of the active scenarios (warp 0 of a one-CTA kernel; deterministic)
__device__ __forceinline__ void build_active_list(const GridDev& g) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  int base = 0;
  for (int s0 = 0; s0 < g.S; s0 += 32) {
    const int s = s0 + lane;
    const bool act = s < g.S && g.state[s].active;
    const unsigned mask = __ballot_sync(0xffffffffu, act);
    if (act) g.active_flat[base + __popc(mask & ((1u << lane) - 1u))] = s;
    base += __popc(mask);
  }
  if (lane == 0) *g.n_active = base;
}

// (a device function: the order loop runs it inside order_end_kernel, sos_abi.cu, together with the tile plan)
__device__ __forceinline__ void converge_block(const GridDev& g, int order_arg, int* order_counter) {
  __shared__ int order_s;
  if (threadIdx.x == 0) {
    // order_arg < 0: take the order number from the device-side counter (CUDA-graph replays cannot
    // change kernel arguments); the counter always tracks the last order handled
    order_s = order_arg >= 0 ? order_arg : *order_counter + 1;
    *order_counter = order_s;
  }
  __syncthreads();
  const int order = order_s;
  for (int s = threadIdx.x; s < g.S; s += blockDim.x) {
    ScenState& st = g.state[s];
    if (st.active) {
      st.n_orders = order;
      const int cap = g.scen[s].order_cap;
      const double r = fmax(st.ratio_toa, st.ratio_surf);
      if (cap > 0 ? order >= cap : !(r >= g.scen[s].threshold)) st.active = 0;
    }
  }
  __syncthreads();
  build_active_list(g);
}

__global__ void converge_kernel(const GridDev g, int order_arg, int* order_counter) { converge_block(g, order_arg, order_counter); }

// ratios with I_n := 1 (the reference initialises In = ones before the loop, :306-309)
__global__ void reset_kernel(const GridDev g, const double* __restrict__ I1, int* order_counter) {
  const int s = blockIdx.x;
  __shared__ double sc[32];
  const int L = g.L, M = g.M, N = g.N, ld = g.ld;
  const double* __restrict__ I = I1 + static_cast<size_t>(s) * L * ld;
  double r0 = -INFINITY, r1 = -INFINITY;
  for (int m = threadIdx.x; m < N; m += blockDim.x) {
    if (m >= M) { const double r = 1.0 / I[m]; if (!isnan(r)) r0 = fmax(r0, r); }
    else { const double r = 1.0 / I[static_cast<size_t>(L - 1) * ld + m]; if (!isnan(r)) r1 = fmax(r1, r); }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    r0 = fmax(r0, __shfl_xor_sync(0xffffffffu, r0, o));
    r1 = fmax(r1, __shfl_xor_sync(0xffffffffu, r1, o));
  }
  if (lane == 0) sc[warp] = r0;
  __syncthreads();
  if (threadIdx.x == 0) { double r = -INFINITY; for (int w = 0; w < nwarps; ++w) r = fmax(r, sc[w]); g.state[s].ratio_toa = r; }
  __syncthreads();
  if (lane == 0) sc[warp] = r1;
  __syncthreads();
  if (threadIdx.x == 0) {
    double r = -INFINITY; for (int w = 0; w < nwarps; ++w) r = fmax(r, sc[w]);
    ScenState& st = g.state[s];
    st.ratio_surf = r;
    st.n_orders = 1;
    st.status = 0;
    if (s == 0) *order_counter = 1;
    const int cap = g.scen[s].order_cap;
    st.active = (cap > 0 ? 1 < cap : fmax(st.ratio_toa, r) >= g.scen[s].threshold) ? 1 : 0;
  }
}

// ratios <-> caller buffer [S][2] (mu-block sharding reduces them across ranks with a MAX all-reduce)
__global__ void ratios_kernel(const GridDev g, double* buf, int set) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= g.S) return;
  if (set) { g.state[s].ratio_toa = buf[2 * s]; g.state[s].ratio_surf = buf[2 * s + 1]; }
  else { buf[2 * s] = g.state[s].ratio_toa; buf[2 * s + 1] = g.state[s].ratio_surf; }
}

// Source coefficients of a whole field (the first order, before the loop): cj[s][t][r] = coef * sum_k I[t, k] Us[k][r]
__global__ void __launch_bounds__(256) project_rows_kernel(const GridDev g, const SrcGen sg, const double* __restrict__ I, double* __restrict__ cj) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s = blockIdx.y, t = blockIdx.x * 8 + warp;
  if (t >= g.L) return;
  const int op = g.scen[s].phase_atm;
  if (sg.rank[op] == 0) return;
  const double* __restrict__ Ut = sg.Ut[op];
  const double* __restrict__ row = I + (static_cast<size_t>(s) * g.L + t) * g.ld;
  double p0 = 0.0, p1 = 0.0;
  if (((g.ld | sg.ldr) & 1) == 0 && ((reinterpret_cast<uintptr_t>(I) | reinterpret_cast<uintptr_t>(Ut)) & 15) == 0) {
    // rows and factor rows start on 16-byte boundaries: two columns per load
    const double2* __restrict__ row2 = reinterpret_cast<const double2*>(row);
    const double2* __restrict__ u0 = reinterpret_cast<const double2*>(Ut);
    const double2* __restrict__ u1 = reinterpret_cast<const double2*>(Ut + sg.ldr);
    const int n2 = g.N >> 1;
#pragma unroll 4
    for (int j = lane; j < n2; j += 32) {
      const double2 x = row2[j], a = u0[j], b = u1[j];
      p0 = fma(x.x, a.x, p0); p0 = fma(x.y, a.y, p0);
      p1 = fma(x.x, b.x, p1); p1 = fma(x.y, b.y, p1);
    }
    if ((g.N & 1) && lane == 0) {
      const int m = g.N - 1;
      p0 = fma(row[m], Ut[m], p0);
      p1 = fma(row[m], Ut[sg.ldr + m], p1);
    }
  } else {
    for (int m = lane; m < g.N; m += 32) {
      const double x = row[m];
      p0 = fma(x, Ut[m], p0);
      p1 = fma(x, Ut[sg.ldr + m], p1);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    p0 += shfl_xor_d(p0, o);
    p1 += shfl_xor_d(p1, o);
  }
  const double coef = g.scen[s].coef_atm;
  if (lane == 0) *reinterpret_cast<double2*>(cj + (static_cast<size_t>(s) * sg.Lp + t) * 2) = make_double2(coef * p0, coef * p1);
}

__global__ void count_active_kernel(const GridDev g) { build_active_list(g); }

}  // namespace sossweep
