/* sos_b200.h -- C ABI of the B200-native Successive-Orders-of-Scattering engine.
 *
 * The reference (Guillaume-SOULIER/SOS-Radiative-Transfer) is pure Python/NumPy and has
 * no FFI; its "operator interface" for the hot path is a set of Python call signatures
 * (SURVEY.md 8b).  Every entry point below names the reference lines it replaces; the
 * ctypes binding a reference maintainer would add is shown in INTEGRATION.md and is what
 * sos-radiative-transfer_b200/_lib.py does.
 *
 * Conventions
 *   - plain C: opaque plan handle, raw pointers, ints, doubles; no torch / C++ types.
 *   - every function returns 0 on success or a negative sos_error; nothing throws.
 *   - pointers named *_d are DEVICE pointers owned by the caller (e.g. torch tensors),
 *     pointers named *_h are HOST pointers read during the call only.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - a "field" is a row-major double array [S*L rows][ld] (row = scenario*L + layer,
 *     N = 2*nb_angles mu-columns used, ld >= N, ld even); S scenarios are stacked along
 *     rows.  This is the reference's (L, 2*nb_angles) C-order array (SOS_Aer_I1_In.py:20)
 *     with a batch dimension in front.
 *   - one plan per (grid, batch); a plan owns its scratch and is not thread-safe; calls on
 *     one plan must be issued on one stream at a time.
 */
#ifndef SOS_B200_H
#define SOS_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOS_ABI_VERSION 1

typedef struct sos_plan sos_plan;

typedef enum {
  SOS_OK = 0,
  SOS_ERR_INVALID = -1,      /* bad argument */
  SOS_ERR_CUDA = -2,         /* a CUDA runtime/driver call failed (see sos_last_cuda_error) */
  SOS_ERR_NOMEM = -3,
  SOS_ERR_UNSUPPORTED = -4,  /* e.g. not an sm_100 device */
  SOS_ERR_STATE = -5,        /* call order violated (e.g. source before set_phase) */
  SOS_ERR_RETRY = -6         /* sos_solve only: the fused order kernel met a case it cannot finish (a mu -> 0+ blend wider
                                than 128 columns); the plan has switched to its general kernels -- restore I_d / In_d
                                (they were consumed) and call sos_solve again */
} sos_error;

typedef enum {
  SOS_SURFACE_NONE = 0,      /* single homogeneous layer: In_NumInt (SOS_Aer_I1_In.py:77-130) */
  SOS_SURFACE_SPECULAR = 1,  /* SOS_Aer_main_specular.py:397,399 */
  SOS_SURFACE_LAMBERT = 2,   /* Lambert-as-coded: SOS_Aer_main_lambertian.py:399,401 */
  SOS_SURFACE_LAMBERT_README = 3, /* the n >= 2 Lambert coupling as the README states it (README.md:215): isotropic upward
                                     radiance -2 rho int_{-1}^{0} I_n(tau*, mu') mu' dmu' > 0 over the WHOLE downward half
                                     (the shipped code has the opposite sign and drops [-h, 0]: Q5).  A separate, named
                                     physics mode: validated by invariants, not by parity with the reference. */
  SOS_SURFACE_LAMBERT_DIFFUSE = 4  /* a Lambertian ground in every order, the direct beam included (three-region plans only;
                                      SOS_ERR_UNSUPPORTED otherwise).  Order 1: no mirror-reflected beam; every upward column
                                      starts at the surface row from the isotropic b = rho (e^{-T/mu0} - 2 int_{-1}^{0} I_1 mu dmu),
                                      the reflection of the direct beam and of order 1's own downward light (a pre-pass of the
                                      first-order entry points writes b per scenario).  Orders n >= 2: the coupling of
                                      SOS_SURFACE_LAMBERT_README.  sos_quadratures adds no collimated reflected beam: the
                                      reflected light is part of the diffuse field. */,
  SOS_SURFACE_ROSSLI = 5           /* a Ross-Li bidirectional ground (RossThick + LiSparse-Reciprocal kernels) in every order
                                      (three-region plans only; SOS_ERR_UNSUPPORTED otherwise):
                                      rho = f_iso + f_vol K_vol + f_geo K_geo with f_iso = sos_scenario.grd_alb.  The f_iso
                                      part is SOS_SURFACE_LAMBERT_DIFFUSE unchanged; every upward column i adds
                                        order 1:  sum_k f_k (e^{-T/mu0} beam_k[i] + sum_c u_c R^k[c][i])
                                        order n:  sum_k f_k sum_c u_c R^k[c][i]
                                      with u_c = -2 w_c mu_c I_n(tau*, mu_c) over the downward half (w = trapezoid weights
                                      of the ascending downward half) and the mode matrices / weights / beam vectors of
                                      sos_plan_set_brdf and sos_plan_set_brdf_scenarios (both required before a first order
                                      or a sweep: SOS_ERR_STATE otherwise).  With f_vol = f_geo = 0 every value is bit for bit
                                      the one of SOS_SURFACE_LAMBERT_DIFFUSE.  No collimated reflected beam in the fluxes. */,
  SOS_SURFACE_OCEAN = 6            /* a wind-roughened ocean (Cox-Munk glint) in every order (three-region plans only;
                                      SOS_ERR_UNSUPPORTED otherwise): rho = grd_alb + rho_glint(mu_i, mu_v, phi; W, n), both
                                      in reflectance-factor units.  grd_alb (whitecaps and water-leaving light) is
                                      SOS_SURFACE_LAMBERT_DIFFUSE unchanged; every upward column i adds
                                        order 1:  f_glint (e^{-T/mu0} beam[i] + sum_c u_c R[c][i])
                                        order n:  f_glint sum_c u_c R[c][i]
                                      with one glint mode matrix R per set (sos_build_glint_modes) and the first weight and
                                      beam vector of sos_plan_set_brdf_scenarios (u as for SOS_SURFACE_ROSSLI; both calls
                                      required: SOS_ERR_STATE otherwise).  With f_glint = 0 every value is bit for bit the one
                                      of SOS_SURFACE_LAMBERT_DIFFUSE.  No collimated reflected beam in the fluxes. */
} sos_surface;

/* device-side status bits (OR-ed per scenario) */
#define SOS_STATUS_BLEND_OVERRUN 1u /* reference would raise IndexError (SOS_Aer_I1_In.py:103) */
#define SOS_STATUS_NONFINITE 2u     /* inf/nan met in a convergence ratio */
#define SOS_STATUS_MAX_ORDERS 4u    /* sos_solve stopped at max_orders with this scenario still above threshold */

/* Grid shared by all scenarios of a batch. */
typedef struct {
  int nb_layers;        /* L */
  int nb_angles;        /* M; N = 2M columns: mu = [linspace(-1,0,M), linspace(0,1,M)] */
  int n_scenarios;      /* S */
  int n_regions;        /* 1 (single layer) or 3 (upper atm / aerosol / lower atm) */
  int region_start[4];  /* first row of each region; region_start[n_regions] = L.
                           3 regions: {0, idx_up, idx_down+1, L} (SOS_Aer_main_specular.py:330,349,368) */
  int surface;          /* sos_surface */
  int ld;               /* leading dimension of fields (elements) */
  int chunk_rows;       /* rows per scan chunk; 0 = let the library choose */
} sos_grid;

/* Per-scenario scalars. */
typedef struct {
  double mu0;           /* SOS_Aer_main_specular.py:23 */
  double grd_alb;       /* :47 */
  double tauStar_tot;   /* :36  (tauStar_atm + tauStar_aer; single layer: tauStar) */
  double coef_atm;      /* source-contraction scale on rows outside the aerosol region: alb_atm (:323);
                           single layer: alb (SOS_Aer_I1_In.py:73) */
  double coef_mix_atm;  /* aerosol rows: alb_atm * dtau_atm/(dtau_atm+dtau_aer)  (:321) */
  double coef_mix_aer;  /* aerosol rows: alb_aer * dtau_aer/(dtau_atm+dtau_aer)  (:321) */
  double threshold;     /* convergence threshold, 1e-4 (:309) */
  int phase_atm;        /* index into the matrices registered with sos_plan_set_phase */
  int phase_aer;
  int extrap_width[3];  /* idx of improved_limit_mu_down per region (:342-345,361-364,380-383;
                           single layer SOS_Aer_I1_In.py:124-127) */
  int order_cap;        /* 0: the reference's stopping rule (ratio of :309 against threshold).  > 0: the scenario sums
                           exactly the orders 1 .. order_cap (active while its order is below the cap; the ratio is not
                           consulted and a 0/0 ratio is not SOS_STATUS_NONFINITE, a non-finite I_n still is).  What an
                           azimuthal Fourier mode m >= 1 uses: it sums the orders its mode 0 summed, and its ratio is
                           meaningless (I_m changes sign; the mu = +-1 columns are exactly 0). */
} sos_scenario;

/* Per-scenario results of sos_solve / sos_converge (host copy). */
typedef struct {
  double ratio_toa;     /* max(In[0,M:]/I[0,M:])  (:309) */
  double ratio_surf;    /* max(In[L-1,:M]/I[L-1,:M]) */
  int n_orders;         /* the reference's `n` at loop exit */
  int active;           /* 1 while the scenario has not converged */
  unsigned status;      /* SOS_STATUS_* bits */
  int reserved;
} sos_result;

int sos_abi_version(void);
const char* sos_strerror(int err);
const char* sos_last_cuda_error(void);

/* mu-grid constants + per-scenario tau profiles (SOS_Aer_tau_profile.py:21-27) are uploaded
 * once.  tau_h: [S][L]; mu_h: [N]; extrap_W_h: 4 extrapolation matrices for the widths
 * int(0.005M), int(0.02M), int(0.04M), int(0.06M) -- see sos_extrap_layout(). */
int sos_plan_create(sos_plan** out, const sos_grid* grid, const double* mu_h, const double* tau_h,
                    const sos_scenario* scen_h, const double* extrap_W_h, int extrap_W_len);
int sos_plan_destroy(sos_plan* plan);
/* Feed an existing plan the NEXT batch of scenarios on the same grid (same L, M, S, regions, surface; phase indices into
 * the matrices already registered): re-uploads tau and the per-scenario scalars, regroups the scenarios by operand,
 * re-mixes the per-scenario aerosol operands of the folded contraction and resets the per-scenario state.  What a
 * sweep driver (SOS_Aer_critical_albedo.py:417-503: one solve per (tau_aer, mu0, albedo) point) calls between batches
 * instead of destroying and re-creating the plan; device buffers, tensor maps and phase operands stay.  Synchronises
 * `stream`. */
int sos_plan_update(sos_plan* plan, const double* tau_h, const sos_scenario* scen_h, void* stream);

/* Extrapolation table layout: for width class c (0..3) the matrix W_c is [idx_c][ns_c] row-major
 * at offset off_c in extrap_W_h, where ns_c = (idx_c<2 ? 2 : min(5, idx_c)) sources
 * (SOS_Aer_In_limit.py:118-141).  Writes idx[4], ns[4], off[4] and returns the total length. */
int sos_extrap_layout(int nb_angles, int* idx, int* ns, int* off);

/* A[k][m] = 0.25 * w_k * P[m][N-1-k]  (the operand of Jn_NumInt as a GEMM, SOS_Aer_I1_In.py:73;
 * w = composite-trapezoid weights of the mu grid).  P_d: [N][ldp], A_d: [N][lda]. */
int sos_build_contraction(sos_plan* plan, const double* P_d, int ldp, double* A_d, int lda, void* stream);

/* Azimuth-averaged phase functions built on the device (SOS_Aer_phase_func.py:68-292): family 0 =
 * Rayleigh (:79-133), 1 = Henyey-Greenstein with asymmetry g (:141-195), 2 = tabulated (FWC: :202-292;
 * tab_x_d ascending cos(scattering angle), tab_y_d values, device arrays).  phi_h / cphi_h: the 25
 * azimuth nodes linspace(0, pi, 25) and their cosines as the host computed them.  Writes P_d [N][ldp]
 * (every column normalised to trapz = 4, :131) and/or P0_d [N] for the solar direction mu0 (normalised
 * to trapz = 2, :105); either may be NULL. */
int sos_build_phase(sos_plan* plan, int family, double g, double mu0, const double* phi_h, const double* cphi_h,
                    const double* tab_x_d, const double* tab_y_d, int tab_n, double* P_d, int ldp, double* P0_d,
                    void* stream);

/* Azimuthal Fourier modes m = 0 .. n_modes-1 of the same phase functions (family and table arguments as in
 * sos_build_phase).  Azimuth nodes: phi_h [n_phi] ascending on [0, pi] (2 <= n_phi <= 1024); cphi_h [1 + n_modes][n_phi]:
 * row 0 = cos(0 - phi_k) (the node cosines, as sos_build_phase takes them), row 1 + m = cos(m phi_k), both computed by
 * the host.  The phase function is evaluated once per (element, node); with A = f(-(cc - x_k)), B = f(-(cc + x_k)),
 * x_k = ss cos(phi_k), mode m integrates trapz_k(cos(m phi_k) (A + (-1)^m B)).  Every mode is normalised by the column
 * integrals of MODE 0: P_m[:, n] = 4 R_m[:, n] / trapz(R_0[:, n], mu), P0_m = 2 P0raw_m / trapz(P0raw_0, mu), so that
 * sum_m (2 - delta_m0) P0_m cos(m phi) = c p(cos Theta) with one constant c.  With the 25 nodes of sos_build_phase,
 * mode 0 is bit for bit what sos_build_phase writes.  P_d: mode m at P_d + m*mode_stride ([N][ldp] each, mode_stride >=
 * N*ldp); P0_d: [n_modes][N]; either may be NULL.  1 <= n_modes <= 64. */
int sos_build_phase_modes(sos_plan* plan, int family, double g, double mu0, int n_phi, const double* phi_h, const double* cphi_h,
                          int n_modes, const double* tab_x_d, const double* tab_y_d, int tab_n, double* P_d, int ldp,
                          size_t mode_stride, double* P0_d, void* stream);

/* Fourier modes m = 0 .. n_modes-1 of the two Ross-Li kernels on the plan's mu grid, for SOS_SURFACE_ROSSLI.
 * R^k_m(mu, mu') = (1/pi) int_0^pi K_k(max(mu, mu_min), max(mu', mu_min), phi - pi) cos(m phi) dphi, where phi is the engine's
 * propagation azimuth relative to the incident light's and psi = phi - pi the Ross-Li relative azimuth (hot spot at psi = 0),
 * so that rho = R_0 + 2 sum_{m >= 1} R_m cos(m phi), the normalisation of the radiance modes.  Kernels of Lucht, Schaaf &
 * Strahler (2000) with h/b = 2, b/r = 1; both zenith cosines clamped to mu_min (0 < mu_min < 1).  Nodes: phi_h [n_nodes]
 * ascending on [0, pi] (2 <= n_nodes <= 1024), trapezoid rule; cos_h [1 + n_modes][n_nodes]: row 0 = cos(phi_k - pi),
 * row 1 + m = cos(m phi_k), both computed by the host.  Writes the TRANSPOSED matrices: element (c, i) = R_m(mu_{M+1+i}, |mu_c|),
 * c = 0 .. M-1 downward columns, i = 0 .. M-2 upward columns, at Rvol_d / Rgeo_d + m * mode_stride + c * ldr + i
 * (ldr >= M-1, mode_stride >= M * ldr).  One thread per element evaluates both kernels once per node.  1 <= n_modes <= 64. */
int sos_build_brdf_modes(sos_plan* plan, int n_nodes, const double* phi_h, const double* cos_h, int n_modes, double mu_min,
                         double* Rvol_d, double* Rgeo_d, int ldr, size_t mode_stride, void* stream);

/* Fourier modes m = 0 .. n_modes-1 of the Cox-Munk glint on the plan's mu grid, for SOS_SURFACE_OCEAN.
 * R_m(mu, mu') = (1/pi) int_0^pi rho_glint(mu, mu', phi) cos(m phi) dphi with phi the engine's propagation azimuth (glint at
 * phi = 0), rho_glint = r(omega) exp(-tan^2 theta_n / sigma2) S / (4 sigma2 mu mu' mu_n^4): isotropic slope variance sigma2 > 0
 * (Cox & Munk: 0.003 + 0.00512 W), unpolarised Fresnel reflectance r for the relative refractive index n_ref > 1, Smith
 * shadowing S (DESIGN §12).  Nodes: phi_h [n_nodes] ascending on [0, pi] (2 <= n_nodes <= 1024), trapezoid rule;
 * cos_h [1 + n_modes][n_nodes]: row 0 = cos(phi_k), row 1 + m = cos(m phi_k).  Writes the transposed layout of
 * sos_build_brdf_modes: element (c, i) = R_m(mu_{M+1+i}, |mu_c|) at R_d + m * mode_stride + c * ldr + i; the entries of the
 * column mu = 0- are 0.  1 <= n_modes <= 64. */
int sos_build_glint_modes(sos_plan* plan, int n_nodes, const double* phi_h, const double* cos_h, int n_modes, double sigma2,
                          double n_ref, double* R_d, int ldr, size_t mode_stride, void* stream);

/* Azimuth synthesis of Fourier-mode fields: out[geo][r][p][col] (+)= sum over s with geo_h[s] = geo of
 * w_h[s][p] * I[s][rows_h[r]][col] (col < N), the sum in ascending s (no atomics: deterministic).  I_d: a field of this plan
 * ([S*L][ld]); geo_h [S] in [0, n_geo) or -1 (member skipped); w_h [S][n_az] (1 for mode 0, 2 cos(m phi_p) for mode m, as
 * the host computed them); rows_h [n_rows] in [0, L); out_d [n_geo][n_rows][n_az][N].  accumulate = 0 overwrites, 1 adds
 * (the mode sub-batches of one geometry solved on several plans add into one output).  Only geometries with at least one
 * member are written. */
int sos_azimuth_synthesis(sos_plan* plan, const double* I_d, const int* geo_h, const double* w_h, int n_geo, const int* rows_h,
                          int n_rows, int n_az, double* out_d, int accumulate, void* stream);

/* Exact direct glint of azimuth-resolved radiance over SOS_SURFACE_OCEAN: for entries k = 0 .. n-1, rows r, azimuths
 * p and upward columns i = M+1 .. N-1 of the plan's grid,
 *   out[geo_h[k]][r][p][i] += e^{-T/mu0} (rho_glint(mu_i, mu0, phi_p) - sum_{m < n_modes} (2 - delta_m0) beam[k][m][i] cos(m phi_p))
 *                             * e^{-(T - tau[k][r]) / mu_i}
 * (out as written by sos_azimuth_synthesis, [n_geo][n_rows][n_az][N]; geo_h [n] in [0, n_geo)): the once-reflected direct
 * beam, transmitted without scattering to the row, with its truncated Fourier series replaced by the exact reflectance.
 * par_h [n][4] = (mu0, tauStar_tot, sigma2, n_ref); tau_h [n][n_rows] = tau at the rows; beam_h [n][n_modes][M-1] = the
 * glint beam vectors of modes 0 .. n_modes-1 (the ones given to sos_plan_set_brdf_scenarios); phi_h [n_az].  One thread
 * per output element, no atomics: deterministic.  1 <= n_modes <= 64. */
int sos_glint_correction(sos_plan* plan, int n, const int* geo_h, const double* par_h, const double* tau_h, int n_rows,
                         const double* beam_h, int n_modes, const double* phi_h, int n_az, int n_geo, double* out_d,
                         void* stream);

/* Exact single scattering of azimuth-resolved radiance (three-region plans; SOS_ERR_UNSUPPORTED otherwise).  The first order
 * of sos_first_order is linear in its coefficient planes; for entries k = 0 .. n-1 (a plan scenario and the geometry it was
 * synthesized into), requested rows r (rows_h [n_rows] in [0, L)), azimuths p and every column of the plan's grid it adds
 *   out[geo][r][p][col] += I1[dC](tau[scenario][rows_h[r]], mu_col)
 * (out as written by sos_azimuth_synthesis, [n_geo][n_rows][n_az][N]): the closed-form first order of the plan's scenario with
 * the coefficient planes dC_atm = alb_atm dP0_atm, dC_mix = dC_atm f_atm + (dP0_aer alb_aer) f_aer built from
 *   dP0(mu, phi_p) = p(cos Theta) / norm - sum_{m < n_modes} (2 - delta_m0) P0m[series][m](mu) cos(m phi_p),
 *   cos Theta = -mu0 mu + sqrt(1 - mu0^2) sqrt(1 - mu^2) cos phi_p,
 * i.e. the truncated Fourier series of the singly scattered radiance replaced by its exact value.  Over a specular ground
 * (and the Lambert kinds) the mirror-reflected beam and the upward carry rho I1[L-1, mirror] are kept; over
 * SOS_SURFACE_LAMBERT_DIFFUSE, SOS_SURFACE_ROSSLI and SOS_SURFACE_OCEAN both are 0 (their order-1 surface terms stay the
 * series).  P0m_h [n_vec][n_modes][N]: the solar mode vectors the radiance was summed with (1 <= n_modes <= 64);
 * tab_h [n_tab]: the tabulated phase functions, abscissae (ascending) at tab_off and values at tab_off + tab_n; phi_h [n_az].
 * One thread per (entry, azimuth, column), no atomics: deterministic. */
typedef struct {
  int scenario;         /* plan scenario (tau, mu0, tauStar_tot, grd_alb) */
  int geo;              /* first index of out */
  int family[2];        /* atmosphere, aerosol: -1 isotropic (dP0 = 0), 0 Rayleigh, 1 Henyey-Greenstein, 2 tabulated */
  int series[2];        /* row of P0m_h */
  int tab_off[2];       /* tabulated: offset of the abscissae in tab_h */
  int tab_n[2];         /* tabulated: number of abscissae */
  double g[2];          /* Henyey-Greenstein asymmetry */
  double norm[2];       /* T > 0: the mode-0 normalisation, trapz_mu of the azimuth ring integral / (4 pi) */
  double w[4];          /* alb_atm, f_atm, alb_aer, f_aer */
} sos_ss_entry;
int sos_single_scatter_correction(sos_plan* plan, int n, const sos_ss_entry* ent_h, const double* P0m_h, int n_vec, int n_modes,
                                  const double* tab_h, int n_tab, const int* rows_h, int n_rows, const double* phi_h, int n_az,
                                  int n_geo, double* out_d, void* stream);

/* Register the contraction matrices (device, [N][lda] each) the scenarios index. */
int sos_plan_set_phase(sos_plan* plan, const double* const* A_d, int n_matrices, int lda);

/* SOS_SURFACE_ROSSLI and SOS_SURFACE_OCEAN plans only (SOS_ERR_UNSUPPORTED otherwise).
 *   sos_plan_set_brdf            register n_sets (1 .. 64) mode matrix pairs (Rvol_d[j], Rgeo_d[j]): device [M][ldr] each in
 *                                the transposed layout of sos_build_brdf_modes (ldr >= M-1), kept alive by the caller.  Drops
 *                                the captured order graphs; the per-scenario data must be given again afterwards.  An ocean
 *                                plan takes one matrix per set (the glint of one (W, n, mode), sos_build_glint_modes) in
 *                                Rvol_d and Rgeo_d = NULL; NULL for a Ross-Li plan, or not NULL for an ocean plan, is
 *                                SOS_ERR_INVALID.
 *   sos_plan_set_brdf_scenarios  per scenario: set_h [S] (the pair it uses, 0 .. n_sets-1), f_h [S][2] = (f_vol, f_geo) >= 0
 *                                and beam_h [S][2][M-1] = (R^vol_m(mu_i, mu0), R^geo_m(mu_i, mu0)) over the upward columns
 *                                i = M+1 .. N-1 for the scenario's mode m.  Copied on `stream` into plan-owned buffers in place:
 *                                captured order graphs stay valid, so it follows sos_plan_update for the next batch.  Ocean:
 *                                f_h[s] = (f_glint >= 0, 0) (a second weight != 0 is SOS_ERR_INVALID), beam_h[s][0] = the
 *                                glint mode R_m(mu_i, mu0); beam_h[s][1] is not read. */
int sos_plan_set_brdf(sos_plan* plan, const double* const* Rvol_d, const double* const* Rgeo_d, int n_sets, int ldr);
int sos_plan_set_brdf_scenarios(sos_plan* plan, const int* set_h, const double* f_h, const double* beam_h, void* stream);

/* Folded contraction (optional, half the multiply-adds).  The operand A[k][m] = w_k/4 P[m][N-1-k] of
 * SOS_Aer_I1_In.py:73 is centrosymmetric (A[N-1-k][N-1-m] = A[k][m]) whenever P(mu, mu') = P(-mu, -mu') --
 * true for every builder of SOS_Aer_phase_func.py -- and the mu grid is symmetric (SOS_Aer_main_specular.py:59-61).
 * Then J[:, j] = u B+ + v B-, J[:, N-1-j] = u B+ - v B- with u, v = I[:, k] +- I[:, N-1-k] and two
 * M x M operands B+-: the same sum, reassociated (agreement ~1e-14 relative).
 *   sos_fold_layout     rows / ld of a folded operand for this nb_angles (returns rows*ld, the element count)
 *   sos_build_folded    F_d [rows][ldf] from A_d; *defect_out (host) = max|A[k][m] - A[N-1-k][N-1-m]| / max|A|.
 *                       Synchronises the stream.  The caller decides (the Python host enables the fold when every
 *                       operand's defect is <= 1e-12; F is built from the symmetrised A).
 *   sos_plan_set_folded register one folded operand per matrix of sos_plan_set_phase (same order); sos_source /
 *                       sos_solve then use the folded kernel for full-column, single-GPU launches and the general
 *                       kernel otherwise.  n_matrices = 0 switches it off.  sos_plan_set_phase resets it.
 *                       For three-region plans it also premixes, per scenario, the two aerosol-row operands
 *                       c1 F[atm] + c2 F[aer] (SOS_Aer_main_specular.py:321) into one plan-owned operand, so that aerosol
 *                       tiles need one pass instead of two (S operands of rows*ldf doubles, skipped above 2 GB;
 *                       environment SOS_FOLD_PREMIX=0 keeps the two-pass tiles).  Launches with fewer tiles than half the SMs
 *                       (single solves) split every output tile in two over the k range (two partials added into a
 *                       zeroed J: order independent; SOS_FOLD_KSPLIT=0 disables it). */
int sos_fold_layout(int nb_angles, int* rows, int* ld);
int sos_build_folded(sos_plan* plan, const double* A_d, int lda, double* F_d, int ldf, double* defect_out, void* stream);
int sos_plan_set_folded(sos_plan* plan, const double* const* F_d, int n_matrices, int ldf);

/* Low-rank operands (optional).  The Rayleigh operand of SOS_Aer_phase_func.py:79-133 is rank 2 and the isotropic one
 * (:68-76) rank 1, exactly up to rounding; every row outside the aerosol layer uses the molecular operand
 * (SOS_Aer_main_specular.py:323).  For an operand registered here with rank r in 1..16 and factors A = Us Vt --
 * Ut_d[i] = (U diag(s))^T and Vt_d[i], both [R][ldr] with R = 4 (r <= 4) or 16 rows, zero beyond r -- the rows that use it
 * alone are contracted as (I Us) Vt: 2 r N multiply-adds per row instead of N^2, HBM bound.  rank[i] = 0 keeps operand i
 * dense.  Takes effect with the folded contraction (call before or after sos_plan_set_folded); sos_plan_set_phase
 * resets it; n_matrices = 0 switches it off.  The caller supplies the factors (the Python host: the closed form of
 * sos_build_lowrank_mu2 below, accepted only when it reproduces the dense operand to rounding). */
int sos_plan_set_lowrank(sos_plan* plan, const double* const* Ut_d, const double* const* Vt_d, const int* rank, int n_matrices,
                         int ldr);
/* Closed-form factors for sos_plan_set_lowrank (no SVD): summed over the two half rings, the azimuth integrand of the
 * Rayleigh builder (SOS_Aer_phase_func.py:97) is 0.75 (2 + 2 mu^2 mu'^2 + 2 (1 - mu^2)(1 - mu'^2) cos^2 phi), so every row k of
 * A[k][m] = w_k/4 P[m][N-1-k] is affine in mu_m^2 whatever the column normalisation (:131) did: A[k][m] = alpha_k + beta_k mu_m^2
 * (isotropic, :68-76: beta = 0).  Reads alpha, beta off two columns of A_d, writes Ut_d = [alpha; beta; 0; 0], Vt_d = [1; mu^2; 0; 0]
 * ([4][ldr], see sos_lowrank_layout), and returns *residual_out = max|A - Ut^T Vt| / max|A| and *rank_out (1 or 2).  The caller
 * enables the factors only if the residual is at rounding level (the Python host: <= 1e-14); any other operand stays dense.
 * Synchronises the stream. */
int sos_lowrank_layout(int nb_angles, int* rows, int* ldr);
int sos_build_lowrank_mu2(sos_plan* plan, const double* A_d, int lda, double* Ut_d, double* Vt_d, int ldr, double* residual_out,
                          int* rank_out, void* stream);

/* First order.
 *  n_regions == 3: inlined closed form of SOS_Aer_main_specular.py:104-292; C_h is [S][2][N]:
 *     C_h[s][0][m] = alb_atm*P0_atm[m], C_h[s][1][m] = alb_atm*P0_atm[m]*f_atm + alb_aer*P0_aer[m]*f_aer
 *  n_regions == 1: I1_NumInt (SOS_Aer_I1_In.py:13-58); C_h[s][0][m] = alb*P0[m] ([S][2][N], plane 1 unused) */
int sos_first_order(sos_plan* plan, const double* C_h, double* I1_d, void* stream);
/* ... the same, every value stored twice: I1_d and I1_copy_d (the field the order loop accumulates into: sos_solve starts
 * from I = I_1, SOS_Aer_main_specular.py:302-304), which saves the device-to-device copy of the field in front of every
 * solve.  I1_copy_d may be NULL (= sos_first_order). */
int sos_first_order2(sos_plan* plan, const double* C_h, double* I1_d, double* I1_copy_d, void* stream);
/* ... the same with the coefficient planes assembled on the device from what a sweep driver actually holds: a table of
 * the distinct solar phase vectors P0tab_h [n_tab][N] of the batch (one row per (phase function, mu0):
 * SOS_Aer_phase_func.py:68-292), per scenario the two rows it uses idx_h [S][2] = (atmosphere, aerosol) and the weights
 * w_h [S][4] = (alb_atm, f_atm, alb_aer, f_aer) (SOS_Aer_main_specular.py:52-53):
 *     C[s][0][m] = P0tab[ia][m]*w0,   C[s][1][m] = (P0tab[ia][m]*w0)*w1 + (P0tab[ie][m]*w2)*w3
 * with every product and the sum rounded separately, i.e. bit for bit the planes sos_first_order takes (n_regions == 1:
 * w = (alb, 0, 0, 0)).  Saves the host the per-element arithmetic on [S][2][N] and the copy of it.  n_tab*N + 5*S must not
 * exceed 2*S*N (SOS_ERR_UNSUPPORTED otherwise: use sos_first_order2). */
int sos_first_order_tab(sos_plan* plan, const double* P0tab_h, int n_tab, const int* idx_h, const double* w_h, double* I1_d,
                        double* I1_copy_d, void* stream);

/* Jn_NumInt (SOS_Aer_I1_In.py:62-74) / SOS_Aer_main_specular.py:315-323 as one FP64 GEMM. */
int sos_source(sos_plan* plan, const double* In1_d, double* J_d, void* stream);

/* The same contraction restricted to layers [row0, row1) (row0 a multiple of 64; single-scenario,
 * single-region plans only): lets a mu-sharded solve start the contraction of the rows whose I_{n-1}
 * has already been all-gathered while the remaining rows are still in flight over NVLink. */
int sos_source_rows(sos_plan* plan, const double* In1_d, double* J_d, int row0, int row1, void* stream);

/* Fused all-gather + contraction for mu-block sharding: In1_peers_d[r] is the SAME field layout
 * [S*L][ld] in the memory of the GPU that owns mu columns [peer_col[r], peer_col[r+1]) (peer memory
 * mapped with sos_ipc_open, or this GPU's own buffer); the kernel fetches every k-range of I_{n-1}
 * straight from its owner by TMA over NVLink, so no separate all-gather is needed.  The caller
 * guarantees (e.g. with the MAX all-reduce of the convergence ratios) that every owner has finished
 * writing its columns.  peer_col: [n_peers + 1], multiples of 16, peer_col[0] = 0, peer_col[n_peers] = N. */
int sos_source_peers(sos_plan* plan, const double* const* In1_peers_d, int n_peers, const int* peer_col, double* J_d,
                     void* stream);
/* CUDA IPC plumbing for the above (one process per GPU): allocate a shareable device buffer and export
 * its 64-byte handle / map a peer's buffer / unmap / free; plus a stream-ordered device copy. */
int sos_ipc_alloc(size_t bytes, void** ptr_d, unsigned char* handle64);
int sos_ipc_open(const unsigned char* handle64, void** ptr_d);
int sos_ipc_close(void* ptr_d);
int sos_ipc_free(void* ptr_d);
int sos_copy_d2d(void* dst_d, const void* src_d, size_t bytes, void* stream);

/* In_NumInt (SOS_Aer_I1_In.py:77-130) / SOS_Aer_main_specular.py:327-449: down scan, mu->0
 * columns, extrapolation, surface coupling, up scan, blend.  If I_d != NULL also I += I_n and
 * the convergence ratios of :309 are refreshed (SOS_Aer_main_specular.py:454-456). */
int sos_sweeps(sos_plan* plan, const double* J_d, double* In_d, double* I_d, void* stream);

/* Convergence bookkeeping for the order that was just accumulated (`n` = its order number):
 * scenarios whose ratio fell below threshold become inactive with n_orders = n.  order < 0: use the
 * plan's device-side order counter + 1 (reset to 1 by sos_reset) -- for CUDA-graph replays. */
int sos_converge(sos_plan* plan, int order, void* stream);

/* Whole order loop (SOS_Aer_main_specular.py:302-458).  I_d holds I1 on entry and I on exit;
 * In_d must hold I1 as well (it is the I_{n-1} operand of order 2) and holds the last order on
 * exit; J_d is scratch.  orders_d (may be NULL) receives every order: [max_saved][S*L][ld]
 * (I_saved, :304-305,458), order n>=2 at index n-2.  poll_every: orders enqueued between two
 * non-blocking polls of the device "all converged" counter (>=1).  results_h: [S]. */
int sos_solve(sos_plan* plan, double* I_d, double* In_d, double* J_d, double* orders_d, int max_saved,
              int max_orders, int poll_every, sos_result* results_h, void* stream);

/* Copy the per-scenario results to the host (synchronises the stream). */
int sos_get_results(sos_plan* plan, sos_result* results_h, void* stream);
/* Reset per-scenario state (active=1, n_orders=1, ratios from I1 with In := 1 as in :306-309). */
int sos_reset(sos_plan* plan, const double* I1_d, void* stream);

/* Quadratures of SOS_Aer_graphe.py: flux_up/flux_down (:154-158, direct beam scaled by
 * direct_scale: 1 there, 1/(4 pi) in :77-78 and SOS_Aer_critical_albedo.py:380-381),
 * net flux (:39-41), mean diffusivity (:8-10) and heating rate (:70-91; z_h: [L] altitudes).
 * Outputs are device arrays [S][L]; any may be NULL. */
int sos_quadratures(sos_plan* plan, const double* I_d, double direct_scale, const double* z_h,
                    double* flux_up_d, double* flux_down_d, double* net_flux_d, double* diffusivity_d,
                    double* heating_d, void* stream);

/* Number of kernel launches issued through this plan so far (bench.py's gpu_launches). */
long long sos_launch_count(const sos_plan* plan);

/* Which code path will sos_solve take on this plan?  Returns 0 / 1 (or the device ordinal), negative on error. */
#define SOS_QUERY_FUSED_ORDER 0       /* sos_solve may rebuild sources inside the sweeps (buffers exist, nothing disabled it) */
#define SOS_QUERY_GENERATED_SOURCE 1  /* ... and does: J is rebuilt from two projections per row on the molecular rows
                                         (csrc/sweep.cuh: SrcGen) instead of being written by a contraction and read back */
#define SOS_QUERY_FOLDED 2            /* folded contraction registered */
#define SOS_QUERY_DEVICE 3            /* CUDA device ordinal the plan lives on */
int sos_plan_query(const sos_plan* plan, int what);

/* mu-block sharding of one large grid (BASELINE config 4): this plan computes only the mu columns
 * [col0, col1) of J and I_n (and accumulates only those columns of I); the caller all-gathers the
 * I_n blocks of all ranks before the next sos_source.  col0 and col1 must be multiples of 128 (or 0 /
 * N); only grids without surface coupling (n_regions == 1, SOS_SURFACE_NONE) can be sharded, and a
 * block boundary must not cut the mu -> 0 zones (SOS_ERR_UNSUPPORTED otherwise). */
int sos_plan_set_columns(sos_plan* plan, int col0, int col1);
/* Layer-block sharding of one large grid over the GPUs of a node (BASELINE configs[3]; the order loop it splits is
 * SOS_Aer_main_specular.py:302-458 on the single-layer operators SOS_Aer_I1_In.py:62-130).  Rank r of n_ranks owns a
 * contiguous block of scan chunks = layers [*row0_out, *row1_out): its source contraction and sweeps touch only those rows
 * (the contraction a few halo rows more), every field keeps the full [L][ld] layout.  Per order the ranks exchange, by
 * stores into each other's memory over NVLink (no host round trip, no NCCL call on the data path):
 *   - the chunk aggregates of the scan (N doubles per chunk and direction), after which every rank runs the same carry
 *     chain over the same numbers as the unsharded solve: results are bit-identical to it;
 *   - the I_n rows next to a block boundary that the neighbour reads as halos, and the two convergence ratios.
 * mailbox_peers_d[q] / In_peers_d[q]: rank q's mailbox (sos_layer_mailbox_bytes() bytes, 128-byte aligned, zeroed once at
 * allocation) and I_n field as mapped into THIS process (sos_ipc_alloc / sos_ipc_open; entry `rank` = this rank's own
 * buffers).  Afterwards sos_solve(plan, I_d, In_peers_d[rank], J_d, ...) runs the sharded order loop: every rank must call
 * it with the same max_orders, I_d and In_d holding the first order on ALL rows; on exit the rank's rows of I_d are final.
 * Only single-scenario, single-region plans without surface coupling, all mu columns.  n_ranks <= 1 restores the whole grid. */
int sos_layer_mailbox_bytes(const sos_plan* plan, size_t* bytes);
int sos_plan_set_layers(sos_plan* plan, int rank, int n_ranks, void* const* mailbox_peers_d, double* const* In_peers_d,
                        int* row0_out, int* row1_out);

/* Copy the per-scenario convergence ratios {ratio_toa, ratio_surf} to (set = 0) or from (set = 1) a
 * device buffer [S][2]: sharded ranks MAX-all-reduce them between sos_sweeps and sos_converge. */
int sos_state_ratios(sos_plan* plan, double* buf_d, int set, void* stream);

/* Optional timing of kernel classes with CUDA events on the launching stream:
 * class 0 = source contraction (all its launches of one order per span), class 1 = layer sweeps (four launches per
 * span), class 2 = the apply pass of the sweeps alone (the HBM-bound kernel; nested inside class 1), class 3 = the
 * dense DMMA kernel of the contraction alone (nested inside class 0).  sos_get_profile synchronises the stream,
 * returns accumulated milliseconds and span counts in ms[SOS_PROFILE_CLASSES] / spans[SOS_PROFILE_CLASSES] and clears
 * the accumulators. */
#define SOS_PROFILE_CLASSES 4
int sos_set_profiling(sos_plan* plan, int enabled);
int sos_get_profile(sos_plan* plan, double* ms, long long* spans, void* stream);

/* FP64 throughput probe used for the roofline denominator (DFMA or DMMA loop, all SMs);
 * returns TFLOP/s in *tflops.  kind: 0 = DFMA, 1 = DMMA m8n8k4. */
int sos_fp64_peak(int kind, int repeats, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* SOS_B200_H */
