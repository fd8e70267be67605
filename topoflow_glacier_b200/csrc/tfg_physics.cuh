// tfg_physics.cuh -- one cell, one timestep of the energy-balance + melt update.
//
// Restates BmiTopoflowGlacier.update() (reference src/topoflow_glacier/bmi/bmi_topoflow_glacier.py:413-465)
// and Clear_Sky_Radiation (reference src/topoflow_glacier/physics/solar_funcs.py:894-953) as a single
// device function.  Quantities that depend on the clock only arrive in TimeRow, quantities that depend on the
// cell only in the Cell accessor (RegCell / SmemCell); both are evaluated on the host with the reference's scalar expressions.
// In StrictF64 mode every operation keeps the reference's order and association (line numbers in comments).
#pragma once
#include "tfg_num.cuh"

namespace tfg {

// Numeric literals of the physics, kept in __constant__ memory: as immediates every float64 literal costs two
// UMOV instructions per use; from the constant bank it is one LDCU (often hoisted out of the time loop).
struct LitTable {
  double inv_esat0, inv_dew_a, esat10, mag_a, mag_b, esat0, c90, ky_a, ky_b, ky_c, ky_nc, sa_a0, sa_a1, sa_b0, sa_b1, s_a0, s_a1, s_b0, s_b1, dew_c, dew_b, wp_a, wp_b, alb_r1, alb_r0, alb_0, alb_k, alb_ice, alb_bare, st_a, st_b, st_c, st_d, st_e, st_f, kelvin, c12, snow_thr, c3600, c001, c01, pi;
};
static __constant__ LitTable kLit = {0.1636661211129296, 0.1636098885816659, 6.11, 17.3, 237.3, 0.611, 90.0, 0.50572, 6.07995, 1.6364, -1.6364, -0.1240, 0.0207, -0.0682, 0.0248, -0.0363, 0.0084, -0.0572, 0.0173, 257.14, 18.678, 1.12, 0.0614, 0.12, 0.05, 0.4, 0.44, 0.3, 0.15, 0.151977, 8.313659, 1.676331, 0.00391838, 0.023101, 4.86035, 273.15, 12.0, 0.03, 3600.0, 0.01, 0.1, 3.141592653589793};
#define LIT(field, value) (P::f32 ? Num<P>(value) : Num<P>(static_cast<typename P::raw>(kLit.field)))
#ifndef TFG_AIRMASS_TABLE   // fast float64: Kasten-Young air mass from the table of tfg_math.cuh (0: closed form, A/B runs)
#define TFG_AIRMASS_TABLE 1
#endif
#ifndef TFG_SPLIT_STEP
#define TFG_SPLIT_STEP 0
#endif
#ifndef TFG_ALBEDO_EARLY  // fast float64 step: the albedo-ageing exponential (:1042-1048) is evaluated beside the W_p / e_sat(T_surf)
#define TFG_ALBEDO_EARLY 1 // exponentials (one group of three shares table index arithmetic and coefficients); bit-identical, +0.7 %
#endif
#ifndef TFG_CT_HOIST   // column-term step: the late terms (W_p, e_sat(T_dew); LW_in, T_wb) are requested a section ahead of their use
#define TFG_CT_HOIST 1
#endif
#ifndef TFG_EXP5   // experiment: all five exponentials of the met block in one group
#define TFG_EXP5 0
#endif
#ifndef TFG_FUSE_ROOT7   // experiment: Brutsaert's 7th root evaluated beside the W_p / e_sat(T_surf) exponentials (fm::exp_tab2_root7);
#define TFG_FUSE_ROOT7 0 // bit-identical, measured slower (28.5 vs 30.0 G: longer live ranges at the register limit)
#endif
#ifndef TFG_FOLD_CONSTS  // fast float64: constant factors folded (a_elev/R* per launch, rho_air Lv 0.622/p0c, 0.611*10): -4 FP64 per step
#define TFG_FOLD_CONSTS 1
#endif
#ifndef TFG_REUSE_COSZ   // fast float64: K_h = I_sc E0 max(cos Z, 0) reuses cos Z (the same fused multiply-add, bit for bit)
#define TFG_REUSE_COSZ 1
#endif
#ifndef TFG_WETBULB_TABLE   // fast float64: Stull wet bulb from the tables of tfg_math.cuh (0: closed form, A/B runs)
#define TFG_WETBULB_TABLE 1
#endif

// host-precomputed scalars (products/ratios formed in the reference's own order)
template <class raw>
struct Consts {
  raw dt;            // cfg.dt [h]
  raw days_per_dt;   // dt / 86400 (sic, :287)
  raw T0;
  raw sea_p0;        // :539
  raw r_star;        // :543
  raw eps, one_m_eps;  // :817
  raw gz;            // g * z  (:640)
  raw z, z0_air, kappa;  // :670
  raw rho_cp_air;    // rho_air * Cp_air (:745)
  raw rho_lv_air;    // rho_air * Lv (:932)
  raw lhc;           // latent_heat_constant (:931)
  raw ws_ratio;      // rho_H2O / rho_snow (:385, :1030)
  raw wi_ratio;      // rho_H2O / rho_ice
  raw rho_cp_snow;   // rho_snow * Cp_snow (:1533)
  raw rho_lf;        // rho_H2O * Lf (:1368)
  raw dust;          // cfg.dust_atten
  raw emis_a;        // (1 - F) * 1.72 (:1179)
  raw emis_b;        // 1 + 0.22 * C**2 (:1180)
  raw canopy;        // F
  raw sigma;         // :1234
  raw es_sigma;      // em_surf * sigma (:1236)
  raw one_m_es;      // 1 - em_surf (:1246)
  raw one_seventh;   // :292
  raw omega;         // 15 deg/h in rad (solar_funcs.py:257-258)
  raw rad2deg;       // 180 / pi (solar_funcs.py:550)
  raw deg2rad;       // pi / 180 (solar_funcs.py:566)
  raw inv_z0, inv_dt, inv_rho_lf;  // fast modes only: reciprocals of z0_air, dt, rho_H2O*Lf
  raw inv_rstar, inv_p0c, kappa2;  // fast modes only: 1/R*, 1/(sea_p0*0.01), kappa^2
  raw cq0;                         // fast float64: rho_air*Lv * latent_heat_constant / (sea_p0*0.01)  (:931-934 folded)
  int satterlund;
};

template <class raw>
struct TimeRow {  // see tfg_time_row in include/tfglacier.h
  raw clock_hour, TE, sin_decl, cos_decl, tan_decl, isc_e0;
  raw cos_hour, sin_hour;  // cos/sin of omega*((clock_hour - 12) - TE); fast modes only
};

template <class raw>
struct CellState {
  raw h_snow, h_swe, h_ice, h_iwe, eccs, ecci, albedo, n_days;
  // float32 mode only: low parts of h_swe / h_iwe.  The water-equivalent balance (:1594-1617) is carried as
  // (double)h + (double)lo and evaluated in float64 inside the float32 kernel: accumulating hourly melt of 1e-4 m into a
  // float32 depth of ~1 m loses the melt-out hour, which is where float32 results left the reference (VERDICT r1 #11)
  raw swe_lo, iwe_lo;
};

// float32 mode: one water-equivalent balance in float64.  h (+ low part) gains `gain`, then loses min(M*3600, h)/3600*dt*3600;
// returns the melt rate actually realised.  Same operation order as the reference, so the melt-out residue logic carries over.
__device__ __forceinline__ float balance64(float& h, float& lo, float gain, float M, float dt) {
  if (gain == 0.0f && M == 0.0f) return 0.0f;   // nothing enters or leaves (frozen pack, snow-covered ice): h + lo stays as it is
  // single-rounding intrinsics throughout: this translation unit allows FMA contraction, and a fused w - (m dt) 3600
  // would return the rounding residue of the product instead of the reference's exact zero at melt-out
  double w = __dadd_rn((double)h, (double)lo);
  w = __dadd_rn(w, (double)gain);
  const double s3 = __dmul_rn((double)M, 3600.0);
  const double s = (s3 < w) ? s3 : w;                 // both finite and >= 0 here: no NaN handling needed
  // s / 3600 correctly rounded (Markstein, as div3600 in tfg_num.cuh): the reference's own float64 operations in its
  // own order, so a pack that melts out leaves a rounding residue exactly when the reference's would
  const double y = 1.0 / 3600.0, q = __dmul_rn(s, y);
  const double m = __fma_rn(__fma_rn(-3600.0, q, s), y, q);
  w = __dsub_rn(w, __dmul_rn(__dmul_rn(m, (double)dt), 3600.0));
  w = (w > 0.0) ? w : 0.0;
  h = (float)w;
  lo = (float)__dsub_rn(w, (double)h);
  return (float)m;
}


// ---- where the per-cell constants and the diagnostic integrals live during a launch ------------------------
// SmemCell keeps them in shared memory, one column per thread, and reads a value where it is used: in registers
// (RegCell) they pin ~44 registers for the whole time loop and hold the float64 kernels at 3 blocks per SM.
enum { kSaElev, kSSinLat, kSCosLat, kSNegTanLat, kSSinEq, kSCosEq, kSNegTanEq, kSDlon, kSTNoon, kSDa, kSTrs,
       kSCB, kSSB, kSCB2, kSSB2, kSVolP, kSVolPR, kSVolPS, kSVolSM, kSVolIM, kSPmax,
       kSaElevR,   // fast float64 only: a_elev / R*, formed once per launch instead of once per step
       kSCount };
// Per-cell surface factors (tfg_bind_cell_params): the rows of the library's [kPCount][n_cells] scratch and, in kernels
// instantiated with per-cell parameters, shared-memory columns kSCount + i.  Each replaces the Consts field of the
// same meaning; the strict step divides by z0_air, the fast steps multiply by its reciprocal (the fast float64 kernel
// needs both: its fallback for insane forcings and SATTERLUND is the strict step).
enum { kPDust, kPEmisA, kPEmisB, kPCanopy, kPEsSigma, kPOneMEs, kPZ0, kPInvZ0, kPCount };

template <class raw>
struct RegCell {
  static constexpr bool kPar = false;
  raw v[kSCount];
  __device__ __forceinline__ raw get(int i) const { return v[i]; }
  __device__ __forceinline__ void set(int i, raw x) { v[i] = x; }
  __device__ __forceinline__ raw par(int, raw k) const { return k; }
};

template <class raw, int BLOCK, bool PAR = false>
struct SmemCell {
  static constexpr bool kPar = PAR;   // per-cell surface factors in columns kSCount + kP*
  unsigned base;  // shared-window address of this thread's column
  // surface factor i of this cell, or the context constant `k` when the kernel runs without per-cell parameters
  __device__ __forceinline__ raw par(int i, raw k) const {
    if constexpr (PAR) return get(kSCount + i); else return k;
  }
  __device__ __forceinline__ raw get(int i) const {
    raw x;
    if constexpr (sizeof(raw) == 8) asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(x) : "r"(base + i * BLOCK * 8));
    else asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(x) : "r"(base + i * BLOCK * 4));
    return x;
  }
  __device__ __forceinline__ void set(int i, raw x) {
    if constexpr (sizeof(raw) == 8) asm volatile("st.volatile.shared.f64 [%0], %1;" ::"r"(base + i * BLOCK * 8), "d"(x));
    else asm volatile("st.volatile.shared.f32 [%0], %1;" ::"r"(base + i * BLOCK * 4), "f"(x));
  }
};

template <class raw>
struct StepOut {
  raw SM, IM, M_total, RH;
  // intermediates (only stored when the caller records them)
  raw p0, e_sat_air, e_air, T_dew, T_surf, e_sat_surf, Ri, Dn, Dh, Qh, W_p, e_surf, Qe, th, Qn_SW, em_air, Qn_LW,
      Q_sum, P_rain, P_snow;
};

// update_saturation_vapor_pressure(MBAR=True), :784-802
template <class P>
__device__ __forceinline__ Num<P> e_sat_mbar(const Consts<typename P::raw>& k, Num<P> T) {
  using R = Num<P>;
  R e_sat;
  if (!k.satterlund) {
    R term1 = (LIT(mag_a, 17.3) * T) / (T + LIT(mag_b, 237.3));
    e_sat = LIT(esat0, 0.611) * nexp(term1);
  } else {
    R term1 = R(2353.0) / (T + 273.15);
    e_sat = divk(npow(R(10.0), R(11.4) - term1), 1000.0);
  }
  return e_sat * 10.0;
}

// The clock- and cell-dependent part of Clear_Sky_Radiation; returns K_cs.
template <class P, class Cell>
__device__ __forceinline__ Num<P> clear_sky(const Consts<typename P::raw>& k, const TimeRow<typename P::raw>& tr,
                                            const Cell& s, Num<P> th, Num<P> W_p, Num<P> albedo) {
  using R = Num<P>;
  const R sin_d(tr.sin_decl), cos_d(tr.cos_decl), tan_d(tr.tan_decl), omega(k.omega);
  const R wt = omega * th;
  R c_wt, c_u;
  if constexpr (P::strict) {
    c_wt = ncos(wt);                                         // cos(omega*th), solar_funcs.py:282, :391
    c_u = ncos(wt + R(s.get(kSDlon)));                              // solar_funcs.py:867
  } else {
    // omega*th = A_t - B_c with A_t = omega*((clock-12)-TE) (host, per step) and B_c = omega*LC (per cell):
    // cos(A - B) = cosA cosB + sinA sinB -- two FMAs instead of a full-range cos()
    const R cA(tr.cos_hour), sA(tr.sin_hour);
    c_wt = fmadd(cA, R(s.get(kSCB)), sA * R(s.get(kSSB)));
    c_u = fmadd(cA, R(s.get(kSCB2)), sA * R(s.get(kSSB2)));
  }
  // sunrise / sunset arguments, solar_funcs.py:325-326 (horizontal) and :796 (equivalent latitude)
  R arg_eq = R(s.get(kSNegTanEq)) * tan_d, arg_h = R(s.get(kSNegTanLat)) * tan_d;
  if constexpr (P::strict) {
    arg_eq = nmin(nmax(R(-1.0), arg_eq), R(1.0));
    arg_h = nmin(nmax(R(-1.0), arg_h), R(1.0));
  }  // fast modes compare cosines with the unclamped arguments: beyond +-1 (polar day / night) the outcome is the same
  bool dark;
  if constexpr (P::strict) {
    // T_sr / T_ss exactly as solar_funcs.py:783-830, then the comparison of :939
    const R q_eq = nacos(arg_eq) / omega;
    const R q_h = nacos(arg_h) / omega;
    const R T_sr = nmax((-q_eq) + R(s.get(kSTNoon)), -q_h);
    const R T_ss = nmin(q_eq + R(s.get(kSTNoon)), q_h);
    dark = (th <= T_sr) || (th >= T_ss);
  } else {
    // th <= -acos(a)/omega  or  th >= acos(a)/omega   <=>   cos(omega*th) <= a   for |omega*th| < pi;
    // outside that range both reference comparisons are true anyway (|T_sr|,|T_ss| <= 12 h).
    const R pi = LIT(pi, 3.141592653589793);
    dark = (c_wt <= arg_h) || (c_u <= arg_eq) || (nabs(wt) >= pi) || (nabs(wt + R(s.get(kSDlon))) >= pi);
  }
  if (dark) return R(0.0);                                   // solar_funcs.py:940-941

  // Zenith_Angle solar_funcs.py:281-284
  R cosZ;
  if constexpr (P::strict) cosZ = (R(s.get(kSSinLat)) * sin_d) + ((R(s.get(kSCosLat)) * cos_d) * c_wt);
  else cosZ = fmadd(R(s.get(kSCosLat)) * cos_d, c_wt, R(s.get(kSSinLat)) * sin_d);
  // Optical_Air_Mass solar_funcs.py:549-568 (Kasten & Young 1989)
  R gamma, t1, t2;
  if constexpr (P::strict) {
    const R Z = nacos(cosZ);
    gamma = LIT(c90, 90.0) - (Z * R(k.rad2deg));
    gamma = sel(R(0.0) > gamma, R(0.0), gamma);
    t1 = nsin(gamma * R(k.deg2rad));
    t2 = LIT(ky_a, 0.50572) / npow(gamma + LIT(ky_b, 6.07995), LIT(ky_c, 1.6364));
  } else {
    // elevation angle gamma = 90deg - Z = asin(cos Z), sin(gamma) = cos Z; a/(gamma+b)^c = a*exp(-c*log(gamma+b))
    t1 = relu(cosZ);
    if constexpr (!TFG_AIRMASS_TABLE || !P::lean) {
      const R elev_rad = nasin01(t1);
      gamma = elev_rad * R(k.rad2deg);
      t2 = LIT(ky_a, 0.50572) * nexp(LIT(ky_nc, -1.6364) * nlog(fmadd(elev_rad, R(k.rad2deg), LIT(ky_b, 6.07995))));
    }
  }
  R M_opt;
  // lean: 1/M = sin(gamma) + t2 as one piecewise polynomial in cos Z (fm::inv_air_mass): no asin, log, exp
  if constexpr (TFG_AIRMASS_TABLE && P::lean) M_opt = R(fm::rcp3(fm::inv_air_mass(t1.v)));
  else M_opt = R(1.0) / (t1 + t2);
  // Atmospheric_Transmissivity solar_funcs.py:608-614
  const R a_sa = fnmadd(LIT(sa_a1, 0.0207), W_p, LIT(sa_a0, -0.1240));
  const R b_sa = fnmadd(LIT(sa_b1, 0.0248), W_p, LIT(sa_b0, -0.0682));
  // Scattering_Attenuation solar_funcs.py:649-653
  const R a_s = fnmadd(LIT(s_a1, 0.0084), W_p, LIT(s_a0, -0.0363));
  const R b_s = fnmadd(LIT(s_b1, 0.0173), W_p, LIT(s_b0, -0.0572));
  R e_tau, e_gam;
  if constexpr (P::lean) {  // the two exponentials side by side (see fm::exp_tab_n)
    const double ex[2] = {fmadd(b_sa, M_opt, a_sa).v, fmadd(b_s, M_opt, a_s).v};
    double ey[2];
    fm::exp_tab_n<2>(ex, ey);
    e_tau = R(ey[0]); e_gam = R(ey[1]);
  } else {
    e_tau = nexp(fmadd(b_sa, M_opt, a_sa)); e_gam = nexp(fmadd(b_s, M_opt, a_s));
  }
  const R tau = nmin(relu(e_tau - R(s.par(kPDust, k.dust))), R(1.0));
  const R gam_s = (R(1.0) - e_gam) + R(s.par(kPDust, k.dust));
  // ET_Radiation_Flux solar_funcs.py:391-412 ; ET_Radiation_Flux_Slope :866-887
  const R isc_e0(tr.isc_e0);
  // (cos_d cos_lat) cos(wt) + sin_d sin_lat is cos Z itself: the products commute exactly, so the lean path reuses it
  R K_h;
  if constexpr (P::lean && TFG_REUSE_COSZ) K_h = relu(isc_e0 * cosZ);
  else K_h = relu(isc_e0 * fmadd(cos_d * R(s.get(kSCosLat)), c_wt, sin_d * R(s.get(kSSinLat))));
  const R K_s = relu(isc_e0 * fmadd(cos_d * R(s.get(kSCosEq)), c_u, R(s.get(kSSinEq)) * sin_d));
  const R half_gam = R(0.5) * gam_s;
  const R K_dif = half_gam * K_h;                            // :667
  const R K_glob = fmadd(tau, K_h, K_dif);                   // :634, :683
  const R K_bs = (half_gam * albedo) * K_glob;               // :711
  return fmadd(tau, K_s, K_dif) + K_bs;                      // :909
}


// =====================================================================================================================
// EXPERIMENT (round 2, not the default path): the fast float64 step in two parts.  Build with -DTFG_SPLIT_STEP=1 (and
// -DTFG_PIPELINE=1 for the software-pipelined loop of tfg_pipe.cuh).  Measured on the bench shape (16 777 216 cells x
// 128 steps, profiles/r2_experiments.md): single-stream split step 29.0 G cell-steps/s (inline step: 30.0 G);
// pipelined loop 22.2 G at 128 registers / 4 blocks per SM, 21.9 G at 96 registers (440 B of spills): the second
// instruction stream costs more in registers (fewer resident warps, spills) than it returns in overlapped latency --
// warps issue in order, so it is thread-level parallelism that hides the FP64 latency of this kernel, not ILP.
//
// `lean_forcing` is everything of update() that does not read the carried state: the met block up to the dew point
// (:519-556, :747-893), the vapour factor of the latent heat flux for BOTH surface temperatures the state can select
// (T_surf = T_dew, or 0 degC over a melting surface, :906-911), incoming longwave (:1167-1234), the clear-sky shortwave
// except its LINEAR dependence on albedo (K_cs = A + albedo*B, solar_funcs.py:894-953), and the snowfall wet bulb
// (:1507-1520).  `lean_state` consumes the ten numbers of `Derived` and advances the state (:626-733 log law and bulk
// exchange, :1006-1059 albedo, :1207-1319 net fluxes, :1321-1617 melt, water equivalents, cold content).
// The split (a) lets a kernel evaluate the forcing part of step t+1 beside the state part of step t -- two independent
// instruction streams per thread, where the single-stream step waits out one FP64 latency after the other -- and
// (b) is the hand-over interface of the producer / consumer kernel (tfg_ws.cuh).  Every instantiation of the fast mode
// goes through these two functions, so recording / aggregate / integral kernels agree bit for bit.
// =====================================================================================================================
enum { kD_P, kD_Tair, kD_uz, kD_Tdew, kD_Xa, kD_Xb, kD_LWin, kD_A, kD_B, kD_ccs, kDHand,   // the ten hand-over values
       kD_RH = kDHand, kD_p0, kD_esat_air, kD_eair, kD_esdew, kD_Wp, kD_emair, kD_th, kDCount };  // + output / recording only
//   kD_P     +P where it rains, -P where it snows (T_air <= T_rain_snow)
//   kD_Xa/Xb rho_air Lv (0.622/p0) (e_air - RH e_sat(T_surf)) for T_surf = T_dew / T_surf = 0 degC: Qe = De * X
//   kD_LWin  em_air sigma T_K^4          kD_A/B  K_cs = A + albedo * B (both 0 at night)
//   kD_ccs   rho_snow Cp_snow (P_snow dt rho_H2O/rho_snow) (T0 - T_wb), 0 unless it snows
template <class raw>
struct Derived {            // in registers (single-stream kernels)
  raw v[kDCount];
  __device__ __forceinline__ raw get(int i) const { return v[i]; }
};
struct SmemDerived {        // one stage of the producer -> consumer ring in shared memory (tfg_ws.cuh): value i of this
  unsigned base;            // thread's cell at base + i * stride bytes, read at the point of use
  unsigned stride;
  __device__ __forceinline__ double get(int i) const {
    if (i >= kDHand) return 0.0;   // output / recording values do not travel (the producer stores RH itself)
    double x;
    asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(x) : "r"(base + (unsigned)i * stride));
    return x;
  }
};

template <class Cell>
__device__ __forceinline__ void lean_forcing(const Consts<double>& k, const TimeRow<double>& tr, const Cell& s, double LC,
                                             double Pp, double T_air, double P_air, double q, double uz, Derived<double>& d) {
  const double T_K = T_air + kLit.kelvin;
  const bool is_snow = T_air <= s.get(kSTrs);                                   // :585, :604
  d.v[kD_P] = is_snow ? -Pp : Pp;
  d.v[kD_Tair] = T_air; d.v[kD_uz] = uz;
  // -- three reciprocals: 1/T_K, the vapour-pressure quotient (:817), the Magnus quotient of the air (:788)
  const double den3[3] = {T_K, fma(k.one_m_eps, q, k.eps), T_air + kLit.mag_b};
  double rc3[3];
  fm::rcp3_n<3>(den3, rc3);
  const double rTK = rc3[0];
  const double e_air = ((q * P_air) * rc3[1]) * kLit.c001;
  // -- exp(-M g elev / (R* T_K)) (:551-556) and exp(-17.3 T/(T+237.3)); log(e_air/6.1121) (:892)
  const double ex2[2] = {-((s.get(kSaElev) * k.inv_rstar) * rTK), -((kLit.mag_a * T_air) * rc3[2])};
  double ey2[2];
  fm::exp_tab_n<2>(ex2, ey2);
  const double log_term = fm::log_tab(e_air * kLit.inv_dew_a);
  const double RH = (e_air * ey2[1]) * kLit.inv_esat0;                          // e_air / (6.11 exp(t1)), :838
  const double T_dew = (kLit.dew_c * log_term) * fm::rcp3(kLit.dew_b - log_term);   // :888-893
  // -- W_p = 1.12 exp(0.0614 T_dew) (:919-920) and e_sat(T_dew) (:784-802)
  const double ex2b[2] = {kLit.wp_b * T_dew, (kLit.mag_a * T_dew) * fm::rcp3(T_dew + kLit.mag_b)};
  double ey2b[2];
  fm::exp_tab_n<2>(ex2b, ey2b);
  const double W_p = kLit.wp_a * ey2b[0];
  const double es_dew = (kLit.esat0 * ey2b[1]) * 10.0;
  const double es_zero = (kLit.esat0 * 1.0) * 10.0;                             // e_sat(0 degC), same operations
  const double cq = ey2[0] * k.cq0;                                             // rho_air Lv * 0.622 / p0, :931-934
  d.v[kD_Xa] = cq * fma(-RH, es_dew, e_air);
  d.v[kD_Xb] = cq * fma(-RH, es_zero, e_air);
  d.v[kD_Tdew] = T_dew; d.v[kD_RH] = RH;
  // -- update_em_air :1167-1180 (Brutsaert), incoming longwave :1234
  const double em_air = fma(s.par(kPEmisA, k.emis_a) * fm::root7((e_air * kLit.c01) * rTK), s.par(kPEmisB, k.emis_b),
                            s.par(kPCanopy, k.canopy));
  const double tk2 = T_K * T_K;
  d.v[kD_LWin] = (em_air * k.sigma) * (tk2 * tk2);
  // -- update_julian_day :990-1004 ; True_Solar_Noon solar_funcs.py:1471 ; Clear_Sky_Radiation solar_funcs.py:894-953
  const double th = tr.clock_hour - ((kLit.c12 + LC) + tr.TE);
  const double wt = k.omega * th;
  const double c_wt = fma(tr.cos_hour, s.get(kSCB), tr.sin_hour * s.get(kSSB));       // cos(omega th) by angle addition
  const double c_u = fma(tr.cos_hour, s.get(kSCB2), tr.sin_hour * s.get(kSSB2));      // cos(omega th + dlon)
  const double arg_eq = s.get(kSNegTanEq) * tr.tan_decl, arg_h = s.get(kSNegTanLat) * tr.tan_decl;
  // th <= -acos(a)/omega or th >= acos(a)/omega  <=>  cos(omega th) <= a  for |omega th| < pi (solar_funcs.py:783-830, :939)
  const bool dark = (c_wt <= arg_h) || (c_u <= arg_eq) || (fabs(wt) >= kLit.pi) || (fabs(wt + s.get(kSDlon)) >= kLit.pi);
  d.v[kD_A] = 0.0; d.v[kD_B] = 0.0;
  if (!dark) {
    const double cos_lat = s.get(kSCosLat), sin_lat = s.get(kSSinLat);
    const double cosZ = fma(cos_lat * tr.cos_decl, c_wt, sin_lat * tr.sin_decl);        // :281-284
    const double t1 = relu(Num<FastF64>(cosZ)).v;
    const double M_opt = fm::rcp3(fm::inv_air_mass(t1));                                 // :549-568 (Kasten & Young)
    const double ex[2] = {fma(fma(-kLit.sa_b1, W_p, kLit.sa_b0), M_opt, fma(-kLit.sa_a1, W_p, kLit.sa_a0)),    // :608-614
                          fma(fma(-kLit.s_b1, W_p, kLit.s_b0), M_opt, fma(-kLit.s_a1, W_p, kLit.s_a0))};      // :649-653
    double ey[2];
    fm::exp_tab_n<2>(ex, ey);
    const double tau = nmin(relu(Num<FastF64>(ey[0] - s.par(kPDust, k.dust))), Num<FastF64>(1.0)).v;
    const double half_gam = 0.5 * ((1.0 - ey[1]) + s.par(kPDust, k.dust));
    const double K_h = relu(Num<FastF64>(tr.isc_e0 * fma(tr.cos_decl * cos_lat, c_wt, tr.sin_decl * sin_lat))).v;      // :391-412
    const double K_s = relu(Num<FastF64>(tr.isc_e0 * fma(tr.cos_decl * s.get(kSCosEq), c_u, s.get(kSSinEq) * tr.sin_decl))).v;  // :866-887
    const double K_dif = half_gam * K_h;                                                 // :667
    d.v[kD_A] = fma(tau, K_s, K_dif);                                                          // :909 without backscatter
    d.v[kD_B] = half_gam * fma(tau, K_h, K_dif);                                               // :711: K_bs = albedo * B
  }
  // -- update_snowfall_cold_content :1507-1537: the wet bulb is only consumed where snow falls
  d.v[kD_ccs] = 0.0;
  if (is_snow && Pp > 0.0) {
    double T_wb;
    if (RH >= 0.046875 && RH <= 2.0) {          // table bins 1..32
      T_wb = fm::stull_wet_bulb_tab(T_air, RH);
    } else {
      using R = Num<FastF64>;
      const R T(T_air), H(RH);
      T_wb = (((((T * natan(R(kLit.st_a) * nsqrt(H + R(kLit.st_b)))) + natan(T + H)) - natan(H - R(kLit.st_c))) +
               ((R(kLit.st_d) * npow15(H)) * natan(R(kLit.st_e) * H))) - R(kLit.st_f)).v;
    }
    d.v[kD_ccs] = (k.rho_cp_snow * ((Pp * k.dt) * k.ws_ratio)) * (k.T0 - T_wb);
  }
  d.v[kD_p0] = fm::div_fast(1.0, ey2[0] * k.inv_p0c); d.v[kD_esat_air] = fm::div_fast(kLit.esat10, ey2[1]); d.v[kD_eair] = e_air;
  d.v[kD_esdew] = es_dew; d.v[kD_Wp] = W_p; d.v[kD_emair] = em_air; d.v[kD_th] = th;
}

template <bool VOL, class Cell, class D, class WindowFn>
__device__ __forceinline__ void lean_state(const Consts<double>& k, Cell& s, CellState<double>& st, const D& d,
                                           WindowFn&& window_sum, StepOut<double>& o) {
  using R = Num<FastF64>;
  const double dt = k.dt;
  double h_snow = st.h_snow, h_swe = st.h_swe, h_ice = st.h_ice, h_iwe = st.h_iwe, Eccs = st.eccs, Ecci = st.ecci;
  const double P_signed = d.get(kD_P);
  const double P_rain = relu(R(P_signed)).v, P_snow = relu(R(-P_signed)).v;
  const double Pp = fabs(P_signed), T_air = d.get(kD_Tair), uz = d.get(kD_uz), T_dew = d.get(kD_Tdew);
  if constexpr (VOL) {  // :567-568, :576, :613-614, :623-624
    const double da = s.get(kSDa);
    s.set(kSVolP, fma(Pp * da, dt, s.get(kSVolP)));
    s.set(kSPmax, nmax(R(s.get(kSPmax)), R(Pp)).v);
    s.set(kSVolPR, fma(P_rain * da, dt, s.get(kSVolPR)));
    s.set(kSVolPS, fma(P_snow * da, dt, s.get(kSVolPS)));
  }
  const double T_K = T_air + kLit.kelvin;
  // -- update_T_surf :906-911: min(T_dew, 0) over snow or ice; e_sat(T_surf) is then e_sat(0) or e_sat(T_dew)
  const bool warm = ((h_snow > 0.0) || (h_ice > 0.0)) && (T_dew > 0.0);
  const double T_surf = warm ? 0.0 : T_dew;
  const double X = warm ? d.get(kD_Xb) : d.get(kD_Xa);
  // -- update_bulk_richardson_number :640-644, update_bulk_aero_conductance :670-733 as ONE quotient:
  //    stable   (top > 0): Dh = Dn / (1 + 10 top/bot) = uz k^2 bot          / (L^2 (bot + 10 top))
  //    unstable (top <= 0): Dh = Dn * (1 - 10 top/bot) = uz k^2 (bot - 10 top) / (L^2 bot)       (top = 0: Dh = Dn)
  const double dT = T_air - T_surf;
  const double top = k.gz * dT;
  double bot = (uz * uz) * T_K;
  bot = (bot == 0.0) ? kLit.c001 : bot;
  const bool stable = top > 0.0;
  const double num = stable ? bot : fma(-10.0, top, bot);
  const double den = stable ? fma(10.0, top, bot) : bot;
  const double L = fm::log_tab(nmax(R((k.z - h_snow) * s.par(kPInvZ0, k.inv_z0)), R(kLit.c001)).v);
  const double uk2 = uz * k.kappa2, LL = L * L;
  const double Dh = (uk2 * num) * fm::rcp3(LL * den);
  const double Qh = (k.rho_cp_air * Dh) * dT;                                   // :744-745
  const double Qe = Dh * X;                                                     // :931-934
  // -- update_albedo("aging") :1023-1059
  const double r = (T_air > 0.0) ? kLit.alb_r1 : kLit.alb_r0;
  const double ring_new = __dmul_rn(__dmul_rn(P_snow, dt), k.ws_ratio);         // :1031-1033
  const double tot = window_sum(ring_new);                                      // :1027-1037
  double n = st.n_days;
  n = (tot < kLit.snow_thr) ? n + k.days_per_dt : 0.0;                          // :1040-1041 (tot is finite on the sane path)
  double albedo = st.albedo;
  if (h_snow > 0.0) albedo = fma(kLit.alb_k, fm::exp_tab((-n) * r), kLit.alb_0);        // :1042-1048
  if (h_snow == 0.0 && h_ice > 0.0) albedo = kLit.alb_ice;                      // :1049-1053
  if (h_snow == 0.0 && h_ice == 0.0) albedo = kLit.alb_bare;                    // :1054-1058
  // -- net shortwave :1122-1139 (K_cs = A + albedo B), net longwave :1231-1248, energy sum :1314
  const double Qn_SW = fma(albedo, d.get(kD_B), d.get(kD_A)) * (1.0 - albedo);
  const double T_surf_K = T_surf + kLit.kelvin, ts2 = T_surf_K * T_surf_K;
  const double LW_in = d.get(kD_LWin);
  const double LW_out = fma(s.par(kPOneMEs, k.one_m_es), LW_in, s.par(kPEsSigma, k.es_sigma) * (ts2 * ts2));
  const double Qn_LW = LW_in - LW_out;
  const double Q_sum = ((Qn_SW + Qn_LW) + Qh) + Qe;
  // -- snow: update_snow_meltrate :1364-1368, enforce_max_snow_meltrate :1465
  const double previous_swe = h_swe;                                            // :1571
  const double E_in = Q_sum * dt;
  double SM = (relu(R(E_in - Eccs)).v * k.inv_dt) * k.inv_rho_lf;
  if constexpr (VOL) s.set(kSVolSM, fma((SM * s.get(kSDa)) * dt, kLit.c3600, s.get(kSVolSM)));   // :1486-1487
  // -- update_swe :1594-1606 (single-rounding operations: decides whether SWE reaches exactly 0)
  h_swe = __dadd_rn(h_swe, __dmul_rn(P_snow, dt));
  SM = div3600(nmin(R(__dmul_rn(SM, kLit.c3600)), R(h_swe))).v;
  h_swe = relu(R(__dsub_rn(h_swe, __dmul_rn(__dmul_rn(SM, dt), kLit.c3600)))).v;
  // -- update_snowfall_cold_content :1533-1537
  if (P_snow > 0.0) Eccs = relu(R((Eccs + d.get(kD_ccs)) - E_in)).v;
  // -- update_ice_meltrate :1418-1428 (NEW h_swe, OLD h_ice), enforce_max_ice_meltrate :1473-1480
  double IM = (relu(R(E_in - Ecci)).v * k.inv_dt) * k.inv_rho_lf;
  IM = ((h_swe == 0.0) && (previous_swe == 0.0)) ? IM : 0.0;
  Ecci = relu(R(Ecci - E_in)).v;
  Ecci = (h_ice == 0.0) ? 0.0 : Ecci;
  IM = nmin(R(IM), R(h_iwe * k.inv_dt)).v;
  if constexpr (VOL) s.set(kSVolIM, fma((IM * s.get(kSDa)) * dt, kLit.c3600, s.get(kSVolIM)));   // :1493-1494
  // -- update_iwe :1612-1617
  IM = div3600(nmin(R(__dmul_rn(IM, kLit.c3600)), R(h_iwe))).v;
  h_iwe = relu(R(__dsub_rn(h_iwe, __dmul_rn(__dmul_rn(IM, dt), kLit.c3600)))).v;
  const double M_total = fma(P_rain, 1.0 / 3600.0, IM + SM);                    // :1441-1445
  h_snow = __dmul_rn(h_swe, k.ws_ratio);                                        // :1711
  h_ice = __dmul_rn(h_iwe, k.wi_ratio);                                         // :1726
  // -- update_snowpack_cold_content :1552-1558
  if (P_snow <= 0.0) Eccs = relu(R(Eccs - E_in)).v;
  if (h_snow == 0.0) Eccs = 0.0;

  st.h_snow = h_snow; st.h_swe = h_swe; st.h_ice = h_ice; st.h_iwe = h_iwe;
  st.eccs = Eccs; st.ecci = Ecci; st.albedo = albedo; st.n_days = n;
  o.SM = SM; o.IM = IM; o.M_total = M_total; o.RH = d.get(kD_RH);
  // intermediates: only read when a caller records them (dead code otherwise)
  const double e_sat_surf = warm ? (kLit.esat0 * 1.0) * 10.0 : d.get(kD_esdew);
  o.p0 = d.get(kD_p0); o.e_sat_air = d.get(kD_esat_air); o.e_air = d.get(kD_eair); o.T_dew = T_dew; o.T_surf = T_surf; o.e_sat_surf = e_sat_surf;
  o.Ri = fm::div_fast(top, bot); o.Dn = fm::div_fast(uk2, LL); o.Dh = Dh; o.Qh = Qh; o.W_p = d.get(kD_Wp);
  o.e_surf = d.get(kD_RH) * e_sat_surf; o.Qe = Qe; o.th = d.get(kD_th); o.Qn_SW = Qn_SW; o.em_air = d.get(kD_emair); o.Qn_LW = Qn_LW;
  o.Q_sum = Q_sum; o.P_rain = P_rain; o.P_snow = P_snow;
}

// ---- column terms -----------------------------------------------------------------------------------------------------
// With a forcing map bound (tfg_bind_forcing_map: how every catchment run is configured -- one met series per
// catchment, many cells) the part of update() that reads nothing but the forcings is the same for every cell of a
// column: vapour pressures, relative humidity, dew point (:423-425, :784-893), precipitable water (:919-920), air
// emissivity and incoming longwave (:1167-1234), the snowfall wet bulb (:1507-1520).  `column_terms_eval` evaluates it
// ONCE PER COLUMN AND TIMESTEP (tfg::column_terms_kernel) with exactly the operations of the per-cell fast step, and the
// melt kernel reads the results: one 128-byte line per column and timestep, which also carries the raw forcings, so
// the per-cell forcing block is not read at all.  What stays per cell: pressure at the cell's elevation, the log law,
// the bulk exchange, albedo, clear-sky shortwave on the cell's slope, the melt / cold-content / water-equivalent updates.
enum { kCtP, kCtTair, kCtUz, kCtRTK, kCtEair, kCtRH, kCtTdew, kCtSane,        // read ahead (next step) by the kernel
       kCtWp, kCtEsDew, kCtLWin, kCtTwb, kCtEmAir, kCtEsatAir, kCtPair, kCtQ,  // read at their point of use
       kCtCount };
static_assert(kCtCount == 16, "one 128-byte line per column and timestep");
struct NoColumnTerms { static constexpr bool on = false; };
struct ColumnTerms {
  static constexpr bool on = true;
  double rTK, e_air, RH, T_dew;   // in registers (prefetched with the forcings)
  const double* line;             // this step's line: the remaining terms are loaded where they are consumed
  __device__ __forceinline__ double get(int i) const { return __ldg(line + i); }
};

// the forcing-only terms of one column and timestep; `sane` as in the melt kernel's fast-path test (otherwise the
// kernel takes the strict step from the raw forcings and none of the terms is read)
// PAR (per-cell parameters bound): the emissivity and longwave slots carry the parameter-free factors x**(1/7) and
// T_K**4 instead, from which the melt kernel forms em_air and LW_in with the cell's parameters (same operations)
template <class P, bool PAR = false>
__device__ __forceinline__ void column_terms_eval(const Consts<double>& k, double Pp, double T_air_, double P_air_, double q_,
                                                  double uz, bool sane, double* out) {
  using R = Num<P>;
  static_assert(P::lean, "column terms exist for the fast float64 mode only");
  double o[kCtCount];
#pragma unroll
  for (int i = 0; i < kCtCount; ++i) o[i] = 0.0;
  o[kCtP] = Pp; o[kCtTair] = T_air_; o[kCtUz] = uz; o[kCtPair] = P_air_; o[kCtQ] = q_;
  if (sane) {
    const R T_air(T_air_), P_air(P_air_), q(q_);
    const R T_K = T_air + LIT(kelvin, 273.15);
    const double den3[3] = {T_K.v, fmadd(R(k.one_m_eps), q, R(k.eps)).v, (T_air + LIT(mag_b, 237.3)).v};
    double rc3[3];
    fm::rcp3_n<3>(den3, rc3);
    const R rTK(rc3[0]);
    const R e = (q * P_air) * R(rc3[1]);
    const R e_air = e * LIT(c001, 0.01);
    const double ex1[1] = {(-((LIT(mag_a, 17.3) * T_air) * R(rc3[2]))).v};
    const double lx1[1] = {(e_air * LIT(inv_dew_a, 0.1636098885816659)).v};
    double ey1[1], ly1[1];
    fm::exp_tab_n<1>(ex1, ey1);
    fm::log_tab_n<1>(lx1, ly1);
    const R en(ey1[0]), log_term(ly1[0]);
    const R RH = (e_air * en) * LIT(inv_esat0, 0.1636661211129296);
    const R T_dew = (LIT(dew_c, 257.14) * log_term) * R(fm::rcp3((LIT(dew_b, 18.678) - log_term).v));
    const double den1[1] = {(T_dew + LIT(mag_b, 237.3)).v};
    double rc1[1];
    fm::rcp3_n<1>(den1, rc1);
    const double ex2[2] = {(LIT(wp_b, 0.0614) * T_dew).v, ((LIT(mag_a, 17.3) * T_dew) * R(rc1[0])).v};
    double ey2[2];
    fm::exp_tab_n<2>(ex2, ey2);
    const R W_p = LIT(wp_a, 1.12) * R(ey2[0]);
    const R es_dew = LIT(esat10, 6.11) * R(ey2[1]);
    const R x = (e_air * LIT(c01, 0.1)) * rTK;
    R em_air, LW_in;
    if constexpr (PAR) {
      em_air = R(fm::root7(x.v));
      LW_in = npow4(T_K);
    } else {
      em_air = fmadd(R(k.emis_a) * R(fm::root7(x.v)), R(k.emis_b), R(k.canopy));
      LW_in = (em_air * R(k.sigma)) * npow4(T_K);
    }
    R T_wb;
    bool stull_fast;
    if constexpr (TFG_WETBULB_TABLE) stull_fast = (RH >= 0.046875) && (RH <= 2.0);
    else stull_fast = (RH >= 0.0) && (RH <= 2.0);
    if (stull_fast) {
      if constexpr (TFG_WETBULB_TABLE) T_wb = R(fm::stull_wet_bulb_tab(T_air.v, RH.v));
      else T_wb = R(fm::stull_wet_bulb(T_air.v, RH.v));
    } else {
      T_wb = ((((T_air * natan(LIT(st_a, 0.151977) * nsqrt(RH + LIT(st_b, 8.313659)))) + natan(T_air + RH)) -
               natan(RH - LIT(st_c, 1.676331))) +
              ((LIT(st_d, 0.00391838) * npow15(RH)) * natan(LIT(st_e, 0.023101) * RH))) -
             LIT(st_f, 4.86035);
    }
    o[kCtRTK] = rTK.v; o[kCtEair] = e_air.v; o[kCtRH] = RH.v; o[kCtTdew] = T_dew.v; o[kCtSane] = 1.0;
    o[kCtWp] = W_p.v; o[kCtEsDew] = es_dew.v; o[kCtLWin] = LW_in.v; o[kCtTwb] = T_wb.v; o[kCtEmAir] = em_air.v;
    o[kCtEsatAir] = (LIT(esat10, 6.11) / en).v;
  }
#pragma unroll
  for (int i = 0; i < kCtCount; i += 2) *reinterpret_cast<double2*>(out + i) = make_double2(o[i], o[i + 1]);
}

// The same terms in the strict arithmetic (libdevice functions, IEEE division, NumPy's NaN rules: the expressions of the
// strict per-cell step, operation for operation), SATTERLUND configurations included.  There is no "sane" test in this
// mode -- a missing value poisons the column's terms exactly as it poisons every cell of the column in the per-cell
// step.  Slot kCtRTK carries e_sat(0 degC) here (the strict step has no use for 1/T_K).
template <class P, bool PAR = false>
__device__ __forceinline__ void column_terms_eval_strict(const Consts<double>& k, double Pp, double T_air_, double P_air_,
                                                         double q_, double uz, double* out) {
  using R = Num<P>;
  static_assert(P::strict, "strict float64 mode");
  const R T_air(T_air_), P_air(P_air_), q(q_);
  const R T_K = T_air + LIT(kelvin, 273.15);
  const R e_sat_air = e_sat_mbar<P>(k, T_air);
  const R e = (q * P_air) / (R(k.eps) + (R(k.one_m_eps) * q));     // :817
  const R e_air = (e / 1000.0) * 10.0;
  const R RH = e_air / e_sat_air;                                  // :838
  const R log_term = nlog(divk(e_air, 6.1121));                    // :888-893
  const R T_dew = (LIT(dew_c, 257.14) * log_term) / (LIT(dew_b, 18.678) - log_term);
  const R W_p = LIT(wp_a, 1.12) * nexp(LIT(wp_b, 0.0614) * T_dew);  // :919-920
  double zero = 0.0;
  asm volatile("" : "+d"(zero));   // opaque: e_sat(0) goes through the device functions like the per-cell step's, not the compiler's folding
  const R es_dew = e_sat_mbar<P>(k, T_dew), es_zero = e_sat_mbar<P>(k, R(zero));
  R em_air, LW_in;                                                 // :1167-1192
  if (!k.satterlund) {
    const R x = divk(e_air, 10.0) / T_K;
    if constexpr (PAR) {   // the parameter-free factors, as in column_terms_eval
      em_air = npow(x, R(k.one_seventh));
    } else {
      const R term1 = R(k.emis_a) * npow(x, R(k.one_seventh));
      em_air = fmadd(term1, R(k.emis_b), R(k.canopy));
    }
  } else {
    em_air = R(1.08) * (R(1.0) - nexp(R(-1.0) * npow(e_air, divk(T_K, 2016.0))));
  }
  if (PAR && !k.satterlund) LW_in = npow4(T_K);
  else LW_in = (em_air * R(k.sigma)) * npow4(T_K);                 // :1234
  const R T_wb = ((((T_air * natan(LIT(st_a, 0.151977) * nsqrt(RH + LIT(st_b, 8.313659)))) + natan(T_air + RH)) -
                   natan(RH - LIT(st_c, 1.676331))) +
                  ((LIT(st_d, 0.00391838) * npow15(RH)) * natan(LIT(st_e, 0.023101) * RH))) -
                 LIT(st_f, 4.86035);                                // :1507-1520
  double o[kCtCount];
  o[kCtP] = Pp; o[kCtTair] = T_air_; o[kCtUz] = uz; o[kCtPair] = P_air_; o[kCtQ] = q_;
  o[kCtRTK] = es_zero.v; o[kCtEair] = e_air.v; o[kCtRH] = RH.v; o[kCtTdew] = T_dew.v; o[kCtSane] = 1.0;
  o[kCtWp] = W_p.v; o[kCtEsDew] = es_dew.v; o[kCtLWin] = LW_in.v; o[kCtTwb] = T_wb.v; o[kCtEmAir] = em_air.v;
  o[kCtEsatAir] = e_sat_air.v;
#pragma unroll
  for (int i = 0; i < kCtCount; i += 2) *reinterpret_cast<double2*>(out + i) = make_double2(o[i], o[i + 1]);
}

// One update().  `window_sum(ring_new)` must return the 72-slot snowfall-window sum AFTER this step's
// entry `ring_new` replaced the oldest one (:1027-1037); the caller owns the window storage.
// `mid_step()` is called once the pressure / humidity / wind forcings are dead (after the turbulent fluxes): the
// kernel issues the next step's forcing loads there, so that they do not hold registers through the met block.
template <class P, bool VOL, class Cell, class WindowFn, class MidFn, class Pre = NoColumnTerms>
__device__ __forceinline__ void cell_step(const Consts<typename P::raw>& k, const TimeRow<typename P::raw>& tr,
                                          Cell& s, Num<P> LC, CellState<typename P::raw>& st,
                                          Num<P> Pp, Num<P> T_air, Num<P> P_air, Num<P> q, Num<P> uz,
                                          WindowFn&& window_sum, MidFn&& mid_step, StepOut<typename P::raw>& o,
                                          const Pre& pre = Pre()) {
  using R = Num<P>;
#if TFG_SPLIT_STEP   // experiment: the fast float64 step through lean_forcing / lean_state (measured 3 % slower, see below)
  if constexpr (P::lean) {
    Derived<double> d;
    lean_forcing(k, tr, s, LC.v, Pp.v, T_air.v, P_air.v, q.v, uz.v, d);
    mid_step();
    lean_state<VOL>(k, s, st, d, window_sum, o);
    return;
  }
#endif
  const R dt(k.dt);
  R h_snow(st.h_snow), h_swe(st.h_swe), h_ice(st.h_ice), h_iwe(st.h_iwe), Eccs(st.eccs), Ecci(st.ecci);

  const R T_K = T_air + LIT(kelvin, 273.15);
  // ---- update_P_rain :585, update_P_snow :604  (P * bool)
  const bool is_rain = T_air > R(s.get(kSTrs));
  const bool is_snow = T_air <= R(s.get(kSTrs));
  R P_rain, P_snow;
  if constexpr (P::strict) {
    P_rain = Pp * R(is_rain ? 1.0 : 0.0);
    P_snow = Pp * R(is_snow ? 1.0 : 0.0);
  } else {
    P_rain = sel(is_snow, R(0.0), Pp);   // sane T_air (no NaN): is_rain == !is_snow
    P_snow = sel(is_snow, Pp, R(0.0));
  }
  if constexpr (VOL) {  // :567-568, :576, :613-614, :623-624
    const R da(s.get(kSDa));
    s.set(kSVolP, fmadd(Pp * da, dt, R(s.get(kSVolP))).v);
    s.set(kSPmax, nmax(R(s.get(kSPmax)), Pp).v);
    s.set(kSVolPR, fmadd(P_rain * da, dt, R(s.get(kSVolPR))).v);
    s.set(kSVolPS, fmadd(P_snow * da, dt, R(s.get(kSVolPS))).v);
  }
  R p0, e_sat_air, e_air, RH, T_dew, T_surf, e_sat_surf, dT, Ri, Dn, Dh, Qh, W_p, e_surf, Qe, rTK;
  R n_early, tot_early, alb_exp;   // lean + TFG_ALBEDO_EARLY: days since snowfall, window sum, exp(-n r)
  double root7_pre = 0.0;   // x**(1/7) of update_em_air, evaluated early beside two exponentials (lean, TFG_FUSE_ROOT7)
  if constexpr (P::lean && Pre::on) {
    // Column terms bound (see column_terms_eval): only what depends on the cell is left of the met block
    static_assert(TFG_ALBEDO_EARLY && TFG_FOLD_CONSTS, "the column-term step is written for the default fast step");
    rTK = R(pre.rTK); e_air = R(pre.e_air); RH = R(pre.RH); T_dew = R(pre.T_dew);
    double2 late0 = make_double2(0.0, 0.0);   // W_p, e_sat(T_dew): consumed at the end of this block
    if constexpr (TFG_CT_HOIST) late0 = __ldg(reinterpret_cast<const double2*>(pre.line + kCtWp));
    const double lx1[1] = {nmax((R(k.z) - h_snow) * R(s.par(kPInvZ0, k.inv_z0)), LIT(c001, 0.01)).v};
    double ly1[1];
    fm::log_tab_n<1>(lx1, ly1);
    const R L(ly1[0]);
    const bool cover = (h_snow > 0.0) || (h_ice > 0.0);
    T_surf = sel(cover, nmin(T_dew, R(0.0)), T_dew);                                         // :906-911
    dT = T_air - T_surf;
    const R top = R(k.gz) * dT;                                                              // :640-644
    R bot = (uz * uz) * T_K;
    bot = sel(bot == 0.0, LIT(c001, 0.01), bot);
    const bool stable = top > 0.0;
    const R num = sel(stable, bot, fnmadd(R(10.0), top, bot));
    const R den = sel(stable, fmadd(R(10.0), top, bot), bot);
    const R uk2 = uz * R(k.kappa2);
    const R LL = L * L;
    const double den1[1] = {(LL * den).v};
    double rc1[1];
    fm::rcp3_n<1>(den1, rc1);
    Dh = (uk2 * num) * R(rc1[0]);
    // albedo ageing (:1023-1048) beside the pressure exponential (:551-556)
    const R r = sel(T_air > 0.0, LIT(alb_r1, 0.12), LIT(alb_r0, 0.05));
    const R ring_new = xmul(xmul(P_snow, dt), R(k.ws_ratio));  // :1031-1033
    tot_early = R(window_sum(ring_new.v));                     // :1027-1037
    n_early = sel(tot_early < LIT(snow_thr, 0.03), R(st.n_days) + R(k.days_per_dt), R(0.0));
    const double ex2[2] = {(-(R(s.get(kSaElevR)) * rTK)).v, ((-n_early) * r).v};
    double ey2[2];
    fm::exp_tab_n<2>(ex2, ey2);
    alb_exp = R(ey2[1]);
    const R inv_p0 = R(ey2[0]) * R(k.inv_p0c);
    if constexpr (!TFG_CT_HOIST) late0 = make_double2(pre.get(kCtWp), pre.get(kCtEsDew));
    W_p = R(late0.x);
    // e_sat(T_surf): T_surf is the dew point, or 0 degC over a melting surface, where exp(17.3 * 0 / 237.3) = 1 exactly
    e_sat_surf = sel(cover && (T_dew > 0.0), LIT(esat10, 6.11) * R(1.0), R(late0.y));
    Qh = (R(k.rho_cp_air) * Dh) * dT;                                                        // :744-745
    e_surf = RH * e_sat_surf;                                                                // :853
    Qe = (Dh * fnmadd(RH, e_sat_surf, e_air)) * (R(ey2[0]) * R(k.cq0));                      // :931-934
    // only read when a caller records them (dead code otherwise)
    p0 = R(1.0) / inv_p0; Ri = top / bot; Dn = uk2 / LL;
    e_sat_air = R(pre.get(kCtEsatAir));
  } else if constexpr (P::lean) {
    // Same quantities with 7 instead of 12 divisions: 1/T_K is shared, 1/p0 and RH come from exp(-x) instead of
    // dividing by exp(x), and the aerodynamic block (:640-733) collapses into one quotient:
    //   stable   (top > 0): Dh = Dn / (1 + 10 top/bot) = uz k^2 bot          / (L^2 (bot + 10 top))
    //   unstable (top <= 0): Dh = Dn * (1 - 10 top/bot) = uz k^2 (bot - 10 top) / (L^2 bot)       (top = 0: Dh = Dn)
    // Independent reciprocals / exponentials / logarithms are evaluated side by side (fm::*_n) so that their
    // dependent FP64 chains overlap.  SATTERLUND configurations never get here (the kernel runs them strictly).
    // -- three reciprocals: 1/T_K, the vapour-pressure quotient (:817), the Magnus quotient of the air (:788)
    const double den3[3] = {T_K.v, fmadd(R(k.one_m_eps), q, R(k.eps)).v, (T_air + LIT(mag_b, 237.3)).v};
    double rc3[3];
    fm::rcp3_n<3>(den3, rc3);
    rTK = R(rc3[0]);
    const R e = (q * P_air) * R(rc3[1]);
    e_air = e * LIT(c001, 0.01);
    // -- exp(-M g elev / (R* T_K)) (:551-556), exp(-17.3 T/(T+237.3)); log(e_air/6.1121) (:892), the log law (:670)
    R ex_p0;
    if constexpr (TFG_FOLD_CONSTS) ex_p0 = -(R(s.get(kSaElevR)) * rTK);
    else ex_p0 = -((R(s.get(kSaElev)) * R(k.inv_rstar)) * rTK);
    const double ex2[2] = {ex_p0.v, (-((LIT(mag_a, 17.3) * T_air) * R(rc3[2]))).v};
    const double lx2[2] = {(e_air * LIT(inv_dew_a, 0.1636098885816659)).v,
                           nmax((R(k.z) - h_snow) * R(s.par(kPInvZ0, k.inv_z0)), LIT(c001, 0.01)).v};
    double ey2[2], ly2[2];
    if constexpr (!(TFG_EXP5 && TFG_ALBEDO_EARLY)) fm::exp_tab_n<2>(ex2, ey2);
    fm::log_tab_n<2>(lx2, ly2);
    const R log_term(ly2[0]), L(ly2[1]);
    T_dew = (LIT(dew_c, 257.14) * log_term) * R(fm::rcp3((LIT(dew_b, 18.678) - log_term).v));
    const bool cover = (h_snow > 0.0) || (h_ice > 0.0);
    T_surf = sel(cover, nmin(T_dew, R(0.0)), T_dew);                                         // :906-911
    dT = T_air - T_surf;
    const R top = R(k.gz) * dT;                                                              // :640-644
    R bot = (uz * uz) * T_K;
    bot = sel(bot == 0.0, LIT(c001, 0.01), bot);
    const bool stable = top > 0.0;
    const R num = sel(stable, bot, fnmadd(R(10.0), top, bot));
    const R den = sel(stable, fmadd(R(10.0), top, bot), bot);
    const R uk2 = uz * R(k.kappa2);
    const R LL = L * L;
    // -- two reciprocals: the Magnus quotient of the surface, the aerodynamic quotient
    const double den2[2] = {(T_surf + LIT(mag_b, 237.3)).v, (LL * den).v};
    double rc2[2];
    fm::rcp3_n<2>(den2, rc2);
    Dh = (uk2 * num) * R(rc2[1]);
    // -- W_p = 1.12 exp(0.0614 T_dew) (:919-920) and e_sat(T_surf) (:784-802)
    const double ex2b[2] = {(LIT(wp_b, 0.0614) * T_dew).v, ((LIT(mag_a, 17.3) * T_surf) * R(rc2[0])).v};
    double ey2b[2];
    if constexpr (TFG_ALBEDO_EARLY) {
      const R r = sel(T_air > 0.0, LIT(alb_r1, 0.12), LIT(alb_r0, 0.05));
      const R ring_new = xmul(xmul(P_snow, dt), R(k.ws_ratio));  // :1031-1033
      tot_early = R(window_sum(ring_new.v));                     // :1027-1037
      n_early = sel(tot_early < LIT(snow_thr, 0.03), R(st.n_days) + R(k.days_per_dt), R(0.0));
      if constexpr (TFG_EXP5) {
        const double ex5[5] = {ex2[0], ex2[1], ex2b[0], ex2b[1], ((-n_early) * r).v};
        double ey5[5];
        fm::exp_tab_n<5>(ex5, ey5);
        ey2[0] = ey5[0]; ey2[1] = ey5[1]; ey2b[0] = ey5[2]; ey2b[1] = ey5[3]; alb_exp = R(ey5[4]);
      } else {
        const double ex3[3] = {ex2b[0], ex2b[1], ((-n_early) * r).v};
        double ey3[3];
        fm::exp_tab_n<3>(ex3, ey3);
        ey2b[0] = ey3[0]; ey2b[1] = ey3[1]; alb_exp = R(ey3[2]);
      }
    } else if constexpr (TFG_FUSE_ROOT7) fm::exp_tab2_root7(ex2b, ey2b, ((e_air * LIT(c01, 0.1)) * rTK).v, root7_pre);
    else fm::exp_tab_n<2>(ex2b, ey2b);
    const R inv_p0 = R(ey2[0]) * R(k.inv_p0c);
    const R en(ey2[1]);
    RH = (e_air * en) * LIT(inv_esat0, 0.1636661211129296);                                 // e_air / (6.11 exp(t1)), :838
    W_p = LIT(wp_a, 1.12) * R(ey2b[0]);
    if constexpr (TFG_FOLD_CONSTS) e_sat_surf = LIT(esat10, 6.11) * R(ey2b[1]);
    else e_sat_surf = (LIT(esat0, 0.611) * R(ey2b[1])) * 10.0;
    Qh = (R(k.rho_cp_air) * Dh) * dT;                                                        // :744-745
    e_surf = RH * e_sat_surf;                                                                // :853
    if constexpr (TFG_FOLD_CONSTS)                                                           // :931-934, constants folded into cq0
      Qe = (Dh * fnmadd(RH, e_sat_surf, e_air)) * (R(ey2[0]) * R(k.cq0));
    else
      Qe = ((R(k.rho_lv_air) * Dh) * fnmadd(RH, e_sat_surf, e_air)) * (R(k.lhc) * inv_p0);
    // only read when a caller records them (dead code otherwise)
    p0 = R(1.0) / inv_p0; Ri = top / bot; Dn = uk2 / LL;
    e_sat_air = LIT(esat10, 6.11) / en;
  } else if constexpr (Pre::on) {
    // Strict step with the column terms bound (column_terms_eval_strict): the per-cell remainder, same operations
    static_assert(P::strict, "column terms: float64 modes");
    p0 = R(k.sea_p0) * nexp(R(s.get(kSaElev)) / (R(k.r_star) * T_K));                        // :551-556
    p0 = (p0 / 1000.0) * 10.0;
    e_sat_air = R(pre.get(kCtEsatAir)); e_air = R(pre.e_air); RH = R(pre.RH); T_dew = R(pre.T_dew);
    const bool cover = (h_snow > 0.0) || (h_ice > 0.0);
    T_surf = sel(cover, nmin(T_dew, R(0.0)), T_dew);                                         // :906-911
    // e_sat(T_surf), :784-802: T_surf is the dew point or, over a melting surface with a dew point above freezing, 0 degC
    e_sat_surf = sel(cover && (T_dew > 0.0), R(pre.rTK), R(pre.get(kCtEsDew)));
    dT = T_air - T_surf;
    const R top = R(k.gz) * dT;                                                              // :640-644
    R bot = (uz * uz) * T_K;
    bot = sel(bot == 0.0, R(0.01), bot);
    Ri = top / bot;
    const R zr = (R(k.z) - h_snow) / R(s.par(kPZ0, k.z0_air));                               // :670-733
    const R arg = R(k.kappa) / nlog(nmax(zr, R(0.01)));
    Dn = uz * (arg * arg);
    if (T_air == T_surf) Dh = Dn;
    else if (Ri > 0.0) Dh = Dn / (R(1.0) + (R(10.0) * Ri));
    else Dh = Dn * (R(1.0) - (R(10.0) * Ri));
    Qh = (R(k.rho_cp_air) * Dh) * dT;                                                        // :744-745
    W_p = R(pre.get(kCtWp));
    e_surf = RH * e_sat_surf;                                                                // :853
    Qe = ((R(k.rho_lv_air) * Dh) * (e_air - e_surf)) * (R(k.lhc) / p0);                      // :931-934
  } else {
    // ---- update_atm_pressure_from_elevation(T_C=True, MBAR=True) :551-556
    p0 = R(k.sea_p0) * nexp(R(s.get(kSaElev)) / (R(k.r_star) * T_K));
    if constexpr (P::strict) p0 = (p0 / 1000.0) * 10.0; else p0 = p0 * 0.01;
    // ---- vapour pressures :423-425
    e_sat_air = e_sat_mbar<P>(k, T_air);
    R e = (q * P_air) / (R(k.eps) + (R(k.one_m_eps) * q));     // :817
    if constexpr (P::strict) e_air = (e / 1000.0) * 10.0; else e_air = e * 0.01;
    RH = e_air / e_sat_air;                            // :838
    // ---- update_dew_point :888-893
    const R log_term = nlog(divk(e_air, 6.1121));
    T_dew = (LIT(dew_c, 257.14) * log_term) / (LIT(dew_b, 18.678) - log_term);
    // ---- update_T_surf :906-911
    const bool cover = (h_snow > 0.0) || (h_ice > 0.0);
    T_surf = sel(cover, nmin(T_dew, R(0.0)), T_dew);
    e_sat_surf = e_sat_mbar<P>(k, T_surf);
    // ---- update_bulk_richardson_number :640-644
    dT = T_air - T_surf;
    const R top = R(k.gz) * dT;
    R bot = (uz * uz) * T_K;
    bot = sel(bot == 0.0, R(0.01), bot);
    Ri = top / bot;
    // ---- update_bulk_aero_conductance :670-733
    R zr;
    if constexpr (P::strict) zr = (R(k.z) - h_snow) / R(s.par(kPZ0, k.z0_air));
    else zr = (R(k.z) - h_snow) * R(s.par(kPInvZ0, k.inv_z0));
    const R arg = R(k.kappa) / nlog(nmax(zr, R(0.01)));
    Dn = uz * (arg * arg);
    if (T_air == T_surf) Dh = Dn;
    else if (Ri > 0.0) Dh = Dn / (R(1.0) + (R(10.0) * Ri));
    else Dh = Dn * (R(1.0) - (R(10.0) * Ri));
    // ---- update_sensible_heat_flux :744-745
    Qh = (R(k.rho_cp_air) * Dh) * dT;
    // ---- update_precipitable_water_content :919-920
    W_p = LIT(wp_a, 1.12) * nexp(LIT(wp_b, 0.0614) * T_dew);
    // ---- update_vapor_pressure(SURFACE=True) :853 ; update_latent_heat_flux :931-934
    e_surf = RH * e_sat_surf;
    Qe = ((R(k.rho_lv_air) * Dh) * (e_air - e_surf)) * (R(k.lhc) / p0);
  }
  mid_step();
  double2 late1 = make_double2(0.0, 0.0);     // column terms LW_in, T_wb: consumed further down
  if constexpr (Pre::on && TFG_CT_HOIST) late1 = __ldg(reinterpret_cast<const double2*>(pre.line + kCtLWin));
  // ---- update_julian_day :990-1004 ; True_Solar_Noon solar_funcs.py:1471
  const R solar_noon = (LIT(c12, 12.0) + LC) + R(tr.TE);
  const R th = R(tr.clock_hour) - solar_noon;
  // ---- update_albedo("aging") :1023-1059
  R n, tot, albedo(st.albedo);
  if constexpr (P::lean && TFG_ALBEDO_EARLY) {
    n = n_early; tot = tot_early;
    albedo = sel(h_snow > 0.0, fmadd(LIT(alb_k, 0.44), alb_exp, LIT(alb_0, 0.4)), albedo);
  } else {
    const R r = sel(T_air > 0.0, LIT(alb_r1, 0.12), LIT(alb_r0, 0.05));
    const R ring_new = xmul(xmul(P_snow, dt), R(k.ws_ratio));  // :1031-1033
    tot = R(window_sum(ring_new.v));                           // :1027-1037
    n = R(st.n_days);
    const R thr = LIT(snow_thr, 0.03);
    if constexpr (P::strict) {
      n = sel(tot >= thr, R(0.0), n);                         // :1040
      n = sel(tot < thr, n + R(k.days_per_dt), n);            // :1041
    } else {
      n = sel(tot < thr, n + R(k.days_per_dt), R(0.0));       // tot is finite on the sane path
    }
    if (h_snow > 0.0) albedo = fmadd(LIT(alb_k, 0.44), nexp((-n) * r), LIT(alb_0, 0.4));  // :1042-1048
  }
  if (h_snow == 0.0 && h_ice > 0.0) albedo = LIT(alb_ice, 0.3);         // :1049-1053
  if (h_snow == 0.0 && h_ice == 0.0) albedo = LIT(alb_bare, 0.15);       // :1054-1058
  // ---- update_net_shortwave_radiation :1122-1139
  const R K_cs = clear_sky<P>(k, tr, s, th, W_p, albedo);
  const R Qn_SW = K_cs * (R(1.0) - albedo);
  // ---- update_em_air :1167-1192
  R em_air;
  if constexpr (Pre::on && Cell::kPar) {
    // per-cell parameters: the line holds the parameter-free factor (x**(1/7)) unless SATTERLUND, which takes none
    if (P::lean || !k.satterlund)
      em_air = fmadd(R(s.par(kPEmisA, k.emis_a)) * R(pre.get(kCtEmAir)), R(s.par(kPEmisB, k.emis_b)), R(s.par(kPCanopy, k.canopy)));
    else
      em_air = R(pre.get(kCtEmAir));
  } else if constexpr (Pre::on) {
    em_air = R(pre.get(kCtEmAir));   // recording only
  } else if (P::lean || !k.satterlund) {
    R x;
    if constexpr (P::lean) x = (e_air * LIT(c01, 0.1)) * rTK; else x = divk(e_air, 10.0) / T_K;
    R term1;
    if constexpr (P::lean && TFG_FUSE_ROOT7) term1 = R(s.par(kPEmisA, k.emis_a)) * R(root7_pre);
    else if constexpr (P::lean) term1 = R(s.par(kPEmisA, k.emis_a)) * R(fm::root7(x.v));   // x > 0 on the sane path
    else term1 = R(s.par(kPEmisA, k.emis_a)) * npow(x, R(k.one_seventh));
    em_air = fmadd(term1, R(s.par(kPEmisB, k.emis_b)), R(s.par(kPCanopy, k.canopy)));
  } else {
    em_air = R(1.08) * (R(1.0) - nexp(R(-1.0) * npow(e_air, divk(T_K, 2016.0))));
  }
  // ---- update_net_longwave_radiation :1231-1248
  const R T_surf_K = T_surf + LIT(kelvin, 273.15);
  R LW_in;
  if constexpr (Pre::on && Cell::kPar) {   // the line holds T_K**4 unless SATTERLUND (then LW_in itself)
    const R line = TFG_CT_HOIST ? R(late1.x) : R(pre.get(kCtLWin));
    if (P::lean || !k.satterlund) LW_in = (em_air * R(k.sigma)) * line;
    else LW_in = line;
  }
  else if constexpr (Pre::on && TFG_CT_HOIST) LW_in = R(late1.x);
  else if constexpr (Pre::on) LW_in = R(pre.get(kCtLWin));
  else LW_in = (em_air * R(k.sigma)) * npow4(T_K);
  R LW_out = R(s.par(kPEsSigma, k.es_sigma)) * npow4(T_surf_K);
  LW_out = fmadd(R(s.par(kPOneMEs, k.one_m_es)), LW_in, LW_out);
  const R Qn_LW = LW_in - LW_out;
  // ---- update_net_energy_flux :1314  (Qa = Qc = 0, :312-313)
  R Q_sum = ((Qn_SW + Qn_LW) + Qh) + Qe;
  if constexpr (P::strict) Q_sum = (Q_sum + R(0.0)) + R(0.0);

  // ---- snow: update_snow_meltrate :1364-1368, enforce_max_snow_meltrate :1465
  const R previous_swe = h_swe;                              // :1571
  const R E_in = Q_sum * dt;
  R SM;
  if constexpr (P::strict) SM = zdiv(zdiv(relu(E_in - Eccs), dt), R(k.rho_lf));
  else SM = (relu(E_in - Eccs) * R(k.inv_dt)) * R(k.inv_rho_lf);   // a product of non-negative factors
  if constexpr (P::strict) SM = relu(SM);
  if constexpr (VOL) s.set(kSVolSM, fmadd((SM * R(s.get(kSDa))) * dt, LIT(c3600, 3600.0), R(s.get(kSVolSM))).v);  // :1486-1487
  // ---- update_swe :1594-1606 (single-rounding ops in every mode: decides whether SWE hits exactly 0)
  const R k3600 = LIT(c3600, 3600.0);
  if constexpr (P::f32) {
    SM = R(balance64(h_swe.v, st.swe_lo, xmul(P_snow, dt).v, SM.v, dt.v));
  } else {
    h_swe = xadd(h_swe, xmul(P_snow, dt));
    SM = div3600(nmin(xmul(SM, k3600), h_swe));
    h_swe = xsub(h_swe, xmul(xmul(SM, dt), k3600));
    h_swe = relu(h_swe);
  }
  // ---- update_snowfall_cold_content :1507-1537 (T_wb is only consumed where P_snow > 0)
  if (P_snow > 0.0) {
    const R new_h_snow = (P_snow * dt) * R(k.ws_ratio);
    R T_wb;
    bool stull_fast = false;
    if constexpr (P::lean && TFG_WETBULB_TABLE) stull_fast = (RH >= 0.046875) && (RH <= 2.0);   // table bins 1..32
    else if constexpr (P::lean || P::f32) stull_fast = (RH >= 0.0) && (RH <= 2.0);
    if constexpr (Pre::on) {
      if constexpr (TFG_CT_HOIST) T_wb = R(late1.y); else T_wb = R(pre.get(kCtTwb));
    } else if (stull_fast) {
      if constexpr (P::f32) T_wb = R(fm::stull_wet_bulb32(T_air.v, RH.v));
      else if constexpr (TFG_WETBULB_TABLE) T_wb = R(fm::stull_wet_bulb_tab(T_air.v, RH.v));
      else T_wb = R(fm::stull_wet_bulb(T_air.v, RH.v));
    } else {
      T_wb = ((((T_air * natan(LIT(st_a, 0.151977) * nsqrt(RH + LIT(st_b, 8.313659)))) + natan(T_air + RH)) -
                       natan(RH - LIT(st_c, 1.676331))) +
                      ((LIT(st_d, 0.00391838) * npow15(RH)) * natan(LIT(st_e, 0.023101) * RH))) -
                     LIT(st_f, 4.86035);
    }
    const R del_T = R(k.T0) - T_wb;
    Eccs = relu(fmadd(R(k.rho_cp_snow) * new_h_snow, del_T, Eccs) - E_in);
  }
  // ---- update_ice_meltrate :1418-1428 (uses the NEW h_swe and the OLD h_ice)
  R IM;
  if constexpr (P::strict) IM = relu(zdiv(zdiv(relu(E_in - Ecci), dt), R(k.rho_lf)));
  else IM = (relu(E_in - Ecci) * R(k.inv_dt)) * R(k.inv_rho_lf);
  IM = sel((h_swe == 0.0) && (previous_swe == 0.0), IM, R(0.0));
  Ecci = relu(Ecci - E_in);
  Ecci = sel(h_ice == 0.0, R(0.0), Ecci);
  // ---- enforce_max_ice_meltrate :1473-1480
  if constexpr (P::strict) IM = relu(nmin(IM, zdiv(h_iwe, dt))); else IM = nmin(IM, h_iwe * R(k.inv_dt));
  if constexpr (VOL) s.set(kSVolIM, fmadd((IM * R(s.get(kSDa))) * dt, LIT(c3600, 3600.0), R(s.get(kSVolIM))).v);  // :1493-1494
  // ---- update_iwe :1612-1617 (single-rounding ops, as for SWE)
  if constexpr (P::f32) {
    IM = R(balance64(h_iwe.v, st.iwe_lo, 0.0f, IM.v, dt.v));
  } else {
    IM = div3600(nmin(xmul(IM, k3600), h_iwe));
    h_iwe = xsub(h_iwe, xmul(xmul(IM, dt), k3600));
    h_iwe = relu(h_iwe);
  }
  // ---- update_combined_meltrate :1441-1445
  R M_total;
  if constexpr (P::strict) M_total = (IM + SM) + divk(P_rain, 3600.0);
  else M_total = fmadd(P_rain, R(1.0 / 3600.0), IM + SM);
  // ---- update_snow_depth :1711, update_ice_depth :1726
  h_snow = xmul(h_swe, R(k.ws_ratio));
  h_ice = xmul(h_iwe, R(k.wi_ratio));
  // ---- update_snowpack_cold_content :1552-1558
  if (P_snow <= 0.0) Eccs = relu(Eccs - E_in);
  if (h_snow == 0.0) Eccs = R(0.0);

  st.h_snow = h_snow.v; st.h_swe = h_swe.v; st.h_ice = h_ice.v; st.h_iwe = h_iwe.v;
  st.eccs = Eccs.v; st.ecci = Ecci.v; st.albedo = albedo.v; st.n_days = n.v;
  o.SM = SM.v; o.IM = IM.v; o.M_total = M_total.v; o.RH = RH.v;
  o.p0 = p0.v; o.e_sat_air = e_sat_air.v; o.e_air = e_air.v; o.T_dew = T_dew.v; o.T_surf = T_surf.v;
  o.e_sat_surf = e_sat_surf.v; o.Ri = Ri.v; o.Dn = Dn.v; o.Dh = Dh.v; o.Qh = Qh.v; o.W_p = W_p.v;
  o.e_surf = e_surf.v; o.Qe = Qe.v; o.th = th.v; o.Qn_SW = Qn_SW.v; o.em_air = em_air.v; o.Qn_LW = Qn_LW.v;
  o.Q_sum = Q_sum.v; o.P_rain = P_rain.v; o.P_snow = P_snow.v;
}

}  // namespace tfg
