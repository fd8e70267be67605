// tfg_lean.cuh -- the fast float64 melt kernel (TFG_F64_FAST): TWO cells per thread.
//
// Same path as tfg_run.cuh (reference bmi_topoflow_glacier.py:413-465 in a fused time loop), restructured for the
// instruction-issue bound the round-1 profile showed (889 warp-instructions per warp-step, only 380 of them FP64):
//   * a thread owns the cells 2i and 2i+1 of the grid, so every constant load, clock-row load, address computation,
//     sanity vote, loop and branch instruction is paid once per TWO cell-steps;
//   * forcing, state and the snowfall window move as 128-bit vectors (ld.global.cs.v2.f64 / st.v2): a warp reads 512
//     contiguous bytes per forcing variable and step;
//   * the per-cell constants of both cells sit side by side in shared memory and are read with one LDS.128;
//   * the elementary functions of the two cells are evaluated side by side (fm::*_n), which doubles the independent
//     FP64 chains per warp;
//   * the divergent snowfall branch (Stull wet bulb) is entered once per thread for whichever of its cells needs it.
// The arithmetic per cell is op for op that of the round-1 lean step (every fused multiply-add is written out, the
// unit is compiled with -fmad=false), so recording / aggregate / integral instantiations agree bit for bit.
// Insane input (NaN forcing, absurd values) sends the whole warp through the strict step of tfg_physics.cuh, as before.
#pragma once
#include "tfg_run.cuh"

namespace tfg {

#ifndef TFG_W
#define TFG_W 2
#endif
#ifndef TFG_LEAN_BLOCK
#define TFG_LEAN_BLOCK 128
#endif
#ifndef TFG_LEAN_MIN_BLOCKS
#define TFG_LEAN_MIN_BLOCKS 3
#endif
constexpr int kW = TFG_W;
constexpr int kLeanBlock = TFG_LEAN_BLOCK;
constexpr int kLeanCells = kLeanBlock * kW;  // cells per block

// ---- W doubles / W predicates, element-wise ------------------------------------------------------------------
#define TFG_EACH _Pragma("unroll") for (int w = 0; w < W; ++w)
template <int W> struct VD {
  double v[W];
  __device__ __forceinline__ VD() {}
  __device__ __forceinline__ explicit VD(double x) { TFG_EACH v[w] = x; }
};
template <int W> struct VB { bool v[W]; };

#define TFG_VBIN(name, expr)                                                                           \
  template <int W> __device__ __forceinline__ VD<W> name(const VD<W>& a, const VD<W>& b) {             \
    VD<W> r; TFG_EACH { const double x = a.v[w], y = b.v[w]; r.v[w] = (expr); } return r;              \
  }                                                                                                    \
  template <int W> __device__ __forceinline__ VD<W> name(const VD<W>& a, double y) {                   \
    VD<W> r; TFG_EACH { const double x = a.v[w]; r.v[w] = (expr); } return r;                          \
  }                                                                                                    \
  template <int W> __device__ __forceinline__ VD<W> name(double x, const VD<W>& b) {                   \
    VD<W> r; TFG_EACH { const double y = b.v[w]; r.v[w] = (expr); } return r;                          \
  }
TFG_VBIN(operator+, x + y)
TFG_VBIN(operator-, x - y)
TFG_VBIN(operator*, x * y)
TFG_VBIN(xadd, __dadd_rn(x, y))   // single-rounding operations no build flag may contract (see tfg_num.cuh)
TFG_VBIN(xsub, __dsub_rn(x, y))
TFG_VBIN(xmul, __dmul_rn(x, y))
#undef TFG_VBIN
template <int W> __device__ __forceinline__ VD<W> operator-(const VD<W>& a) { VD<W> r; TFG_EACH r.v[w] = -a.v[w]; return r; }

// a*b + c and c - a*b, fused (the unit is compiled with -fmad=false: fusion is decided here, not by the compiler)
#define TFG_VFMA(name, expr)                                                                                          \
  template <int W> __device__ __forceinline__ VD<W> name(const VD<W>& a, const VD<W>& b, const VD<W>& c) {            \
    VD<W> r; TFG_EACH { const double x = a.v[w], y = b.v[w], z = c.v[w]; r.v[w] = (expr); } return r;                 \
  }                                                                                                                   \
  template <int W> __device__ __forceinline__ VD<W> name(double x, const VD<W>& b, const VD<W>& c) {                  \
    VD<W> r; TFG_EACH { const double y = b.v[w], z = c.v[w]; r.v[w] = (expr); } return r;                             \
  }                                                                                                                   \
  template <int W> __device__ __forceinline__ VD<W> name(const VD<W>& a, double y, const VD<W>& c) {                  \
    VD<W> r; TFG_EACH { const double x = a.v[w], z = c.v[w]; r.v[w] = (expr); } return r;                             \
  }                                                                                                                   \
  template <int W> __device__ __forceinline__ VD<W> name(const VD<W>& a, const VD<W>& b, double z) {                  \
    VD<W> r; TFG_EACH { const double x = a.v[w], y = b.v[w]; r.v[w] = (expr); } return r;                             \
  }                                                                                                                   \
  template <int W> __device__ __forceinline__ VD<W> name(double x, const VD<W>& b, double z) {                        \
    VD<W> r; TFG_EACH { const double y = b.v[w]; r.v[w] = (expr); } return r;                                         \
  }                                                                                                                   \
  template <int W> __device__ __forceinline__ VD<W> name(const VD<W>& a, double y, double z) {                        \
    VD<W> r; TFG_EACH { const double x = a.v[w]; r.v[w] = (expr); } return r;                                         \
  }
TFG_VFMA(vfma, fma(x, y, z))
TFG_VFMA(vfnma, fma(-x, y, z))
#undef TFG_VFMA

#define TFG_VCMP(name, expr)                                                                      \
  template <int W> __device__ __forceinline__ VB<W> name(const VD<W>& a, const VD<W>& b) {        \
    VB<W> r; TFG_EACH { const double x = a.v[w], y = b.v[w]; r.v[w] = (expr); } return r;         \
  }                                                                                               \
  template <int W> __device__ __forceinline__ VB<W> name(const VD<W>& a, double y) {              \
    VB<W> r; TFG_EACH { const double x = a.v[w]; r.v[w] = (expr); } return r;                     \
  }
TFG_VCMP(operator<, x < y)
TFG_VCMP(operator<=, x <= y)
TFG_VCMP(operator>, x > y)
TFG_VCMP(operator>=, x >= y)
TFG_VCMP(operator==, x == y)
#undef TFG_VCMP
template <int W> __device__ __forceinline__ VB<W> operator&&(const VB<W>& a, const VB<W>& b) { VB<W> r; TFG_EACH r.v[w] = a.v[w] && b.v[w]; return r; }
template <int W> __device__ __forceinline__ VB<W> operator||(const VB<W>& a, const VB<W>& b) { VB<W> r; TFG_EACH r.v[w] = a.v[w] || b.v[w]; return r; }
template <int W> __device__ __forceinline__ bool any(const VB<W>& a) { bool r = false; TFG_EACH r = r || a.v[w]; return r; }
template <int W> __device__ __forceinline__ bool all(const VB<W>& a) { bool r = true; TFG_EACH r = r && a.v[w]; return r; }

template <int W> __device__ __forceinline__ VD<W> vsel(const VB<W>& c, const VD<W>& a, const VD<W>& b) { VD<W> r; TFG_EACH r.v[w] = c.v[w] ? a.v[w] : b.v[w]; return r; }
template <int W> __device__ __forceinline__ VD<W> vsel(const VB<W>& c, const VD<W>& a, double b) { VD<W> r; TFG_EACH r.v[w] = c.v[w] ? a.v[w] : b; return r; }
template <int W> __device__ __forceinline__ VD<W> vsel(const VB<W>& c, double a, const VD<W>& b) { VD<W> r; TFG_EACH r.v[w] = c.v[w] ? a : b.v[w]; return r; }
template <int W> __device__ __forceinline__ VD<W> vsel(const VB<W>& c, double a, double b) { VD<W> r; TFG_EACH r.v[w] = c.v[w] ? a : b; return r; }

// setp + selp min / max and the integer relu of tfg_num.cuh (fast float64 forms), element-wise
template <int W> __device__ __forceinline__ VD<W> vmax(const VD<W>& a, const VD<W>& b) { VD<W> r; TFG_EACH r.v[w] = nmax(Num<FastF64>(a.v[w]), Num<FastF64>(b.v[w])).v; return r; }
template <int W> __device__ __forceinline__ VD<W> vmax(const VD<W>& a, double b) { VD<W> r; TFG_EACH r.v[w] = nmax(Num<FastF64>(a.v[w]), Num<FastF64>(b)).v; return r; }
template <int W> __device__ __forceinline__ VD<W> vmin(const VD<W>& a, const VD<W>& b) { VD<W> r; TFG_EACH r.v[w] = nmin(Num<FastF64>(a.v[w]), Num<FastF64>(b.v[w])).v; return r; }
template <int W> __device__ __forceinline__ VD<W> vmin(const VD<W>& a, double b) { VD<W> r; TFG_EACH r.v[w] = nmin(Num<FastF64>(a.v[w]), Num<FastF64>(b)).v; return r; }
template <int W> __device__ __forceinline__ VD<W> vrelu(const VD<W>& a) { VD<W> r; TFG_EACH r.v[w] = relu(Num<FastF64>(a.v[w])).v; return r; }
template <int W> __device__ __forceinline__ VD<W> vabs(const VD<W>& a) { VD<W> r; TFG_EACH r.v[w] = fabs(a.v[w]); return r; }

// K groups of W arguments through the N-at-once routines of tfg_math.cuh (K*W independent chains side by side)
template <int W> __device__ __forceinline__ void vexp2(const VD<W>& a, const VD<W>& b, VD<W>& ea, VD<W>& eb) {
  double x[2 * W], y[2 * W];
  TFG_EACH { x[w] = a.v[w]; x[W + w] = b.v[w]; }
  fm::exp_tab_n<2 * W>(x, y);
  TFG_EACH { ea.v[w] = y[w]; eb.v[w] = y[W + w]; }
}
template <int W> __device__ __forceinline__ VD<W> vexp(const VD<W>& a) { VD<W> r; fm::exp_tab_n<W>(a.v, r.v); return r; }
template <int W> __device__ __forceinline__ VD<W> vlog(const VD<W>& a) { VD<W> r; fm::log_tab_n<W>(a.v, r.v); return r; }
template <int W> __device__ __forceinline__ void vlog2(const VD<W>& a, const VD<W>& b, VD<W>& la, VD<W>& lb) {
  double x[2 * W], y[2 * W];
  TFG_EACH { x[w] = a.v[w]; x[W + w] = b.v[w]; }
  fm::log_tab_n<2 * W>(x, y);
  TFG_EACH { la.v[w] = y[w]; lb.v[w] = y[W + w]; }
}
template <int W> __device__ __forceinline__ VD<W> vrcp(const VD<W>& a) { VD<W> r; fm::rcp3_n<W>(a.v, r.v); return r; }
template <int W> __device__ __forceinline__ void vrcp2(const VD<W>& a, const VD<W>& b, VD<W>& ra, VD<W>& rb) {
  double x[2 * W], y[2 * W];
  TFG_EACH { x[w] = a.v[w]; x[W + w] = b.v[w]; }
  fm::rcp3_n<2 * W>(x, y);
  TFG_EACH { ra.v[w] = y[w]; rb.v[w] = y[W + w]; }
}
template <int W> __device__ __forceinline__ void vrcp3(const VD<W>& a, const VD<W>& b, const VD<W>& c, VD<W>& ra, VD<W>& rb, VD<W>& rc) {
  double x[3 * W], y[3 * W];
  TFG_EACH { x[w] = a.v[w]; x[W + w] = b.v[w]; x[2 * W + w] = c.v[w]; }
  fm::rcp3_n<3 * W>(x, y);
  TFG_EACH { ra.v[w] = y[w]; rb.v[w] = y[W + w]; rc.v[w] = y[2 * W + w]; }
}

// a / 3600 with a single rounding (Markstein, see div3600 in tfg_num.cuh): one range test for all W values
template <int W> __device__ __forceinline__ VD<W> vdiv3600(const VD<W>& a) {
  bool fast = true;
  TFG_EACH {
    const unsigned hi = (unsigned)__double2hiint(a.v[w]) & 0x7fffffffu;
    fast = fast && (hi >= 0x04100000u || (hi | (unsigned)__double2loint(a.v[w])) == 0u);
  }
  VD<W> r;
  if (fast) {
    const double y = 1.0 / 3600.0;
    TFG_EACH { const double q = __dmul_rn(a.v[w], y); r.v[w] = __fma_rn(__fma_rn(-3600.0, q, a.v[w]), y, q); }
  } else {
    TFG_EACH r.v[w] = div3600(Num<FastF64>(a.v[w])).v;
  }
  return r;
}

// ---- per-cell constants of the W cells of a thread: rows of [thread][w] pairs in shared memory ------------------
template <int W>
struct LeanCells {
  unsigned base;  // shared-window address of element 0 of this thread's pair in row 0
  static constexpr int kRowBytes = kLeanCells * 8;
  __device__ __forceinline__ VD<W> get(int i) const {
    VD<W> x;
    if constexpr (W == 2) {
      asm volatile("ld.volatile.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x.v[0]), "=d"(x.v[1]) : "r"(base + i * kRowBytes));
    } else {
      TFG_EACH asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(x.v[w]) : "r"(base + i * kRowBytes + w * 8));
    }
    return x;
  }
  __device__ __forceinline__ void set(int i, const VD<W>& x) const {
    if constexpr (W == 2) {
      asm volatile("st.volatile.shared.v2.f64 [%0], {%1, %2};" ::"r"(base + i * kRowBytes), "d"(x.v[0]), "d"(x.v[1]));
    } else {
      TFG_EACH asm volatile("st.volatile.shared.f64 [%0], %1;" ::"r"(base + i * kRowBytes + w * 8), "d"(x.v[w]));
    }
  }
  // the same storage seen as the single-cell accessor of tfg_physics.cuh (strict fallback step)
  __device__ __forceinline__ SmemCell<double, kLeanCells> elem(int w) const { return SmemCell<double, kLeanCells>{base + (unsigned)w * 8u}; }
};

#define LLIT(field) (kLit.field)

// Clear_Sky_Radiation (solar_funcs.py:894-953), fast form of tfg_physics.cuh clear_sky for W cells; `day` = cells in daylight
template <int W>
__device__ __forceinline__ VD<W> lean_clear_sky(const Consts<double>& k, const TimeRow<double>& tr, const LeanCells<W>& s,
                                                const VD<W>& th, const VD<W>& W_p, const VD<W>& albedo) {
  const double sin_d = tr.sin_decl, cos_d = tr.cos_decl, tan_d = tr.tan_decl;
  const VD<W> wt = k.omega * th;
  // cos(omega*th) and cos(omega*th + dlon) by angle addition (per-step cos/sin A, per-cell cos/sin B)
  const VD<W> c_wt = vfma(tr.cos_hour, s.get(kSCB), tr.sin_hour * s.get(kSSB));
  const VD<W> c_u = vfma(tr.cos_hour, s.get(kSCB2), tr.sin_hour * s.get(kSSB2));
  const VD<W> arg_eq = s.get(kSNegTanEq) * tan_d, arg_h = s.get(kSNegTanLat) * tan_d;
  const double pi = LLIT(pi);
  const VB<W> dark = (c_wt <= arg_h) || (c_u <= arg_eq) || (vabs(wt) >= VD<W>(pi)) || (vabs(wt + s.get(kSDlon)) >= VD<W>(pi));
  VD<W> K_cs(0.0);
  if (all(dark)) return K_cs;                                   // solar_funcs.py:940-941
  const VD<W> cos_lat = s.get(kSCosLat), sin_lat = s.get(kSSinLat);
  const VD<W> cosZ = vfma(cos_lat * cos_d, c_wt, sin_lat * sin_d);    // Zenith_Angle :281-284
  // Optical_Air_Mass :549-568: sin(gamma) = cos Z, gamma = asin(cos Z); a/(gamma+b)^c = a*exp(-c*log(gamma+b))
  const VD<W> t1 = vrelu(cosZ);
  VD<W> elev_rad;
  TFG_EACH elev_rad.v[w] = fm::asin01(t1.v[w]);
  const VD<W> t2 = LLIT(ky_a) * vexp(LLIT(ky_nc) * vlog(vfma(elev_rad, k.rad2deg, LLIT(ky_b))));
  const VD<W> M_opt = vrcp(t1 + t2);
  const VD<W> a_sa = vfnma(LLIT(sa_a1), W_p, LLIT(sa_a0)), b_sa = vfnma(LLIT(sa_b1), W_p, LLIT(sa_b0));   // :608-614
  const VD<W> a_s = vfnma(LLIT(s_a1), W_p, LLIT(s_a0)), b_s = vfnma(LLIT(s_b1), W_p, LLIT(s_b0));         // :649-653
  VD<W> e_tau, e_gam;
  vexp2(vfma(b_sa, M_opt, a_sa), vfma(b_s, M_opt, a_s), e_tau, e_gam);
  const VD<W> tau = vmin(vrelu(e_tau - k.dust), 1.0);
  const VD<W> gam_s = (1.0 - e_gam) + k.dust;
  const double isc_e0 = tr.isc_e0;
  const VD<W> K_h = vrelu(isc_e0 * vfma(cos_d * cos_lat, c_wt, sin_d * sin_lat));                 // :391-412
  const VD<W> K_s = vrelu(isc_e0 * vfma(cos_d * s.get(kSCosEq), c_u, s.get(kSSinEq) * sin_d));    // :866-887
  const VD<W> half_gam = 0.5 * gam_s;
  const VD<W> K_dif = half_gam * K_h;                            // :667
  const VD<W> K_glob = vfma(tau, K_h, K_dif);                    // :634, :683
  const VD<W> K_bs = (half_gam * albedo) * K_glob;               // :711
  K_cs = vfma(tau, K_s, K_dif) + K_bs;                           // :909
  return vsel(dark, 0.0, K_cs);
}

// One update() of W cells (the lean branch of cell_step in tfg_physics.cuh, element-wise).  `window_sum(w, x)` returns
// the snowfall-window sum of cell w after its newest entry x was stored; `mid_step()` issues the next step's loads.
template <int W, bool VOL, class WindowFn, class MidFn>
__device__ __forceinline__ void lean_step(const Consts<double>& k, const TimeRow<double>& tr, const LeanCells<W>& s,
                                          const VD<W>& LC, CellState<double> (&st)[W], const VD<W>& Pp,
                                          const VD<W>& T_air, const VD<W>& P_air, const VD<W>& q, const VD<W>& uz,
                                          WindowFn&& window_sum, MidFn&& mid_step, StepOut<double> (&o)[W], VD<W>& tot_out) {
  using V = VD<W>;
  const double dt = k.dt;
  V h_snow, h_swe, h_ice, h_iwe, Eccs, Ecci, albedo, n;
  TFG_EACH {
    h_snow.v[w] = st[w].h_snow; h_swe.v[w] = st[w].h_swe; h_ice.v[w] = st[w].h_ice; h_iwe.v[w] = st[w].h_iwe;
    Eccs.v[w] = st[w].eccs; Ecci.v[w] = st[w].ecci; albedo.v[w] = st[w].albedo; n.v[w] = st[w].n_days;
  }
  const V T_K = T_air + LLIT(kelvin);
  // ---- update_P_rain :585, update_P_snow :604
  const VB<W> is_snow = T_air <= s.get(kSTrs);
  const V P_rain = vsel(is_snow, 0.0, Pp), P_snow = vsel(is_snow, Pp, 0.0);
  if constexpr (VOL) {  // :567-568, :576, :613-614, :623-624
    const V da = s.get(kSDa);
    s.set(kSVolP, vfma(Pp * da, dt, s.get(kSVolP)));
    s.set(kSPmax, vmax(s.get(kSPmax), Pp));
    s.set(kSVolPR, vfma(P_rain * da, dt, s.get(kSVolPR)));
    s.set(kSVolPS, vfma(P_snow * da, dt, s.get(kSVolPS)));
  }
  // ---- met block: 7 divisions (see the lean branch of cell_step for the algebra), all chains of the W cells abreast
  V rTK, r_q, r_mag;
  vrcp3(T_K, vfma(k.one_m_eps, q, k.eps), T_air + LLIT(mag_b), rTK, r_q, r_mag);
  const V e_air = ((q * P_air) * r_q) * LLIT(c001);                                           // :817
  V e_p0, en, log_term, L;
  vexp2(-((s.get(kSaElev) * k.inv_rstar) * rTK), -((LLIT(mag_a) * T_air) * r_mag), e_p0, en);   // :551-556, :788
  vlog2(e_air * LLIT(inv_dew_a), vmax((k.z - h_snow) * k.inv_z0, LLIT(c001)), log_term, L);     // :892, :670
  const V inv_p0 = e_p0 * k.inv_p0c;
  const V RH = (e_air * en) * LLIT(inv_esat0);                                                // :838
  const V T_dew = (LLIT(dew_c) * log_term) * vrcp(LLIT(dew_b) - log_term);                    // :888-893
  const VB<W> cover = (h_snow > 0.0) || (h_ice > 0.0);
  const V T_surf = vsel(cover, vmin(T_dew, 0.0), T_dew);                                      // :906-911
  const V dT = T_air - T_surf;
  const V top = k.gz * dT;                                                                    // :640-644
  V bot = (uz * uz) * T_K;
  bot = vsel(bot == 0.0, LLIT(c001), bot);
  const VB<W> stable = top > 0.0;
  const V num = vsel(stable, bot, vfnma(10.0, top, bot));
  const V den = vsel(stable, vfma(10.0, top, bot), bot);
  const V uk2 = uz * k.kappa2;
  const V LL = L * L;
  V r_surf, r_aero;
  vrcp2(T_surf + LLIT(mag_b), LL * den, r_surf, r_aero);
  const V Dh = (uk2 * num) * r_aero;                                                          // :670-733
  V e_wp, e_ss;
  vexp2(LLIT(wp_b) * T_dew, (LLIT(mag_a) * T_surf) * r_surf, e_wp, e_ss);
  const V W_p = LLIT(wp_a) * e_wp;                                                            // :919-920
  const V e_sat_surf = (LLIT(esat0) * e_ss) * 10.0;                                           // :784-802
  const V Qh = (k.rho_cp_air * Dh) * dT;                                                      // :744-745
  const V e_surf = RH * e_sat_surf;                                                           // :853
  const V Qe = ((k.rho_lv_air * Dh) * vfnma(RH, e_sat_surf, e_air)) * (k.lhc * inv_p0);       // :931-934
  mid_step();
  // ---- update_julian_day :990-1004 ; True_Solar_Noon solar_funcs.py:1471
  const V solar_noon = (LLIT(c12) + LC) + tr.TE;
  const V th = tr.clock_hour - solar_noon;
  // ---- update_albedo("aging") :1023-1059
  const V r = vsel(T_air > 0.0, LLIT(alb_r1), LLIT(alb_r0));
  const V ring_new = xmul(xmul(P_snow, dt), k.ws_ratio);                                      // :1031-1033
  V tot;
  TFG_EACH tot.v[w] = window_sum(w, ring_new.v[w]);                                           // :1027-1037
  tot_out = tot;
  n = vsel(tot < LLIT(snow_thr), n + k.days_per_dt, 0.0);                                     // :1040-1041 (finite tot)
  const VB<W> snowy = h_snow > 0.0;
  if (any(snowy)) albedo = vsel(snowy, vfma(LLIT(alb_k), vexp((-n) * r), LLIT(alb_0)), albedo);   // :1042-1048
  albedo = vsel((h_snow == 0.0) && (h_ice > 0.0), LLIT(alb_ice), albedo);                     // :1049-1053
  albedo = vsel((h_snow == 0.0) && (h_ice == 0.0), LLIT(alb_bare), albedo);                   // :1054-1058
  // ---- update_net_shortwave_radiation :1122-1139
  const V K_cs = lean_clear_sky<W>(k, tr, s, th, W_p, albedo);
  const V Qn_SW = K_cs * (1.0 - albedo);
  // ---- update_em_air :1167-1180 (Brutsaert), update_net_longwave_radiation :1231-1248
  const V x7 = (e_air * LLIT(c01)) * rTK;
  V root;
  TFG_EACH root.v[w] = fm::root7(x7.v[w]);
  const V em_air = vfma(k.emis_a * root, k.emis_b, k.canopy);
  const V T_surf_K = T_surf + LLIT(kelvin);
  const V tk2 = T_K * T_K, ts2 = T_surf_K * T_surf_K;
  const V LW_in = (em_air * k.sigma) * (tk2 * tk2);
  V LW_out = k.es_sigma * (ts2 * ts2);
  LW_out = vfma(k.one_m_es, LW_in, LW_out);
  const V Qn_LW = LW_in - LW_out;
  // ---- update_net_energy_flux :1314 (Qa = Qc = 0)
  const V Q_sum = ((Qn_SW + Qn_LW) + Qh) + Qe;
  // ---- snow: update_snow_meltrate :1364-1368, enforce_max_snow_meltrate :1465
  const V previous_swe = h_swe;                                                               // :1571
  const V E_in = Q_sum * dt;
  V SM = (vrelu(E_in - Eccs) * k.inv_dt) * k.inv_rho_lf;
  if constexpr (VOL) s.set(kSVolSM, vfma((SM * s.get(kSDa)) * dt, LLIT(c3600), s.get(kSVolSM)));   // :1486-1487
  // ---- update_swe :1594-1606 (single-rounding operations: decides whether SWE reaches exactly 0)
  const double k3600 = LLIT(c3600);
  h_swe = xadd(h_swe, xmul(P_snow, dt));
  SM = vdiv3600(vmin(xmul(SM, k3600), h_swe));
  h_swe = vrelu(xsub(h_swe, xmul(xmul(SM, dt), k3600)));
  // ---- update_snowfall_cold_content :1507-1537 (T_wb only where P_snow > 0: entered once per thread per needing cell)
  const VB<W> snowing = P_snow > 0.0;
  if (any(snowing)) {
    V T_wb(0.0);
    TFG_EACH {
      if (snowing.v[w]) {
        const double rh = RH.v[w], ta = T_air.v[w];
        if (rh >= 0.0 && rh <= 2.0) {
          T_wb.v[w] = fm::stull_wet_bulb(ta, rh);
        } else {
          using R = Num<FastF64>;
          const R T(ta), H(rh);
          T_wb.v[w] = (((((T * natan(R(LLIT(st_a)) * nsqrt(H + R(LLIT(st_b))))) + natan(T + H)) - natan(H - R(LLIT(st_c)))) +
                        ((R(LLIT(st_d)) * npow15(H)) * natan(R(LLIT(st_e)) * H))) - R(LLIT(st_f))).v;
        }
      }
    }
    const V new_h_snow = (P_snow * dt) * k.ws_ratio;
    const V del_T = k.T0 - T_wb;
    Eccs = vsel(snowing, vrelu(vfma(k.rho_cp_snow * new_h_snow, del_T, Eccs) - E_in), Eccs);
  }
  // ---- update_ice_meltrate :1418-1428 (NEW h_swe, OLD h_ice)
  V IM = (vrelu(E_in - Ecci) * k.inv_dt) * k.inv_rho_lf;
  IM = vsel((h_swe == 0.0) && (previous_swe == 0.0), IM, 0.0);
  Ecci = vrelu(Ecci - E_in);
  Ecci = vsel(h_ice == 0.0, 0.0, Ecci);
  IM = vmin(IM, h_iwe * k.inv_dt);                                                            // :1473-1480
  if constexpr (VOL) s.set(kSVolIM, vfma((IM * s.get(kSDa)) * dt, LLIT(c3600), s.get(kSVolIM)));   // :1493-1494
  // ---- update_iwe :1612-1617
  IM = vdiv3600(vmin(xmul(IM, k3600), h_iwe));
  h_iwe = vrelu(xsub(h_iwe, xmul(xmul(IM, dt), k3600)));
  // ---- update_combined_meltrate :1441-1445
  const V M_total = vfma(P_rain, 1.0 / 3600.0, IM + SM);
  // ---- update_snow_depth :1711, update_ice_depth :1726
  h_snow = xmul(h_swe, k.ws_ratio);
  h_ice = xmul(h_iwe, k.wi_ratio);
  // ---- update_snowpack_cold_content :1552-1558
  Eccs = vsel(P_snow <= 0.0, vrelu(Eccs - E_in), Eccs);
  Eccs = vsel(h_snow == 0.0, 0.0, Eccs);

  TFG_EACH {
    st[w].h_snow = h_snow.v[w]; st[w].h_swe = h_swe.v[w]; st[w].h_ice = h_ice.v[w]; st[w].h_iwe = h_iwe.v[w];
    st[w].eccs = Eccs.v[w]; st[w].ecci = Ecci.v[w]; st[w].albedo = albedo.v[w]; st[w].n_days = n.v[w];
    o[w].SM = SM.v[w]; o[w].IM = IM.v[w]; o[w].M_total = M_total.v[w]; o[w].RH = RH.v[w];
    // intermediates: only read by the recording instantiation (dead code otherwise)
    o[w].p0 = fm::div_fast(1.0, inv_p0.v[w]); o[w].Ri = fm::div_fast(top.v[w], bot.v[w]); o[w].Dn = fm::div_fast(uk2.v[w], LL.v[w]);
    o[w].e_sat_air = fm::div_fast(LLIT(esat10), en.v[w]);
    o[w].e_air = e_air.v[w]; o[w].T_dew = T_dew.v[w]; o[w].T_surf = T_surf.v[w]; o[w].e_sat_surf = e_sat_surf.v[w];
    o[w].Dh = Dh.v[w]; o[w].Qh = Qh.v[w]; o[w].W_p = W_p.v[w]; o[w].e_surf = e_surf.v[w]; o[w].Qe = Qe.v[w];
    o[w].th = th.v[w]; o[w].Qn_SW = Qn_SW.v[w]; o[w].em_air = em_air.v[w]; o[w].Qn_LW = Qn_LW.v[w];
    o[w].Q_sum = Q_sum.v[w]; o[w].P_rain = P_rain.v[w]; o[w].P_snow = P_snow.v[w];
  }
}

// 64-bit / 128-bit access to a pair of consecutive cells
template <bool VEC> __device__ __forceinline__ void ld_pair(const double* a, int64_t g0, const int64_t (&c)[2], bool pair, double (&x)[2]) {
  if (VEC && pair) { const double2 t = *reinterpret_cast<const double2*>(a + g0); x[0] = t.x; x[1] = t.y; }
  else { x[0] = a[c[0]]; x[1] = a[c[1]]; }
}
template <bool VEC> __device__ __forceinline__ void ldg_pair(const double* a, int64_t g0, const int64_t (&c)[2], bool pair, double (&x)[2]) {
  if (VEC && pair) { const double2 t = __ldg(reinterpret_cast<const double2*>(a + g0)); x[0] = t.x; x[1] = t.y; }
  else { x[0] = __ldg(a + c[0]); x[1] = __ldg(a + c[1]); }
}
template <bool VEC> __device__ __forceinline__ void st_pair(double* a, int64_t g0, const bool (&act)[2], bool pair, double x0, double x1) {
  if (VEC && pair) { *reinterpret_cast<double2*>(a + g0) = make_double2(x0, x1); }
  else { if (act[0]) a[g0] = x0; if (act[1]) a[g0 + 1] = x1; }
}

template <bool REC, bool AGG, bool VOL, bool VEC>
__global__ void __launch_bounds__(kLeanBlock, TFG_LEAN_MIN_BLOCKS) run_kernel_lean(const __grid_constant__ RunParams<double> p) {
  static_assert(kW == 2, "the pair loads / stores below are written for two cells per thread");
  constexpr int W = kW;
  using V = VD<W>;
  const int64_t N = p.n_cells;
  const int64_t g0 = ((int64_t)blockIdx.x * kLeanBlock + threadIdx.x) * W;  // first cell of this thread
  bool active[W];
  int64_t c[W];
  TFG_EACH { active[w] = g0 + w < N; c[w] = active[w] ? g0 + w : N - 1; }
  const bool pair = active[W - 1];  // both cells exist (VEC: N is even, so a thread has both or none)

  for (int i = threadIdx.x; i < fm::kTabDoubles; i += kLeanBlock)   // exp / log lookup tables -> dynamic shared memory
    fm::tfg_tabs[i] = (i < 64) ? fm::kExpTab[i] : fm::kLogTab[(i - 64) >> 1][(i - 64) & 1];
  __syncthreads();
  __shared__ alignas(16) double sm_cell[kSCount][kLeanCells];
  LeanCells<W> s;
  s.base = (unsigned)__cvta_generic_to_shared(&sm_cell[0][threadIdx.x * W]);
  {
    const double* tabs[11] = {p.a_elev, p.sin_lat, p.cos_lat, p.neg_tan_lat, p.sin_eq, p.cos_eq, p.neg_tan_eq, p.dlon, p.t_noon, p.da_m2, p.t_rs};
#pragma unroll
    for (int i = 0; i < 11; ++i) { V x; ldg_pair<VEC>(tabs[i], g0, c, pair, x.v); s.set(kSaElev + i, x); }
    s.set(kSCB, V(0.0)); s.set(kSSB, V(0.0)); s.set(kSCB2, V(0.0)); s.set(kSSB2, V(0.0));
  }
  V lon;
  ldg_pair<VEC>(p.lon, g0, c, pair, lon.v);
  int tz[W];
  TFG_EACH tz[w] = p.tz_idx ? (int)__ldg(p.tz_idx + c[w]) : 0;

  CellState<double> st[W];
  {
    double x[W];
#define TFG_LD(field) ld_pair<VEC>(p.field, g0, c, pair, x); TFG_EACH st[w].field = x[w];
    TFG_LD(h_snow) TFG_LD(h_swe) TFG_LD(h_ice) TFG_LD(h_iwe) TFG_LD(eccs) TFG_LD(ecci) TFG_LD(albedo) TFG_LD(n_days)
#undef TFG_LD
  }
  const bool have_vol = VOL && p.vol_P != nullptr;
  {
    const double* vols[6] = {p.vol_P, p.vol_PR, p.vol_PS, p.vol_SM, p.vol_IM, p.P_max};
#pragma unroll
    for (int i = 0; i < 6; ++i) { V x(0.0); if (have_vol) ld_pair<VEC>(vols[i], g0, c, pair, x.v); s.set(kSVolP + i, x); }
  }

  const int slots = p.ring_slots;
  int slot = (int)(p.step0 % slots);
  const bool exact = p.exact_ring != 0;
  // incremental window sum, re-derived exactly (reference summation order) inside a guard band of the 0.03 m threshold
  // of :1040 -- see tfg_run.cuh; a fixed band of 1e-9 m covers 600 roundings of sums below 1e4 m
  V tot(0.0);
  double n_round = (double)slots + 16.0;
  constexpr double kMaxRoundings = 600.0;
  bool carried = false;
  if (!exact && p.win_carry != nullptr) {
    double n0[W];
    ld_pair<VEC>(p.win_carry + 2 * N, g0, c, pair, n0);
    bool ok = true;
    TFG_EACH ok = ok && (n0[w] + (double)(2 * p.n_steps) <= kMaxRoundings);  // false for the NaN that marks "no valid sum"
    if (ok) {
      ld_pair<VEC>(p.win_carry, g0, c, pair, tot.v);
      n_round = fmax(n0[0], n0[W - 1]);
      carried = true;
    }
  }
  if (!exact && !carried) {
    for (int j = 0; j < slots; ++j) {
      V x;
      ld_pair<VEC>(p.ring + (int64_t)j * N, g0, c, pair, x.v);
      tot = xadd(tot, x);
    }
  }

  int basin[W] = {0, 0};
  bool warp_uniform = false;
  const bool have_agg = AGG && p.basin_agg != nullptr && p.basin_id != nullptr;
  if (have_agg) {
    TFG_EACH basin[w] = __ldg(p.basin_id + c[w]);
    warp_uniform = __all_sync(0xffffffffu, basin[0] == __shfl_sync(0xffffffffu, basin[0], 0) && basin[W - 1] == basin[0]);
  }

  // forcing block [step][var][column]: column = cell, or the cell's entry of the forcing map
  const int64_t FN = p.n_cols;
  const bool mapped = p.forcing_col != nullptr;
  int64_t col[W];
  TFG_EACH col[w] = mapped ? (int64_t)__ldg(p.forcing_col + c[w]) : c[w];
  const bool fvec = VEC && pair && !mapped;      // 128-bit forcing loads (rows are 16-byte aligned: N even, base aligned)
  const double* f = p.forcing;
  auto load_forcing = [&](int step_t, V (&dst)[TFG_N_FORCING]) {
    const double* fn = f + (int64_t)step_t * (TFG_N_FORCING * FN);
    if (fvec) {
#pragma unroll
      for (int v = 0; v < TFG_N_FORCING; ++v) {
        const double2 t = __ldcs(reinterpret_cast<const double2*>(fn + (int64_t)v * FN + g0));
        dst[v].v[0] = t.x; dst[v].v[1] = t.y;
      }
    } else {
#pragma unroll
      for (int v = 0; v < TFG_N_FORCING; ++v) TFG_EACH dst[v].v[w] = __ldcs(fn + (int64_t)v * FN + col[w]);
    }
  };
  V fc[TFG_N_FORCING], fnx[TFG_N_FORCING];
  load_forcing(0, fc);

  V r_old;
  ld_pair<VEC>(p.ring + (int64_t)slot * N, g0, c, pair, r_old.v);
  V LC(0.0);
  double gmt_prev[W];
  TFG_EACH gmt_prev[w] = __longlong_as_double(0x7ff8000000000000ll);  // NaN: the first step always sets the zone

  auto finite = [](double v) { return ((unsigned)__double2hiint(v) & 0x7ff00000u) != 0x7ff00000u; };
  bool statics_sane = true, state_ok = true;
  TFG_EACH {
    state_ok = state_ok && finite(st[w].h_snow) && finite(st[w].h_swe) && finite(st[w].h_ice) && finite(st[w].h_iwe) &&
               finite(st[w].eccs) && finite(st[w].ecci) && finite(st[w].albedo) && finite(st[w].n_days);
    statics_sane = statics_sane && finite(lon.v[w]);
  }
  {
    const V ae = s.get(kSaElev);
    TFG_EACH statics_sane = statics_sane && fabs(ae.v[w]) < 2.0e5;   // |elev| < 700 km
    for (int i = kSSinLat; i <= kSTrs; ++i) { const V x = s.get(i); TFG_EACH statics_sane = statics_sane && finite(x.v[w]); }
  }

  StepOut<double> o[W];
  V tot_now(0.0);
  for (int t = 0; t < p.n_steps; ++t) {
    const TimeRow<double>& row = p.rows[t];
    TFG_EACH {
      const double gmt = p.gmt[t * p.n_tz + tz[w]];
      if (!(gmt == gmt_prev[w])) {  // first step, or DST switch (the offset is piece-wise constant in time)
        gmt_prev[w] = gmt;
        LC.v[w] = ((gmt * 15.0) - lon.v[w]) * (1.0 / 15.0);   // True_Solar_Noon, solar_funcs.py:1466-1468
        const double B = p.k.omega * LC.v[w];
        double sb, cb, sb2, cb2;
        auto e = s.elem(w);
        sincos(B, &sb, &cb); sincos(B - e.get(kSDlon), &sb2, &cb2);
        e.set(kSSB, sb); e.set(kSCB, cb); e.set(kSSB2, sb2); e.set(kSCB2, cb2);
      }
    }
    const bool wrap = (slot + 1 == slots);
    const int slot_next = wrap ? 0 : slot + 1;
    double* ring_cur = p.ring + (int64_t)slot * N;
    V ring_new_all(0.0);
    bool stored[W] = {false, false};
    // window sum of cell w after its newest entry is in place (np.roll(-1) + write of the newest slot, :1027-1037)
    auto window = [&](int w, double ring_new) -> double {
      ring_new_all.v[w] = ring_new;
      stored[w] = true;
      if (exact || !fvec) { if (active[w]) ring_cur[g0 + w] = ring_new; }
      else if (w == W - 1) *reinterpret_cast<double2*>(ring_cur + g0) = make_double2(ring_new_all.v[0], ring_new);
      double tn;
      if (exact) {
        if (fvec && w < W - 1) ring_cur[g0 + w] = ring_new;   // (unreachable: exact launches store per cell above)
        tn = window_sum_exact<FastF64>(p.ring + c[w], N, slots, slot).v;
      } else {
        tot.v[w] = __dadd_rn(__dsub_rn(tot.v[w], r_old.v[w]), ring_new);
        // magnitude test on the high word: sums >= 1e4 m and NaN / inf of either sign take the exact path every step,
        // so a non-finite entry poisons the sum only while it is inside the window (as the reference's re-summation)
        const bool near = (fabs(tot.v[w] - LLIT(snow_thr)) <= 1e-9) ||
                          (((unsigned)__double2hiint(tot.v[w]) & 0x7fffffffu) >= 0x40c38800u);
        if (near) {
          if (fvec && w < W - 1) ring_cur[g0 + w] = ring_new;   // the exact sum reads this cell's newest slot from memory
          tot.v[w] = window_sum_exact<FastF64>(p.ring + c[w], N, slots, slot).v;
          n_round = 16.0;
        }
        tn = tot.v[w];
      }
      return tn;
    };
    bool prefetched = false;
    auto prefetch = [&]() {  // next step's forcings, issued mid-step
      if (prefetched) return;
      prefetched = true;
#pragma unroll
      for (int v = 0; v < TFG_N_FORCING; ++v) fnx[v] = fc[v];
      if (t + 1 < p.n_steps) load_forcing(t + 1, fnx);
    };
    // The lean math cores assume physically sane arguments.  Bit tests on the high words (no FP64 pipe):
    // P in [0, 10) m/h, |T_air| < 90 degC, P_air in [1e3, 2e5) Pa, q in [1e-7, 0.2), uz = 0 or in [1e-100, 200)
    auto in_range = [](double v, double lo, double hi) {
      const unsigned h = (unsigned)__double2hiint(v), l = (unsigned)__double2hiint(lo), u = (unsigned)__double2hiint(hi);
      return (h - l) < (u - l);
    };
    bool sane = statics_sane && state_ok;
    TFG_EACH {
      sane = sane && ((unsigned)__double2hiint(fc[0].v[w]) < (unsigned)__double2hiint(10.0)) &&
             (((unsigned)__double2hiint(fc[1].v[w]) & 0x7fffffffu) < (unsigned)__double2hiint(90.0)) &&
             in_range(fc[2].v[w], 1e3, 2e5) && in_range(fc[3].v[w], 1e-7, 0.2) &&
             (in_range(fc[4].v[w], 1e-100, 200.0) || fc[4].v[w] == 0.0);
    }
    if (__all_sync(0xffffffffu, sane) && !p.k.satterlund) {
      lean_step<W, VOL>(p.k, row, s, LC, st, fc[0], fc[1], fc[2], fc[3], fc[4], window, prefetch, o, tot_now);
    } else {
      // Same step in the strict arithmetic (libdevice, IEEE division, NumPy's NaN rules): whatever the input -- missing
      // data, absurd values, SATTERLUND configurations -- the cells behave like the reference, NaN poisoning included.
      using S = Num<StrictF64>;
      TFG_EACH {
        auto cell = s.elem(w);
        const S LCs = ((S(gmt_prev[w]) * 15.0) - S(lon.v[w])) / 15.0;
        auto win_w = [&](double x) { const double tn = window(w, x); tot_now.v[w] = tn; return tn; };
        cell_step<StrictF64, VOL>(p.k, row, cell, LCs, st[w], S(fc[0].v[w]), S(fc[1].v[w]), S(fc[2].v[w]), S(fc[3].v[w]),
                                  S(fc[4].v[w]), win_w, prefetch, o[w]);
      }
      state_ok = true;
      TFG_EACH state_ok = state_ok && finite(st[w].h_snow) && finite(st[w].h_swe) && finite(st[w].h_ice) &&
                          finite(st[w].h_iwe) && finite(st[w].eccs) && finite(st[w].ecci) && finite(st[w].albedo) &&
                          finite(st[w].n_days);
    }
    if (!exact) n_round += 2.0;
    // next step's oldest window entry (after this step's store)
    ld_pair<VEC>(p.ring + (int64_t)slot_next * N, g0, c, pair, r_old.v);

    if constexpr (REC) {
      if (p.record != nullptr) {
        TFG_EACH {
          if (!active[w]) continue;
          double* rp = p.record + ((int64_t)t * p.n_rec) * N + c[w];
          const uint64_t m = p.record_mask;
          int r = 0;
#define TFG_PUT(bit, val)              \
  if ((m >> (bit)) & 1ull) {           \
    rp[(int64_t)r * N] = (val);        \
    ++r;                               \
  }
          TFG_PUT(TFG_REC_H_SNOW, st[w].h_snow) TFG_PUT(TFG_REC_H_SWE, st[w].h_swe) TFG_PUT(TFG_REC_SM, o[w].SM)
          TFG_PUT(TFG_REC_H_ICE, st[w].h_ice) TFG_PUT(TFG_REC_H_IWE, st[w].h_iwe) TFG_PUT(TFG_REC_IM, o[w].IM)
          TFG_PUT(TFG_REC_M_TOTAL, o[w].M_total) TFG_PUT(TFG_REC_RH, o[w].RH) TFG_PUT(TFG_REC_P0, o[w].p0)
          TFG_PUT(TFG_REC_E_SAT_AIR, o[w].e_sat_air) TFG_PUT(TFG_REC_E_AIR, o[w].e_air) TFG_PUT(TFG_REC_T_DEW, o[w].T_dew)
          TFG_PUT(TFG_REC_T_SURF, o[w].T_surf) TFG_PUT(TFG_REC_E_SAT_SURF, o[w].e_sat_surf) TFG_PUT(TFG_REC_RI, o[w].Ri)
          TFG_PUT(TFG_REC_DN, o[w].Dn) TFG_PUT(TFG_REC_DH, o[w].Dh) TFG_PUT(TFG_REC_QH, o[w].Qh) TFG_PUT(TFG_REC_W_P, o[w].W_p)
          TFG_PUT(TFG_REC_E_SURF, o[w].e_surf) TFG_PUT(TFG_REC_QE, o[w].Qe) TFG_PUT(TFG_REC_TSN_OFFSET, o[w].th)
          TFG_PUT(TFG_REC_ALBEDO, st[w].albedo) TFG_PUT(TFG_REC_N_DAYS, st[w].n_days) TFG_PUT(TFG_REC_QN_SW, o[w].Qn_SW)
          TFG_PUT(TFG_REC_EM_AIR, o[w].em_air) TFG_PUT(TFG_REC_QN_LW, o[w].Qn_LW) TFG_PUT(TFG_REC_Q_SUM, o[w].Q_sum)
          TFG_PUT(TFG_REC_ECCS, st[w].eccs) TFG_PUT(TFG_REC_ECCI, st[w].ecci) TFG_PUT(TFG_REC_SNOW3DAY, tot_now.v[w])
          TFG_PUT(TFG_REC_P_RAIN, o[w].P_rain) TFG_PUT(TFG_REC_P_SNOW, o[w].P_snow)
#undef TFG_PUT
        }
      }
    }
    if constexpr (AGG) {
      if (have_agg) {
        // area-weighted basin sums (np.sum sites :567-568,:1486-1494 and the driver's `* da_m2`): the two cells of a
        // thread first, then a warp-shuffle tree when the 64 cells of the warp sit inside one basin, one RED per warp
        // and quantity; per-cell atomics for warps that straddle basins
        const V da = s.get(kSDa);
        double v0[W], v1[W], v2[W];
        TFG_EACH {
          v0[w] = active[w] ? o[w].M_total * da.v[w] : 0.0;
          v1[w] = active[w] ? st[w].h_swe * da.v[w] : 0.0;
          v2[w] = active[w] ? st[w].h_iwe * da.v[w] : 0.0;
        }
        if (warp_uniform) {
          const double a0 = v0[0] + v0[1], a1 = v1[0] + v1[1], a2 = v2[0] + v2[1];
          const int64_t entry = ((int64_t)t * p.n_basin + basin[0]) * TFG_N_AGG;
          double* dst = static_cast<double*>(p.basin_agg) + entry;
          long long* acc = static_cast<long long*>(p.basin_agg) + 2 * entry;
          // three sums in one butterfly (lanes 0-7: a0, 8-15: a1, 16-23: a2): 6 shuffles instead of 15
          const unsigned full = 0xffffffffu;
          const int lane = threadIdx.x & 31;
          const bool hi = (lane & 16) != 0;
          double k0 = hi ? a2 : a0, k1 = hi ? 0.0 : a1;
          k0 += __shfl_xor_sync(full, hi ? a0 : a2, 16);
          k1 += __shfl_xor_sync(full, hi ? a1 : 0.0, 16);
          const bool hi2 = (lane & 8) != 0;
          double kk = hi2 ? k1 : k0;
          kk += __shfl_xor_sync(full, hi2 ? k0 : k1, 8);
          kk += __shfl_xor_sync(full, kk, 4);
          kk += __shfl_xor_sync(full, kk, 2);
          kk += __shfl_xor_sync(full, kk, 1);
          if ((lane & 7) == 0 && lane < 24) {
            if (p.agg_exact) agg_add_exact(acc + 2 * (lane >> 3), kk, p.agg_up[lane >> 3], p.agg_lo, p.agg_bad);
            else atomicAdd(dst + (lane >> 3), kk);
          }
        } else {
          TFG_EACH {
            if (!active[w]) continue;
            const int64_t entry = ((int64_t)t * p.n_basin + basin[w]) * TFG_N_AGG;
            double* dst = static_cast<double*>(p.basin_agg) + entry;
            long long* acc = static_cast<long long*>(p.basin_agg) + 2 * entry;
            if (p.agg_exact) {
              agg_add_exact(acc + 0, v0[w], p.agg_up[0], p.agg_lo, p.agg_bad); agg_add_exact(acc + 2, v1[w], p.agg_up[1], p.agg_lo, p.agg_bad);
              agg_add_exact(acc + 4, v2[w], p.agg_up[2], p.agg_lo, p.agg_bad);
            } else {
              atomicAdd(dst + 0, v0[w]); atomicAdd(dst + 1, v1[w]); atomicAdd(dst + 2, v2[w]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int v = 0; v < TFG_N_FORCING; ++v) fc[v] = fnx[v];
    slot = slot_next;
  }

  if (p.win_carry != nullptr) {
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    // exact launches move the window without the running sum: re-seed next time
    st_pair<VEC>(p.win_carry + 2 * N, g0, active, pair, exact ? nanv : n_round, exact ? nanv : n_round);
    if (!exact) {
      st_pair<VEC>(p.win_carry, g0, active, pair, tot.v[0], tot.v[1]);
      st_pair<VEC>(p.win_carry + N, g0, active, pair, fabs(tot.v[0]), fabs(tot.v[1]));
    }
  }
#define TFG_ST(field) st_pair<VEC>(p.field, g0, active, pair, st[0].field, st[1].field);
  TFG_ST(h_snow) TFG_ST(h_swe) TFG_ST(h_ice) TFG_ST(h_iwe) TFG_ST(eccs) TFG_ST(ecci) TFG_ST(albedo) TFG_ST(n_days)
#undef TFG_ST
  st_pair<VEC>(p.SM, g0, active, pair, o[0].SM, o[1].SM);
  st_pair<VEC>(p.IM, g0, active, pair, o[0].IM, o[1].IM);
  st_pair<VEC>(p.M_total, g0, active, pair, o[0].M_total, o[1].M_total);
  st_pair<VEC>(p.RH, g0, active, pair, o[0].RH, o[1].RH);
  if (have_vol) {
    double* vols[6] = {p.vol_P, p.vol_PR, p.vol_PS, p.vol_SM, p.vol_IM, p.P_max};
#pragma unroll
    for (int i = 0; i < 6; ++i) { const V x = s.get(kSVolP + i); st_pair<VEC>(vols[i], g0, active, pair, x.v[0], x.v[1]); }
  }
}

inline cudaError_t launch_run_lean(const RunParams<double>& p, bool rec, bool agg, bool vol, cudaStream_t stream) {
  const unsigned grid = (unsigned)((p.n_cells + kLeanCells - 1) / kLeanCells);
  const size_t dyn = fm::kTabDoubles * sizeof(double);
  // 128-bit access needs an even cell count (every row of a [k][N] block then starts 16-byte aligned) and aligned bases
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  bool vec = (p.n_cells % 2 == 0) && al(p.forcing) && al(p.ring) && al(p.h_snow) && al(p.a_elev) && al(p.win_carry) &&
             (p.forcing_col != nullptr || p.n_cols == p.n_cells);
  const void* ptrs[] = {p.sin_lat, p.cos_lat, p.neg_tan_lat, p.lon, p.sin_eq, p.cos_eq, p.neg_tan_eq, p.dlon, p.t_noon, p.da_m2, p.t_rs,
                        p.h_swe, p.h_ice, p.h_iwe, p.eccs, p.ecci, p.albedo, p.n_days, p.SM, p.IM, p.M_total, p.RH,
                        p.vol_P, p.vol_PR, p.vol_PS, p.vol_SM, p.vol_IM, p.P_max};
  for (const void* q : ptrs) vec = vec && al(q);
#define TFG_GO(R, A, L)                                                                          \
  do {                                                                                           \
    if (vec) run_kernel_lean<R, A, L, true><<<grid, kLeanBlock, dyn, stream>>>(p);               \
    else run_kernel_lean<R, A, L, false><<<grid, kLeanBlock, dyn, stream>>>(p);                  \
  } while (0)
  if (rec) TFG_GO(true, true, true);
  else if (agg && vol) TFG_GO(false, true, true);
  else if (agg) TFG_GO(false, true, false);
  else if (vol) TFG_GO(false, false, true);
  else TFG_GO(false, false, false);
#undef TFG_GO
  return cudaGetLastError();
}

}  // namespace tfg
