// tfg_abi.cu -- the extern "C" surface of libtfglacier.so (include/tfglacier.h): context, binding,
// dispatch of the fused melt kernel, forcing ingestion/conversion and the synthetic-forcing generator.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <string>
#include <vector>

#include "tfg_run.cuh"

namespace {

thread_local std::string g_err;

int fail(const char* what, cudaError_t e = cudaSuccess) {
  g_err = what;
  if (e != cudaSuccess) {
    g_err += ": ";
    g_err += cudaGetErrorString(e);
  }
  return -1;
}

#define TFG_CUDA(call)                                   \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return fail(#call, e__);     \
  } while (0)

}  // namespace

struct tfg_ctx {
  int device = 0;
  int mode = TFG_F64_STRICT;
  bool have_consts = false, have_static = false, have_state = false;
  tfg_constants c{};
  tfg_statics s{};
  tfg_state st{};
  int64_t n_cells = 0;
  // host copies of the clock-only tables (owned by the library); each launch carries its rows as kernel parameters
  std::vector<double> h_rows, h_gmt;
  int64_t n_time = 0;
  int n_tz = 1;
  int use_tma = 0;  // forcing tiles staged by the TMA copy engine (tfg_set_option)
  int64_t exact_agg = 0;  // TFG_OPT_EXACT_AGG value (0 = floating-point atomics)
  const int32_t* forcing_col = nullptr;  // tfg_bind_forcing_map
  void* win_carry = nullptr;             // tfg_bind_window_carry
  void* mass_lo = nullptr;               // tfg_bind_mass_residual
  int64_t n_cols = 0;
  int column_terms = 1;                  // TFG_OPT_COLUMN_TERMS
  double* col_terms = nullptr;           // [<= kMaxLaunchSteps][n_cols][16] scratch of the column-term pass (owned)
  size_t col_terms_bytes = 0;
  int64_t col_term_launches = 0;         // launches that went through the column-term pass (tfg_column_term_launches)
  void* cell_par = nullptr;              // [tfg::kPCount][n_cells] per-cell surface factors, context element type (owned)
  size_t cell_par_bytes = 0;
  int* cell_par_bad = nullptr;           // device flags of tfg_bind_cell_params' range check (owned)
  bool have_cell_par = false;            // tfg_bind_cell_params: the scratch holds this context's factors
  tfg_objective obj{};                   // tfg_bind_objective (caller's arrays)
  bool have_obj = false;
  int* obj_bad = nullptr;                // device flag of tfg_bind_objective's range check of obs_col (owned)
  void* fadj = nullptr;                  // [2][n_cells] T_air offset and P multiplier, context element type (owned)
  size_t fadj_bytes = 0;
  int* fadj_bad = nullptr;               // device flags of tfg_bind_forcing_adjust's range check (owned)
  bool have_fadj = false;                // tfg_bind_forcing_adjust: the scratch holds this context's adjustments
  // forcing noise (tfg_bind_forcing_noise)
  tfg_forcing_noise noise{};             // host fields; the arrays are the library's copies below
  bool have_noise = false;
  double noise_c[2] = {0.0, 0.0};        // sqrt(1 - rho^2) of T_air and P, formed once here
  int64_t* noise_ids = nullptr;          // [n_streams] global stream ids (owned)
  int32_t* noise_cell = nullptr;         // [n_cells] stream index of each cell (owned)
  double* noise_z = nullptr;             // [2][n_streams] z_T, z_P of step noise_next - 1 (owned)
  int64_t noise_streams_cap = 0, noise_cells_cap = 0;
  int64_t noise_next = -1;               // step whose z the cache continues to; -1: regenerate from step0
  void* noise_buf = nullptr;             // [<= kMaxLaunchSteps][2][n_streams] dT, fP of a launch, element type (owned)
  size_t noise_buf_bytes = 0;
  int* noise_bad = nullptr;              // device flags of tfg_bind_forcing_noise's checks (owned)
};

namespace {

// Single-rounding operations on the host and on the device alike (the device compiler would otherwise contract
// a*b + c into one FMA, and a per-cell factor would then differ from the constant the host derived).
__host__ __device__ inline double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
__host__ __device__ inline double add_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
__host__ __device__ inline double div_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}

// The factors the five surface parameters enter the kernels through, in the rows of tfg::kP*.  derive() forms them from
// the context constants, cell_params_kernel from per-cell arrays: one statement of them keeps the two bit-identical.
__host__ __device__ inline void surface_factors(double dust, double canopy, double cloud, double z0, double em_surf,
                                                double sigma, double out[tfg::kPCount]) {
  out[tfg::kPDust] = dust;
  out[tfg::kPEmisA] = mul_rn(add_rn(1.0, -canopy), 1.72);                 // (1 - F) * 1.72 (:1179)
  out[tfg::kPEmisB] = add_rn(1.0, mul_rn(0.22, mul_rn(cloud, cloud)));   // 1 + 0.22 * C**2 (:1180)
  out[tfg::kPCanopy] = canopy;
  out[tfg::kPEsSigma] = mul_rn(em_surf, sigma);                          // em_surf * sigma (:1236)
  out[tfg::kPOneMEs] = add_rn(1.0, -em_surf);                            // 1 - em_surf (:1246)
  out[tfg::kPZ0] = z0;
  out[tfg::kPInvZ0] = div_rn(1.0, z0);
}

template <class raw>
tfg::Consts<raw> derive(const tfg_constants& c) {
  // every product / ratio is formed exactly as the reference forms it (file:line in tfg_physics.cuh)
  tfg::Consts<double> k;
  k.dt = c.dt_hours;
  k.days_per_dt = c.dt_hours / 86400.0;
  k.T0 = c.T0;
  k.sea_p0 = c.sea_level_p0;
  k.r_star = c.uni_gas_const;
  k.eps = c.eps;
  k.one_m_eps = 1.0 - c.eps;
  k.gz = c.g * c.z_wind;
  k.z = c.z_wind;
  k.z0_air = c.z0_air;
  k.kappa = c.kappa;
  k.rho_cp_air = c.rho_air * c.Cp_air;
  k.rho_lv_air = c.rho_air * c.Lv;
  k.lhc = c.latent_heat_constant;
  k.ws_ratio = c.rho_H2O / c.rho_snow;
  k.wi_ratio = c.rho_H2O / c.rho_ice;
  k.rho_cp_snow = c.rho_snow * c.Cp_snow;
  k.rho_lf = c.rho_H2O * c.Lf;
  double sf[tfg::kPCount];
  surface_factors(c.dust_atten, c.canopy_factor, c.cloud_factor, c.z0_air, c.em_surf, c.sigma, sf);
  k.dust = sf[tfg::kPDust];
  k.emis_a = sf[tfg::kPEmisA];
  k.emis_b = sf[tfg::kPEmisB];
  k.canopy = sf[tfg::kPCanopy];
  k.sigma = c.sigma;
  k.es_sigma = sf[tfg::kPEsSigma];
  k.one_m_es = sf[tfg::kPOneMEs];
  k.one_seventh = 1.0 / 7.0;
  const double pi = 3.141592653589793;
  k.omega = (360.0 / 24.0) * (pi / 180.0);
  k.rad2deg = 180.0 / pi;
  k.deg2rad = pi / 180.0;
  k.inv_z0 = sf[tfg::kPInvZ0];
  k.inv_dt = 1.0 / c.dt_hours;
  k.inv_rho_lf = 1.0 / k.rho_lf;
  k.inv_rstar = 1.0 / c.uni_gas_const;
  k.inv_p0c = 1.0 / (c.sea_level_p0 * 0.01);
  k.kappa2 = c.kappa * c.kappa;
  k.cq0 = (k.rho_lv_air * k.lhc) * k.inv_p0c;
  k.satterlund = c.satterlund;
  tfg::Consts<raw> r;
#define CP(f) r.f = static_cast<raw>(k.f)
  CP(dt); CP(days_per_dt); CP(T0); CP(sea_p0); CP(r_star); CP(eps); CP(one_m_eps); CP(gz); CP(z); CP(z0_air);
  CP(kappa); CP(rho_cp_air); CP(rho_lv_air); CP(lhc); CP(ws_ratio); CP(wi_ratio); CP(rho_cp_snow); CP(rho_lf);
  CP(dust); CP(emis_a); CP(emis_b); CP(canopy); CP(sigma); CP(es_sigma); CP(one_m_es); CP(one_seventh); CP(omega);
  CP(rad2deg); CP(deg2rad); CP(inv_z0); CP(inv_dt); CP(inv_rho_lf); CP(inv_rstar); CP(inv_p0c); CP(kappa2); CP(cq0);
#undef CP
  r.satterlund = k.satterlund;
  return r;
}

template <class raw>
tfg::RunParams<raw> make_params(const tfg_ctx* x, const void* forcing, int64_t step0, int32_t n_steps, void* record,
                                uint64_t mask, void* agg, int32_t n_basin, long long* agg_bad) {
  tfg::RunParams<raw> p{};
  p.n_cells = x->n_cells;
  p.step0 = step0;
  p.n_steps = n_steps;
  p.ring_slots = x->c.ring_slots;
  p.n_tz = x->n_tz;
  p.exact_ring = (n_steps == 1);
  p.use_tma = x->use_tma;
  p.forcing = static_cast<const raw*>(forcing);
  p.forcing_col = x->forcing_col;
  p.win_carry = static_cast<raw*>(x->win_carry);
  p.mass_lo = static_cast<raw*>(x->mass_lo);
  p.n_cols = x->forcing_col ? x->n_cols : x->n_cells;
#define S(f) p.f = static_cast<const raw*>(x->s.f)
  S(a_elev); S(sin_lat); S(cos_lat); S(neg_tan_lat); S(lon); S(dlon); S(t_noon); S(da_m2);
#undef S
  p.sin_eq = static_cast<const raw*>(x->s.sin_lat_eq);
  p.cos_eq = static_cast<const raw*>(x->s.cos_lat_eq);
  p.neg_tan_eq = static_cast<const raw*>(x->s.neg_tan_lat_eq);
  p.t_rs = static_cast<const raw*>(x->s.t_rain_snow);
  p.basin_id = x->s.basin_id;
  p.tz_idx = x->s.tz_idx;
#define T(f) p.f = static_cast<raw*>(x->st.f)
  T(h_snow); T(h_swe); T(h_ice); T(h_iwe); T(eccs); T(ecci); T(albedo); T(n_days); T(SM); T(IM); T(M_total); T(RH);
  T(vol_P); T(vol_PR); T(vol_PS); T(vol_SM); T(vol_IM); T(P_max); T(ring);
#undef T
  for (int32_t t = 0; t < n_steps; ++t) {
    const double* r = &x->h_rows[(size_t)(step0 + t) * 8];
    p.rows[t] = tfg::TimeRow<raw>{(raw)r[0], (raw)r[1], (raw)r[2], (raw)r[3], (raw)r[4], (raw)r[5], (raw)r[6], (raw)r[7]};
    for (int z = 0; z < x->n_tz; ++z) p.gmt[t * x->n_tz + z] = (raw)x->h_gmt[(size_t)(step0 + t) * x->n_tz + z];
  }
  p.gmt_varies = 0;
  for (int32_t t = 1; t < n_steps && !p.gmt_varies; ++t)
    for (int z = 0; z < x->n_tz; ++z)
      if (!(p.gmt[t * x->n_tz + z] == p.gmt[z])) p.gmt_varies = 1;   // also true for NaN offsets
  p.record = static_cast<raw*>(record);
  p.record_mask = mask;
  p.n_rec = __builtin_popcountll(mask);
  p.basin_agg = agg;
  p.agg_exact = x->exact_agg != 0;
  p.agg_bad = agg_bad;
  for (int q = 0; q < TFG_N_AGG; ++q)  // 2^(40 - E_q): scales a partial sum into the hi fixed-point word
    p.agg_up[q] = ldexp(1.0, 40 - ((int)((x->exact_agg >> (8 * q)) & 0xff) - 128));
  const int lo_bits = (int)((x->exact_agg >> 32) & 0xff);  // L, the low word's fraction bits; 0 = 42
  p.agg_lo = ldexp(1.0, lo_bits ? lo_bits : 42);
  p.n_basin = n_basin;
  p.k = derive<raw>(x->c);
  p.cell_par = x->have_cell_par ? static_cast<const raw*>(x->cell_par) : nullptr;
  p.fadj = x->have_fadj ? static_cast<const raw*>(x->fadj) : nullptr;
  // objective: the scored part of [step0, step0 + n_steps) is its intersection with the observation window; a launch
  // outside the window leaves obj_acc NULL and runs the kernels without an objective
  if (x->have_obj) {
    const tfg_objective& o = x->obj;
    const int64_t lo = std::max<int64_t>(step0, o.obs_step0), hi = std::min<int64_t>(step0 + n_steps, o.obs_step0 + o.n_obs_steps);
    if (lo < hi) {
      p.obj_acc = o.acc;
      p.obj_obs = o.obs + (lo - o.obs_step0) * o.n_obs_cols;
      p.obj_col = o.obs_col;
      p.obj_ncols = o.n_obs_cols;
      p.obj_t_lo = (int32_t)(lo - step0);
      p.obj_t_hi = (int32_t)(hi - step0);
      p.obj_quantity = o.quantity;
    }
  }
  return p;
}

// ---- per-cell surface parameters (tfg_bind_cell_params) -----------------------------------------------------------
// Ranges of the configuration schema (topoflow_glacier_b200/config.py); bit i of *bad = parameter i out of range.
__global__ void cell_params_kernel(const tfg_cell_params in, const tfg_constants c, void* out, bool f32, int64_t N, int* bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double* src[5] = {in.dust_atten, in.canopy_factor, in.cloud_factor, in.z0_air, in.em_surf};
  const double dflt[5] = {c.dust_atten, c.canopy_factor, c.cloud_factor, c.z0_air, c.em_surf};
  const double lo[5] = {0.0, 0.0, 0.0, 1e-4, 0.9}, hi[5] = {0.2, 1.0, 1.0, 0.1, 1.0};
  double v[5];
  int flags = 0;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    v[j] = src[j] ? src[j][i] : dflt[j];
    if (src[j] && !(v[j] >= lo[j] && v[j] <= hi[j])) flags |= 1 << j;   // NaN and +-inf fail too
  }
  if (flags) atomicOr(bad, flags);
  double f[tfg::kPCount];
  surface_factors(v[0], v[1], v[2], v[3], v[4], c.sigma, f);
#pragma unroll
  for (int r = 0; r < tfg::kPCount; ++r) {
    if (f32) static_cast<float*>(out)[r * N + i] = (float)f[r];
    else static_cast<double*>(out)[r * N + i] = f[r];
  }
}

// ---- forcing adjustments (tfg_bind_forcing_adjust): range check, then one rounding to the element type ------------
// bit 0 of *bad: T_air_offset outside [-30, 30] K or not finite; bit 1: P_multiplier outside [0, 10] or not finite
__global__ void forcing_adjust_kernel(const tfg_forcing_adjust in, void* out, bool f32, int64_t N, int* bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double off = in.T_air_offset ? in.T_air_offset[i] : 0.0, mul = in.P_multiplier ? in.P_multiplier[i] : 1.0;
  const int flags = (!(off >= -30.0 && off <= 30.0) ? 1 : 0) | (!(mul >= 0.0 && mul <= 10.0) ? 2 : 0);  // NaN fails too
  if (flags) atomicOr(bad, flags);
  if (f32) { static_cast<float*>(out)[i] = (float)off; static_cast<float*>(out)[N + i] = (float)mul; }
  else { static_cast<double*>(out)[i] = off; static_cast<double*>(out)[N + i] = mul; }
}

// ---- objective (tfg_bind_objective): *bad = 1 if an observation column index is outside [0, n_cols) -------------
__global__ void obs_col_check_kernel(const int32_t* col, int64_t N, int64_t n_cols, int* bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N && !(col[i] >= 0 && (int64_t)col[i] < n_cols)) atomicOr(bad, 1);
}

// ---- K2: raw met columns -> live forcings (examples/run_topoflow_glacier.py:40-73) -------------------
template <class src_t, class raw>
__global__ void convert_kernel(const src_t* __restrict__ in, raw* __restrict__ out, int64_t n_steps, int64_t N) {
  const int64_t total = n_steps * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / N, c = i - t * N;
    const src_t* r = in + t * 6 * N + c;
    // float32 sources (AORC / NWM style met data) widen exactly; arithmetic is float64 as in the driver
    const double rain = (double)__ldcs(r), t2d = (double)__ldcs(r + N), psfc = (double)__ldcs(r + 2 * N),
                 q2d = (double)__ldcs(r + 3 * N), u = (double)__ldcs(r + 4 * N), v = (double)__ldcs(r + 5 * N);
    raw* o = out + t * TFG_N_FORCING * N + c;
    o[0] = (raw)__dmul_rn(rain, 0.001);                         // precip * 10**(-3)
    o[N] = (raw)__dadd_rn(-273.15, t2d);                        // K_to_C + T2D
    o[2 * N] = (raw)psfc;
    o[3 * N] = (raw)q2d;
    o[4 * N] = (raw)__dsqrt_rn(__dadd_rn(__dmul_rn(u, u), __dmul_rn(v, v)));  // (U**2 + V**2) ** 0.5
  }
}

struct PackScale { double scale[6], offset[6]; };
template <class raw>
__global__ void convert_packed_kernel(const int16_t* __restrict__ in, raw* __restrict__ out, int64_t n_steps, int64_t N,
                                      const PackScale ps) {
  const int64_t total = n_steps * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / N, c = i - t * N;
    const int16_t* r = in + t * 6 * N + c;
    double v[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) v[j] = __dadd_rn(__dmul_rn((double)__ldcs(r + j * N), ps.scale[j]), ps.offset[j]);
    raw* o = out + t * TFG_N_FORCING * N + c;
    o[0] = (raw)__dmul_rn(v[0], 0.001);
    o[N] = (raw)__dadd_rn(-273.15, v[1]);
    o[2 * N] = (raw)v[2];
    o[3 * N] = (raw)v[3];
    o[4 * N] = (raw)__dsqrt_rn(__dadd_rn(__dmul_rn(v[4], v[4]), __dmul_rn(v[5], v[5])));
  }
}

// ---- causal box/FIR filter along time: the "mock routing" of the reference example --------------------------
// out[t][j] = sum_{k < taps} w[k] * in[t-k][j]   (np.convolve(x, w, "full")[:T], examples/run_topoflow_glacier.py:129-131)
__global__ void fir_kernel(const double* __restrict__ in, double* __restrict__ out, const double* __restrict__ w,
                           int taps, int64_t T, int64_t M) {
  const int64_t total = T * M;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / M, j = i - t * M;
    double acc = 0.0;
    for (int k = 0; k < taps && k <= t; ++k) acc = fma(w[k], in[(t - k) * M + j], acc);
    out[i] = acc;
  }
}

// ---- FP64 pipe peak: what the compute roofline of the melt kernel is measured against -------------------------
// 8 independent DFMA chains per thread, 1024 threads per SM-resident wave; reports DFMA warp-instructions / s.
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double seed) {
  double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 12345.678) out[0] = a0;  // keep the chains alive
}

// ---- synthetic forcing (bench only): Philox4x32-10 keyed by (seed, cell, step) ------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

template <class raw>
__global__ void synth_kernel(raw* __restrict__ out, const raw* __restrict__ elev, int64_t step0, int32_t n_steps,
                             int64_t N, uint64_t seed, int64_t storm_cells) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N) return;
  const float lapse = -6.5e-3f * ((float)elev[c] - 2400.0f);
  for (int t = 0; t < n_steps; ++t) {
    const int64_t step = step0 + t;
    uint32_t a[4], b[4];
    philox4x32_10((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)step, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), a);
    philox4x32_10((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)step, 1u, (uint32_t)seed, (uint32_t)(seed >> 32), b);
    if (storm_cells > 1) {  // precipitation occurrence shared by `storm_cells` consecutive cells (a weather system)
      uint32_t w[4];
      const int64_t cw = c / storm_cells;
      philox4x32_10((uint32_t)cw, (uint32_t)(cw >> 32), (uint32_t)step, 2u, (uint32_t)seed, (uint32_t)(seed >> 32), w);
      b[1] = w[1];
    }
    // Box-Muller pairs
    const float r0 = sqrtf(-2.0f * __logf(u01(a[0]))), r1 = sqrtf(-2.0f * __logf(u01(a[2])));
    float s0, c0, s1, c1;
    __sincosf(6.2831853f * u01(a[1]), &s0, &c0);
    __sincosf(6.2831853f * u01(a[3]), &s1, &c1);
    const float nT = r0 * c0, nP = r0 * s0, nU = r1 * c1, nV = r1 * s1;
    const int hour = (int)(step % 24);
    const int doy = (int)((274 + step / 24) % 365);
    const float T2D = 273.15f + 2.0f + 9.0f * __sinf(6.2831853f * (float)(doy - 105) / 365.0f) +
                      4.0f * __sinf(6.2831853f * (float)(hour - 15) / 24.0f) + 2.0f * nT + lapse;
    const float PSFC = 88900.0f + 400.0f * nP;
    const float Tc = T2D - 273.15f;
    const float esat = 611.0f * __expf(17.3f * Tc / (Tc + 237.3f));
    const float qsat = 0.622f * esat / (PSFC - 0.378f * esat);
    const float q = fminf(fmaxf(0.8f * qsat * (0.5f + 0.5f * u01(b[0])), 5e-4f), 0.012f);
    const float rain = (u01(b[1]) < 0.12f) ? -0.5f * __logf(u01(b[2])) : 0.0f;  // mm/h
    raw* o = out + (int64_t)t * TFG_N_FORCING * N + c;
    o[0] = (raw)((double)rain * 0.001);
    o[N] = (raw)((double)T2D - 273.15);
    o[2 * N] = (raw)PSFC;
    o[3 * N] = (raw)q;
    o[4 * N] = (raw)(3.0f * sqrtf(nU * nU + nV * nV));
  }
}

// ---- forcing noise (tfg_bind_forcing_noise) -------------------------------------------------------------------------
constexpr int64_t kNoiseStepLimit = int64_t(1) << 32;   // a step is one 32-bit counter word
constexpr size_t kNoiseScratchCap = size_t(1) << 31;    // 2 GB of [steps][2][n_streams], as the column-term scratch

struct NoiseGen {
  uint64_t seed;
  int64_t s0;
  double sd_T, rho_T, c_T, sd_P, rho_P, c_P, half_var_P;   // c = sqrt(1 - rho^2), half_var_P = sd_P^2 / 2 (host)
};

// The two standard normals of stream id g at absolute step s (include/tfglacier.h states the definition)
__device__ __forceinline__ void noise_normals(uint64_t seed, int64_t g, int64_t s, double& eT, double& eP) {
  uint32_t w[4];
  philox4x32_10((uint32_t)g, (uint32_t)((uint64_t)g >> 32), (uint32_t)s, 0x4E4F4953u, (uint32_t)seed,
                (uint32_t)(seed >> 32), w);
  const uint64_t a = ((uint64_t)w[0] << 21) | (w[1] >> 11), b = ((uint64_t)w[2] << 21) | (w[3] >> 11);
  const double ua = (double)(a + 1) * 0x1p-53, ub = (double)b * 0x1p-53;   // exact: 53-bit integers
  const double r = sqrt(__dmul_rn(-2.0, log(ua)));
  double sp, cp;
  sincospi(__dmul_rn(2.0, ub), &sp, &cp);
  eT = __dmul_rn(r, cp);
  eP = __dmul_rn(r, sp);
}

// One thread per stream walks absolute steps [from, step0 + n_steps) and writes dT, fP of steps >= step0 to
// outT / outP[(s - step0) * row + j].  from == g.s0 starts the recursion at z(s0) = e(s0); from > g.s0 continues from
// z[j], z[n_streams + j] (= z(from - 1)).  z != nullptr: the last z is stored back there.
template <class raw>
__global__ void __launch_bounds__(128) forcing_noise_kernel(const NoiseGen g, const int64_t* __restrict__ ids,
                                                            int64_t n_streams, int64_t from, int64_t step0, int32_t n_steps,
                                                            double* __restrict__ z, raw* __restrict__ outT,
                                                            raw* __restrict__ outP, int64_t row) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_streams) return;
  const int64_t id = ids[j];
  double zT = 0.0, zP = 0.0;
  if (from > g.s0) { zT = z[j]; zP = z[n_streams + j]; }
  for (int64_t s = from; s < step0 + n_steps; ++s) {
    double eT, eP;
    noise_normals(g.seed, id, s, eT, eP);
    if (s == g.s0) { zT = eT; zP = eP; }
    else {
      zT = __dadd_rn(__dmul_rn(g.rho_T, zT), __dmul_rn(g.c_T, eT));
      zP = __dadd_rn(__dmul_rn(g.rho_P, zP), __dmul_rn(g.c_P, eP));
    }
    if (s >= step0) {
      const int64_t o = (s - step0) * row + j;
      outT[o] = (raw)__dmul_rn(g.sd_T, zT);
      outP[o] = (raw)exp(__dadd_rn(__dmul_rn(g.sd_P, zP), -g.half_var_P));
    }
  }
  if (z) { z[j] = zT; z[n_streams + j] = zP; }
}

// The library's copies of the stream ids (NULL: 0 .. n_streams-1) and of the cell -> stream map (NULL: cell i reads
// stream i).  Bit 0 of *bad: a stream id < 0; bit 1: a cell_stream entry outside [0, n_streams)
__global__ void noise_index_kernel(const int64_t* ids, int64_t n_streams, const int32_t* cell_stream, int64_t N,
                                   int64_t* ids_out, int32_t* cell_out, int* bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n_streams > N ? n_streams : N);
       i += (int64_t)gridDim.x * blockDim.x) {
    int flags = 0;
    if (i < n_streams) {
      const int64_t g = ids ? ids[i] : i;
      if (g < 0) flags |= 1;
      ids_out[i] = g;
    }
    if (i < N) {
      const int32_t k = cell_stream ? cell_stream[i] : (int32_t)i;
      if (!(k >= 0 && (int64_t)k < n_streams)) flags |= 2;
      cell_out[i] = k;
    }
    if (flags) atomicOr(bad, flags);
  }
}

NoiseGen noise_gen(const tfg_ctx* x) {
  const tfg_forcing_noise& n = x->noise;
  return NoiseGen{n.seed, n.step0, n.T_air_sd, n.T_air_rho, x->noise_c[0], n.P_sd, n.P_rho, x->noise_c[1],
                  0.5 * (n.P_sd * n.P_sd)};
}

// Steps per launch while noise is bound: the [steps][2][n_streams] scratch stays within kNoiseScratchCap
int32_t noise_launch_steps(const tfg_ctx* x) {
  const int64_t cap = (int64_t)(kNoiseScratchCap / ((size_t)x->noise.n_streams * 2 * tfg_elem_size(x)));
  return (int32_t)std::max<int64_t>(1, std::min<int64_t>(tfg::kMaxLaunchSteps, cap));
}

// Noise pre-pass of one launch, on the launch's stream: dT and fP of its steps into the scratch, continuing the cached
// z when the launch follows the last one, else regenerating it from step0.  `want_steps` sizes a new scratch.
template <class raw>
cudaError_t noise_pass(tfg_ctx* x, tfg::RunParams<raw>& p, int32_t want_steps, cudaStream_t s) {
  const int64_t S = x->noise.n_streams;
  const size_t need = (size_t)p.n_steps * 2 * (size_t)S * sizeof(raw);
  if (x->noise_buf_bytes < need) {
    if (x->noise_buf) cudaFree(x->noise_buf);
    x->noise_buf = nullptr;
    x->noise_buf_bytes = 0;
    const size_t want = std::max<size_t>(need, (size_t)want_steps * 2 * (size_t)S * sizeof(raw));
    cudaError_t e = cudaMalloc(&x->noise_buf, want);
    if (e != cudaSuccess) return e;
    x->noise_buf_bytes = want;
  }
  raw* buf = static_cast<raw*>(x->noise_buf);
  const int64_t from = (x->noise_next == p.step0) ? p.step0 : x->noise.step0;
  x->noise_next = -1;
  forcing_noise_kernel<raw><<<(unsigned)((S + 127) / 128), 128, 0, s>>>(noise_gen(x), x->noise_ids, S, from, p.step0,
                                                                         p.n_steps, x->noise_z, buf, buf + S, 2 * S);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  x->noise_next = p.step0 + p.n_steps;
  p.noise = buf;
  p.cell_stream = x->noise_cell;
  p.n_streams = S;
  return cudaSuccess;
}

}  // namespace

extern "C" {

int tfg_abi_version(void) { return TFG_ABI_VERSION; }
const char* tfg_last_error(void) { return g_err.c_str(); }

int tfg_create(tfg_ctx** out, int device, int mode) {
  if (!out) return fail("tfg_create: out is NULL");
  if (mode != TFG_F64_STRICT && mode != TFG_F64_FAST && mode != TFG_F32) return fail("tfg_create: unknown mode");
  int n = 0;
  TFG_CUDA(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) return fail("tfg_create: no such CUDA device");
  TFG_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  TFG_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail("tfg_create: libtfglacier is built for sm_100a (B200) only");
  tfg_ctx* x = new tfg_ctx();
  x->device = device;
  x->mode = mode;
  *out = x;
  return 0;
}

void tfg_destroy(tfg_ctx* x) {
  if (!x) return;
  cudaSetDevice(x->device);
  if (x->col_terms) cudaFree(x->col_terms);
  if (x->cell_par) cudaFree(x->cell_par);
  if (x->cell_par_bad) cudaFree(x->cell_par_bad);
  if (x->obj_bad) cudaFree(x->obj_bad);
  if (x->fadj) cudaFree(x->fadj);
  if (x->fadj_bad) cudaFree(x->fadj_bad);
  if (x->noise_ids) cudaFree(x->noise_ids);
  if (x->noise_cell) cudaFree(x->noise_cell);
  if (x->noise_z) cudaFree(x->noise_z);
  if (x->noise_buf) cudaFree(x->noise_buf);
  if (x->noise_bad) cudaFree(x->noise_bad);
  delete x;
}

int tfg_mode(const tfg_ctx* x) { return x ? x->mode : -1; }
int64_t tfg_column_term_launches(const tfg_ctx* x) { return x ? x->col_term_launches : -1; }
size_t tfg_elem_size(const tfg_ctx* x) { return (x && x->mode == TFG_F32) ? 4 : 8; }

int tfg_set_option(tfg_ctx* x, int option, int64_t value) {
  if (!x) return fail("tfg_set_option: NULL context");
  if (option == TFG_OPT_TMA_STAGING) { x->use_tma = value != 0; return 0; }
  if (option == TFG_OPT_EXACT_AGG) {
    if (value != 0 && (((value >> 32) & 0xff) > 62 || (value >> 40) != 0))
      return fail("tfg_set_option: TFG_OPT_EXACT_AGG: low-word bits L (bits 32-39) must be at most 62, bits 40-63 zero");
    x->exact_agg = value;
    return 0;
  }
  if (option == TFG_OPT_COLUMN_TERMS) { x->column_terms = value != 0; return 0; }
  return fail("tfg_set_option: unknown option");
}

int tfg_set_constants(tfg_ctx* x, const tfg_constants* c) {
  if (!x || !c) return fail("tfg_set_constants: NULL argument");
  if (!(c->dt_hours > 0)) return fail("tfg_set_constants: dt_hours must be > 0");
  if (c->ring_slots < 1 || c->ring_slots > TFG_RING_SLOTS_MAX) return fail("tfg_set_constants: bad ring_slots");
  x->c = *c;
  x->have_consts = true;
  x->have_cell_par = false;  // the factors of unnamed parameters came from the old constants: bind again
  return 0;
}

int tfg_bind_static(tfg_ctx* x, int64_t n_cells, const tfg_statics* s) {
  if (!x || !s) return fail("tfg_bind_static: NULL argument");
  if (n_cells <= 0) return fail("tfg_bind_static: n_cells must be > 0");
  if (n_cells >= (int64_t(1) << 31)) return fail("tfg_bind_static: at most 2^31 - 1 cells per shard (a cell's state alone is ~1 KB: 180 GB of HBM hold < 2^28)");
  const void* req[] = {s->a_elev, s->sin_lat, s->cos_lat, s->neg_tan_lat, s->lon, s->sin_lat_eq, s->cos_lat_eq,
                       s->neg_tan_lat_eq, s->dlon, s->t_noon, s->da_m2, s->t_rain_snow};
  for (const void* p : req)
    if (!p) return fail("tfg_bind_static: a required table is NULL");
  x->s = *s;
  x->n_cells = n_cells;
  x->have_static = true;
  x->have_cell_par = false;  // sized for the old cell count: bind again
  x->have_obj = false;       // likewise the objective's per-cell arrays
  x->have_fadj = false;      // and the forcing adjustments
  x->have_noise = false;     // and the forcing noise
  return 0;
}

int tfg_bind_forcing_noise(tfg_ctx* x, const tfg_forcing_noise* n, void* stream) {
  if (!x) return fail("tfg_bind_forcing_noise: NULL context");
  x->have_noise = false;
  if (!n) return 0;
#if defined(TFG_LEAN_W2) || TFG_WS || TFG_PIPELINE || TFG_SPLIT_STEP
  return fail("tfg_bind_forcing_noise: this build runs an experimental kernel variant, which has no forcing noise");
#endif
  if (!x->have_static) return fail("tfg_bind_forcing_noise: call after tfg_bind_static");
  auto within = [](double v, double lo, double hi) { return v >= lo && v <= hi; };   // NaN and +-inf fail too
  if (!within(n->T_air_sd, 0.0, 5.0)) return fail("tfg_bind_forcing_noise: T_air_sd must be finite and within [0, 5] K");
  if (!within(n->T_air_rho, 0.0, 1.0)) return fail("tfg_bind_forcing_noise: T_air_rho must be finite and within [0, 1]");
  if (!within(n->P_sd, 0.0, 1.5)) return fail("tfg_bind_forcing_noise: P_sd must be finite and within [0, 1.5]");
  if (!within(n->P_rho, 0.0, 1.0)) return fail("tfg_bind_forcing_noise: P_rho must be finite and within [0, 1]");
  if (n->step0 < 0 || n->step0 >= kNoiseStepLimit) return fail("tfg_bind_forcing_noise: step0 must be in [0, 2^32)");
  if (n->n_streams <= 0 || n->n_streams > INT32_MAX)
    return fail("tfg_bind_forcing_noise: n_streams must be in [1, 2^31 - 1]");
  if (!n->cell_stream && n->n_streams != x->n_cells)
    return fail("tfg_bind_forcing_noise: n_streams must equal n_cells when cell_stream is NULL (cell i reads stream i)");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (x->noise_streams_cap < n->n_streams) {
    if (x->noise_ids) TFG_CUDA(cudaFree(x->noise_ids));
    if (x->noise_z) TFG_CUDA(cudaFree(x->noise_z));
    x->noise_ids = nullptr; x->noise_z = nullptr; x->noise_streams_cap = 0;
    TFG_CUDA(cudaMalloc(&x->noise_ids, (size_t)n->n_streams * sizeof(int64_t)));
    TFG_CUDA(cudaMalloc(&x->noise_z, 2 * (size_t)n->n_streams * sizeof(double)));
    x->noise_streams_cap = n->n_streams;
  }
  if (x->noise_cells_cap < x->n_cells) {
    if (x->noise_cell) TFG_CUDA(cudaFree(x->noise_cell));
    x->noise_cell = nullptr; x->noise_cells_cap = 0;
    TFG_CUDA(cudaMalloc(&x->noise_cell, (size_t)x->n_cells * sizeof(int32_t)));
    x->noise_cells_cap = x->n_cells;
  }
  if (!x->noise_bad) TFG_CUDA(cudaMalloc(&x->noise_bad, sizeof(int)));
  TFG_CUDA(cudaMemsetAsync(x->noise_bad, 0, sizeof(int), s));
  const int64_t total = std::max<int64_t>(n->n_streams, x->n_cells);
  noise_index_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, 148 * 32), 256, 0, s>>>(
      n->stream_id, n->n_streams, n->cell_stream, x->n_cells, x->noise_ids, x->noise_cell, x->noise_bad);
  TFG_CUDA(cudaGetLastError());
  int bad = 0;
  TFG_CUDA(cudaMemcpyAsync(&bad, x->noise_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  TFG_CUDA(cudaStreamSynchronize(s));
  if (bad) {
    std::string m = "tfg_bind_forcing_noise:";
    if (bad & 1) m += " stream_id has negative entries;";
    if (bad & 2) m += " cell_stream has entries outside [0, n_streams);";
    m.pop_back();
    return fail(m.c_str());
  }
  x->noise = *n;
  x->noise.stream_id = x->noise_ids;
  x->noise.cell_stream = x->noise_cell;
  x->noise_c[0] = std::sqrt(1.0 - n->T_air_rho * n->T_air_rho);
  x->noise_c[1] = std::sqrt(1.0 - n->P_rho * n->P_rho);
  x->noise_next = -1;
  x->have_noise = true;
  return 0;
}

int tfg_forcing_noise_series(tfg_ctx* x, int64_t step0, int32_t n_steps, void* dT, void* fP, void* stream) {
  if (!x || !dT || !fP) return fail("tfg_forcing_noise_series: NULL argument");
  if (!x->have_noise) return fail("tfg_forcing_noise_series: no forcing noise bound");
  if (n_steps <= 0) return fail("tfg_forcing_noise_series: n_steps must be > 0");
  if (step0 < x->noise.step0) return fail("tfg_forcing_noise_series: step0 is before the bound noise's step0");
  if (step0 + n_steps > kNoiseStepLimit) return fail("tfg_forcing_noise_series: steps must stay below 2^32");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t S = x->noise.n_streams;
  const unsigned grid = (unsigned)((S + 127) / 128);
  if (x->mode == TFG_F32)
    forcing_noise_kernel<float><<<grid, 128, 0, s>>>(noise_gen(x), x->noise_ids, S, x->noise.step0, step0, n_steps, nullptr,
                                                     static_cast<float*>(dT), static_cast<float*>(fP), S);
  else
    forcing_noise_kernel<double><<<grid, 128, 0, s>>>(noise_gen(x), x->noise_ids, S, x->noise.step0, step0, n_steps,
                                                      nullptr, static_cast<double*>(dT), static_cast<double*>(fP), S);
  TFG_CUDA(cudaGetLastError());
  return 0;
}

int tfg_bind_forcing_adjust(tfg_ctx* x, const tfg_forcing_adjust* a, void* stream) {
  if (!x) return fail("tfg_bind_forcing_adjust: NULL context");
  x->have_fadj = false;
  if (!a) return 0;
#if defined(TFG_LEAN_W2) || TFG_WS || TFG_PIPELINE || TFG_SPLIT_STEP
  return fail("tfg_bind_forcing_adjust: this build runs an experimental kernel variant, which has no forcing adjustments");
#endif
  if (!x->have_static) return fail("tfg_bind_forcing_adjust: call after tfg_bind_static");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t need = 2 * (size_t)x->n_cells * tfg_elem_size(x);
  if (x->fadj_bytes < need) {
    if (x->fadj) TFG_CUDA(cudaFree(x->fadj));
    x->fadj = nullptr;
    x->fadj_bytes = 0;
    TFG_CUDA(cudaMalloc(&x->fadj, need));
    x->fadj_bytes = need;
  }
  if (!x->fadj_bad) TFG_CUDA(cudaMalloc(&x->fadj_bad, sizeof(int)));
  TFG_CUDA(cudaMemsetAsync(x->fadj_bad, 0, sizeof(int), s));
  forcing_adjust_kernel<<<(unsigned)((x->n_cells + 255) / 256), 256, 0, s>>>(*a, x->fadj, x->mode == TFG_F32, x->n_cells,
                                                                             x->fadj_bad);
  TFG_CUDA(cudaGetLastError());
  int bad = 0;
  TFG_CUDA(cudaMemcpyAsync(&bad, x->fadj_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  TFG_CUDA(cudaStreamSynchronize(s));
  if (bad) {
    std::string m = "tfg_bind_forcing_adjust: values not finite or outside their range:";
    if (bad & 1) m += " T_air_offset [-30, 30]";
    if (bad & 2) m += " P_multiplier [0, 10]";
    return fail(m.c_str());
  }
  x->have_fadj = true;
  return 0;
}

int tfg_bind_cell_params(tfg_ctx* x, const tfg_cell_params* p, void* stream) {
  if (!x) return fail("tfg_bind_cell_params: NULL context");
  x->have_cell_par = false;
  if (!p) return 0;
#if defined(TFG_LEAN_W2) || TFG_WS || TFG_PIPELINE || TFG_SPLIT_STEP
  return fail("tfg_bind_cell_params: this build runs an experimental kernel variant, which has no per-cell parameters");
#endif
  if (!x->have_static || !x->have_consts) return fail("tfg_bind_cell_params: call after tfg_set_constants and tfg_bind_static");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t need = (size_t)tfg::kPCount * (size_t)x->n_cells * tfg_elem_size(x);
  if (x->cell_par_bytes < need) {
    if (x->cell_par) TFG_CUDA(cudaFree(x->cell_par));
    x->cell_par = nullptr;
    x->cell_par_bytes = 0;
    TFG_CUDA(cudaMalloc(&x->cell_par, need));
    x->cell_par_bytes = need;
  }
  if (!x->cell_par_bad) TFG_CUDA(cudaMalloc(&x->cell_par_bad, sizeof(int)));
  TFG_CUDA(cudaMemsetAsync(x->cell_par_bad, 0, sizeof(int), s));
  cell_params_kernel<<<(unsigned)((x->n_cells + 255) / 256), 256, 0, s>>>(*p, x->c, x->cell_par, x->mode == TFG_F32,
                                                                         x->n_cells, x->cell_par_bad);
  TFG_CUDA(cudaGetLastError());
  int bad = 0;
  TFG_CUDA(cudaMemcpyAsync(&bad, x->cell_par_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  TFG_CUDA(cudaStreamSynchronize(s));
  if (bad) {
    static const char* names[5] = {"dust_atten [0, 0.2]", "canopy_factor [0, 1]", "cloud_factor [0, 1]", "z0_air [1e-4, 0.1]",
                                   "em_surf [0.9, 1]"};
    std::string m = "tfg_bind_cell_params: values not finite or outside their range:";
    for (int j = 0; j < 5; ++j)
      if (bad & (1 << j)) { m += " "; m += names[j]; }
    return fail(m.c_str());
  }
  x->have_cell_par = true;
  return 0;
}

int tfg_bind_objective(tfg_ctx* x, const tfg_objective* o, void* stream) {
  if (!x) return fail("tfg_bind_objective: NULL context");
  x->have_obj = false;
  if (!o) return 0;
#if defined(TFG_LEAN_W2) || TFG_WS || TFG_PIPELINE || TFG_SPLIT_STEP
  return fail("tfg_bind_objective: this build runs an experimental kernel variant, which has no objective");
#endif
  if (!x->have_static) return fail("tfg_bind_objective: call after tfg_bind_static");
  if (o->quantity < TFG_REC_H_SNOW || o->quantity > TFG_REC_RH)
    return fail("tfg_bind_objective: quantity must be one of the eight BMI outputs, TFG_REC_H_SNOW .. TFG_REC_RH (0-7)");
  if (!o->obs) return fail("tfg_bind_objective: obs is NULL");
  if (!o->acc) return fail("tfg_bind_objective: acc is NULL");
  if (o->n_obs_steps <= 0) return fail("tfg_bind_objective: n_obs_steps must be > 0");
  if (o->n_obs_cols <= 0) return fail("tfg_bind_objective: n_obs_cols must be > 0");
  if (!o->obs_col && o->n_obs_cols != x->n_cells)
    return fail("tfg_bind_objective: n_obs_cols must equal n_cells when obs_col is NULL (column = cell)");
  if (o->obs_col) {
    TFG_CUDA(cudaSetDevice(x->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!x->obj_bad) TFG_CUDA(cudaMalloc(&x->obj_bad, sizeof(int)));
    TFG_CUDA(cudaMemsetAsync(x->obj_bad, 0, sizeof(int), s));
    obs_col_check_kernel<<<(unsigned)((x->n_cells + 255) / 256), 256, 0, s>>>(o->obs_col, x->n_cells, o->n_obs_cols, x->obj_bad);
    TFG_CUDA(cudaGetLastError());
    int bad = 0;
    TFG_CUDA(cudaMemcpyAsync(&bad, x->obj_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
    TFG_CUDA(cudaStreamSynchronize(s));
    if (bad) return fail("tfg_bind_objective: obs_col has entries outside [0, n_obs_cols)");
  }
  x->obj = *o;
  x->have_obj = true;
  return 0;
}

int tfg_bind_window_carry(tfg_ctx* x, void* carry) {
  if (!x) return fail("tfg_bind_window_carry: NULL context");
  x->win_carry = carry;
  return 0;
}

int tfg_bind_mass_residual(tfg_ctx* x, void* lo) {
  if (!x) return fail("tfg_bind_mass_residual: NULL context");
  if (lo && x->mode != TFG_F32) return fail("tfg_bind_mass_residual: only the float32 mode carries low parts");
  x->mass_lo = lo;
  return 0;
}

int tfg_bind_forcing_map(tfg_ctx* x, const int32_t* forcing_col, int64_t n_cols) {
  if (!x) return fail("tfg_bind_forcing_map: NULL context");
  if (forcing_col && n_cols <= 0) return fail("tfg_bind_forcing_map: n_cols must be > 0");
  x->forcing_col = forcing_col;
  x->n_cols = forcing_col ? n_cols : 0;
  return 0;
}

int tfg_bind_state(tfg_ctx* x, const tfg_state* s) {
  if (!x || !s) return fail("tfg_bind_state: NULL argument");
  void* req[] = {s->h_snow, s->h_swe, s->h_ice, s->h_iwe, s->eccs, s->ecci, s->albedo, s->n_days,
                 s->SM, s->IM, s->M_total, s->RH, s->ring};
  for (void* p : req)
    if (!p) return fail("tfg_bind_state: a required array is NULL");
  void* vol[] = {s->vol_P, s->vol_PR, s->vol_PS, s->vol_SM, s->vol_IM, s->P_max};
  int nv = 0;
  for (void* p : vol) nv += (p != nullptr);
  if (nv != 0 && nv != 6) return fail("tfg_bind_state: pass all six diagnostic integrals or none");
  x->st = *s;
  x->have_state = true;
  return 0;
}

int tfg_bind_time(tfg_ctx* x, const tfg_time_row* rows, const double* gmt, int64_t n_steps, int n_tz, void* stream) {
  if (!x || !rows || !gmt) return fail("tfg_bind_time: NULL argument");
  if (n_steps <= 0 || n_tz < 1 || n_tz > TFG_MAX_TZ) return fail("tfg_bind_time: bad n_steps / n_tz");
  (void)stream;
  x->h_rows.assign(reinterpret_cast<const double*>(rows), reinterpret_cast<const double*>(rows) + (size_t)n_steps * 8);
  x->h_gmt.assign(gmt, gmt + (size_t)n_steps * n_tz);
  x->n_time = n_steps;
  x->n_tz = n_tz;
  return 0;
}

int tfg_run(tfg_ctx* x, const void* forcing, int64_t step0, int32_t n_steps, void* record, uint64_t record_mask,
            void* basin_agg, int32_t n_basin, void* stream) {
  if (!x || !forcing) return fail("tfg_run: NULL argument");
  if (!x->have_consts || !x->have_static || !x->have_state || x->h_rows.empty())
    return fail("tfg_run: constants, statics, state and time tables must be bound first");
  if (n_steps <= 0 || step0 < 0) return fail("tfg_run: bad step range");
  if (step0 + n_steps > x->n_time) return fail("tfg_run: step range exceeds the bound time table");
  if (record && (record_mask == 0 || (record_mask >> TFG_REC_COUNT) != 0)) return fail("tfg_run: bad record_mask");
  if (basin_agg && (n_basin <= 0 || !x->s.basin_id)) return fail("tfg_run: aggregates need basin_id and n_basin");
  if (x->have_noise && step0 < x->noise.step0) return fail("tfg_run: the launch starts before the forcing noise's step0");
  if (x->have_noise && step0 + n_steps > kNoiseStepLimit) return fail("tfg_run: forcing noise: steps must stay below 2^32");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool rec = record != nullptr, agg = basin_agg != nullptr, vol = x->st.vol_P != nullptr;
  cudaError_t e = cudaSuccess;
  const size_t es = tfg_elem_size(x);
  // a launch carries at most kMaxLaunchSteps clock rows; longer runs are a sequence of launches on the same stream
  // (bit-identical to one launch: state and snowfall window are carried through HBM either way).  With forcing noise
  // bound, launches are shorter where its scratch would exceed kNoiseScratchCap.
  const int32_t per_launch = x->have_noise ? noise_launch_steps(x) : tfg::kMaxLaunchSteps;
  for (int32_t t0 = 0; t0 < n_steps && e == cudaSuccess; t0 += per_launch) {
    const int32_t nt = std::min<int32_t>(per_launch, n_steps - t0);
    const int32_t want = std::min<int32_t>(per_launch, n_steps);
    const void* f = static_cast<const char*>(forcing) + (size_t)t0 * TFG_N_FORCING * (x->forcing_col ? x->n_cols : x->n_cells) * es;
    void* r = record ? static_cast<char*>(record) + (size_t)t0 * __builtin_popcountll(record_mask) * x->n_cells * es : nullptr;
    // float64 sums: 8 B per entry; exact mode: two int64 words per entry (the trailing counter stays at the end)
    void* a = basin_agg ? static_cast<char*>(basin_agg) + (size_t)t0 * n_basin * TFG_N_AGG * (x->exact_agg ? 16 : 8) : nullptr;
    long long* agg_bad = (basin_agg && x->exact_agg) ? static_cast<long long*>(basin_agg) + (size_t)n_steps * n_basin * TFG_N_AGG * 2 : nullptr;
    if (x->mode == TFG_F32) {
      auto p = make_params<float>(x, f, step0 + t0, nt, r, record_mask, a, n_basin, agg_bad);
      if (x->have_noise) e = noise_pass(x, p, want, s);
      if (e == cudaSuccess) e = tfg::launch_run_f32(p, rec, agg, vol, s);
    } else {
      auto p = make_params<double>(x, f, step0 + t0, nt, r, record_mask, a, n_basin, agg_bad);
      if (x->have_noise) e = noise_pass(x, p, want, s);
      const bool strict = x->mode == TFG_F64_STRICT;
      // Forcing map with few columns per cell: the forcing-only part of the step is evaluated once per column and
      // timestep (column_terms_kernel, in the arithmetic of the context's mode) and the melt kernel reads one line per
      // step instead of redoing it per cell.  Same device functions either way: results do not depend on this switch
      // (test_column_terms_*).  Not for launches so small that a second kernel launch costs more than it saves
      // (per-step BMI updates of a few cells); the fast mode leaves SATTERLUND configurations to its strict step.
      // Forcing adjustments and forcing noise make the forcing differ per cell (or stream), so the pass is not taken
      // while either is bound.
      const size_t need = (size_t)nt * (size_t)x->n_cols * tfg::kCtCount * sizeof(double);
      if (e == cudaSuccess && x->column_terms && x->forcing_col && !x->have_fadj && !x->have_noise && !x->use_tma && (strict || !x->c.satterlund) && x->n_cols * 8 <= x->n_cells &&
          (int64_t)nt * x->n_cells >= 65536 && need <= (size_t(1) << 31)) {
        if (x->col_terms_bytes < need) {   // grows to the largest launch seen; a failed allocation leaves the plain path
          if (x->col_terms) cudaFree(x->col_terms);
          x->col_terms = nullptr; x->col_terms_bytes = 0;
          const size_t want = (size_t)std::min<int64_t>(tfg::kMaxLaunchSteps, std::max<int32_t>(nt, n_steps)) * (size_t)x->n_cols *
                              tfg::kCtCount * sizeof(double);
          if (cudaMalloc(&x->col_terms, want) == cudaSuccess) x->col_terms_bytes = want;
          else (void)cudaGetLastError();
        }
        if (x->col_terms_bytes >= need) {
          const bool par = p.cell_par != nullptr;
          e = strict ? tfg::launch_column_terms_strict(static_cast<const double*>(f), x->col_terms, nt, x->n_cols, p.k, par, s)
                     : tfg::launch_column_terms_fast(static_cast<const double*>(f), x->col_terms, nt, x->n_cols, p.k, par, s);
          p.col_terms = x->col_terms;
          ++x->col_term_launches;
        }
      }
      if (e == cudaSuccess) e = strict ? tfg::launch_run_strict(p, rec, agg, vol, s) : tfg::launch_run_fast(p, rec, agg, vol, s);
    }
  }
  if (e != cudaSuccess) return fail("tfg_run: kernel launch", e);
  return 0;
}

int tfg_ingest_async(tfg_ctx* x, const void* pinned_src, void* dev_dst, size_t bytes, void* stream, void* done_event) {
  if (!x || !pinned_src || !dev_dst) return fail("tfg_ingest_async: NULL argument");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  TFG_CUDA(cudaMemcpyAsync(dev_dst, pinned_src, bytes, cudaMemcpyHostToDevice, s));
  if (done_event) TFG_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(done_event), s));
  return 0;
}

int tfg_host_alloc(void** out, size_t bytes, int write_combined) {
  if (!out || bytes == 0) return fail("tfg_host_alloc: bad argument");
  TFG_CUDA(cudaHostAlloc(out, bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
  return 0;
}

int tfg_host_free(void* block) {
  if (block) TFG_CUDA(cudaFreeHost(block));
  return 0;
}

int tfg_host_is_pinned(const void* p) {
  cudaPointerAttributes a{};
  if (!p || cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
  return a.type == cudaMemoryTypeHost ? 1 : 0;
}

int tfg_stream_wait_event(tfg_ctx* x, void* stream, void* event) {
  if (!x || !event) return fail("tfg_stream_wait_event: NULL argument");
  TFG_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), static_cast<cudaEvent_t>(event), 0));
  return 0;
}

int tfg_convert_forcing(tfg_ctx* x, const void* raw, int raw_elem_size, void* out, int64_t n_steps, int64_t n_cells,
                        void* stream) {
  if (!x || !raw || !out) return fail("tfg_convert_forcing: NULL argument");
  if (n_steps <= 0 || n_cells <= 0) return fail("tfg_convert_forcing: empty block");
  if (raw_elem_size != 4 && raw_elem_size != 8) return fail("tfg_convert_forcing: raw_elem_size must be 4 or 8");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t total = n_steps * n_cells;
  const unsigned grid = (unsigned)((total + 255) / 256 < 148 * 32 ? (total + 255) / 256 : 148 * 32);
  const bool f32out = x->mode == TFG_F32;
  if (raw_elem_size == 8) {
    const double* r = static_cast<const double*>(raw);
    if (f32out) convert_kernel<double, float><<<grid, 256, 0, s>>>(r, static_cast<float*>(out), n_steps, n_cells);
    else convert_kernel<double, double><<<grid, 256, 0, s>>>(r, static_cast<double*>(out), n_steps, n_cells);
  } else {
    const float* r = static_cast<const float*>(raw);
    if (f32out) convert_kernel<float, float><<<grid, 256, 0, s>>>(r, static_cast<float*>(out), n_steps, n_cells);
    else convert_kernel<float, double><<<grid, 256, 0, s>>>(r, static_cast<double*>(out), n_steps, n_cells);
  }
  TFG_CUDA(cudaGetLastError());
  return 0;
}

int tfg_convert_forcing_packed(tfg_ctx* x, const int16_t* raw, const double* scale, const double* offset, void* out,
                               int64_t n_steps, int64_t n_cells, void* stream) {
  if (!x || !raw || !out || !scale || !offset) return fail("tfg_convert_forcing_packed: NULL argument");
  if (n_steps <= 0 || n_cells <= 0) return fail("tfg_convert_forcing_packed: empty block");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PackScale ps;
  for (int j = 0; j < 6; ++j) { ps.scale[j] = scale[j]; ps.offset[j] = offset[j]; }
  const int64_t total = n_steps * n_cells;
  const unsigned grid = (unsigned)((total + 255) / 256 < 148 * 32 ? (total + 255) / 256 : 148 * 32);
  if (x->mode == TFG_F32) convert_packed_kernel<float><<<grid, 256, 0, s>>>(raw, static_cast<float*>(out), n_steps, n_cells, ps);
  else convert_packed_kernel<double><<<grid, 256, 0, s>>>(raw, static_cast<double*>(out), n_steps, n_cells, ps);
  TFG_CUDA(cudaGetLastError());
  return 0;
}

int tfg_route_fir(tfg_ctx* x, const double* series, double* out, const double* weights, int32_t taps, int64_t n_steps,
                  int64_t n_series, void* stream) {
  if (!x || !series || !out || !weights) return fail("tfg_route_fir: NULL argument");
  if (taps < 1 || n_steps < 1 || n_series < 1) return fail("tfg_route_fir: empty problem");
  TFG_CUDA(cudaSetDevice(x->device));
  const int64_t total = n_steps * n_series;
  const unsigned grid = (unsigned)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  fir_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(series, out, weights, taps, n_steps, n_series);
  TFG_CUDA(cudaGetLastError());
  return 0;
}

int tfg_measure_fp64_peak(tfg_ctx* x, double* dfma_thread_ops_per_s, void* stream) {
  if (!x || !dfma_thread_ops_per_s) return fail("tfg_measure_fp64_peak: NULL argument");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  double* d = nullptr;
  TFG_CUDA(cudaMalloc(&d, sizeof(double)));
  cudaEvent_t a, b;
  TFG_CUDA(cudaEventCreate(&a));
  TFG_CUDA(cudaEventCreate(&b));
  const int iters = 4096, blocks = 148 * 8, threads = 256;
  dfma_peak_kernel<<<blocks, threads, 0, s>>>(d, 64, 1.0);  // warm-up
  float best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    TFG_CUDA(cudaEventRecord(a, s));
    dfma_peak_kernel<<<blocks, threads, 0, s>>>(d, iters, 1.0);
    TFG_CUDA(cudaEventRecord(b, s));
    TFG_CUDA(cudaEventSynchronize(b));
    float ms = 0;
    TFG_CUDA(cudaEventElapsedTime(&ms, a, b));
    best = ms < best ? ms : best;
  }
  TFG_CUDA(cudaGetLastError());
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(d);
  *dfma_thread_ops_per_s = (double)blocks * threads * iters * 64.0 / (best * 1e-3);
  return 0;
}

int tfg_synth_forcing(tfg_ctx* x, void* forcing, int64_t step0, int32_t n_steps, int64_t n_cells, const void* elev,
                      uint64_t seed, int64_t storm_cells, void* stream) {
  if (!x || !forcing || !elev) return fail("tfg_synth_forcing: NULL argument");
  if (n_steps <= 0 || n_cells <= 0) return fail("tfg_synth_forcing: empty block");
  TFG_CUDA(cudaSetDevice(x->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const unsigned grid = (unsigned)((n_cells + 255) / 256);
  if (x->mode == TFG_F32)
    synth_kernel<float><<<grid, 256, 0, s>>>(static_cast<float*>(forcing), static_cast<const float*>(elev), step0,
                                             n_steps, n_cells, seed, storm_cells);
  else
    synth_kernel<double><<<grid, 256, 0, s>>>(static_cast<double*>(forcing), static_cast<const double*>(elev), step0,
                                              n_steps, n_cells, seed, storm_cells);
  TFG_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
