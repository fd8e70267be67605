/*
 * tfglacier.h -- C ABI of libtfglacier.so, the sm_100a implementation of the
 * per-cell, per-timestep energy-balance + snow/ice melt update of topoflow-glacier.
 *
 * The reference has NO foreign-function interface for this path: its boundary is the
 * Python class BmiTopoflowGlacier (src/topoflow_glacier/bmi/bmi_topoflow_glacier.py:115).
 * Each entry point below names the reference code it replaces; the Python host
 * (topoflow_glacier_b200/bmi.py) keeps the reference's BMI method names and calls these
 * through ctypes.  See INTEGRATION.md for the binding a maintainer adds.
 *
 * Conventions
 *   - every pointer marked "dev" is a raw CUDA device pointer (e.g. torch.Tensor.data_ptr());
 *     the library never allocates, frees or retains caller memory beyond a bound pointer;
 *   - element type of every "dev" array is double (TFG_F64_*) or float (TFG_F32) as chosen in
 *     tfg_create(); constants and time tables are always passed as double on the host side;
 *   - all per-cell arrays are SoA of length n_cells; 2-D blocks are row-major with the cell
 *     index fastest ([step][var][cell]);
 *   - every function returns 0 on success, <0 on error (tfg_last_error() gives the text);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); launches are
 *     asynchronous with respect to the host.
 */
#ifndef TFGLACIER_H
#define TFGLACIER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFG_ABI_VERSION 1
#if defined(__GNUC__)
#define TFG_API __attribute__((visibility("default")))
#else
#define TFG_API
#endif

/* arithmetic modes */
#define TFG_F64_STRICT 0 /* float64; + - * / sqrt IEEE-rounded in the reference's order (no FMA contraction) */
#define TFG_F64_FAST 1   /* float64; algebraically equivalent shortcuts, FMA allowed (see DESIGN.md)        */
#define TFG_F32 2        /* float32 state/forcing, fast intrinsics; own tolerance                            */

#define TFG_N_FORCING 5 /* P [m/h], T_air [degC], P_air [Pa], Hum_sp [kg/kg], uz [m/s]                      */
#define TFG_RING_SLOTS_MAX 72
#define TFG_MAX_TZ 8
#define TFG_N_AGG 3 /* per-basin sums: M_total*da_m2, h_swe*da_m2, h_iwe*da_m2                            */

/* indices of recordable per-step quantities (bit i of `record_mask`, row order in the record buffer) */
enum tfg_rec {
  TFG_REC_H_SNOW = 0, TFG_REC_H_SWE, TFG_REC_SM, TFG_REC_H_ICE, TFG_REC_H_IWE, TFG_REC_IM, TFG_REC_M_TOTAL,
  TFG_REC_RH, /* ^ the eight BMI outputs, bmi_topoflow_glacier.py:28-37 */
  TFG_REC_P0, TFG_REC_E_SAT_AIR, TFG_REC_E_AIR, TFG_REC_T_DEW, TFG_REC_T_SURF, TFG_REC_E_SAT_SURF, TFG_REC_RI,
  TFG_REC_DN, TFG_REC_DH, TFG_REC_QH, TFG_REC_W_P, TFG_REC_E_SURF, TFG_REC_QE, TFG_REC_TSN_OFFSET,
  TFG_REC_ALBEDO, TFG_REC_N_DAYS, TFG_REC_QN_SW, TFG_REC_EM_AIR, TFG_REC_QN_LW, TFG_REC_Q_SUM, TFG_REC_ECCS,
  TFG_REC_ECCI, TFG_REC_SNOW3DAY, TFG_REC_P_RAIN, TFG_REC_P_SNOW,
  TFG_REC_COUNT
};

typedef struct tfg_ctx tfg_ctx;

/* Physical constants read by the path: TopoflowGlacierConfig defaults, bmi/config.py:27-101,
 * plus the hard-coded wind height z = 10 m (bmi_topoflow_glacier.py:301).                       */
typedef struct tfg_constants {
  double dt_hours; /* cfg.dt (integer hours in the reference)                                    */
  double T0, h_active_layer;
  double rho_air, rho_snow, rho_ice, rho_H2O;
  double Cp_air, Cp_snow, Cp_ice;
  double g, Lf, Lv, eps, kappa, latent_heat_constant, sigma;
  double sea_level_p0, uni_gas_const, M_mass_air;
  double z0_air, em_surf, dust_atten, canopy_factor, cloud_factor;
  double z_wind;
  int32_t satterlund;
  int32_t ring_slots; /* int(3*24/dt), bmi_topoflow_glacier.py:296; <= TFG_RING_SLOTS_MAX         */
} tfg_constants;

/* Clock-only part of one update(): replaces update_julian_day (bmi_topoflow_glacier.py:957-1004),
 * Day_Angle/Declination/Eccentricity_Correction (solar_funcs.py:156-247) and Equation_Of_Time
 * (solar_funcs.py:1301-1429), which the host evaluates once per step with the reference's own
 * scalar expressions.                                                                           */
typedef struct tfg_time_row {
  double clock_hour; /* (jd - int(jd)) * 24                                                      */
  double TE;         /* equation of time [h]                                                     */
  double sin_decl, cos_decl, tan_decl;
  double isc_e0;     /* I_sc * E0                                                                */
  double cos_hour, sin_hour; /* cos/sin of omega*((clock_hour - 12) - TE), omega = 15 deg/h; read by the
                              * fast modes only (angle-addition form of cos(omega*th), DESIGN.md)       */
} tfg_time_row;

/* Cell-only tables: replaces set_aspect_angle/set_slope_angle (bmi_topoflow_glacier.py:1082-1113),
 * Equivalent_Latitude / Longitude_Offset / Noon_Offset_Slope (solar_funcs.py:718-778) and the
 * per-cell factors of update_atm_pressure_from_elevation (:552).  All dev, length n_cells.        */
typedef struct tfg_statics {
  const void* a_elev;      /* (-M*g)*elev                                                         */
  const void* sin_lat;
  const void* cos_lat;
  const void* neg_tan_lat; /* -tan(lat)                                                           */
  const void* lon;         /* degrees east                                                        */
  const void* sin_lat_eq;
  const void* cos_lat_eq;
  const void* neg_tan_lat_eq; /* -tan(lat_eq after the deg round trip, solar_funcs.py:793,320)    */
  const void* dlon;        /* rad                                                                 */
  const void* t_noon;      /* h                                                                   */
  const void* da_m2;
  const void* t_rain_snow; /* degC                                                                */
  const int32_t* basin_id; /* may be NULL when no aggregates are requested                        */
  const uint8_t* tz_idx;   /* may be NULL (all cells use zone 0)                                  */
} tfg_statics;

/* Carried state + BMI outputs + diagnostic integrals; all dev, length n_cells, updated in place.
 * Replaces the (1,) arrays of Context (physics/context.py:18-71) and the attributes initialised at
 * bmi_topoflow_glacier.py:298-395.                                                                */
typedef struct tfg_state {
  void* h_snow; void* h_swe; void* h_ice; void* h_iwe; /* carried + BMI outputs                   */
  void* eccs; void* ecci; void* albedo; void* n_days;  /* carried                                 */
  void* SM; void* IM; void* M_total; void* RH;         /* BMI outputs of the last step            */
  void* vol_P; void* vol_PR; void* vol_PS; void* vol_SM; void* vol_IM; void* P_max; /* NULL = skip */
  void* ring;   /* [ring_slots][n_cells] 3-day snowfall window; slot of absolute step s is s % slots */
} tfg_state;

/* ---- lifetime ------------------------------------------------------------------------------- */
TFG_API int tfg_abi_version(void);
TFG_API const char* tfg_last_error(void);
/* one context per (process, device); `mode` is one of TFG_F64_STRICT / TFG_F64_FAST / TFG_F32 */
TFG_API int tfg_create(tfg_ctx** out, int device, int mode);
TFG_API void tfg_destroy(tfg_ctx* ctx);
TFG_API int tfg_mode(const tfg_ctx* ctx);
/* tuning switches; TFG_OPT_TMA_STAGING: forcing tiles reach shared memory through cp.async.bulk + mbarrier
 * (4 stages) instead of per-thread prefetching loads; results are bit-identical either way */
#define TFG_OPT_TMA_STAGING 1
/* TFG_OPT_EXACT_AGG: order-independent basin aggregates.  value = 0 switches it off; otherwise
 * value = L<<32 | 1<<24 | (E2+128)<<16 | (E1+128)<<8 | (E0+128), E_q the binary exponent that bounds a 32-cell partial
 * sum of aggregate q (|partial| < 2^E_q), L in [1, 62] the fraction bits of the low word (L = 0 means 42; bits 40-63
 * must be 0).  tfg_run then reads `basin_agg` as int64 [n_steps][n_basin][TFG_N_AGG][2] followed by ONE trailing
 * int64 counter: every contribution v is split into two fixed-point words, hi = trunc(v * 2^(40-E_q)) and
 * lo = trunc(frac(v * 2^(40-E_q)) * 2^L) (value = hi * 2^(E_q-40) + lo * 2^(E_q-40-L)), that are added with integer
 * atomics, so the sums do not depend on the order of the atomics, on the launch geometry or on how cells are sharded
 * over GPUs (32-cell aligned shards), and an integer all-reduce of the accumulators is exact.  Contributions that are
 * not finite or reach 2^E_q are left out and counted in the trailing word.
 * Headroom: with C contributions to one (step, basin, aggregate) the low word stays below C * 2^L and the high word
 * below C * 2^40; the caller picks L <= 62 - ceil(log2 C) (a warp of 32 cells inside one basin is one contribution,
 * every cell of a warp that straddles basins is one).  Words that leave the int64 range wrap without notice. */
#define TFG_OPT_EXACT_AGG 2
/* TFG_OPT_COLUMN_TERMS (default 1; TFG_F64_FAST and TFG_F64_STRICT contexts with a forcing map of at most n_cells / 8 columns): the part of
 * update() that reads nothing but the forcings (vapour pressures, relative humidity, dew point, precipitable water,
 * air emissivity, incoming longwave, snowfall wet bulb: bmi_topoflow_glacier.py:423-425, :784-893, :919-920,
 * :1167-1234, :1507-1520) is evaluated once per forcing COLUMN and timestep by a small pass in front of each launch and
 * read back by the melt kernel, instead of once per cell.  The same device functions run either way: results are
 * bit-identical with the switch off (value = 0).  tfg_column_term_launches counts the launches that took the pass. */
#define TFG_OPT_COLUMN_TERMS 3
TFG_API int tfg_set_option(tfg_ctx* ctx, int option, int64_t value);
TFG_API int64_t tfg_column_term_launches(const tfg_ctx* ctx);
TFG_API size_t tfg_elem_size(const tfg_ctx* ctx);

/* ---- binding (replaces BmiTopoflowGlacier.initialize, bmi_topoflow_glacier.py:274-411) ------- */
TFG_API int tfg_set_constants(tfg_ctx* ctx, const tfg_constants* c);
TFG_API int tfg_bind_static(tfg_ctx* ctx, int64_t n_cells, const tfg_statics* s);
TFG_API int tfg_bind_state(tfg_ctx* ctx, const tfg_state* s);
/* Optional [3][n_cells] scratch (context element type, initialise the third row to NaN): the kernel keeps the running
 * sum of the 3-day snowfall window there between launches, so that a launch of a few timesteps does not re-read all
 * ring_slots entries of every cell; an exact re-sum still happens whenever the sum is within rounding distance of the
 * 0.03 m threshold (bmi_topoflow_glacier.py:1040), so decisions -- and hence all state -- are unchanged.  Set the third
 * row to NaN after changing the window from outside.  NULL switches it off.                                        */
TFG_API int tfg_bind_window_carry(tfg_ctx* ctx, void* carry);
/* float32 mode only, optional [2][n_cells] float scratch (zero it first): the low parts of h_swe / h_iwe.  With it the
 * water-equivalent balances (bmi_topoflow_glacier.py:1594-1617) are carried as float + float and evaluated in float64
 * inside the float32 kernel, so that the hour a pack melts out does not drift with float32 accumulation.  NULL = plain
 * float32 balances.                                                                                                   */
TFG_API int tfg_bind_mass_residual(tfg_ctx* ctx, void* lo);
/* Optional forcing map: cell i reads column forcing_col[i] (dev int32 [n_cells], values in [0, n_cols)) of forcing
 * blocks that are then [n_steps][5][n_cols] -- the cells of one catchment share the catchment's forcing series, as the
 * reference's one-CSV-per-catchment drivers do (examples/run_topoflow_glacier.py:30-49), without replicating it per
 * cell on the host or over PCIe.  NULL restores the default, one column per cell.  Call after tfg_bind_static.    */
TFG_API int tfg_bind_forcing_map(tfg_ctx* ctx, const int32_t* forcing_col, int64_t n_cols);
/* Optional per-cell surface parameters: each field is a dev float64 array of length n_cells (in every mode), or NULL
 * for "use the context constant" of the same name.  Where each one enters the reference:
 *   dust_atten     atmospheric transmissivity and scattering of clear-sky radiation (solar_funcs.py:894-953)
 *   canopy_factor  Brutsaert air emissivity, em_air = (1 - F) 1.72 (e/T)^(1/7) (1 + 0.22 C^2) + F (:1167-1180)
 *   cloud_factor   the same expression, through C
 *   z0_air         log-law aerodynamic conductance, ln((z - h_snow) / z0_air) (:670)
 *   em_surf        outgoing longwave, em_surf sigma T_surf^4 + (1 - em_surf) LW_in (:1236-1246)
 * Ranges of the configuration schema: dust_atten [0, 0.2], canopy_factor [0, 1], cloud_factor [0, 1],
 * z0_air [1e-4, 0.1], em_surf [0.9, 1].                                                                      */
typedef struct tfg_cell_params {
  const double* dust_atten;
  const double* canopy_factor;
  const double* cloud_factor;
  const double* z0_air;
  const double* em_surf;
} tfg_cell_params;

/* Bind (p != NULL) or unbind (p == NULL) per-cell surface parameters; call after tfg_bind_static and tfg_set_constants,
 * and again after either changes.  May be called between launches (a calibration loop).  The library derives the
 * factors the kernels read (the per-cell counterparts of what tfg_set_constants derives from the constants) into a
 * scratch it owns, on `stream`, and checks every value on the device: a non-finite value or one outside the ranges
 * above is an error, after which no parameters are bound.  The call waits for that check; the caller's arrays are not
 * read again afterwards.  A cell whose parameters equal the constants gives the bits of an unbound run.          */
TFG_API int tfg_bind_cell_params(tfg_ctx* ctx, const tfg_cell_params* p, void* stream);

/* Optional objective: while one is bound, every tfg_run launch compares one BMI output of every cell with an observed
 * series and adds four float64 sums per cell into `acc`, so that a calibration or sensitivity run scores each
 * candidate (cell) on the device instead of recording a series per cell-step.
 *   quantity  TFG_REC_H_SNOW .. TFG_REC_RH (the eight BMI outputs); the value compared for absolute step k is the one
 *             the record buffer holds for step k (what get_value returns after that update())
 *   obs       dev float64 [n_obs_steps][n_obs_cols] in every mode; row j belongs to absolute step obs_step0 + j.  A
 *             non-finite value means "not observed": that step is not scored for the cells reading that column
 *             (daily observations of an hourly model, a spin-up period).  Steps outside the window are not scored.
 *   obs_col   dev int32 [n_cells] in [0, n_obs_cols): cell i reads column obs_col[i]; NULL = column i (n_obs_cols
 *             must then equal n_cells)
 *   acc       dev float64 [TFG_N_OBJ][n_cells], ACCUMULATED INTO (zero it to start); owned by the caller.  Rows:
 *             S_s = sum s, S_ss = sum s*s, S_so = sum s*o, S_ee = sum (s-o)*(s-o).  Each scored step runs exactly
 *             d = s - o; S_s += s; S_ss += s*s; S_so += s*o; S_ee += d*d in float64 (a float32 s widened exactly), each
 *             operation rounded once, so the sums depend only on the per-step values and their order: they are the
 *             same bits for any launch split, for the per-step path and for any sharding, and a host float64 loop over
 *             a recorded series reproduces them.  A cell whose state is NaN is still scored where its observation is
 *             finite, so its sums become NaN.
 * NSE, KGE, RMSE and bias follow from the sums and the observations' own moments (topoflow_glacier_b200/objective.py). */
#define TFG_N_OBJ 4 /* rows of tfg_objective.acc */
typedef struct tfg_objective {
  int32_t quantity;                   /* TFG_REC_H_SNOW .. TFG_REC_RH                                          */
  const double* obs;                  /* dev [n_obs_steps][n_obs_cols]; non-finite = not observed               */
  int64_t obs_step0, n_obs_steps, n_obs_cols;
  const int32_t* obs_col;             /* dev [n_cells] in [0, n_obs_cols), or NULL (column = cell)              */
  double* acc;                        /* dev [TFG_N_OBJ][n_cells], accumulated into                            */
} tfg_objective;
/* Bind (o != NULL) or unbind (o == NULL) an objective; call after tfg_bind_static (binding statics again unbinds it).
 * The host fields are checked, and obs_col's range on the device, on `stream`; the call waits for that check.  On
 * error nothing is bound and tfg_last_error() names the field.  The arrays are read by every later tfg_run.        */
TFG_API int tfg_bind_objective(tfg_ctx* ctx, const tfg_objective* o, void* stream);

/* Optional per-cell forcing adjustments: each field is a dev float64 array of length n_cells (in every mode), or NULL
 * for the identity (offset 0, multiplier 1).  At every step cell i reads its forcing -- its own column, or column
 * forcing_col[i] with a forcing map -- and then uses
 *   T_air' = T_air + T_air_offset[i]      [degC + K]
 *   P'     = P * P_multiplier[i]          [m/h]
 * each ONE IEEE operation in the context's element type; the library rounds the offsets and multipliers to that type
 * once, at bind time (float64 in both float64 modes, float32 in TFG_F32).  A run with adjustments is therefore
 * bit-identical to a run whose per-cell forcing was adjusted in advance with the same two operations.  P_air, Hum_sp
 * and uz are NOT adjusted: air pressure and humidity stay what the forcing says (the cell's own air pressure at its
 * elevation is formed from a_elev, as without adjustments).  The adjusted values are what every later operation sees,
 * including the fast float64 mode's test for physically sane forcings and its strict fallback: an offset that takes
 * |T_air'| to 90 degC or more, or a multiplier that takes P' to 10 m/h or more, takes the strict step, as the same
 * forcing given per cell would.  A cell with offset 0 and multiplier 1 gets the bits of an unbound run, except that a
 * forcing T_air of -0.0 becomes +0.0 (IEEE: -0.0 + 0.0 = +0.0).  Ranges: T_air_offset [-30, 30] K (a 4.5 km band at
 * 6.5 K/km; elevation bands: T_air_offset = -T_lapse_rate * (elev_cell - elev_series)), P_multiplier [0, 10].  The
 * input values a caller sets (the forcing block, the BMI input variables) are not changed; the adjustment happens
 * inside the step.  With adjustments bound the TFG_OPT_COLUMN_TERMS pass is not taken (the forcing-only terms then
 * differ per cell).                                                                                                  */
typedef struct tfg_forcing_adjust {
  const double* T_air_offset;  /* dev float64 [n_cells] or NULL (0) */
  const double* P_multiplier;  /* dev float64 [n_cells] or NULL (1) */
} tfg_forcing_adjust;
/* Bind (a != NULL) or unbind (a == NULL) forcing adjustments; call after tfg_bind_static (binding statics again unbinds
 * them).  May be called between launches.  The library checks every value on the device, on `stream`, and waits for
 * that check: a non-finite value or one outside the ranges above is an error, after which nothing is bound and
 * tfg_last_error() names the field.  It then keeps the values, in its element type, in a [2][n_cells] scratch it
 * owns; the caller's arrays are not read again.                                                                      */
TFG_API int tfg_bind_forcing_adjust(tfg_ctx* ctx, const tfg_forcing_adjust* a, void* stream);

/* host tables for steps [0, n_steps): rows[n_steps], gmt_offset_hours[n_steps][n_tz]; copied by the library
 * (each launch carries its <= 128 rows in the kernel parameter block); replaces solar.gmt_offset_hours,
 * solar_funcs.py:1616-1637, evaluated on the host                                                 */
TFG_API int tfg_bind_time(tfg_ctx* ctx, const tfg_time_row* rows, const double* gmt_offset_hours, int64_t n_steps,
                  int n_tz, void* stream);

/* ---- the hot path --------------------------------------------------------------------------- */
/* Replaces `for _ in range(n_steps): update()` (bmi_topoflow_glacier.py:413-465, :489-490):
 * advances every cell n_steps timesteps starting at absolute step `step0` (0 = first update after
 * initialize) in ONE launch, state held in registers across steps.
 *   forcing      dev [n_steps][5][n_cells] (TFG_N_FORCING order); [n_steps][5][n_cols] with a forcing map
 *   record       dev [n_steps][popcount(record_mask)][n_cells] or NULL: per-step series of the
 *                quantities whose tfg_rec bit is set, rows in ascending bit order
 *   basin_agg    dev [n_steps][n_basin][TFG_N_AGG] float64 or NULL: ACCUMULATED INTO (zero it first);
 *                replaces np.sum(...) at :567-568,:1486-1494 and the driver-side `* da_m2`
 *                (examples/run_topoflow_glacier.py:115); int64 fixed-point accumulators under TFG_OPT_EXACT_AGG
 * With an objective bound (tfg_bind_objective), the steps of [step0, step0 + n_steps) inside its window are scored.
 * n_steps == 1 re-sums the snowfall window exactly every step (the literal update()).          */
TFG_API int tfg_run(tfg_ctx* ctx, const void* forcing, int64_t step0, int32_t n_steps, void* record, uint64_t record_mask,
            void* basin_agg, int32_t n_basin, void* stream);

/* ---- forcing ingestion (replaces the driver loop, examples/run_topoflow_glacier.py:40-73) ---- */
/* cudaMemcpyAsync of one pinned host block to the device on `stream`, then records `done_event`
 * (cudaEvent_t as void*, may be NULL).                                                          */
TFG_API int tfg_ingest_async(tfg_ctx* ctx, const void* pinned_src, void* dev_dst, size_t bytes, void* stream,
                     void* done_event);
/* Page-locked host staging memory for the sources of tfg_ingest_async (cudaHostAlloc; no context needed).  With
 * write_combined != 0 the block is write-combined: host writes stream past the CPU caches and the device's reads over
 * PCIe need no cache snoop -- meant for buffers the host only fills (host READS of such memory are slow).           */
TFG_API int tfg_host_alloc(void** out, size_t bytes, int write_combined);
TFG_API int tfg_host_free(void* block);
/* 1 if `p` points into page-locked host memory (cudaHostAlloc / cudaHostRegister, whoever allocated it), else 0 */
TFG_API int tfg_host_is_pinned(const void* p);
/* raw met columns -> live forcings, on the device:
 *   raw dev [n_steps][6][n_cells] float64 (raw_elem_size 8) or float32 (4; widened exactly, e.g. AORC/NWM
 *       single-precision sources): RAINRATE [mm/h], T2D [K], PSFC [Pa], Q2D, U2D, V2D
 *   out dev [n_steps][5][n_cells] (context element type):
 *   P = RAINRATE*1e-3, T_air = -273.15 + T2D, P_air, Hum_sp, uz = sqrt(U2D^2 + V2D^2)             */
TFG_API int tfg_convert_forcing(tfg_ctx* ctx, const void* raw, int raw_elem_size, void* out, int64_t n_steps,
                                int64_t n_cells, void* stream);
/* the same from PACKED columns, as NetCDF met archives store them (scale_factor / add_offset per variable, e.g. the
 * NWM / AORC forcing files behind the per-catchment CSVs of examples/run_topoflow_glacier.py:30-49): raw dev int16
 * [n_steps][6][n_cells]; value = (double)raw * scale[v] + offset[v] (two IEEE operations, so a host statement
 * raw * scale + offset in float64 gives the same bits), then the unit conversions above.  12 bytes per cell-step cross
 * PCIe instead of 24 (float32) or 48 (float64).  scale / offset are HOST arrays of 6 doubles.                      */
TFG_API int tfg_convert_forcing_packed(tfg_ctx* ctx, const int16_t* raw, const double* scale, const double* offset, void* out,
                                       int64_t n_steps, int64_t n_cells, void* stream);
/* wait (device-side) on `stream` for an event recorded by tfg_ingest_async on another stream     */
TFG_API int tfg_stream_wait_event(tfg_ctx* ctx, void* stream, void* event);

/* ---- hydrograph post-processing (SURVEY.md 8f) ------------------------------------------------ */
/* causal FIR along time of n_series float64 series stored [n_steps][n_series] (device):
 * out[t][j] = sum_{k<taps} weights[k]*series[t-k][j]; with 20 taps of 0.05 this is the "mock routing"
 * np.convolve(output_m_total, weights, "full")[:T] of examples/run_topoflow_glacier.py:129-131     */
TFG_API int tfg_route_fir(tfg_ctx* ctx, const double* series, double* out, const double* weights, int32_t taps,
                          int64_t n_steps, int64_t n_series, void* stream);

/* ---- measurement helper ---------------------------------------------------------------------- */
/* DFMA microbenchmark (8 independent chains per thread, full chip): thread-level DFMA/s, i.e. FP64 FLOP/s / 2.
 * bench.py divides it by the kernel's FP64 instruction count per cell-step to get the compute roofline.      */
TFG_API int tfg_measure_fp64_peak(tfg_ctx* ctx, double* dfma_thread_ops_per_s, void* stream);

/* ---- synthetic workloads for bench.py (SURVEY.md 8d cfg 4/5) ---------------------------------- */
/* counter-based (Philox4x32-10) hourly forcing keyed by (seed, cell, absolute step); storm_cells > 1 makes
 * `storm_cells` consecutive cells share the precipitation occurrence (spatially coherent weather), 1 = iid     */
TFG_API int tfg_synth_forcing(tfg_ctx* ctx, void* forcing, int64_t step0, int32_t n_steps, int64_t n_cells,
                      const void* elev_m /* dev [n_cells], context element type */, uint64_t seed,
                      int64_t storm_cells, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TFGLACIER_H */
