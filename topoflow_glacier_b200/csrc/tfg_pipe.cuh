// tfg_pipe.cuh -- the fast float64 melt kernel with a software-pipelined time loop.
//
// Same path and same arithmetic as run_kernel<FastF64> (tfg_run.cuh): one thread = one cell, state in registers for the
// whole launch.  The difference is the ORDER of the work inside the loop.  update() falls into a part that does not read
// the carried state (lean_forcing, tfg_physics.cuh: ~60 % of the FP64 work) and a part that does (lean_state).  Here the
// loop body evaluates the forcing part of step t+1 and the state part of step t in ONE basic block: two independent
// instruction streams per thread, so that the FP64 latency of one chain is filled with the other (ncu: `wait` -- a
// dependent FP64 instruction waiting out the pipe -- was the top stall of the single-stream kernel at 5 warps per
// scheduler).  Results are bit-identical to the single-stream kernel (same two device functions).
// Steps whose forcing or state is not physically sane (missing data, absurd values) run through the strict step of
// tfg_physics.cuh, one stream at a time, exactly as in run_kernel.
#pragma once
#include "tfg_run.cuh"

namespace tfg {

#ifndef TFG_PIPE_MIN_BLOCKS
#define TFG_PIPE_MIN_BLOCKS 4
#endif

template <bool REC, bool AGG, bool VOL>
__global__ void __launch_bounds__(kBlock, TFG_PIPE_MIN_BLOCKS) run_kernel_pipe(const __grid_constant__ RunParams<double> p) {
  using P = FastF64;
  using R = Num<P>;
  const int64_t gid = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  const bool active = gid < p.n_cells;
  const int64_t c = active ? gid : p.n_cells - 1;
  const int64_t N = p.n_cells;

  for (int i = threadIdx.x; i < fm::kTabDoubles; i += kBlock)   // exp / log lookup tables -> dynamic shared memory
    fm::tfg_tabs[i] = (i < 64) ? fm::kExpTab[i] : fm::kLogTab[(i - 64) >> 1][(i - 64) & 1];
  __syncthreads();
  __shared__ double sm_cell[kSCount][kBlock];   // per-cell constants + diagnostic integrals, one column per thread
  SmemCell<double, kBlock> s;
  s.base = (unsigned)__cvta_generic_to_shared(&sm_cell[0][threadIdx.x]);
  s.set(kSaElev, __ldg(p.a_elev + c)); s.set(kSSinLat, __ldg(p.sin_lat + c)); s.set(kSCosLat, __ldg(p.cos_lat + c));
  s.set(kSNegTanLat, __ldg(p.neg_tan_lat + c)); s.set(kSSinEq, __ldg(p.sin_eq + c)); s.set(kSCosEq, __ldg(p.cos_eq + c));
  s.set(kSNegTanEq, __ldg(p.neg_tan_eq + c)); s.set(kSDlon, __ldg(p.dlon + c)); s.set(kSTNoon, __ldg(p.t_noon + c));
  s.set(kSDa, __ldg(p.da_m2 + c)); s.set(kSTrs, __ldg(p.t_rs + c));
  s.set(kSCB, 0); s.set(kSSB, 0); s.set(kSCB2, 0); s.set(kSSB2, 0);
  const double lon = __ldg(p.lon + c);
  const int tz = p.tz_idx ? (int)__ldg(p.tz_idx + c) : 0;

  CellState<double> st;
  st.h_snow = p.h_snow[c]; st.h_swe = p.h_swe[c]; st.h_ice = p.h_ice[c]; st.h_iwe = p.h_iwe[c];
  st.eccs = p.eccs[c]; st.ecci = p.ecci[c]; st.albedo = p.albedo[c]; st.n_days = p.n_days[c];
  st.swe_lo = st.iwe_lo = 0;
  const bool have_vol = VOL && p.vol_P != nullptr;
  s.set(kSVolP, have_vol ? p.vol_P[c] : 0); s.set(kSVolPR, have_vol ? p.vol_PR[c] : 0);
  s.set(kSVolPS, have_vol ? p.vol_PS[c] : 0); s.set(kSVolSM, have_vol ? p.vol_SM[c] : 0);
  s.set(kSVolIM, have_vol ? p.vol_IM[c] : 0); s.set(kSPmax, have_vol ? p.P_max[c] : 0);

  // incremental window sum (see run_kernel): re-derived exactly inside a fixed 1e-9 m band around the 0.03 m threshold
  const int slots = p.ring_slots;
  int slot = (int)(p.step0 % slots);
  double* ring = p.ring + c;
  double tot = 0.0, n_round = (double)slots + 16.0;
  constexpr double kMaxRoundings = 600.0;
  bool carried = false;
  if (p.win_carry != nullptr) {
    const double n0 = p.win_carry[2 * N + c];
    if (n0 + (double)(2 * p.n_steps) <= kMaxRoundings) {  // false for the NaN that marks "no valid sum"
      tot = p.win_carry[c]; n_round = n0;
      carried = true;
    }
  }
  if (!carried)
    for (int j = 0; j < slots; ++j) tot = __dadd_rn(tot, ring[(int64_t)j * N]);

  int basin = 0;
  bool warp_uniform = false;
  const bool have_agg = AGG && p.basin_agg != nullptr && p.basin_id != nullptr;
  if (have_agg) {
    basin = __ldg(p.basin_id + c);
    warp_uniform = __all_sync(0xffffffffu, basin == __shfl_sync(0xffffffffu, basin, 0));
  }

  const int64_t FN = p.n_cols;
  const double* f = p.forcing + (p.forcing_col ? (int64_t)__ldg(p.forcing_col + c) : c);
  auto finite = [](double v) { return ((unsigned)__double2hiint(v) & 0x7ff00000u) != 0x7ff00000u; };
  auto in_range = [](double v, double lo, double hi) {
    const unsigned h = (unsigned)__double2hiint(v), l = (unsigned)__double2hiint(lo), u = (unsigned)__double2hiint(hi);
    return (h - l) < (u - l);
  };
  // P in [0, 10) m/h, |T_air| < 90 degC, P_air in [1e3, 2e5) Pa, q in [1e-7, 0.2), uz = 0 or in [1e-100, 200)
  auto forcing_sane = [&](double f0, double f1, double f2, double f3, double f4) {
    return ((unsigned)__double2hiint(f0) < (unsigned)__double2hiint(10.0)) &&
           (((unsigned)__double2hiint(f1) & 0x7fffffffu) < (unsigned)__double2hiint(90.0)) && in_range(f2, 1e3, 2e5) &&
           in_range(f3, 1e-7, 0.2) && (in_range(f4, 1e-100, 200.0) || f4 == 0.0);
  };
  auto state_finite = [&]() {
    return finite(st.h_snow) && finite(st.h_swe) && finite(st.h_ice) && finite(st.h_iwe) && finite(st.eccs) &&
           finite(st.ecci) && finite(st.albedo) && finite(st.n_days);
  };
  bool state_ok = state_finite();
  bool statics_sane = fabs(s.get(kSaElev)) < 2.0e5 && finite(lon);
  for (int i = kSSinLat; i <= kSTrs; ++i) statics_sane = statics_sane && finite(s.get(i));

  double LC = 0.0;
  double gmt_prev = __longlong_as_double(0x7ff8000000000000ll);   // NaN: the first step always sets the zone
  auto set_zone = [&](double gmt) {       // True_Solar_Noon, solar_funcs.py:1466-1468 + the per-cell angle-addition pair
    LC = ((gmt * 15.0) - lon) * (1.0 / 15.0);
    const double B = p.k.omega * LC;
    double sb, cb, sb2, cb2;
    sincos(B, &sb, &cb); sincos(B - s.get(kSDlon), &sb2, &cb2);
    s.set(kSSB, sb); s.set(kSCB, cb); s.set(kSSB2, sb2); s.set(kSCB2, cb2);
  };
  // forcing part of step `ts` from the five raw values; false = not sane, nothing computed
  auto forcing_part = [&](int ts, double f0, double f1, double f2, double f3, double f4, Derived<double>& d) -> bool {
    const double gmt = p.gmt[ts * p.n_tz + tz];
    if (!(gmt == gmt_prev)) { gmt_prev = gmt; set_zone(gmt); }   // first step, or DST switch
    const bool ok = __all_sync(0xffffffffu, forcing_sane(f0, f1, f2, f3, f4) && statics_sane) && !p.k.satterlund;
    if (ok) lean_forcing(p.k, p.rows[ts], s, LC, f0, f1, f2, f3, f4, d);
    return ok;
  };

  double f0 = __ldcs(f), f1 = __ldcs(f + FN), f2 = __ldcs(f + 2 * FN), f3 = __ldcs(f + 3 * FN), f4 = __ldcs(f + 4 * FN);
  Derived<double> d_cur;
  bool fs_cur = forcing_part(0, f0, f1, f2, f3, f4, d_cur);
  if (p.n_steps > 1) {
    const double* fn = f + (int64_t)(TFG_N_FORCING * FN);
    f0 = __ldcs(fn); f1 = __ldcs(fn + FN); f2 = __ldcs(fn + 2 * FN); f3 = __ldcs(fn + 3 * FN); f4 = __ldcs(fn + 4 * FN);
  }
  double r_old = ring[(int64_t)slot * N];

  StepOut<double> o;
  double tot_now = 0.0;
  for (int t = 0; t < p.n_steps; ++t) {
    const bool wrap = (slot + 1 == slots);
    const int slot_next = wrap ? 0 : slot + 1;
    bool applied = false;
    auto window = [&](double ring_new) -> double {   // np.roll(-1) + write of the newest slot + np.sum, :1027-1037
      if (applied) return tot_now;
      applied = true;
      if (active) ring[(int64_t)slot * N] = ring_new;
      tot = __dadd_rn(__dsub_rn(tot, r_old), ring_new);
      // sums >= 1e4 m and NaN / inf of either sign take the exact path every step (see run_kernel)
      const bool near = (fabs(tot - kLit.snow_thr) <= 1e-9) || (((unsigned)__double2hiint(tot) & 0x7fffffffu) >= 0x40c38800u);
      if (near) { tot = window_sum_exact<P>(ring, N, slots, slot).v; n_round = 16.0; }
      tot_now = tot;
      return tot;
    };
    Derived<double> d_next;
    bool fs_next = false;
    const bool have_next = t + 1 < p.n_steps;
    const bool lean_now = fs_cur && __all_sync(0xffffffffu, state_ok);
    if (lean_now) {
      // ---- the common case, ONE basic block: forcing part of step t+1 beside the state part of step t ----------
      if (have_next) fs_next = forcing_part(t + 1, f0, f1, f2, f3, f4, d_next);
      if (t + 2 < p.n_steps) {   // raw forcing of step t+2 (the registers of step t+1 are free again)
        const double* fn = f + (int64_t)(t + 2) * (TFG_N_FORCING * FN);
        f0 = __ldcs(fn); f1 = __ldcs(fn + FN); f2 = __ldcs(fn + 2 * FN); f3 = __ldcs(fn + 3 * FN); f4 = __ldcs(fn + 4 * FN);
      }
      lean_state<VOL>(p.k, s, st, d_cur, window, o);
    } else {
      // ---- strict step t (libdevice, IEEE division, NumPy's NaN rules) from the raw forcing, re-read ------------
      using S = Num<StrictF64>;
      const double* fc = f + (int64_t)t * (TFG_N_FORCING * FN);
      const double g0 = __ldcs(fc), g1 = __ldcs(fc + FN), g2 = __ldcs(fc + 2 * FN), g3 = __ldcs(fc + 3 * FN), g4 = __ldcs(fc + 4 * FN);
      const S LCs = ((S(p.gmt[t * p.n_tz + tz]) * 15.0) - S(lon)) / 15.0;
      auto win_s = [&](double x) { return window(x); };
      cell_step<StrictF64, VOL>(p.k, p.rows[t], s, LCs, st, S(g0), S(g1), S(g2), S(g3), S(g4), win_s, []() {}, o);
      state_ok = state_finite();
      if (have_next) fs_next = forcing_part(t + 1, f0, f1, f2, f3, f4, d_next);
      if (t + 2 < p.n_steps) {
        const double* fn = f + (int64_t)(t + 2) * (TFG_N_FORCING * FN);
        f0 = __ldcs(fn); f1 = __ldcs(fn + FN); f2 = __ldcs(fn + 2 * FN); f3 = __ldcs(fn + 3 * FN); f4 = __ldcs(fn + 4 * FN);
      }
    }
    n_round += 2.0;
    r_old = ring[(int64_t)slot_next * N];   // next step's oldest entry (after this step's store)

    if constexpr (REC) {
      if (active && p.record != nullptr) {
        double* rp = p.record + ((int64_t)t * p.n_rec) * N + c;
        const uint64_t m = p.record_mask;
        int r = 0;
#define TFG_PUT(bit, val)              \
  if ((m >> (bit)) & 1ull) {           \
    rp[(int64_t)r * N] = (val);        \
    ++r;                               \
  }
        TFG_PUT(TFG_REC_H_SNOW, st.h_snow) TFG_PUT(TFG_REC_H_SWE, st.h_swe) TFG_PUT(TFG_REC_SM, o.SM)
        TFG_PUT(TFG_REC_H_ICE, st.h_ice) TFG_PUT(TFG_REC_H_IWE, st.h_iwe) TFG_PUT(TFG_REC_IM, o.IM)
        TFG_PUT(TFG_REC_M_TOTAL, o.M_total) TFG_PUT(TFG_REC_RH, o.RH) TFG_PUT(TFG_REC_P0, o.p0)
        TFG_PUT(TFG_REC_E_SAT_AIR, o.e_sat_air) TFG_PUT(TFG_REC_E_AIR, o.e_air) TFG_PUT(TFG_REC_T_DEW, o.T_dew)
        TFG_PUT(TFG_REC_T_SURF, o.T_surf) TFG_PUT(TFG_REC_E_SAT_SURF, o.e_sat_surf) TFG_PUT(TFG_REC_RI, o.Ri)
        TFG_PUT(TFG_REC_DN, o.Dn) TFG_PUT(TFG_REC_DH, o.Dh) TFG_PUT(TFG_REC_QH, o.Qh) TFG_PUT(TFG_REC_W_P, o.W_p)
        TFG_PUT(TFG_REC_E_SURF, o.e_surf) TFG_PUT(TFG_REC_QE, o.Qe) TFG_PUT(TFG_REC_TSN_OFFSET, o.th)
        TFG_PUT(TFG_REC_ALBEDO, st.albedo) TFG_PUT(TFG_REC_N_DAYS, st.n_days) TFG_PUT(TFG_REC_QN_SW, o.Qn_SW)
        TFG_PUT(TFG_REC_EM_AIR, o.em_air) TFG_PUT(TFG_REC_QN_LW, o.Qn_LW) TFG_PUT(TFG_REC_Q_SUM, o.Q_sum)
        TFG_PUT(TFG_REC_ECCS, st.eccs) TFG_PUT(TFG_REC_ECCI, st.ecci) TFG_PUT(TFG_REC_SNOW3DAY, tot_now)
        TFG_PUT(TFG_REC_P_RAIN, o.P_rain) TFG_PUT(TFG_REC_P_SNOW, o.P_snow)
#undef TFG_PUT
      }
    }
    if constexpr (AGG) {
      if (have_agg) {   // area-weighted basin sums, see run_kernel
        const double da = s.get(kSDa);
        double v0 = active ? o.M_total * da : 0.0;
        double v1 = active ? st.h_swe * da : 0.0;
        double v2 = active ? st.h_iwe * da : 0.0;
        const int64_t entry = ((int64_t)t * p.n_basin + basin) * TFG_N_AGG;
        double* dst = static_cast<double*>(p.basin_agg) + entry;
        long long* acc = static_cast<long long*>(p.basin_agg) + 2 * entry;
        if (warp_uniform) {
          const unsigned full = 0xffffffffu;
          const int lane = threadIdx.x & 31;
          const bool hi = (lane & 16) != 0;
          double k0 = hi ? v2 : v0, k1 = hi ? 0.0 : v1;
          k0 += __shfl_xor_sync(full, hi ? v0 : v2, 16);
          k1 += __shfl_xor_sync(full, hi ? v1 : 0.0, 16);
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
        } else if (active) {
          if (p.agg_exact) {
            agg_add_exact(acc + 0, v0, p.agg_up[0], p.agg_lo, p.agg_bad); agg_add_exact(acc + 2, v1, p.agg_up[1], p.agg_lo, p.agg_bad);
            agg_add_exact(acc + 4, v2, p.agg_up[2], p.agg_lo, p.agg_bad);
          } else {
            atomicAdd(dst + 0, v0); atomicAdd(dst + 1, v1); atomicAdd(dst + 2, v2);
          }
        }
      }
    }
    d_cur = d_next;
    fs_cur = fs_next;
    slot = slot_next;
  }

  if (active && p.win_carry != nullptr) {
    p.win_carry[c] = tot; p.win_carry[N + c] = fabs(tot); p.win_carry[2 * N + c] = n_round;
  }
  if (active) {
    p.h_snow[c] = st.h_snow; p.h_swe[c] = st.h_swe; p.h_ice[c] = st.h_ice; p.h_iwe[c] = st.h_iwe;
    p.eccs[c] = st.eccs; p.ecci[c] = st.ecci; p.albedo[c] = st.albedo; p.n_days[c] = st.n_days;
    p.SM[c] = o.SM; p.IM[c] = o.IM; p.M_total[c] = o.M_total; p.RH[c] = o.RH;
    if (have_vol) {
      p.vol_P[c] = s.get(kSVolP); p.vol_PR[c] = s.get(kSVolPR); p.vol_PS[c] = s.get(kSVolPS);
      p.vol_SM[c] = s.get(kSVolSM); p.vol_IM[c] = s.get(kSVolIM); p.P_max[c] = s.get(kSPmax);
    }
  }
}

// launches of one step re-sum the window exactly (the literal update()) and stay with run_kernel, as do TMA-staged ones
inline cudaError_t launch_run_pipe(const RunParams<double>& p, bool rec, bool agg, bool vol, cudaStream_t stream) {
  const unsigned grid = (unsigned)((p.n_cells + kBlock - 1) / kBlock);
  const size_t dyn = fm::kTabDoubles * sizeof(double);
  if (rec) run_kernel_pipe<true, true, true><<<grid, kBlock, dyn, stream>>>(p);
  else if (agg && vol) run_kernel_pipe<false, true, true><<<grid, kBlock, dyn, stream>>>(p);
  else if (agg) run_kernel_pipe<false, true, false><<<grid, kBlock, dyn, stream>>>(p);
  else if (vol) run_kernel_pipe<false, false, true><<<grid, kBlock, dyn, stream>>>(p);
  else run_kernel_pipe<false, false, false><<<grid, kBlock, dyn, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace tfg
