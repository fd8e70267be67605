// tfg_ws.cuh -- EXPERIMENT (round 2, build with -DTFG_WS=1; not the default): the fast float64 melt kernel, warp-specialised
// into producer warps and consumer warps.  Bit-identical to the split single-stream kernel, no deadlocks, and slower:
// 25.5 G cell-steps/s with one producer warp per consumer warp at 80 registers (24 warps/SM), 22.0 G at 64 registers
// (32 warps/SM, 300 B of spills), 12.7 G with one producer warp per two consumer warps -- against 30.0 G for the
// single-stream kernel (profiles/r2_experiments.md).  A warp of this code issues one instruction per ~15 cycles on its
// own; it would take >= 10 warps per scheduler to hide that, and the ring, the barriers and the duplicated prologue cost
// more than the 20 % of extra warps return.
//
// Same path and the same two device functions as the single-stream fast kernel (tfg_physics.cuh: lean_forcing,
// lean_state), so results are bit-identical to it.  What changes is WHO evaluates them.  The round-2 experiments
// (profiles/r2_experiments.md) showed that this kernel hides its FP64 latency with thread-level parallelism and that every
// attempt to add instruction-level parallelism lost more in registers than it won; 96 registers per thread cap the
// single-stream kernel at 20 warps per SM.  update() falls into a part that never reads the carried state (met block,
// vapour terms, incoming longwave, clear-sky shortwave up to its linear dependence on albedo, the snowfall wet bulb:
// ~40 % of the instructions) and a part that does (log law, albedo, net fluxes, melt, water equivalents, window,
// aggregates).  Here a block of 128 cells is served by 4 CONSUMER warps, which own the state of one cell per thread for
// the whole launch, and 2 PRODUCER warps, which own nothing: a producer lane evaluates the forcing part of its two cells
// (one in each of the two consumer warps it serves) a few timesteps ahead and hands ten numbers per cell-step to the
// consumer thread of that cell through a ring of stages in shared memory.  Neither role needs the other's registers:
// both fit in 80, and the SM holds 24 warps whose instruction streams are 560 and 650 instructions per step instead of
// 20 warps with 865.
//
//   producer warp w, step t:  wait empty[t % S][w]  ->  5 forcing loads, lean_forcing  ->  10 st.shared  ->  arrive full[t % S][w]
//   consumer warp w, step t:  wait full[t % S][w]   ->  lean_state reading the stage at the point of use  ->  arrive empty[t % S][w]
//
// The mbarriers couple a producer warp with ITS consumer warp only; the four pairs of a block drift freely.
// Steps whose forcing or state is not physically sane run through the strict step on the consumer, from the raw forcing.
#pragma once
#include "tfg_run.cuh"

namespace tfg {

#ifndef TFG_WS_STAGES
#define TFG_WS_STAGES 3
#endif
#ifndef TFG_WS_MIN_BLOCKS
#define TFG_WS_MIN_BLOCKS 4
#endif
#ifndef TFG_WS_RATIO   // consumer warps served by one producer warp: the state part is ~1.7x the forcing part in instructions,
#define TFG_WS_RATIO 2 // so one producer warp keeps two consumer warps busy
#endif
constexpr int kWsCells = 128;                 // cells per block = consumer threads
constexpr int kWsRatio = TFG_WS_RATIO;
constexpr int kWsThreads = kWsCells + kWsCells / kWsRatio;
constexpr int kWsStages = TFG_WS_STAGES;
constexpr int kWsWarps = kWsCells / 32;
// dynamic shared memory: exp / log tables | cell constants + integrals [kSCount][128] | ring [S][10][128] | flags | barriers
constexpr size_t kWsSmem = (size_t)(fm::kTabDoubles + kSCount * kWsCells + kWsStages * kDHand * kWsCells) * sizeof(double) +
                           (size_t)kWsStages * kWsWarps * (sizeof(int) + 2 * sizeof(uint64_t));

__device__ __forceinline__ void mbar_arrive_release(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait_acquire(uint64_t* bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\tWS_WAIT:\n\t"
      "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 P1, [%0], %1, %2;\n\t"   // suspends the warp (no issue slots) up
      "@P1 bra WS_DONE;\n\tbra WS_WAIT;\n\tWS_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"(20000u)   // to ~20 us per try
      : "memory");
}

template <bool AGG, bool VOL>
__global__ void __launch_bounds__(kWsThreads, TFG_WS_MIN_BLOCKS) run_kernel_ws(const __grid_constant__ RunParams<double> p) {
  using P = FastF64;
  const bool producer = threadIdx.x >= kWsCells;
  const int lane = threadIdx.x & 31;
  const int64_t N = p.n_cells;
  // consumer: one cell; producer warp pw serves the consumer warps pw*kWsRatio ... + kWsRatio-1, one cell per lane in each
  const int pw = producer ? (threadIdx.x - kWsCells) >> 5 : 0;
  const int tid = producer ? (pw * kWsRatio) * 32 + lane : threadIdx.x;   // first (or only) cell of this thread within the block
  const int wp = tid >> 5;                                                 // consumer warp of that cell

  double* sm_cell = fm::tfg_tabs + fm::kTabDoubles;                      // [kSCount][kWsCells]
  double* sm_ring = sm_cell + kSCount * kWsCells;                        // [stage][value][cell]
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(sm_ring + kWsStages * kDHand * kWsCells);   // [stage][consumer warp]
  uint64_t* bar_empty = bar_full + kWsStages * kWsWarps;
  int* sm_flag = reinterpret_cast<int*>(bar_empty + kWsStages * kWsWarps);                     // [stage][consumer warp]: 1 = not sane

  for (int i = threadIdx.x; i < fm::kTabDoubles; i += kWsThreads)
    fm::tfg_tabs[i] = (i < 64) ? fm::kExpTab[i] : fm::kLogTab[(i - 64) >> 1][(i - 64) & 1];
  if (threadIdx.x < kWsStages * kWsWarps) {
    mbar_init(&bar_full[threadIdx.x], 1);
    mbar_init(&bar_empty[threadIdx.x], 1);
  }
  auto cell_of = [&](int tcell) { const int64_t g = (int64_t)blockIdx.x * kWsCells + tcell; return g < N ? g : N - 1; };
  auto column = [&](int tcell) { return SmemCell<double, kWsCells>{(unsigned)__cvta_generic_to_shared(sm_cell + tcell)}; };
  if (producer) {   // the producer fills the constants it reads, the consumer its own: no cross-role dependence but the barrier below
#pragma unroll
    for (int h = 0; h < kWsRatio; ++h) {
      auto sc = column(tid + 32 * h);
      const int64_t ch = cell_of(tid + 32 * h);
      sc.set(kSaElev, __ldg(p.a_elev + ch)); sc.set(kSSinLat, __ldg(p.sin_lat + ch)); sc.set(kSCosLat, __ldg(p.cos_lat + ch));
      sc.set(kSNegTanLat, __ldg(p.neg_tan_lat + ch)); sc.set(kSSinEq, __ldg(p.sin_eq + ch)); sc.set(kSCosEq, __ldg(p.cos_eq + ch));
      sc.set(kSNegTanEq, __ldg(p.neg_tan_eq + ch)); sc.set(kSDlon, __ldg(p.dlon + ch)); sc.set(kSTNoon, __ldg(p.t_noon + ch));
      sc.set(kSTrs, __ldg(p.t_rs + ch));
      sc.set(kSCB, 0); sc.set(kSSB, 0); sc.set(kSCB2, 0); sc.set(kSSB2, 0);
    }
  } else {
    auto sc = column(tid);
    const int64_t ch = cell_of(tid);
    const bool have_vol = VOL && p.vol_P != nullptr;
    sc.set(kSDa, __ldg(p.da_m2 + ch));
    sc.set(kSVolP, have_vol ? p.vol_P[ch] : 0); sc.set(kSVolPR, have_vol ? p.vol_PR[ch] : 0);
    sc.set(kSVolPS, have_vol ? p.vol_PS[ch] : 0); sc.set(kSVolSM, have_vol ? p.vol_SM[ch] : 0);
    sc.set(kSVolIM, have_vol ? p.vol_IM[ch] : 0); sc.set(kSPmax, have_vol ? p.P_max[ch] : 0);
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();   // tables, constants and barriers are in place; from here on the two roles only meet at their mbarriers

  const int64_t FN = p.n_cols;
  auto finite = [](double v) { return ((unsigned)__double2hiint(v) & 0x7ff00000u) != 0x7ff00000u; };
  const unsigned ring_stride = kWsCells * sizeof(double);

  if (producer) {
    // ============================ PRODUCER: the state-free part of update(), a few steps ahead ============================
    const double* f[kWsRatio];
    int64_t cc[kWsRatio];
    double lon[kWsRatio], LC[kWsRatio], gmt_prev[kWsRatio];
    int tz[kWsRatio];
    bool act[kWsRatio], statics_sane[kWsRatio];
#pragma unroll
    for (int h = 0; h < kWsRatio; ++h) {
      const int tc = tid + 32 * h;
      auto sc = column(tc);
      cc[h] = cell_of(tc);
      act[h] = (int64_t)blockIdx.x * kWsCells + tc < N;
      f[h] = p.forcing + (p.forcing_col ? (int64_t)__ldg(p.forcing_col + cc[h]) : cc[h]);
      lon[h] = __ldg(p.lon + cc[h]);
      tz[h] = p.tz_idx ? (int)__ldg(p.tz_idx + cc[h]) : 0;
      LC[h] = 0.0;
      gmt_prev[h] = __longlong_as_double(0x7ff8000000000000ll);   // NaN: the first step always sets the zone
      bool ok = fabs(sc.get(kSaElev)) < 2.0e5 && finite(lon[h]);  // finite tables, |elev| < 700 km
      for (int i = kSSinLat; i <= kSTNoon; ++i) ok = ok && finite(sc.get(i));
      statics_sane[h] = ok && finite(sc.get(kSTrs)) && finite(__ldg(p.da_m2 + cc[h]));
    }
    auto in_range = [](double v, double lo, double hi) {
      const unsigned h = (unsigned)__double2hiint(v), l = (unsigned)__double2hiint(lo), u = (unsigned)__double2hiint(hi);
      return (h - l) < (u - l);
    };
    // work items in order (t, h): the forcings of the NEXT item are requested while the current one is evaluated
    double f0 = __ldcs(f[0]), f1 = __ldcs(f[0] + FN), f2 = __ldcs(f[0] + 2 * FN), f3 = __ldcs(f[0] + 3 * FN), f4 = __ldcs(f[0] + 4 * FN);
    for (int t = 0; t < p.n_steps; ++t) {
      const int sg = t % kWsStages;
      auto work_item = [&](auto H) {   // h as a compile-time constant: the per-cell arrays above stay in registers
        constexpr int h = decltype(H)::value;
        const int tc = tid + 32 * h, w = wp + h;
        auto sc = column(tc);
        const double gmt = p.gmt[t * p.n_tz + tz[h]];
        if (!(gmt == gmt_prev[h])) {   // first step, or DST switch: True_Solar_Noon (solar_funcs.py:1466-1468) + the angle-addition pair
          gmt_prev[h] = gmt;
          LC[h] = ((gmt * 15.0) - lon[h]) * (1.0 / 15.0);
          const double B = p.k.omega * LC[h];
          double sb, cb, sb2, cb2;
          sincos(B, &sb, &cb); sincos(B - sc.get(kSDlon), &sb2, &cb2);
          sc.set(kSSB, sb); sc.set(kSCB, cb); sc.set(kSSB2, sb2); sc.set(kSCB2, cb2);
        }
        // P in [0, 10) m/h, |T_air| < 90 degC, P_air in [1e3, 2e5) Pa, q in [1e-7, 0.2), uz = 0 or in [1e-100, 200)
        const bool sane = ((unsigned)__double2hiint(f0) < (unsigned)__double2hiint(10.0)) &&
                          (((unsigned)__double2hiint(f1) & 0x7fffffffu) < (unsigned)__double2hiint(90.0)) &&
                          in_range(f2, 1e3, 2e5) && in_range(f3, 1e-7, 0.2) && (in_range(f4, 1e-100, 200.0) || f4 == 0.0) &&
                          statics_sane[h];
        const bool ok = __all_sync(0xffffffffu, sane);
        Derived<double> d;
        if (ok) lean_forcing(p.k, p.rows[t], sc, LC[h], f0, f1, f2, f3, f4, d);
        {   // next work item's forcings (this item's are consumed)
          constexpr int hn = (h + 1 == kWsRatio) ? 0 : h + 1;
          const int tn = (h + 1 == kWsRatio) ? t + 1 : t;
          if (tn < p.n_steps) {
            const double* fn = f[hn] + (int64_t)tn * (TFG_N_FORCING * FN);
            f0 = __ldcs(fn); f1 = __ldcs(fn + FN); f2 = __ldcs(fn + 2 * FN); f3 = __ldcs(fn + 3 * FN); f4 = __ldcs(fn + 4 * FN);
          }
        }
        mbar_wait_acquire(&bar_empty[sg * kWsWarps + w], (unsigned)(((t / kWsStages) & 1) ^ 1));   // stage free (fresh barrier: passes)
        if (ok) {
          const unsigned dst = (unsigned)__cvta_generic_to_shared(sm_ring + tc) + (unsigned)sg * (kDHand * ring_stride);
#pragma unroll
          for (int i = 0; i < kDHand; ++i) asm volatile("st.volatile.shared.f64 [%0], %1;" ::"r"(dst + i * ring_stride), "d"(d.v[i]));
          if (t == p.n_steps - 1 && act[h]) p.RH[cc[h]] = d.v[kD_RH];   // BMI output of the last step (does not travel through the ring)
        }
        __syncwarp();
        if (lane == 0) {
          sm_flag[sg * kWsWarps + w] = ok ? 0 : 1;
          mbar_arrive_release(&bar_full[sg * kWsWarps + w]);
        }
      };
      work_item(std::integral_constant<int, 0>{});
      if constexpr (kWsRatio > 1) work_item(std::integral_constant<int, kWsRatio - 1>{});
      static_assert(kWsRatio <= 2, "one or two consumer warps per producer warp");
    }
    return;
  }

  // ============================ CONSUMER: carried state, one cell per thread for the whole launch ============================
  const int64_t c = cell_of(tid);
  const bool active = (int64_t)blockIdx.x * kWsCells + tid < N;
  SmemCell<double, kWsCells> s = column(tid);
  const double* f = p.forcing + (p.forcing_col ? (int64_t)__ldg(p.forcing_col + c) : c);
  const double lon = __ldg(p.lon + c);
  const int tz = p.tz_idx ? (int)__ldg(p.tz_idx + c) : 0;
  const unsigned ring0 = (unsigned)__cvta_generic_to_shared(sm_ring + tid);
  CellState<double> st;
  st.h_snow = p.h_snow[c]; st.h_swe = p.h_swe[c]; st.h_ice = p.h_ice[c]; st.h_iwe = p.h_iwe[c];
  st.eccs = p.eccs[c]; st.ecci = p.ecci[c]; st.albedo = p.albedo[c]; st.n_days = p.n_days[c];
  st.swe_lo = st.iwe_lo = 0;
  const bool have_vol = VOL && p.vol_P != nullptr;
  auto state_finite = [&]() {
    return finite(st.h_snow) && finite(st.h_swe) && finite(st.h_ice) && finite(st.h_iwe) && finite(st.eccs) &&
           finite(st.ecci) && finite(st.albedo) && finite(st.n_days);
  };
  bool state_ok = state_finite();

  // incremental window sum (see run_kernel): re-derived exactly inside a fixed 1e-9 m band around the 0.03 m threshold
  const int slots = p.ring_slots;
  int slot = (int)(p.step0 % slots);
  double* ring = p.ring + c;
  double tot = 0.0, n_round = (double)slots + 16.0;
  constexpr double kMaxRoundings = 600.0;
  bool carried = false;
  if (p.win_carry != nullptr) {
    const double n0 = p.win_carry[2 * N + c];
    if (n0 + (double)(2 * p.n_steps) <= kMaxRoundings) {   // false for the NaN that marks "no valid sum"
      tot = p.win_carry[c]; n_round = n0;
      carried = true;
    }
  }
  if (!carried)
    for (int j = 0; j < slots; ++j) tot = __dadd_rn(tot, ring[(int64_t)j * N]);
  double r_old = ring[(int64_t)slot * N];

  int basin = 0;
  bool warp_uniform = false;
  const bool have_agg = AGG && p.basin_agg != nullptr && p.basin_id != nullptr;
  if (have_agg) {
    basin = __ldg(p.basin_id + c);
    warp_uniform = __all_sync(0xffffffffu, basin == __shfl_sync(0xffffffffu, basin, 0));
  }

  StepOut<double> o;
  bool last_strict = false;
  for (int t = 0; t < p.n_steps; ++t) {
    const int sg = t % kWsStages;
    const bool wrap = (slot + 1 == slots);
    const int slot_next = wrap ? 0 : slot + 1;
    auto window = [&](double ring_new) -> double {   // np.roll(-1) + write of the newest slot + np.sum, :1027-1037
      if (active) ring[(int64_t)slot * N] = ring_new;
      tot = __dadd_rn(__dsub_rn(tot, r_old), ring_new);
      // sums >= 1e4 m and NaN / inf of either sign take the exact path every step (see run_kernel)
      const bool near = (fabs(tot - kLit.snow_thr) <= 1e-9) || (((unsigned)__double2hiint(tot) & 0x7fffffffu) >= 0x40c38800u);
      if (near) { tot = window_sum_exact<P>(ring, N, slots, slot).v; n_round = 16.0; }
      return tot;
    };
    mbar_wait_acquire(&bar_full[sg * kWsWarps + wp], (unsigned)((t / kWsStages) & 1));
    const bool insane = *reinterpret_cast<volatile int*>(&sm_flag[sg * kWsWarps + wp]) != 0;
    last_strict = insane || !__all_sync(0xffffffffu, state_ok);
    if (!last_strict) {
      const SmemDerived d{ring0 + (unsigned)sg * (kDHand * ring_stride), ring_stride};
      lean_state<VOL>(p.k, s, st, d, window, o);
    } else {
      // strict step (libdevice, IEEE division, NumPy's NaN rules) from the raw forcing: missing data and absurd values
      // poison a cell exactly as they do in the reference
      using S = Num<StrictF64>;
      const double* fc = f + (int64_t)t * (TFG_N_FORCING * FN);
      const double g0 = __ldcs(fc), g1 = __ldcs(fc + FN), g2 = __ldcs(fc + 2 * FN), g3 = __ldcs(fc + 3 * FN), g4 = __ldcs(fc + 4 * FN);
      const S LCs = ((S(p.gmt[t * p.n_tz + tz]) * 15.0) - S(lon)) / 15.0;
      // the strict step reads the producer-side constants through the same columns
      cell_step<StrictF64, VOL>(p.k, p.rows[t], s, LCs, st, S(g0), S(g1), S(g2), S(g3), S(g4), window, []() {}, o);
      state_ok = state_finite();
    }
    __syncwarp();
    if (lane == 0) mbar_arrive_release(&bar_empty[sg * kWsWarps + wp]);   // the stage may be refilled
    n_round += 2.0;
    r_old = ring[(int64_t)slot_next * N];   // next step's oldest entry (after this step's store)

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
    slot = slot_next;
  }

  if (active && p.win_carry != nullptr) {
    p.win_carry[c] = tot; p.win_carry[N + c] = fabs(tot); p.win_carry[2 * N + c] = n_round;
  }
  if (active) {
    p.h_snow[c] = st.h_snow; p.h_swe[c] = st.h_swe; p.h_ice[c] = st.h_ice; p.h_iwe[c] = st.h_iwe;
    p.eccs[c] = st.eccs; p.ecci[c] = st.ecci; p.albedo[c] = st.albedo; p.n_days[c] = st.n_days;
    p.SM[c] = o.SM; p.IM[c] = o.IM; p.M_total[c] = o.M_total;
    if (last_strict) p.RH[c] = o.RH;   // otherwise the producer stored it
    if (have_vol) {
      p.vol_P[c] = s.get(kSVolP); p.vol_PR[c] = s.get(kSVolPR); p.vol_PS[c] = s.get(kSVolPS);
      p.vol_SM[c] = s.get(kSVolSM); p.vol_IM[c] = s.get(kSVolIM); p.P_max[c] = s.get(kSPmax);
    }
  }
}

// Recording launches, one-step launches (exact window re-sum), TMA staging and SATTERLUND configurations stay with the
// single-stream kernel, which evaluates the same two device functions.
inline cudaError_t launch_run_ws(const RunParams<double>& p, bool agg, bool vol, cudaStream_t stream) {
  const unsigned grid = (unsigned)((p.n_cells + kWsCells - 1) / kWsCells);
  // more than 48 KB of dynamic shared memory is opt-in, per function and device
  auto opt_in = [](const void* fn) { return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem); };
  cudaError_t e = agg ? (vol ? opt_in((const void*)run_kernel_ws<true, true>) : opt_in((const void*)run_kernel_ws<true, false>))
                      : (vol ? opt_in((const void*)run_kernel_ws<false, true>) : opt_in((const void*)run_kernel_ws<false, false>));
  if (e != cudaSuccess) return e;
  if (agg && vol) run_kernel_ws<true, true><<<grid, kWsThreads, kWsSmem, stream>>>(p);
  else if (agg) run_kernel_ws<true, false><<<grid, kWsThreads, kWsSmem, stream>>>(p);
  else if (vol) run_kernel_ws<false, true><<<grid, kWsThreads, kWsSmem, stream>>>(p);
  else run_kernel_ws<false, false><<<grid, kWsThreads, kWsSmem, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace tfg
