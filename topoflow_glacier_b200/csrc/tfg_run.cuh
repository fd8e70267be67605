// tfg_run.cuh -- the fused, time-looping melt kernel (K1) and its launcher.
//
// One thread owns one cell for the whole launch: static tables and carried state are loaded once,
// stay in registers for n_steps timesteps, and are written back once.  Per step a thread reads only
// its five forcings (coalesced, [step][var][cell], streaming loads prefetched one step ahead) plus one
// slot of the 3-day snowfall window.  This replaces the reference's per-step driver loop
// (examples/run_topoflow_glacier.py:64-109) around BmiTopoflowGlacier.update()
// (bmi_topoflow_glacier.py:413-465).
#pragma once
#include <type_traits>

#include "tfg_physics.cuh"
#include "../../include/tfglacier.h"

namespace tfg {

#ifndef TFG_BLOCK
#define TFG_BLOCK 128
#endif
#ifndef TFG_MIN_BLOCKS
#define TFG_MIN_BLOCKS 5
#endif
#ifndef TFG_MIN_BLOCKS_F32
#define TFG_MIN_BLOCKS_F32 8
#endif
#ifndef TFG_CPASYNC  // 1: next-step forcings staged in shared memory by cp.async instead of register prefetches (measured slower)
#define TFG_CPASYNC 0
#endif
#ifndef TFG_CT_REGPF   // column-term kernel: 1 = next step's line prefetched into registers mid-step; 0 = one L1 prefetch of the line
#define TFG_CT_REGPF 0 // mid-step and 128-bit loads at the top of the step (the line is shared by the warp: 38.8 vs 38.3 G)
#endif
#ifndef TFG_WALK_LEAN  // 1: the fast float64 kernel carries the window-slot pointer (as the float32 kernel does) instead of re-deriving it
#define TFG_WALK_LEAN 0   // measured slower (30.6 vs 31.2 G): two more live registers at the 96-register limit
#endif
#ifndef TFG_DA_ZERO    // 1: replica lanes past the last cell carry area 0, so the basin sums need no `active` predicate
#define TFG_DA_ZERO 1
#endif
#ifndef TFG_ZONE_ONCE  // 1: a launch without a DST switch sets each cell's zone terms once instead of comparing the offset every step
#define TFG_ZONE_ONCE 1
#endif
#ifndef TFG_MIN_BLOCKS_LEAN  // fast float64 kernel: cell constants in shared memory, clock rows in the parameter block -> 96 registers
#define TFG_MIN_BLOCKS_LEAN 5
#endif
constexpr int kBlock = TFG_BLOCK;
constexpr int kMaxLaunchSteps = 128;  // timesteps per launch (longer runs are split by tfg_run); 16.5 KB of parameters

template <class raw>
struct RunParams {
  int64_t n_cells, step0;
  int32_t n_steps, ring_slots, n_tz, exact_ring, use_tma;
  int32_t gmt_varies;  // 0: every zone keeps its UTC offset over this launch (no DST switch inside): the zone is set once
  const raw* forcing;
  const int32_t* forcing_col;  // optional: cell -> column of the forcing block (cells of one catchment share a column)
  int64_t n_cols;              // columns of the forcing block (= n_cells without a map)
  const raw *a_elev, *sin_lat, *cos_lat, *neg_tan_lat, *lon, *sin_eq, *cos_eq, *neg_tan_eq, *dlon, *t_noon, *da_m2,
      *t_rs;
  const int32_t* basin_id;
  const uint8_t* tz_idx;
  raw *h_snow, *h_swe, *h_ice, *h_iwe, *eccs, *ecci, *albedo, *n_days, *SM, *IM, *M_total, *RH;
  raw *vol_P, *vol_PR, *vol_PS, *vol_SM, *vol_IM, *P_max;
  raw* ring;
  raw* mass_lo;    // optional [2][n_cells] (float32 mode): low parts of h_swe / h_iwe, see CellState
  raw* win_carry;  // optional [3][n_cells]: incremental window sum, its largest magnitude and its rounding count, carried
                   // from launch to launch so that short launches need not re-read all 72 slots (NaN count = re-seed)
  // Clock-only tables of THIS launch, passed in the kernel parameter block (constant bank): the step index is
  // warp-uniform, so a row is read with uniform loads straight into the operand slots of the FP64 instructions
  // instead of occupying 16 vector registers per thread for the whole step.
  TimeRow<raw> rows[kMaxLaunchSteps];             // indexed by step - step0
  raw gmt[kMaxLaunchSteps * TFG_MAX_TZ];          // [step - step0][n_tz]
  raw* record;
  uint64_t record_mask;
  int32_t n_rec;
  void* basin_agg;      // float64 sums, or int64 {hi, lo} fixed-point accumulators when agg_exact
  int32_t n_basin, agg_exact;
  double agg_up[TFG_N_AGG];  // 2^(40 - E_q)
  long long* agg_bad;   // exact mode: count of contributions left out (non-finite or >= 2^E_q)
  // 16-byte aligned: ptxas pairs neighbouring constants into 128-bit uniform loads; with the block 8 bytes off the fast
  // kernel loses 2 % (measured: profiles/r2_experiments.md).  New members go behind it.
  alignas(16) Consts<raw> k;
  const raw* col_terms;        // optional [n_steps][n_cols][kCtCount] (fast float64 mode, forcing map bound): the column
                               // terms of this launch (column_terms_kernel); the kernel then does not read `forcing`
  const raw* cell_par;         // optional [kPCount][n_cells] per-cell surface factors (tfg_bind_cell_params)
  // objective (tfg_bind_objective): local steps [obj_t_lo, obj_t_hi) of this launch are scored; obj_obs is the
  // observation row of local step obj_t_lo.  obj_acc == nullptr: no objective (the OBJ instantiations are not chosen)
  double* obj_acc;             // [TFG_N_OBJ][n_cells], accumulated into
  const double* obj_obs;       // [obj_t_hi - obj_t_lo][obj_ncols] (rows of this launch)
  const int32_t* obj_col;      // [n_cells] or nullptr (column = cell)
  int64_t obj_ncols;
  int32_t obj_t_lo, obj_t_hi, obj_quantity;
  double agg_lo;               // 2^L: fraction bits of the low word of exact aggregates (with agg_up; here, behind the
                               // members above, so that the kernels without aggregates keep their parameter offsets)
  const raw* fadj;             // optional [2][n_cells] T_air offset and P multiplier (tfg_bind_forcing_adjust); last, so
                               // that the kernels without adjustments keep their parameter offsets
};

// One IEEE operation in the element type, never contracted into a neighbouring multiply-add: the forcing adjustment
// must give the bits of a forcing adjusted in advance (tfg_bind_forcing_adjust)
__device__ __forceinline__ double add_once(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_once(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double mul_once(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_once(float a, float b) { return __fmul_rn(a, b); }

template <class raw> __device__ __forceinline__ raw ld_stream(const raw* p) { return __ldcs(p); }

// The fast step is written for physically meaningful forcings (no guards, no NaN rules); anything else -- missing data,
// absurd values -- takes the strict step.  Integer tests on the high words: one ALU instruction per bound.
template <class raw>
__device__ __forceinline__ bool forcings_sane(raw f0, raw f1, raw f2, raw f3, raw f4) {
  auto in_range = [](raw v, double lo, double hi) {
    const unsigned h = (unsigned)__double2hiint(v), l = (unsigned)__double2hiint(lo), u = (unsigned)__double2hiint(hi);
    return (h - l) < (u - l);
  };
  return ((unsigned)__double2hiint(f0) < (unsigned)__double2hiint(10.0)) &&
         (((unsigned)__double2hiint(f1) & 0x7fffffffu) < (unsigned)__double2hiint(90.0)) &&
         in_range(f2, 1e3, 2e5) && in_range(f3, 1e-7, 0.2) && (in_range(f4, 1e-100, 200.0) || f4 == 0.0);
}

// One element global -> shared without a register in between (LDGSTS): the next step's forcings are in flight for a
// whole timestep, and as register prefetches they would pin ten registers for that long.
template <class raw> __device__ __forceinline__ void cp_async_elem(raw* dst_smem, const raw* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((unsigned)__cvta_generic_to_shared(dst_smem)), "l"(src),
               "n"((int)sizeof(raw))
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// ---- TMA bulk-copy staging of forcing tiles (cp.async.bulk + mbarrier, SASS: UBLKCP / SYNCS) -----------------
// A block of kBlock cells needs, per timestep, five contiguous rows of kBlock elements (one per forcing).  One
// elected thread asks the copy engine for them kStages steps ahead; the rows land in shared memory and complete
// a "full" mbarrier; every thread reads its five values and arrives on an "empty" mbarrier so the stage can be
// refilled.  No register staging, no per-thread address arithmetic, and the prefetch distance is kStages-1 steps.
constexpr int kStages = 4;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\tLAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}


// np.sum over the window in logical order (oldest first), i.e. NumPy's pairwise kernel for n <= 128:
// eight interleaved accumulators, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the remainder.
// `newest` is the physical slot written this step; logical j lives in physical (newest+1+j) % slots.
template <class P>
__device__ __noinline__ Num<P> window_sum_exact(const typename P::raw* ring, int64_t N, int slots, int newest) {
  using R = Num<P>;
  int p = newest + 1;
  if (p >= slots) p -= slots;
  auto next = [&]() {
    R v(ring[(int64_t)p * N]);
    if (++p >= slots) p = 0;
    return v;
  };
  if (slots < 8) {
    R res(0.0);
    for (int i = 0; i < slots; ++i) res = res + next();
    return res;
  }
  R r0 = next(), r1 = next(), r2 = next(), r3 = next(), r4 = next(), r5 = next(), r6 = next(), r7 = next();
  int i = 8;
  for (; i < slots - (slots % 8); i += 8) {
    r0 = r0 + next(); r1 = r1 + next(); r2 = r2 + next(); r3 = r3 + next();
    r4 = r4 + next(); r5 = r5 + next(); r6 = r6 + next(); r7 = r7 + next();
  }
  R res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
  for (; i < slots; ++i) res = res + next();
  return res;
}

// One contribution to an exact basin aggregate: v * up = a + r with a = trunc (|a| < 2^40), b = trunc(r * lo), lo = 2^L;
// both words are added with integer atomics (associative, hence order-independent).  The host chooses L so that the
// low word of C contributions, |sum| < C * 2^L, stays below 2^63 (MeltEngine.agg_exponents).
__device__ __forceinline__ void agg_add_exact(long long* acc, double v, double up, double lo, long long* bad) {
  const double s = v * up;  // a power-of-two scaling: exact
  if (!(fabs(s) < 1099511627776.0)) {  // also catches NaN
    if (bad) atomicAdd(reinterpret_cast<unsigned long long*>(bad), 1ull);
    return;
  }
  const long long a = __double2ll_rz(s);
  const long long b = __double2ll_rz((s - (double)a) * lo);
  if (a) atomicAdd(reinterpret_cast<unsigned long long*>(acc), (unsigned long long)a);
  if (b) atomicAdd(reinterpret_cast<unsigned long long*>(acc) + 1, (unsigned long long)b);
}

// The objective's four float64 sums of this thread's cell, one shared-memory column each for the whole launch (as
// SmemCell keeps the cell constants): volatile accesses, so that they do not occupy registers across the time loop.
struct ObjSums {
  unsigned base;  // shared-window address of this thread's column of row 0
  __device__ __forceinline__ double get(int i) const {
    double x;
    asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(x) : "r"(base + i * kBlock * 8));
    return x;
  }
  __device__ __forceinline__ void set(int i, double x) {
    asm volatile("st.volatile.shared.f64 [%0], %1;" ::"r"(base + i * kBlock * 8), "d"(x));
  }
};

template <class P, bool REC, bool AGG, bool VOL, bool TMA = false, bool PRE = false, bool PAR = false, bool OBJ = false,
          bool ADJ = false>
__global__ void __launch_bounds__(kBlock, P::lean ? TFG_MIN_BLOCKS_LEAN : (P::f32 ? TFG_MIN_BLOCKS_F32 : TFG_MIN_BLOCKS)) run_kernel(const __grid_constant__ RunParams<typename P::raw> p) {
  using raw = typename P::raw;
  using R = Num<P>;
  const int64_t gid = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  const bool active = gid < p.n_cells;
  const int64_t c = active ? gid : p.n_cells - 1;
  const int64_t N = p.n_cells;

  if constexpr (P::lean) {  // lookup tables of the table-driven exp / log (tfg_math.cuh) -> dynamic shared memory
    for (int i = threadIdx.x; i < fm::kTabDoubles; i += kBlock)
      fm::tfg_tabs[i] = (i < 64) ? fm::kExpTab[i] : fm::kLogTab[(i - 64) >> 1][(i - 64) & 1];
    __syncthreads();
  }
  // per-cell constants + diagnostic integrals live in shared memory (one column per thread)
  constexpr bool kSmem = true;  // RegCell (registers) remains available for experiments
  static_assert(kSmem || !PAR, "per-cell parameters live in shared memory");
  static_assert(!(PAR && TMA), "per-cell parameters run the register-prefetch kernel");
  // PAR: the per-cell surface factors in kPCount more columns (only in these instantiations: the others keep their footprint)
  // ADJ: the cell's T_air offset and P multiplier in two more columns behind them, read where the forcing is read (two
  // more registers across the time loop would cost more, in a kernel at its register limit)
  static_assert(kSmem || !ADJ, "forcing adjustments live in shared memory");
  static_assert(!(ADJ && (TMA || PRE)), "forcing adjustments run the register-prefetch kernel on the forcing itself");
  constexpr int kSAdj = kSCount + (PAR ? kPCount : 0);   // column of the T_air offset; the P multiplier follows
  __shared__ raw sm_cell[kSmem ? kSAdj + (ADJ ? 2 : 0) : 1][kBlock];
  using Cell = typename std::conditional<kSmem, SmemCell<raw, kBlock, PAR>, RegCell<raw>>::type;
  Cell s;
  if constexpr (kSmem) s.base = (unsigned)__cvta_generic_to_shared(&sm_cell[0][threadIdx.x]);
  if constexpr (PAR) {
#pragma unroll
    for (int i = 0; i < kPCount; ++i) s.set(kSCount + i, __ldg(p.cell_par + (int64_t)i * p.n_cells + c));
  }
  if constexpr (ADJ) { s.set(kSAdj, __ldg(p.fadj + c)); s.set(kSAdj + 1, __ldg(p.fadj + p.n_cells + c)); }
  s.set(kSaElev, __ldg(p.a_elev + c)); s.set(kSSinLat, __ldg(p.sin_lat + c)); s.set(kSCosLat, __ldg(p.cos_lat + c));
  s.set(kSNegTanLat, __ldg(p.neg_tan_lat + c)); s.set(kSSinEq, __ldg(p.sin_eq + c)); s.set(kSCosEq, __ldg(p.cos_eq + c));
  s.set(kSNegTanEq, __ldg(p.neg_tan_eq + c)); s.set(kSDlon, __ldg(p.dlon + c)); s.set(kSTNoon, __ldg(p.t_noon + c));
  s.set(kSDa, (TFG_DA_ZERO && !active) ? raw(0) : __ldg(p.da_m2 + c)); s.set(kSTrs, __ldg(p.t_rs + c));
  s.set(kSCB, 0); s.set(kSSB, 0); s.set(kSCB2, 0); s.set(kSSB2, 0);
  s.set(kSaElevR, (raw)(s.get(kSaElev) * p.k.inv_rstar));
  // OBJ: the objective's sums, float64 in every mode, carried on from the caller's accumulators (one running sum per
  // quantity over all launches: the result does not depend on how a run is split into launches)
  static_assert(!(OBJ && TMA), "an objective runs the register-prefetch kernel");
  __shared__ double sm_obj[OBJ ? TFG_N_OBJ : 1][OBJ ? kBlock : 1];
  ObjSums osum;
  if constexpr (OBJ) {
    osum.base = (unsigned)__cvta_generic_to_shared(&sm_obj[0][threadIdx.x]);
#pragma unroll
    for (int i = 0; i < TFG_N_OBJ; ++i) osum.set(i, p.obj_acc[(int64_t)i * p.n_cells + c]);
  }
  const R lon(__ldg(p.lon + c));
  const int tz = p.tz_idx ? (int)__ldg(p.tz_idx + c) : 0;

  CellState<raw> st;
  st.h_snow = p.h_snow[c]; st.h_swe = p.h_swe[c]; st.h_ice = p.h_ice[c]; st.h_iwe = p.h_iwe[c];
  st.eccs = p.eccs[c]; st.ecci = p.ecci[c]; st.albedo = p.albedo[c]; st.n_days = p.n_days[c];
  st.swe_lo = st.iwe_lo = 0;
  if constexpr (P::f32) { if (p.mass_lo != nullptr) { st.swe_lo = p.mass_lo[c]; st.iwe_lo = p.mass_lo[N + c]; } }
  const bool have_vol = VOL && p.vol_P != nullptr;
  s.set(kSVolP, have_vol ? p.vol_P[c] : 0); s.set(kSVolPR, have_vol ? p.vol_PR[c] : 0);
  s.set(kSVolPS, have_vol ? p.vol_PS[c] : 0); s.set(kSVolSM, have_vol ? p.vol_SM[c] : 0);
  s.set(kSVolIM, have_vol ? p.vol_IM[c] : 0); s.set(kSPmax, have_vol ? p.P_max[c] : 0);

  // warps that hold no real cell at all (tail block only) stop here: every block-wide barrier is behind us
  // (TMA staging, whose mbarriers count 128 arrivals, is only used when n_cells is a multiple of the block size)
  const bool warp_has_cells = (int64_t)blockIdx.x * kBlock + (threadIdx.x & ~31u) < p.n_cells;
  if (!warp_has_cells) return;
  const int slots = p.ring_slots;
  int slot = (int)(p.step0 % slots);
  raw* ring = p.ring + c;
  const bool exact = p.exact_ring != 0;
  // incremental window sum: seeded from the stored window, re-derived exactly (reference summation
  // order) whenever it comes within a guard band of the 0.03 m threshold of :1040
  R tot(0.0), tot_hi(0.0);
  const R guard(P::f32 ? 1.2e-7 : 2.3e-16);  // two units of round-off per counted operation
  R n_round((double)slots + 16.0);  // seeding additions + the reference sum's own depth
  // The fast mode's fixed band (below) covers 600 roundings of sums up to 1e4 m; the scaled bands of the other modes
  // stay narrow up to a few hundred.  A carried sum is used while this launch keeps the count below that.
  constexpr double kMaxRoundings = P::lean ? 600.0 : 400.0;
  bool carried = false;
  if (!exact && p.win_carry != nullptr) {
    const R n0(p.win_carry[2 * N + c]);
    if (n0.v + (raw)(2 * p.n_steps) <= (raw)kMaxRoundings) {  // false for the NaN that marks "no valid sum"
      tot = R(p.win_carry[c]); tot_hi = R(p.win_carry[N + c]); n_round = n0;
      carried = true;
    }
  }
  if (!exact && !carried) {
    for (int j = 0; j < slots; ++j) tot = xadd(tot, R(ring[(int64_t)j * N]));
    tot_hi = nabs(tot);
  }

  int basin = 0;
  bool warp_uniform = false;
  const bool have_agg = AGG && p.basin_agg != nullptr && p.basin_id != nullptr;
  if (have_agg) {
    basin = __ldg(p.basin_id + c);
    warp_uniform = __all_sync(0xffffffffu, basin == __shfl_sync(0xffffffffu, basin, 0));
  }

  // forcing block [step][var][column]: column = cell, or the cell's entry of the forcing map
  static_assert(!PRE || (!P::f32 && !TMA), "column terms: float64 modes, no TMA staging");
  const int64_t FN = p.n_cols;
  // PRE: one line of kCtCount values per column and timestep instead of five forcing rows
  const raw* f = PRE ? p.col_terms + (int64_t)__ldg(p.forcing_col + c) * kCtCount
                     : p.forcing + (p.forcing_col ? (int64_t)__ldg(p.forcing_col + c) : c);
  raw f0, f1, f2, f3, f4;        // PRE: P, T_air, 1/T_K, e_air, uz
  raw e0 = 0, e1 = 0, e2 = 0;    // PRE: RH, T_dew, "forcings sane"
  auto load_line = [](const raw* l, raw& a0, raw& a1, raw& a2, raw& a3, raw& a4, raw& b0, raw& b1, raw& b2) {
    if constexpr (PRE) {
      const double2 q0 = __ldg(reinterpret_cast<const double2*>(l + kCtP)), q1 = __ldg(reinterpret_cast<const double2*>(l + kCtUz)),
                    q2 = __ldg(reinterpret_cast<const double2*>(l + kCtEair)), q3 = __ldg(reinterpret_cast<const double2*>(l + kCtTdew));
      a0 = q0.x; a1 = q0.y; a4 = q1.x; a2 = q1.y; a3 = q2.x; b0 = q2.y; b1 = q3.x; b2 = q3.y;
    }
  };
  __shared__ alignas(128) raw sm_force[TMA ? kStages : 1][TFG_N_FORCING][TMA ? kBlock : 1];
  __shared__ uint64_t bar_full[kStages], bar_empty[kStages];
  const raw* fblock = p.forcing + (int64_t)blockIdx.x * kBlock;  // first cell of this block, step 0, variable 0
  // default path: every thread copies its own five forcings of step t+1 into its column of a two-deep
  // shared-memory stage while step t is computed (no cross-thread traffic, hence no barrier)
  constexpr bool kCp = TFG_CPASYNC && !TMA;
  __shared__ raw sm_next[kCp ? 2 : 1][TFG_N_FORCING][kCp ? kBlock : 1];
  auto stage_forcing = [&](int step_t) {
    const raw* fn = f + (int64_t)step_t * (TFG_N_FORCING * FN);
#pragma unroll
    for (int v = 0; v < TFG_N_FORCING; ++v) cp_async_elem(&sm_next[step_t & 1][v][threadIdx.x], fn + (int64_t)v * FN);
    cp_async_commit();
  };
  auto issue_stage = [&](int step_t) {  // elected thread: five row copies for timestep step_t
    const int sg = step_t % kStages;
    mbar_expect_tx(&bar_full[sg], (unsigned)(TFG_N_FORCING * kBlock * sizeof(raw)));
#pragma unroll
    for (int v = 0; v < TFG_N_FORCING; ++v)
      bulk_g2s(&sm_force[sg][v][0], fblock + ((int64_t)step_t * TFG_N_FORCING + v) * N, (unsigned)(kBlock * sizeof(raw)),
               &bar_full[sg]);
  };
  if constexpr (TMA) {
    if (threadIdx.x == 0) {
      for (int i = 0; i < kStages; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], kBlock); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0)
      for (int i = 0; i < kStages && i < p.n_steps; ++i) issue_stage(i);
  } else if constexpr (kCp) {
    stage_forcing(0);
  } else if constexpr (PRE) {
    load_line(f, f0, f1, f2, f3, f4, e0, e1, e2);
  } else {
    f0 = ld_stream(f); f1 = ld_stream(f + FN); f2 = ld_stream(f + 2 * FN); f3 = ld_stream(f + 3 * FN);
    f4 = ld_stream(f + 4 * FN);
  }
  // float32 kernel: the slot pointer walks through the window (no 64-bit multiply per step); the float64 kernels
  // are register-bound and recompute the address instead of carrying two more pointers
  constexpr bool kWalk = P::f32 || (P::lean && TFG_WALK_LEAN);
  raw* ring_cur = ring + (int64_t)slot * N;
  raw r_old = *ring_cur;
  R LC(0.0);
  auto set_zone = [&](raw gmt) {
    if constexpr (P::strict) {
      LC = ((R(gmt) * 15.0) - lon) / 15.0;  // True_Solar_Noon, solar_funcs.py:1466-1468
    } else {
      LC = ((R(gmt) * 15.0) - lon) * R(1.0 / 15.0);
      const raw B = p.k.omega * LC.v;
      raw sb, cb, sb2, cb2;
      if constexpr (P::f32) { __sincosf(B, &sb, &cb); __sincosf(B - s.get(kSDlon), &sb2, &cb2); }
      else { sincos(B, &sb, &cb); sincos(B - s.get(kSDlon), &sb2, &cb2); }
      s.set(kSSB, sb); s.set(kSCB, cb); s.set(kSSB2, sb2); s.set(kSCB2, cb2);
    }
  };
  raw gmt_prev = __longlong_as_double(0x7ff8000000000000ll);  // NaN: the first step always sets the zone

  if (TFG_ZONE_ONCE && !p.gmt_varies) {  // the common case: one UTC offset per zone for the whole launch
    gmt_prev = p.gmt[tz];
    set_zone(gmt_prev);
  }
  bool statics_sane = true, state_ok = true;
  auto finite = [](raw v) { return ((unsigned)__double2hiint((double)v) & 0x7ff00000u) != 0x7ff00000u; };
  if constexpr (P::lean) {  // finite tables, |a_elev| < 2e5 (|elev| < 700 km), finite carried state
    state_ok = finite(st.h_snow) && finite(st.h_swe) && finite(st.h_ice) && finite(st.h_iwe) && finite(st.eccs) &&
               finite(st.ecci) && finite(st.albedo) && finite(st.n_days);
    statics_sane = fabs(s.get(kSaElev)) < 2.0e5 && finite(lon.v);
    for (int i = kSSinLat; i <= kSTrs; ++i) statics_sane = statics_sane && finite(s.get(i));
  }
  StepOut<raw> o;
  for (int t = 0; t < p.n_steps; ++t) {
    raw g0 = 0, g1 = 0, g2 = 0, g3 = 0, g4 = 0, g5 = 0, g6 = 0, g7 = 0;
    if constexpr (TMA) {
      const int sg = t % kStages;
      mbar_wait(&bar_full[sg], (unsigned)((t / kStages) & 1));
      f0 = sm_force[sg][0][threadIdx.x]; f1 = sm_force[sg][1][threadIdx.x]; f2 = sm_force[sg][2][threadIdx.x];
      f3 = sm_force[sg][3][threadIdx.x]; f4 = sm_force[sg][4][threadIdx.x];
      mbar_arrive(&bar_empty[sg]);
      // refill the stage of the PREVIOUS step (most warps are past it already): prefetch distance kStages - 1
      if (threadIdx.x == 0 && t >= 1 && t - 1 + kStages < p.n_steps) {
        mbar_wait(&bar_empty[(t - 1) % kStages], (unsigned)(((t - 1) / kStages) & 1));
        issue_stage(t - 1 + kStages);
      }
    } else if constexpr (!kCp) {
      // the next step's forcings are requested from inside the step (prefetch below)
    } else {
      cp_async_wait_all();  // this thread's copies of step t have landed
      f0 = sm_next[t & 1][0][threadIdx.x]; f1 = sm_next[t & 1][1][threadIdx.x]; f2 = sm_next[t & 1][2][threadIdx.x];
      f3 = sm_next[t & 1][3][threadIdx.x]; f4 = sm_next[t & 1][4][threadIdx.x];
      if (t + 1 < p.n_steps) stage_forcing(t + 1);
    }
    if constexpr (ADJ) {  // T_air' = T_air + offset, P' = P * multiplier: what the sanity test and both steps see
      f1 = add_once(f1, s.get(kSAdj));
      f0 = mul_once(f0, s.get(kSAdj + 1));
    }
    if constexpr (PRE && !TFG_CT_REGPF) { if (t > 0) load_line(f + (int64_t)t * (kCtCount * FN), f0, f1, f2, f3, f4, e0, e1, e2); }
    const TimeRow<raw>& row = p.rows[t];
    if (!TFG_ZONE_ONCE || p.gmt_varies) {  // a DST switch falls into this launch (twice a year): follow the offset step by step
      const raw gmt = p.gmt[t * p.n_tz + tz];
      if (!(gmt == gmt_prev)) {  // the offset is piece-wise constant in time
        gmt_prev = gmt;
        set_zone(gmt);
      }
    }
    const bool wrap = (slot + 1 == slots);
    const int slot_next = wrap ? 0 : slot + 1;
    raw* ring_next;
    if constexpr (kWalk) ring_next = ring_cur + (wrap ? -(int64_t)(slots - 1) * N : N);  // a warp-uniform stride: no cell index needed
    else ring_next = ring + (int64_t)slot_next * N;
    raw r_next = 0;
    R tot_now;
    auto window = [&](raw ring_new_raw) -> raw {
      const R ring_new(ring_new_raw);
      // np.roll(-1) + write of the newest slot, :1027-1033.  Not predicated on `active` (which ptxas re-derives from
      // S2R + 64-bit compares at every use): threads past the last cell replicate cell N-1 IN THE SAME WARP, in lockstep
      // and with identical inputs, so they store the identical value at the same instant; warps without any real cell
      // have left the kernel (see `warp_has_cells`), because a replica warp running a step ahead would overwrite a slot
      // the real cell has not read yet
      *(kWalk ? ring_cur : ring + (int64_t)slot * N) = ring_new.v;
      if (exact) {
        tot_now = window_sum_exact<P>(ring, N, slots, slot);
      } else {
        tot = xadd(xsub(tot, R(r_old)), ring_new);
        bool near_threshold;
        if constexpr (P::lean) {
          // the incremental sum drifts by < 330 roundings of the largest sum seen during a launch (72 seed
          // additions + 2 per step, <= 128 steps): below 1e4 m that is < 4e-10 m, so a fixed band around the
          // threshold suffices; larger sums (absurd forcing) take the exact path every step
          // (the magnitude test on the high word also catches NaN / inf of either sign: a non-finite entry must
          // poison the sum only while it is inside the window, as in the reference's re-summation every step)
          near_threshold = (nabs(tot - LIT(snow_thr, 0.03)) <= 1e-9) ||
                           (((unsigned)__double2hiint(tot.v) & 0x7fffffffu) >= 0x40c38800u);
        } else {
          // drift bound: (seed additions + 2 per step) roundings of the largest sum seen since the last exact sum
          tot_hi = nmax(tot_hi, nabs(tot));
          n_round = n_round + R(2.0);
          // !(x <= y) instead of x > y: a non-finite running sum (NaN compares false) takes the exact path too, so
          // that it recovers as soon as the bad entry has left the window (as the reference's per-step re-sum does)
          near_threshold = !(nabs(tot - 0.03) > (guard * n_round) * tot_hi) || !(nabs(tot) < R(1e30));
        }
        if (near_threshold) {
          tot = window_sum_exact<P>(ring, N, slots, slot);
          tot_hi = nabs(tot);
          n_round = R(16.0);  // the exact sum itself: 8 lanes of 9 additions + 3 levels, in reference order
        }
        tot_now = tot;
      }
      r_next = *ring_next;  // next step's oldest entry (after this step's store)
      return tot_now.v;
    };
    auto prefetch = [&]() {  // next step's forcings, issued mid-step (see cell_step)
      if constexpr (!TMA && !kCp) {
        g0 = f0; g1 = f1; g2 = f2; g3 = f3; g4 = f4;
        if constexpr (PRE && !TFG_CT_REGPF) {
          if (t + 1 < p.n_steps) asm volatile("prefetch.global.L1 [%0];" ::"l"(f + (int64_t)(t + 1) * (kCtCount * FN)));
        } else if constexpr (PRE) {
          g5 = e0; g6 = e1; g7 = e2;
          if (t + 1 < p.n_steps) load_line(f + (int64_t)(t + 1) * (kCtCount * FN), g0, g1, g2, g3, g4, g5, g6, g7);
        } else if (t + 1 < p.n_steps) {
          const raw* fn = f + (int64_t)(t + 1) * (TFG_N_FORCING * FN);
          g0 = ld_stream(fn); g1 = ld_stream(fn + FN); g2 = ld_stream(fn + 2 * FN); g3 = ld_stream(fn + 3 * FN);
          g4 = ld_stream(fn + 4 * FN);
        }
      }
    };
    if constexpr (P::lean) {
      // The lean math cores assume physically sane arguments.  Bit tests on the high words (no FP64 pipe):
      // P in [0, 10) m/h, |T_air| < 90 degC, P_air in [1e3, 2e5) Pa, q in [1e-7, 0.2), uz = 0 or in [1e-100, 200)
      bool sane;
      if constexpr (PRE) sane = (__double2hiint(e2) != 0) && statics_sane;   // the column's forcings were tested once, by column_terms_kernel
      else sane = forcings_sane(f0, f1, f2, f3, f4) && statics_sane;
      // (SATTERLUND = True, a rarely used configuration switch, also takes the strict step: the lean one is
      // written for the default Magnus / Brutsaert formulas only, which keeps it free of configuration branches)
      if (__all_sync(0xffffffffu, sane && state_ok) && !p.k.satterlund) {
        if constexpr (PRE) {
          const ColumnTerms pre{f2, f3, e0, e1, f + (int64_t)t * (kCtCount * FN)};
          cell_step<P, VOL>(p.k, row, s, LC, st, R(f0), R(f1), R(0.0), R(0.0), R(f4), window, prefetch, o, pre);
        } else {
          cell_step<P, VOL>(p.k, row, s, LC, st, R(f0), R(f1), R(f2), R(f3), R(f4), window, prefetch, o);
        }
      } else {
        // Same step in the strict arithmetic (libdevice, IEEE division, NumPy's NaN rules): whatever the input
        // -- missing data, absurd values -- the cell behaves like the reference, NaN poisoning included.
        using S = Num<StrictF64>;
        const S LCs = ((S(gmt_prev) * 15.0) - S(lon.v)) / 15.0;
        if constexpr (PRE) {  // the line carries the raw pressure and humidity for this case
          const raw* line = f + (int64_t)t * (kCtCount * FN);
          f2 = __ldg(line + kCtPair); f3 = __ldg(line + kCtQ);
        }
        cell_step<StrictF64, VOL>(p.k, row, s, LCs, st, S(f0), S(f1), S(f2), S(f3), S(f4), window, prefetch, o);
        state_ok = finite(st.h_snow) && finite(st.h_swe) && finite(st.h_ice) && finite(st.h_iwe) &&
                   finite(st.eccs) && finite(st.ecci) && finite(st.albedo) && finite(st.n_days);
      }
    } else if constexpr (PRE) {   // strict float64 with column terms (no sanity test: NaN rules apply as they come)
      const ColumnTerms pre{f2, f3, e0, e1, f + (int64_t)t * (kCtCount * FN)};
      cell_step<P, VOL>(p.k, row, s, LC, st, R(f0), R(f1), R(0.0), R(0.0), R(f4), window, prefetch, o, pre);
    } else {
      cell_step<P, VOL>(p.k, row, s, LC, st, R(f0), R(f1), R(f2), R(f3), R(f4), window, prefetch, o);
    }

    if constexpr (REC) {
      if (active && p.record != nullptr) {
        raw* rp = p.record + ((int64_t)t * p.n_rec) * N + c;
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
        TFG_PUT(TFG_REC_ECCS, st.eccs) TFG_PUT(TFG_REC_ECCI, st.ecci) TFG_PUT(TFG_REC_SNOW3DAY, tot_now.v)
        TFG_PUT(TFG_REC_P_RAIN, o.P_rain) TFG_PUT(TFG_REC_P_SNOW, o.P_snow)
#undef TFG_PUT
      }
    }
    if constexpr (OBJ) {
      // the step's value of the chosen BMI output against the observation of the cell's column; a non-finite
      // observation is "not observed" (the cell's own value may be NaN: a poisoned cell is scored, and its sums say so)
      if (t >= p.obj_t_lo && t < p.obj_t_hi) {   // warp-uniform
        const int64_t col = p.obj_col ? (int64_t)__ldg(p.obj_col + c) : c;
        const double ob = __ldg(p.obj_obs + (int64_t)(t - p.obj_t_lo) * p.obj_ncols + col);
        if (((unsigned)__double2hiint(ob) & 0x7ff00000u) != 0x7ff00000u) {
          raw v;
          switch (p.obj_quantity) {   // a kernel parameter: warp-uniform
            case TFG_REC_H_SNOW: v = st.h_snow; break;
            case TFG_REC_H_SWE: v = st.h_swe; break;
            case TFG_REC_SM: v = o.SM; break;
            case TFG_REC_H_ICE: v = st.h_ice; break;
            case TFG_REC_H_IWE: v = st.h_iwe; break;
            case TFG_REC_IM: v = o.IM; break;
            case TFG_REC_M_TOTAL: v = o.M_total; break;
            default: v = o.RH; break;
          }
          const double sv = (double)v, d = __dsub_rn(sv, ob);   // float32: widened exactly
          osum.set(0, __dadd_rn(osum.get(0), sv));
          osum.set(1, __dadd_rn(osum.get(1), __dmul_rn(sv, sv)));
          osum.set(2, __dadd_rn(osum.get(2), __dmul_rn(sv, ob)));
          osum.set(3, __dadd_rn(osum.get(3), __dmul_rn(d, d)));
        }
      }
    }
    if constexpr (AGG) {
      if (have_agg) {
        // area-weighted basin sums (np.sum sites :567-568,:1486-1494 and the driver's `* da_m2`):
        // warp-shuffle tree when the warp sits inside one basin, one RED per warp and quantity
        const double da = (double)s.get(kSDa);
        const bool counted = TFG_DA_ZERO || active;
        double v0 = counted ? (double)o.M_total * da : 0.0;
        double v1 = counted ? (double)st.h_swe * da : 0.0;
        double v2 = counted ? (double)st.h_iwe * da : 0.0;
        const int64_t entry = ((int64_t)t * p.n_basin + basin) * TFG_N_AGG;
        double* dst = static_cast<double*>(p.basin_agg) + entry;
        long long* acc = static_cast<long long*>(p.basin_agg) + 2 * entry;
        if (warp_uniform) {
          // three sums in one butterfly: after the first two exchanges every lane is responsible for ONE of the
          // quantities (lanes 0-7: v0, 8-15: v1, 16-23: v2), so 12 shuffles instead of 30
          const unsigned full = 0xffffffffu;
          const int lane = threadIdx.x & 31;
          const bool hi = (lane & 16) != 0;
          double k0 = hi ? v2 : v0, k1 = hi ? 0.0 : v1;
          k0 += __shfl_xor_sync(full, hi ? v0 : v2, 16);
          k1 += __shfl_xor_sync(full, hi ? v1 : 0.0, 16);
          const bool hi2 = (lane & 8) != 0;
          double k = hi2 ? k1 : k0;
          k += __shfl_xor_sync(full, hi2 ? k0 : k1, 8);
          k += __shfl_xor_sync(full, k, 4);
          k += __shfl_xor_sync(full, k, 2);
          k += __shfl_xor_sync(full, k, 1);
          if ((lane & 7) == 0 && lane < 24) {
            if (p.agg_exact) agg_add_exact(acc + 2 * (lane >> 3), k, p.agg_up[lane >> 3], p.agg_lo, p.agg_bad);
            else atomicAdd(dst + (lane >> 3), k);
          }
        } else if (active) {
          if (p.agg_exact) {
            agg_add_exact(acc + 0, v0, p.agg_up[0], p.agg_lo, p.agg_bad);
            agg_add_exact(acc + 2, v1, p.agg_up[1], p.agg_lo, p.agg_bad);
            agg_add_exact(acc + 4, v2, p.agg_up[2], p.agg_lo, p.agg_bad);
          } else {
            atomicAdd(dst + 0, v0); atomicAdd(dst + 1, v1); atomicAdd(dst + 2, v2);
          }
        }
      }
    }
    if constexpr (PRE && !TFG_CT_REGPF) {
    } else {
      if constexpr (!TMA && !kCp) { f0 = g0; f1 = g1; f2 = g2; f3 = g3; f4 = g4; }
      if constexpr (PRE) { e0 = g5; e1 = g6; e2 = g7; }
    }
    r_old = r_next;
    slot = slot_next;
    if constexpr (kWalk) ring_cur = ring_next;
  }

  if (active && p.win_carry != nullptr) {
    if (exact) {
      p.win_carry[2 * N + c] = (raw)nan("");  // the window moved without the running sum: re-seed next time
    } else {
      if constexpr (P::lean) n_round = n_round + R((double)(2 * p.n_steps));  // not counted per step in this mode
      p.win_carry[c] = tot.v; p.win_carry[N + c] = nmax(tot_hi, nabs(tot)).v; p.win_carry[2 * N + c] = n_round.v;
    }
  }
  if (active) {
    p.h_snow[c] = st.h_snow; p.h_swe[c] = st.h_swe; p.h_ice[c] = st.h_ice; p.h_iwe[c] = st.h_iwe;
    p.eccs[c] = st.eccs; p.ecci[c] = st.ecci; p.albedo[c] = st.albedo; p.n_days[c] = st.n_days;
    p.SM[c] = o.SM; p.IM[c] = o.IM; p.M_total[c] = o.M_total; p.RH[c] = o.RH;
    if constexpr (P::f32) { if (p.mass_lo != nullptr) { p.mass_lo[c] = st.swe_lo; p.mass_lo[N + c] = st.iwe_lo; } }
    if (have_vol) {
      p.vol_P[c] = s.get(kSVolP); p.vol_PR[c] = s.get(kSVolPR); p.vol_PS[c] = s.get(kSVolPS);
      p.vol_SM[c] = s.get(kSVolSM); p.vol_IM[c] = s.get(kSVolIM); p.P_max[c] = s.get(kSPmax);
    }
    if constexpr (OBJ) {
#pragma unroll
      for (int i = 0; i < TFG_N_OBJ; ++i) p.obj_acc[(int64_t)i * N + c] = osum.get(i);
    }
  }
}

// host-side dispatch over the compile-time switches; defined once per arithmetic mode (one TU each)
// Column terms of one launch: thread = (timestep, column) of the forcing block [n_steps][5][n_cols]; writes one line of
// kCtCount doubles (see tfg_physics.cuh).  Compiled in the fast translation unit, with the melt kernel's own device
// functions, so the values equal what the per-cell step computes (tests: mapped forcing == replicated forcing, bit for bit).
template <class P, bool PAR = false>
__global__ void __launch_bounds__(256) column_terms_kernel(const double* __restrict__ forcing, double* __restrict__ out,
                                                           int32_t n_steps, int64_t n_cols, const Consts<double> k) {
  if constexpr (P::lean) {
    for (int i = threadIdx.x; i < fm::kTabDoubles; i += blockDim.x)
      fm::tfg_tabs[i] = (i < 64) ? fm::kExpTab[i] : fm::kLogTab[(i - 64) >> 1][(i - 64) & 1];
    __syncthreads();
  }
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n_steps * n_cols) return;
  const int64_t t = idx / n_cols, col = idx - t * n_cols;
  const double* f = forcing + t * (TFG_N_FORCING * n_cols) + col;
  const double f0 = f[0], f1 = f[n_cols], f2 = f[2 * n_cols], f3 = f[3 * n_cols], f4 = f[4 * n_cols];
  if constexpr (P::lean) column_terms_eval<P, PAR>(k, f0, f1, f2, f3, f4, forcings_sane(f0, f1, f2, f3, f4), out + idx * kCtCount);
  else column_terms_eval_strict<P, PAR>(k, f0, f1, f2, f3, f4, out + idx * kCtCount);
}

// par: the melt kernel runs with per-cell parameters, so the line carries their parameter-free factors (column_terms_eval)
template <class P>
cudaError_t launch_column_terms(const double* forcing, double* out, int32_t n_steps, int64_t n_cols, const Consts<double>& k,
                                bool par, cudaStream_t stream) {
  const int64_t total = (int64_t)n_steps * n_cols;
  const unsigned grid = (unsigned)((total + 255) / 256);
  const size_t dyn = P::lean ? fm::kTabDoubles * sizeof(double) : 0;
  if (par) column_terms_kernel<P, true><<<grid, 256, dyn, stream>>>(forcing, out, n_steps, n_cols, k);
  else column_terms_kernel<P><<<grid, 256, dyn, stream>>>(forcing, out, n_steps, n_cols, k);
  return cudaGetLastError();
}

template <class P, bool PAR>
cudaError_t launch_run_as(const RunParams<typename P::raw>& p, bool rec, bool agg, bool vol, cudaStream_t stream) {
  const unsigned grid = (unsigned)((p.n_cells + kBlock - 1) / kBlock);
  // TMA staging needs whole blocks and 16-byte aligned rows; otherwise the register-prefetch kernel runs (always with
  // per-cell parameters, as with a forcing map)
  const bool tma = !PAR && p.use_tma && !rec && !p.forcing_col && (p.n_cells % kBlock == 0) && p.n_steps >= 2 &&
                   ((reinterpret_cast<uintptr_t>(p.forcing) & 15) == 0) &&
                   ((p.n_cells * sizeof(typename P::raw)) % 16 == 0);
  const size_t dyn = P::lean ? fm::kTabDoubles * sizeof(double) : 0;
  if (p.fadj != nullptr) {
    // forcing adjustments bound: the two kernel shapes of the objective, with and without it (tfg_run never binds
    // column terms then: the forcing-only terms differ per cell)
    if (p.obj_acc != nullptr) {
      if (rec) run_kernel<P, true, true, true, false, false, PAR, true, true><<<grid, kBlock, dyn, stream>>>(p);
      else run_kernel<P, false, true, true, false, false, PAR, true, true><<<grid, kBlock, dyn, stream>>>(p);
    } else {
      if (rec) run_kernel<P, true, true, true, false, false, PAR, false, true><<<grid, kBlock, dyn, stream>>>(p);
      else run_kernel<P, false, true, true, false, false, PAR, false, true><<<grid, kBlock, dyn, stream>>>(p);
    }
    return cudaGetLastError();
  }
  if (p.obj_acc != nullptr) {
    // objective bound: two kernel shapes only, both of which test basin_agg and vol_P at run time (register prefetch,
    // like PAR); the recording one for launches that record
    if constexpr (!P::f32) {
      if (p.col_terms != nullptr) {
        if (rec) run_kernel<P, true, true, true, false, true, PAR, true><<<grid, kBlock, dyn, stream>>>(p);
        else run_kernel<P, false, true, true, false, true, PAR, true><<<grid, kBlock, dyn, stream>>>(p);
        return cudaGetLastError();
      }
    }
    if (rec) run_kernel<P, true, true, true, false, false, PAR, true><<<grid, kBlock, dyn, stream>>>(p);
    else run_kernel<P, false, true, true, false, false, PAR, true><<<grid, kBlock, dyn, stream>>>(p);
    return cudaGetLastError();
  }
  if constexpr (!P::f32) {
    if (p.col_terms != nullptr) {  // column terms bound (forcing map): the kernel reads them instead of the forcing block
      if (rec) run_kernel<P, true, true, true, false, true, PAR><<<grid, kBlock, dyn, stream>>>(p);
      else if (agg && vol) run_kernel<P, false, true, true, false, true, PAR><<<grid, kBlock, dyn, stream>>>(p);
      else if (agg) run_kernel<P, false, true, false, false, true, PAR><<<grid, kBlock, dyn, stream>>>(p);
      else if (vol) run_kernel<P, false, false, true, false, true, PAR><<<grid, kBlock, dyn, stream>>>(p);
      else run_kernel<P, false, false, false, false, true, PAR><<<grid, kBlock, dyn, stream>>>(p);
      return cudaGetLastError();
    }
  }
  if (rec) run_kernel<P, true, true, true, false, false, PAR><<<grid, kBlock, dyn, stream>>>(p);
  else if (tma) {
    if constexpr (!PAR) {
      if (agg && vol) run_kernel<P, false, true, true, true><<<grid, kBlock, dyn, stream>>>(p);
      else if (agg) run_kernel<P, false, true, false, true><<<grid, kBlock, dyn, stream>>>(p);
      else if (vol) run_kernel<P, false, false, true, true><<<grid, kBlock, dyn, stream>>>(p);
      else run_kernel<P, false, false, false, true><<<grid, kBlock, dyn, stream>>>(p);
    }
  }
  else if (agg && vol) run_kernel<P, false, true, true, false, false, PAR><<<grid, kBlock, dyn, stream>>>(p);
  else if (agg) run_kernel<P, false, true, false, false, false, PAR><<<grid, kBlock, dyn, stream>>>(p);
  else if (vol) run_kernel<P, false, false, true, false, false, PAR><<<grid, kBlock, dyn, stream>>>(p);
  else run_kernel<P, false, false, false, false, false, PAR><<<grid, kBlock, dyn, stream>>>(p);
  return cudaGetLastError();
}

// per-cell surface parameters bound (tfg_bind_cell_params): the PAR instantiations, chosen from the input; an objective
// bound (p.obj_acc): the OBJ instantiations; forcing adjustments bound (p.fadj): the ADJ instantiations (launch_run_as)
template <class P>
cudaError_t launch_run(const RunParams<typename P::raw>& p, bool rec, bool agg, bool vol, cudaStream_t stream) {
  return p.cell_par != nullptr ? launch_run_as<P, true>(p, rec, agg, vol, stream) : launch_run_as<P, false>(p, rec, agg, vol, stream);
}

cudaError_t launch_run_strict(const RunParams<double>& p, bool rec, bool agg, bool vol, cudaStream_t stream);
cudaError_t launch_run_fast(const RunParams<double>& p, bool rec, bool agg, bool vol, cudaStream_t stream);
cudaError_t launch_run_f32(const RunParams<float>& p, bool rec, bool agg, bool vol, cudaStream_t stream);
cudaError_t launch_column_terms_fast(const double* forcing, double* out, int32_t n_steps, int64_t n_cols, const Consts<double>& k,
                                     bool par, cudaStream_t stream);
cudaError_t launch_column_terms_strict(const double* forcing, double* out, int32_t n_steps, int64_t n_cols, const Consts<double>& k,
                                       bool par, cudaStream_t stream);

}  // namespace tfg
