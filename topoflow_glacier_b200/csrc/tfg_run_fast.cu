// float64 with algebraic shortcuts and written-out FMAs (TFG_F64_FAST)
#ifndef TFG_WS         // 1: experimental warp-specialised producer / consumer kernel (tfg_ws.cuh) for fused launches: bit-identical
#define TFG_WS 0       //    to the split single-stream kernel, measured slower (profiles/r2_experiments.md); 0 = default
#endif
#if TFG_WS && !defined(TFG_SPLIT_STEP)
#define TFG_SPLIT_STEP 1   // every route of the fast mode then evaluates lean_forcing + lean_state: bit-identical results
#endif
#ifndef TFG_PIPELINE   // 1: experimental software-pipelined time loop (tfg_pipe.cuh, needs -DTFG_SPLIT_STEP=1; measured slower)
#define TFG_PIPELINE 0
#endif
#ifdef TFG_LEAN_W2
// Experimental two-cells-per-thread kernel with 128-bit forcing / state / window access (tfg_lean.cuh).  Bit-identical
// results, 8 % fewer instructions per cell-step, but 168 registers (3 blocks per SM) and a hot loop of 26 KB that misses
// the instruction cache: 22.5 G cell-steps/s against 27.9 G for the one-cell kernel (profiles/r2_w2_experiment.txt).
#include "tfg_lean.cuh"
#else
#include "tfg_pipe.cuh"
#include "tfg_ws.cuh"
#endif
namespace tfg {
cudaError_t launch_run_fast(const RunParams<double>& p, bool rec, bool agg, bool vol, cudaStream_t stream) {
#ifdef TFG_LEAN_W2
  return launch_run_lean(p, rec, agg, vol, stream);
#else
  // Recording launches, one-step launches (exact window re-sum: the literal update()), TMA staging and SATTERLUND
  // configurations stay with the single-stream kernel; all routes evaluate the same device functions.
  const bool fused = !p.exact_ring && !p.use_tma && !p.col_terms;
  if (TFG_WS && fused && !rec && !p.k.satterlund && p.n_steps >= 2) return launch_run_ws(p, agg, vol, stream);
  if (TFG_PIPELINE && fused) return launch_run_pipe(p, rec, agg, vol, stream);
  return launch_run<FastF64>(p, rec, agg, vol, stream);
#endif
}
cudaError_t launch_column_terms_fast(const double* forcing, double* out, int32_t n_steps, int64_t n_cols, const Consts<double>& k,
                                     bool par, cudaStream_t stream) {
  return launch_column_terms<FastF64>(forcing, out, n_steps, n_cols, k, par, stream);
}
}  // namespace tfg
