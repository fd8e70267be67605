// float64, reference-order IEEE arithmetic (TFG_F64_STRICT)
#include "tfg_run.cuh"
namespace tfg {
cudaError_t launch_run_strict(const RunParams<double>& p, bool rec, bool agg, bool vol, cudaStream_t stream) {
  return launch_run<StrictF64>(p, rec, agg, vol, stream);
}
cudaError_t launch_column_terms_strict(const double* forcing, double* out, int32_t n_steps, int64_t n_cols, const Consts<double>& k,
                                       bool par, cudaStream_t stream) {
  return launch_column_terms<StrictF64>(forcing, out, n_steps, n_cols, k, par, stream);
}
}  // namespace tfg
