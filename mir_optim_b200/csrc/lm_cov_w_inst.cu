// lm_cov_w_inst.cu -- the weighted instantiations of the covariance kernel (lm_cov.cuh, CtaWeighted), both precisions;
// a translation unit of their own so that they compile beside the unweighted ones (lm_cov.cu).
#include "lm_cov.cuh"
#include "runtime.cuh"

namespace mirb200 {

template int launch_cov_builtin<double, true>(const mir_model_desc&, double, CovArgs, const char*, cudaStream_t);
template int launch_cov_builtin<float, true>(const mir_model_desc&, float, CovArgs, const char*, cudaStream_t);

}  // namespace mirb200
