// lm_cta_w_inst.cu -- the weighted instantiations of the general batched LM kernel (lm_cta.cuh, CtaWeighted), both
// precisions; a translation unit of their own so that they compile beside the unweighted ones (lm_cta_inst.cu).
#include "lm_cta.cuh"
#include "runtime.cuh"

namespace mirb200 {

template int launch_cta_builtin<double, true>(const mir_model_desc&, size_t, const Num<double>::Settings&, const SmallBatchArgs&, cudaStream_t);
template int launch_cta_builtin<float, true>(const mir_model_desc&, size_t, const Num<float>::Settings&, const SmallBatchArgs&, cudaStream_t);

}  // namespace mirb200
