// lm_cta_r_inst.cu -- the robust-loss instantiations of the general batched LM kernel (lm_cta.cuh, CtaRobust: soft_l1 and
// huber, weighted or not), both precisions; a translation unit of their own, beside lm_cta_inst.cu and lm_cta_w_inst.cu.
#include "lm_cta.cuh"
#include "runtime.cuh"

namespace mirb200 {

template int launch_cta_builtin<double, kCtaRobust>(const mir_model_desc&, size_t, const Num<double>::Settings&, const SmallBatchArgs&, cudaStream_t);
template int launch_cta_builtin<float, kCtaRobust>(const mir_model_desc&, size_t, const Num<float>::Settings&, const SmallBatchArgs&, cudaStream_t);

}  // namespace mirb200
