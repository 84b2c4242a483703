// lm_cta_inst.cu -- model dispatch of the general batched LM kernel (lm_cta.cuh), both precisions.  The weighted
// instantiations (MIR_MODEL_WEIGHTED) are compiled in lm_cta_w_inst.cu.
#include "lm_cta.cuh"
#include "runtime.cuh"

namespace mirb200 {

extern template int launch_cta_builtin<double, true>(const mir_model_desc&, size_t, const Num<double>::Settings&, const SmallBatchArgs&, cudaStream_t);
extern template int launch_cta_builtin<float, true>(const mir_model_desc&, size_t, const Num<float>::Settings&, const SmallBatchArgs&, cudaStream_t);

template <class T>
int launch_cta_model(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    if (model.model >= (uint32_t)MIR_MODEL_USER_BASE) return launch_user_model<T>(model, n, st, args, stream);
    if (model.flags & MIR_MODEL_WEIGHTED) return launch_cta_builtin<T, true>(model, n, st, args, stream);
    return launch_cta_builtin<T, false>(model, n, st, args, stream);
}
template int launch_cta_model<double>(const mir_model_desc&, size_t, const Num<double>::Settings&, const SmallBatchArgs&, cudaStream_t);
template int launch_cta_model<float>(const mir_model_desc&, size_t, const Num<float>::Settings&, const SmallBatchArgs&, cudaStream_t);

}  // namespace mirb200
