// lm_cta_inst.cu -- model dispatch of the general batched LM kernel (lm_cta.cuh), both precisions.
#include "lm_cta.cuh"
#include "runtime.cuh"

namespace mirb200 {

template <class T>
int launch_cta_model(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    if (model.model >= (uint32_t)MIR_MODEL_USER_BASE) return launch_user_model<T>(model, n, st, args, stream);
    return visit_cta_model<T>(model, "mir_optim_b200: model id not available in the batched path", [&](auto tag) {
        using M = typename decltype(tag)::type;
        if (n > 128) { set_error("mir_optim_b200: the batched path supports n <= 128"); return (int)MIR_B200_EUNSUPPORTED; }
        if (!M::valid((int)n, (int)args.m)) { set_error("mir_optim_b200: (m, n) not valid for this model"); return (int)MIR_B200_EINVAL; }
        const bool fd = (args.flags & MIR_MODEL_FD_JACOBIAN) || !M::kAnalytic;
        const RuntimeKernel kern{fd ? (const void*)lm_cta_kernel<M, T, true> : (const void*)lm_cta_kernel<M, T, false>, "lm_cta_kernel launch"};
        return launch_cta_fit<T>(kern, st, args, model, n, M::prep_elems((int)n), stream);
    });
}
template int launch_cta_model<double>(const mir_model_desc&, size_t, const Num<double>::Settings&, const SmallBatchArgs&, cudaStream_t);
template int launch_cta_model<float>(const mir_model_desc&, size_t, const Num<float>::Settings&, const SmallBatchArgs&, cudaStream_t);

}  // namespace mirb200
