// lm_nvrtc.cu -- residual models supplied as CUDA source at run time (SURVEY 8f-2; the reference takes arbitrary
// f / g, least_squares.d:78-80, 803-867).  mir_b200_model_compile registers the source; the first launch per precision
// compiles `lm_cta_kernel<CtaUser<UserModel<T>, T>, T, FD>` (the general batched LM kernel, lm_cta.cuh, whose sources
// are embedded in the library by embed_headers.py) with NVRTC for sm_100a, loads the cubin with the driver API and
// caches the functions.  The covariance kernel (`lm_cov_cta_kernel`, lm_cov.cuh) is a separate program, compiled at
// the first covariance call per precision, so registration does no extra work for it; so are the weighted forms of both
// (`lm_cta_kernel<CtaWeighted<CtaUser<...>>>`, `lm_cov_cta_weighted_kernel<CtaWeighted<CtaUser<...>>>`, MIR_MODEL_WEIGHTED), compiled
// at the first weighted call.  All launch with the policy of
// the built-in kernels (launch_persistent, lm_cta.cuh), through the driver API.  libnvrtc and libcuda are bound with
// dlopen: the library has no link-time dependency on them.
#include <dlfcn.h>

#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "lm_cov.cuh"
#include "runtime.cuh"

namespace mirb200 {

extern const char* const kEmbeddedNames[];
extern const char* const kEmbeddedSources[];
extern const int kEmbeddedCount;

namespace {

// ---- NVRTC / driver API, bound at run time --------------------------------------------------------------------------
using nvrtcProgram = void*;
struct Rtc {
    void* h = nullptr; void* hcu = nullptr;
    int (*createProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*destroyProgram)(nvrtcProgram*) = nullptr;
    int (*compileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
    int (*getProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
    int (*getProgramLog)(nvrtcProgram, char*) = nullptr;
    int (*getCUBINSize)(nvrtcProgram, size_t*) = nullptr;
    int (*getCUBIN)(nvrtcProgram, char*) = nullptr;
    int (*addNameExpression)(nvrtcProgram, const char*) = nullptr;
    int (*getLoweredName)(nvrtcProgram, const char*, const char**) = nullptr;
    const char* (*getErrorString)(int) = nullptr;
    // driver
    int (*cuModuleLoadData)(void**, const void*) = nullptr;
    int (*cuModuleUnload)(void*) = nullptr;
    int (*cuModuleGetFunction)(void**, void*, const char*) = nullptr;
    int (*cuFuncSetAttribute)(void*, int, int) = nullptr;
    int (*cuOccupancy)(int*, void*, int, size_t) = nullptr;
    int (*cuLaunchKernel)(void*, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void*, void**, void**) = nullptr;
    int (*cuGetErrorString)(int, const char**) = nullptr;
    bool ok = false, okCu = false;     // NVRTC usable (compilation) / driver API usable (loading and launching)
    std::string why, whyCu;
};

Rtc& rtc()
{
    static Rtc r;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* nm : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"}) { r.h = dlopen(nm, RTLD_NOW | RTLD_LOCAL); if (r.h) break; }
        if (!r.h) { const char* e = dlerror(); r.why = std::string("dlopen(libnvrtc.so.12) failed: ") + (e ? e : "?"); return; }
        r.hcu = dlopen("libcuda.so.1", RTLD_NOW | RTLD_LOCAL);
        if (!r.hcu) { const char* e = dlerror(); r.whyCu = std::string("dlopen(libcuda.so.1) failed: ") + (e ? e : "?"); }
        auto S = [&](void* h, const char* n) { return dlsym(h, n); };
#define BIND(field, handle, name) r.field = reinterpret_cast<decltype(r.field)>(S(handle, name))
        BIND(createProgram, r.h, "nvrtcCreateProgram"); BIND(destroyProgram, r.h, "nvrtcDestroyProgram"); BIND(compileProgram, r.h, "nvrtcCompileProgram");
        BIND(getProgramLogSize, r.h, "nvrtcGetProgramLogSize"); BIND(getProgramLog, r.h, "nvrtcGetProgramLog");
        BIND(getCUBINSize, r.h, "nvrtcGetCUBINSize"); BIND(getCUBIN, r.h, "nvrtcGetCUBIN");
        BIND(addNameExpression, r.h, "nvrtcAddNameExpression"); BIND(getLoweredName, r.h, "nvrtcGetLoweredName"); BIND(getErrorString, r.h, "nvrtcGetErrorString");
        if (r.hcu) {
            BIND(cuModuleLoadData, r.hcu, "cuModuleLoadData"); BIND(cuModuleUnload, r.hcu, "cuModuleUnload"); BIND(cuModuleGetFunction, r.hcu, "cuModuleGetFunction");
            BIND(cuFuncSetAttribute, r.hcu, "cuFuncSetAttribute"); BIND(cuOccupancy, r.hcu, "cuOccupancyMaxActiveBlocksPerMultiprocessor");
            BIND(cuLaunchKernel, r.hcu, "cuLaunchKernel"); BIND(cuGetErrorString, r.hcu, "cuGetErrorString");
        }
#undef BIND
        r.ok = r.createProgram && r.destroyProgram && r.compileProgram && r.getProgramLogSize && r.getProgramLog && r.getCUBINSize && r.getCUBIN &&
               r.addNameExpression && r.getLoweredName;
        if (!r.ok) r.why = "libnvrtc lacks a required entry point";
        r.okCu = r.cuModuleLoadData && r.cuModuleGetFunction && r.cuFuncSetAttribute && r.cuOccupancy && r.cuLaunchKernel;
        if (!r.okCu && r.whyCu.empty()) r.whyCu = "libcuda lacks a required entry point";
    });
    return r;
}

struct Compiled { void* module = nullptr; void* fn[2] = {nullptr, nullptr}; };   // fn[FD]
// the programs compiled per user model: the LM kernel (at registration for double), the covariance kernel and the
// weighted forms of both (lazily)
enum Program { kProgLM = 0, kProgCov = 1, kProgLMW = 2, kProgCovW = 3, kProgCount = 4 };
struct UserModelEntry {
    std::string source;
    std::mutex mu;                                  // compilation / loading of THIS model (others are not held up)
    // key = (device ordinal * 2 + (float ? 1 : 0)) * kProgCount + program: a module belongs to one context
    std::map<int, std::unique_ptr<Compiled>> loaded;
    std::vector<char> cubin[kProgCount][2]; std::string names[kProgCount][2][2];   // [program][precision], kept for other devices
};
std::mutex g_mu;
std::map<uint32_t, std::shared_ptr<UserModelEntry>> g_models;
uint32_t g_next = (uint32_t)MIR_MODEL_USER_BASE;

// NVRTC compile (no device needed); cubin returned in `cubin`, lowered kernel names in names[FD]
int compile_source(const std::string& user, bool isFloat, Program which, std::vector<char>& cubin, std::string names[2])
{
    Rtc& r = rtc();
    if (!r.ok) { set_error("mir_optim_b200: run-time compilation unavailable: " + r.why); return MIR_B200_EUNSUPPORTED; }
    const char* T = isFloat ? "float" : "double";
    const bool lm = which == kProgLM || which == kProgLMW, weighted = which == kProgLMW || which == kProgCovW;
    const std::string header = lm ? "lm_cta.cuh" : "lm_cov.cuh";
    const std::string kernel = lm ? "mirb200::lm_cta_kernel" : weighted ? "mirb200::lm_cov_cta_weighted_kernel" : "mirb200::lm_cov_cta_kernel";
    std::string src = "#include \"" + header + "\"\n#line 1 \"user_model.cu\"\n" + user + "\n";
    std::string model = std::string("mirb200::CtaUser<UserModel<") + T + ">, " + T + ">";
    if (weighted) model = "mirb200::CtaWeighted<" + model + ", " + T + ">";
    const std::string e0 = kernel + "<" + model + ", " + T + ", false>";
    const std::string e1 = kernel + "<" + model + ", " + T + ", true>";
    nvrtcProgram prog = nullptr;
    int rc = r.createProgram(&prog, src.c_str(), "mir_user_model.cu", kEmbeddedCount, kEmbeddedSources, kEmbeddedNames);
    if (rc) { set_error(std::string("mir_optim_b200: nvrtcCreateProgram: ") + (r.getErrorString ? r.getErrorString(rc) : "?")); return MIR_B200_ECUDA; }
    r.addNameExpression(prog, e0.c_str()); r.addNameExpression(prog, e1.c_str());
    const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-default-device", "--device-int128"};
    rc = r.compileProgram(prog, 3, opts);
    if (rc) {
        size_t n = 0; r.getProgramLogSize(prog, &n);
        std::string log(n, '\0'); if (n) r.getProgramLog(prog, &log[0]);
        if (log.size() > 6000) log.resize(6000);
        set_error("mir_optim_b200: the model source does not compile:\n" + log);
        r.destroyProgram(&prog);
        return MIR_B200_EINVAL;
    }
    const char* ln = nullptr;
    if (r.getLoweredName(prog, e0.c_str(), &ln) == 0 && ln) names[0] = ln;
    if (r.getLoweredName(prog, e1.c_str(), &ln) == 0 && ln) names[1] = ln;
    size_t sz = 0; r.getCUBINSize(prog, &sz);
    cubin.resize(sz);
    if (sz) r.getCUBIN(prog, cubin.data());
    r.destroyProgram(&prog);
    if (!sz || names[0].empty() || names[1].empty()) { set_error("mir_optim_b200: NVRTC produced no code for the kernel"); return MIR_B200_ECUDA; }
    return MIR_B200_OK;
}

int cu_fail(const char* what, int rc)
{
    const char* s = nullptr;
    if (rtc().cuGetErrorString) rtc().cuGetErrorString(rc, &s);
    set_error(std::string("mir_optim_b200: ") + what + ": " + (s ? s : "driver error") + " (" + std::to_string(rc) + ")");
    return MIR_B200_ECUDA;
}

int get_compiled(uint32_t id, bool isFloat, Program prog, Compiled** out)
{
    std::shared_ptr<UserModelEntry> e;
    {
        std::lock_guard<std::mutex> g(g_mu);
        auto it = g_models.find(id);
        if (it == g_models.end()) { set_error("mir_optim_b200: unknown user model id"); return MIR_B200_EINVAL; }
        e = it->second;
    }
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    std::lock_guard<std::mutex> g(e->mu);
    std::unique_ptr<Compiled>& c = e->loaded[(dev * 2 + (isFloat ? 1 : 0)) * kProgCount + prog];
    if (!c) {
        const int pi = isFloat ? 1 : 0;
        if (e->cubin[prog][pi].empty()) { const int rc = compile_source(e->source, isFloat, prog, e->cubin[prog][pi], e->names[prog][pi]); if (rc) return rc; }
        Rtc& r = rtc();
        if (!r.okCu) { set_error("mir_optim_b200: cannot load a compiled model: " + r.whyCu); return MIR_B200_ENODEVICE; }
        auto cc = std::make_unique<Compiled>();
        int cr = r.cuModuleLoadData(&cc->module, e->cubin[prog][pi].data());
        if (cr) return cu_fail("cuModuleLoadData (user model)", cr);
        for (int fd = 0; fd < 2; ++fd) {
            cr = r.cuModuleGetFunction(&cc->fn[fd], cc->module, e->names[prog][pi][fd].c_str());
            if (cr) return cu_fail("cuModuleGetFunction (user model)", cr);
        }
        c = std::move(cc);
    }
    *out = c.get();
    return MIR_B200_OK;
}

// a kernel compiled at run time, for launch_persistent (lm_cta.cuh; driver API); `what` names the launch in its error
struct DriverKernel {
    void* fn; const char* what;
    static int rc(int cr, const char* call) { return cr ? cu_fail(call, cr) : MIR_B200_OK; }
    int set_smem(size_t smem) const { return rc(rtc().cuFuncSetAttribute(fn, 8 /* CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES */, (int)smem), "cuFuncSetAttribute"); }
    int occupancy(int* blocks, size_t smem) const { return rc(rtc().cuOccupancy(blocks, fn, CTA_NT, smem), "cuOccupancyMaxActiveBlocksPerMultiprocessor"); }
    int launch(unsigned grid, size_t smem, cudaStream_t s, void** params) const
    {
        return rc(rtc().cuLaunchKernel(fn, grid, 1, 1, CTA_NT, 1, 1, (unsigned)smem, s, params, nullptr), what);
    }
};

}  // namespace

template <class T>
int launch_user_model(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    if (n > 128) { set_error("mir_optim_b200: the batched path supports n <= 128"); return MIR_B200_EUNSUPPORTED; }
    Compiled* c = nullptr;
    if (int rc = get_compiled(model.model, sizeof(T) == 4, (model.flags & MIR_MODEL_WEIGHTED) ? kProgLMW : kProgLM, &c)) return rc;
    void* fn = c->fn[(args.flags & MIR_MODEL_FD_JACOBIAN) ? 1 : 0];      // (a model without jacobian() runs finite differences either way)
    return launch_cta_fit<T>(DriverKernel{fn, "cuLaunchKernel (user model)"}, st, args, model, n, 1, stream);
}
template int launch_user_model<double>(const mir_model_desc&, size_t, const Num<double>::Settings&, const SmallBatchArgs&, cudaStream_t);
template int launch_user_model<float>(const mir_model_desc&, size_t, const Num<float>::Settings&, const SmallBatchArgs&, cudaStream_t);

template <class T>
int launch_user_cov(const mir_model_desc& model, T jacEps, CovArgs ca, cudaStream_t stream)
{
    Compiled* c = nullptr;
    if (int rc = get_compiled(model.model, sizeof(T) == 4, (model.flags & MIR_MODEL_WEIGHTED) ? kProgCovW : kProgCov, &c)) return rc;
    void* fn = c->fn[(model.flags & MIR_MODEL_FD_JACOBIAN) ? 1 : 0];      // (a model without jacobian() runs finite differences either way)
    return launch_cov<T>(DriverKernel{fn, "cuLaunchKernel (user model covariance)"}, jacEps, ca, 1, stream);
}
template int launch_user_cov<double>(const mir_model_desc&, double, CovArgs, cudaStream_t);
template int launch_user_cov<float>(const mir_model_desc&, float, CovArgs, cudaStream_t);

}  // namespace mirb200

using namespace mirb200;

extern "C" {

int mir_b200_model_compile(const char* source, uint32_t* model_id)
{
    clear_error();
    if (!source || !model_id) { set_error("mir_b200_model_compile: null argument"); return MIR_B200_EINVAL; }
    // validate now (double precision; NVRTC needs no device), so that syntax errors surface at registration
    auto e = std::make_shared<UserModelEntry>();
    e->source = source;
    const int rc = compile_source(e->source, false, kProgLM, e->cubin[kProgLM][0], e->names[kProgLM][0]);
    if (rc) return rc;
    std::lock_guard<std::mutex> g(g_mu);
    *model_id = g_next++;
    g_models[*model_id] = e;
    return MIR_B200_OK;
}

int mir_b200_model_release(uint32_t model_id)
{
    std::lock_guard<std::mutex> g(g_mu);
    auto it = g_models.find(model_id);
    if (it == g_models.end()) return MIR_B200_EINVAL;
    // kernels of this model may still be running: modules are unloaded after the devices that hold them are idle
    int cur = 0; cudaGetDevice(&cur);
    for (auto& kv : it->second->loaded) {
        if (!kv.second || !kv.second->module || !rtc().cuModuleUnload) continue;
        if (cudaSetDevice(kv.first / (2 * kProgCount)) == cudaSuccess) { cudaDeviceSynchronize(); rtc().cuModuleUnload(kv.second->module); }
    }
    cudaSetDevice(cur);
    g_models.erase(it);
    return MIR_B200_OK;
}

}  // extern "C"
