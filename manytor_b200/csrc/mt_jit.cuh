// Run-time specialisation of the generic DH chain (the reference's "pluggable fk", README.md:20).
//
// A preset arm (mt_step.cuh) gets its DH table folded at compile time; this file gives ANY table the
// same treatment without rebuilding the library: at mt_create the table is printed into a
// `Preset<ID>` specialisation, NVRTC compiles `step_kernel<ID, X, RAND, WOBS, F16, FINAL>` for sm_100a from the
// very same headers the library was built from (embedded as strings by manytor_b200/build.py), and
// the cubin is loaded through the runtime's library API.  ~0.8 s per variant, cached per process.
// NVRTC is dlopen'ed: when it is absent the handle simply keeps the run-time-table kernels.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdio>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "mt_embedded.inc"   // kEmbeddedHeaderNames[], kEmbeddedHeaderSources[], kEmbeddedHeaderCount
#include "mt_step.cuh"

namespace mt {

struct Nvrtc {
    typedef struct _nvrtcProgram *Program;
    int (*CreateProgram)(Program *, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
    int (*DestroyProgram)(Program *) = nullptr;
    int (*CompileProgram)(Program, int, const char *const *) = nullptr;
    int (*GetProgramLogSize)(Program, size_t *) = nullptr;
    int (*GetProgramLog)(Program, char *) = nullptr;
    int (*GetCUBINSize)(Program, size_t *) = nullptr;
    int (*GetCUBIN)(Program, char *) = nullptr;
    int (*AddNameExpression)(Program, const char *) = nullptr;
    int (*GetLoweredName)(Program, const char *, const char **) = nullptr;
    bool ok = false;

    static Nvrtc &get() {
        static Nvrtc n;
        static std::once_flag once;
        std::call_once(once, [] {
            void *h = nullptr;
            for (const char *name : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12",
                                     "/usr/local/cuda/lib64/libnvrtc.so"}) {
                h = dlopen(name, RTLD_NOW | RTLD_LOCAL);
                if (h) break;
            }
            if (!h) return;
#define MT_SYM(field, sym) n.field = reinterpret_cast<decltype(n.field)>(dlsym(h, sym)); if (!n.field) return;
            MT_SYM(CreateProgram, "nvrtcCreateProgram")
            MT_SYM(DestroyProgram, "nvrtcDestroyProgram")
            MT_SYM(CompileProgram, "nvrtcCompileProgram")
            MT_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
            MT_SYM(GetProgramLog, "nvrtcGetProgramLog")
            MT_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
            MT_SYM(GetCUBIN, "nvrtcGetCUBIN")
            MT_SYM(AddNameExpression, "nvrtcAddNameExpression")
            MT_SYM(GetLoweredName, "nvrtcGetLoweredName")
#undef MT_SYM
            n.ok = true;
        });
        return n;
    }
};

// host headers NVRTC does not have: just enough for mt_*.cuh
static const char *const kShimNames[] = {"stdint.h", "cuda_runtime.h", "type_traits"};
static const char *const kShimSources[] = {
    "typedef signed char int8_t; typedef unsigned char uint8_t; typedef short int16_t; typedef unsigned short uint16_t;\n"
    "typedef int int32_t; typedef unsigned int uint32_t; typedef long long int64_t; typedef unsigned long long uint64_t;\n"
    "typedef unsigned long long uintptr_t;\n",
    "\n",
    "namespace std { template <class T, T v> struct integral_constant { static constexpr T value = v; typedef T value_type; }; }\n"};

struct JitKernel {
    cudaLibrary_t lib = nullptr;
    cudaKernel_t kernel = nullptr;
};

// The Preset<> specialisation text of a (snapped) table: the cache key and the JIT input.
static std::string preset_source(int id, int J, const JointConst *rows) {
    std::string s = "template <> struct Preset<" + std::to_string(id) + "> {\n    static constexpr bool value = true;\n"
                    "    __host__ __device__ static constexpr JointConst row(int i) {\n        switch (i) {\n";
    char buf[256];
    for (int i = 0; i < J; ++i) {
        std::snprintf(buf, sizeof(buf), "            %s return JointConst{%.9ef, %.9ef, %.9ef, %.9ef, %.9ef, %.9ef};\n",
                      i + 1 < J ? ("case " + std::to_string(i) + ":").c_str() : "default:", rows[i].a, rows[i].d, rows[i].ca,
                      rows[i].sa, rows[i].co, rows[i].so);
        s += buf;
    }
    s += "        }\n    }\n};\n";
    return s;
}

// Compile (or fetch from the per-process cache) step_kernel<id, x_template, rnd, wobs, f16, final> for the table
// described by `preset`.  Returns an empty JitKernel and fills `err` on failure.
// `rollout_mode` >= 0 selects the multi-step rollout_kernel<id, x_template, wobs, f16, RolloutMode(rollout_mode), final>
// (`rnd` is ignored).  The cache key holds the template arguments, so handles with the same table and different
// observation formats, final outputs or rollout modes get different kernels.
static JitKernel jit_step_kernel(const std::string &preset, int id, int x_template, bool rnd, bool wobs, bool f16,
                                 bool final, std::string &err, int rollout_mode = -1) {
    static std::mutex mu;
    static std::map<std::string, JitKernel> cache;
    static const char *const kModes[] = {"mt::RolloutMode::kDrawLast", "mt::RolloutMode::kDrawTrajectory",
                                         "mt::RolloutMode::kActionsTrajectory"};
    const bool rollout = rollout_mode >= 0;
    const char *obs = wobs ? (f16 ? "true, true" : "true, false") : "false, false";
    const std::string targs = (rollout ? std::to_string(id) + ", " + std::to_string(x_template) + ", " + obs + ", " + kModes[rollout_mode]
                                       : std::to_string(id) + ", " + std::to_string(x_template) + ", " + (rnd ? "true" : "false") +
                                             ", " + obs) + (final ? ", true" : ", false");
    const std::string kname = rollout ? "rollout_kernel" : "step_kernel";
    const std::string inst = "mt::" + kname + "<" + targs + ">";
    const std::string key = preset + inst;
    std::lock_guard<std::mutex> lock(mu);
    auto hit = cache.find(key);
    if (hit != cache.end()) return hit->second;
    JitKernel out;
    Nvrtc &rtc = Nvrtc::get();
    if (!rtc.ok) {
        err = "libnvrtc not found";
        return out;
    }
    const std::string src = "#include \"mt_step.cuh\"\nnamespace mt {\n" + preset + "template __global__ void " + kname + "<" +
                            targs + ">(const __grid_constant__ StepParams);\n}\n";
    std::vector<const char *> names(kEmbeddedHeaderNames, kEmbeddedHeaderNames + kEmbeddedHeaderCount);
    std::vector<const char *> sources(kEmbeddedHeaderSources, kEmbeddedHeaderSources + kEmbeddedHeaderCount);
    for (int i = 0; i < 3; ++i) {
        names.push_back(kShimNames[i]);
        sources.push_back(kShimSources[i]);
    }
    Nvrtc::Program prog = nullptr;
    if (rtc.CreateProgram(&prog, src.c_str(), "mt_jit_arm.cu", (int)names.size(), sources.data(), names.data()) != 0) {
        err = "nvrtcCreateProgram failed";
        return out;
    }
    rtc.AddNameExpression(prog, inst.c_str());
    const char *opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-default-device", "-lineinfo"};
    const int rc = rtc.CompileProgram(prog, 4, opts);
    if (rc != 0) {
        size_t n = 0;
        rtc.GetProgramLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) rtc.GetProgramLog(prog, &log[0]);
        err = "nvrtc compilation failed: " + log.substr(0, 400);
        rtc.DestroyProgram(&prog);
        return out;
    }
    const char *lowered = nullptr;
    size_t n = 0;
    if (rtc.GetLoweredName(prog, inst.c_str(), &lowered) != 0 || !lowered || rtc.GetCUBINSize(prog, &n) != 0 || n == 0) {
        err = "nvrtc produced no cubin";
        rtc.DestroyProgram(&prog);
        return out;
    }
    std::vector<char> cubin(n);
    rtc.GetCUBIN(prog, cubin.data());
    const std::string lowered_name = lowered;
    rtc.DestroyProgram(&prog);
    cudaError_t ce = cudaLibraryLoadData(&out.lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (ce == cudaSuccess) ce = cudaLibraryGetKernel(&out.kernel, out.lib, lowered_name.c_str());
    if (ce != cudaSuccess) {
        err = std::string("loading the JIT cubin failed: ") + cudaGetErrorString(ce);
        (void)cudaGetLastError();
        out = JitKernel();
        return out;
    }
    cache[key] = out;
    return out;
}

}  // namespace mt
