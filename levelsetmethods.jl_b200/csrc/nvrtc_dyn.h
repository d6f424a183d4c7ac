// nvrtc_dyn.h — NVRTC bound at run time with dlopen (like nccl_dyn.h), so that liblsm_b200.so keeps loading on a machine
// without the run-time compiler; only the expression-coefficient entry points (lsm_expr_check, lsm_field_set_expr) need it.
#pragma once
#include <cstdlib>
#include <dlfcn.h>
#include <mutex>
#include <string>
#include <nvrtc.h>   // types and enums only

namespace lsm {

struct NvrtcApi {
    void* handle = nullptr;
    nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
    nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
    nvrtcResult (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
    nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
    nvrtcResult (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
    nvrtcResult (*DestroyProgram)(nvrtcProgram*) = nullptr;
    const char* (*GetErrorString)(nvrtcResult) = nullptr;

    bool load(const char** why) {
        static std::mutex mu;
        std::lock_guard<std::mutex> lk(mu);
        if (handle) return true;
        std::string home = getenv("CUDA_HOME") ? std::string(getenv("CUDA_HOME")) + "/lib64/libnvrtc.so.12" : std::string();
        const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", home.empty() ? nullptr : home.c_str()};
        for (const char* n : names) {
            if (!n) continue;
            handle = dlopen(n, RTLD_NOW | RTLD_LOCAL);
            if (handle) break;
        }
        if (!handle) { *why = dlerror(); return false; }
#define LSM_SYM(field, sym) field = reinterpret_cast<decltype(field)>(dlsym(handle, sym)); \
        if (!field) { *why = "missing NVRTC symbol " sym; dlclose(handle); handle = nullptr; return false; }
        LSM_SYM(CreateProgram, "nvrtcCreateProgram")
        LSM_SYM(CompileProgram, "nvrtcCompileProgram")
        LSM_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
        LSM_SYM(GetProgramLog, "nvrtcGetProgramLog")
        LSM_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
        LSM_SYM(GetCUBIN, "nvrtcGetCUBIN")
        LSM_SYM(DestroyProgram, "nvrtcDestroyProgram")
        LSM_SYM(GetErrorString, "nvrtcGetErrorString")
#undef LSM_SYM
        return true;
    }
};

inline NvrtcApi& nvrtc() { static NvrtcApi api; return api; }

}  // namespace lsm
