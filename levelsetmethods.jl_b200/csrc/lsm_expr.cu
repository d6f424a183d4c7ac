// lsm_expr.cu — coefficients written as CUDA C++ expressions in x1..xN and t: the device form of a function-valued coefficient
// f(x, t) (levelsetterms.jl:42-43, _eval_field).  Validation, source generation, NVRTC compilation for sm_100a, the process-wide
// cache of compiled kernels and the launch of the generated pointwise kernel.  The engine side (when a field is materialised,
// how its CFL maximum is consumed) is in lsm_api.cu.
//
// The generated kernel evaluates every expression in double at x_d = lc_d + i_d h_d (i_d the 0-based GLOBAL node index, as
// fill_shape_kernel and grid.coords compute it), rounds to the field's dtype on store, and reduces the CFL quantity of the rounded
// values with the per-node formula and IEEE-bits maximum of cfl_kernel (lsm_generic.cu).  It is compiled with --fmad=false and
// without fast-math, so the written operation order is the executed one and + - * / sqrt fabs fmin fmax are bit-identical to
// the same formula in NumPy float64.
#include <cctype>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/lsm_b200.h"
#include "lsm_kernels.h"
#include "nvrtc_dyn.h"

namespace lsm {

struct ExprKernel {
    std::vector<char> cubin;
    bool uses_t = false;
    cudaLibrary_t lib = nullptr;     // loaded on first use by a field (needs a device; compiling does not)
    cudaKernel_t kern = nullptr;
};

namespace {

// The only parameter of the generated kernel; its host twin is ExprArgs (lsm_kernels.h): same members, same order.
const char* const ARGS_SRC =
    "struct lsm_args {\n"
    "    void* dst; unsigned long long* cfl; long long cstride;\n"
    "    int n[3]; int first_last; int f64; int cfl_kind;\n"
    "    double lc[3]; double h[3]; double t;\n"
    "};\n"
    "static_assert(sizeof(lsm_args) == 104, \"lsm_args layout\");\n";
static_assert(sizeof(ExprArgs) == 104, "ExprArgs layout");

std::mutex g_mu;                                                  // lsm_multi_* drive the ranks from several host threads
std::map<std::string, std::unique_ptr<ExprKernel>> g_cache;        // generated source -> kernel; lives as long as the process

std::string quoted(const char* e) {
    std::string s(e);
    if (s.size() > 80) s = s.substr(0, 77) + "...";
    return "\"" + s + "\"";
}

struct Tok { char kind; std::string s; };     // 'i' identifier, 'n' integer literal, 'f' floating literal, 'o' operator character

// Host-side checks of one expression (see lsm_expr_check in include/lsm_b200.h); tokens are only as fine as these checks need.
int32_t validate(int k, const char* e, bool* uses_t, std::string* err) {
    char buf[256];
    auto bad = [&](const char* why) {
        snprintf(buf, sizeof buf, "expression %d (%s): %s", k + 1, quoted(e).c_str(), why);
        *err = buf;
        return (int32_t)LSM_ERR_ARG;
    };
    bool blank = true;
    for (const char* p = e; *p; ++p) if (!isspace((unsigned char)*p)) blank = false;
    if (blank) return bad("empty expression");
    for (const char* p = e; *p; ++p)
        if (strchr(";{}#\"'\\`", *p)) {
            snprintf(buf, sizeof buf, "the character '%c' is not allowed: an expression is a single C++ expression", *p);
            std::string why = buf;
            return bad(why.c_str());
        }
    std::vector<Tok> toks;
    const size_t n = strlen(e);
    for (size_t i = 0; i < n;) {
        const unsigned char c = (unsigned char)e[i];
        if (isspace(c)) { ++i; continue; }
        if (isalpha(c) || c == '_') {
            size_t j = i;
            while (j < n && (isalnum((unsigned char)e[j]) || e[j] == '_')) ++j;
            toks.push_back({'i', std::string(e + i, j - i)});
            i = j;
        } else if (isdigit(c) || (c == '.' && i + 1 < n && isdigit((unsigned char)e[i + 1]))) {
            const bool hex = c == '0' && i + 1 < n && (e[i + 1] == 'x' || e[i + 1] == 'X');
            size_t j = i;
            bool flt = false;
            while (j < n && (isalnum((unsigned char)e[j]) || e[j] == '_' || e[j] == '.')) {
                const char d = e[j];
                if (d == '.') flt = true;
                const bool expo = hex ? (d == 'p' || d == 'P') : (d == 'e' || d == 'E');
                if (expo) { flt = true; if (j + 1 < n && (e[j + 1] == '+' || e[j + 1] == '-')) ++j; }
                ++j;
            }
            toks.push_back({flt ? 'f' : 'n', std::string(e + i, j - i)});
            i = j;
        } else {
            toks.push_back({'o', std::string(1, (char)c)});
            ++i;
        }
    }
    for (const Tok& t : toks) {
        if (t.kind != 'i') continue;
        if (t.s.compare(0, 4, "lsm_") == 0 || t.s.compare(0, 2, "__") == 0) {
            snprintf(buf, sizeof buf, "the identifier '%.40s' is reserved (names starting with lsm_ or __ belong to the generated code)", t.s.c_str());
            std::string why = buf;
            return bad(why.c_str());
        }
        if (t.s == "t") *uses_t = true;
    }
    // integer literal / integer literal: C++ truncates (1/3 == 0) where Julia and Python give 0.333...
    for (size_t i = 0; i + 2 < toks.size(); ++i) {
        if (toks[i].kind != 'n' || toks[i + 1].kind != 'o' || toks[i + 1].s != "/") continue;
        size_t j = i + 2;
        while (j < toks.size() && toks[j].kind == 'o' && (toks[j].s == "+" || toks[j].s == "-")) ++j;
        if (j < toks.size() && toks[j].kind == 'n') {
            snprintf(buf, sizeof buf, "integer division %.20s/%.20s truncates in C++; write a floating literal such as %.20s.0", toks[i].s.c_str(),
                     toks[j].s.c_str(), toks[i].s.c_str());
            std::string why = buf;
            return bad(why.c_str());
        }
    }
    return LSM_OK;
}

std::string generate(int ndim, int ncomp, const char* const* exprs) {
    const std::string N = std::to_string(ndim), C = std::to_string(ncomp);
    std::string s = "// lsm_b200 expression coefficient: ndim " + N + ", ncomp " + C + "\n";
    s += ARGS_SRC;
    s += "extern \"C\" __global__ void __launch_bounds__(256) lsm_expr_fill(const lsm_args lsm_a) {\n"
         "    [[maybe_unused]] const double pi = 3.141592653589793;\n"
         "    [[maybe_unused]] const double t = lsm_a.t;\n"
         "    const long long lsm_total = (long long)lsm_a.n[0] * lsm_a.n[1] * lsm_a.n[2];\n"
         "    unsigned long long lsm_best = 0ULL;\n"
         "    for (long long lsm_i = (long long)blockIdx.x * blockDim.x + threadIdx.x; lsm_i < lsm_total; lsm_i += (long long)gridDim.x * blockDim.x) {\n"
         "        int lsm_I[3];\n"
         "        lsm_I[0] = (int)(lsm_i % lsm_a.n[0]);\n"
         "        const long long lsm_q = lsm_i / lsm_a.n[0];\n"
         "        lsm_I[1] = (int)(lsm_q % lsm_a.n[1]);\n"
         "        lsm_I[2] = (int)(lsm_q / lsm_a.n[1]);\n"
         "        lsm_I[" + std::to_string(ndim - 1) + "] += lsm_a.first_last;\n";
    for (int d = 0; d < ndim; ++d)
        s += "        [[maybe_unused]] const double x" + std::to_string(d + 1) + " = lsm_a.lc[" + std::to_string(d) + "] + (double)lsm_I[" + std::to_string(d) +
             "] * lsm_a.h[" + std::to_string(d) + "];\n";
    for (int c = 0; c < ncomp; ++c)     // one line per expression: the log of a compile error quotes it
        s += "        const double lsm_e" + std::to_string(c) + " = (" + std::string(exprs[c]) + ");\n";
    s += "        double lsm_v[" + C + "];\n"
         "        if (lsm_a.f64) {\n";
    for (int c = 0; c < ncomp; ++c)
        s += "            ((double*)lsm_a.dst)[" + std::to_string(c) + " * lsm_a.cstride + lsm_i] = lsm_e" + std::to_string(c) + "; lsm_v[" +
             std::to_string(c) + "] = lsm_e" + std::to_string(c) + ";\n";
    s += "        } else {\n";
    for (int c = 0; c < ncomp; ++c)
        s += "            { const float lsm_r = (float)lsm_e" + std::to_string(c) + "; ((float*)lsm_a.dst)[" + std::to_string(c) +
             " * lsm_a.cstride + lsm_i] = lsm_r; lsm_v[" + std::to_string(c) + "] = (double)lsm_r; }\n";
    s += "        }\n"
         "        double lsm_s = 0.0;\n"
         "        if (lsm_a.cfl_kind == 1) {\n"                                  // advection: sum_d |u_d| / h_d
         "            for (int lsm_d = 0; lsm_d < " + C + "; ++lsm_d) {\n"
         "                const double lsm_w = fabs(lsm_v[lsm_d]) / lsm_a.h[lsm_d];\n"
         "                lsm_s = lsm_d == 0 ? lsm_w : lsm_s + lsm_w;\n"
         "            }\n"
         "        } else if (lsm_a.cfl_kind == 2) {\n"                           // normal motion, curvature: |v|
         "            lsm_s = fabs(lsm_v[0]);\n"
         "        }\n"
         "        const unsigned long long lsm_b = isnan(lsm_s) ? 0x7FF8000000000000ULL : (unsigned long long)__double_as_longlong(lsm_s);\n"
         "        lsm_best = lsm_b > lsm_best ? lsm_b : lsm_best;\n"
         "    }\n"
         "    if (lsm_a.cfl_kind == 0) return;\n"
         "    for (int lsm_o = 16; lsm_o > 0; lsm_o >>= 1) {\n"
         "        const unsigned long long lsm_x = __shfl_xor_sync(0xffffffffu, lsm_best, lsm_o);\n"
         "        lsm_best = lsm_x > lsm_best ? lsm_x : lsm_best;\n"
         "    }\n"
         "    __shared__ unsigned long long lsm_wbest[8];\n"
         "    const int lsm_lane = threadIdx.x & 31, lsm_warp = threadIdx.x >> 5;\n"
         "    if (lsm_lane == 0) lsm_wbest[lsm_warp] = lsm_best;\n"
         "    __syncthreads();\n"
         "    if (lsm_warp == 0) {\n"
         "        lsm_best = lsm_lane < (int)(blockDim.x >> 5) ? lsm_wbest[lsm_lane] : 0ULL;\n"
         "        for (int lsm_o = 4; lsm_o > 0; lsm_o >>= 1) {\n"
         "            const unsigned long long lsm_x = __shfl_xor_sync(0xffffffffu, lsm_best, lsm_o);\n"
         "            lsm_best = lsm_x > lsm_best ? lsm_x : lsm_best;\n"
         "        }\n"
         "        if (lsm_lane == 0) atomicMax(lsm_a.cfl, lsm_best);\n"
         "    }\n"
         "}\n";
    return s;
}

int32_t compile(const std::string& src, ExprKernel* k, std::string* err) {
    const char* why = "";
    if (!nvrtc().load(&why)) { *err = std::string("cannot load NVRTC (libnvrtc.so.12), which expression coefficients need: ") + why; return LSM_ERR_UNSUPPORTED; }
    NvrtcApi& R = nvrtc();
    nvrtcProgram prog = nullptr;
    nvrtcResult r = R.CreateProgram(&prog, src.c_str(), "lsm_expr.cu", 0, nullptr, nullptr);
    if (r != NVRTC_SUCCESS) { *err = std::string("nvrtcCreateProgram failed: ") + R.GetErrorString(r); return LSM_ERR_CUDA; }
    // no fast-math: correctly rounded division and sqrt; no FMA contraction: the written operation order is the executed one
    const char* opts[] = {"-arch=sm_100a", "--fmad=false", "-std=c++17"};
    r = R.CompileProgram(prog, 3, opts);
    int32_t rc = LSM_OK;
    if (r != NVRTC_SUCCESS) {
        size_t ls = 0;
        R.GetProgramLogSize(prog, &ls);
        std::string log(ls, '\0');
        if (ls) R.GetProgramLog(prog, &log[0]);
        while (!log.empty() && log.back() == '\0') log.pop_back();
        *err = std::string("the expression does not compile (NVRTC: ") + R.GetErrorString(r) + "):\n" + log;
        rc = r == NVRTC_ERROR_COMPILATION ? LSM_ERR_ARG : LSM_ERR_CUDA;
    } else {
        size_t cs = 0;
        R.GetCUBINSize(prog, &cs);
        k->cubin.resize(cs);
        if (cs == 0 || R.GetCUBIN(prog, k->cubin.data()) != NVRTC_SUCCESS) { *err = "NVRTC produced no sm_100a code"; rc = LSM_ERR_CUDA; }
    }
    R.DestroyProgram(&prog);
    return rc;
}

}  // namespace

int32_t expr_get(int ndim, int ncomp, const char* const* exprs, bool load, const ExprKernel** out, std::string* err) {
    char buf[256];
    if (!exprs) { *err = "null expression list"; return LSM_ERR_ARG; }
    if (ndim < 1 || ndim > 3) { snprintf(buf, sizeof buf, "ndim must be 1, 2 or 3 (got %d)", ndim); *err = buf; return LSM_ERR_ARG; }
    if (ncomp != 1 && ncomp != ndim) { snprintf(buf, sizeof buf, "ncomp must be 1 or ndim = %d (got %d)", ndim, ncomp); *err = buf; return LSM_ERR_ARG; }
    int count = 0;
    while (count <= ncomp && exprs[count]) ++count;
    if (count != ncomp) {
        snprintf(buf, sizeof buf, "%s expressions for %d component(s): give one per component, then a NULL pointer",
                 count > ncomp ? "more than ncomp" : "fewer than ncomp", ncomp);
        *err = buf;
        return LSM_ERR_ARG;
    }
    bool uses_t = false;
    for (int c = 0; c < ncomp; ++c) { const int32_t rc = validate(c, exprs[c], &uses_t, err); if (rc != LSM_OK) return rc; }
    const std::string src = generate(ndim, ncomp, exprs);
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_cache.find(src);
    ExprKernel* k = it == g_cache.end() ? nullptr : it->second.get();
    if (!k) {
        std::unique_ptr<ExprKernel> nk(new ExprKernel());
        nk->uses_t = uses_t;
        const int32_t rc = compile(src, nk.get(), err);
        if (rc != LSM_OK) return rc;
        k = nk.get();
        g_cache.emplace(src, std::move(nk));
    }
    if (load && !k->kern) {
        cudaError_t e = cudaLibraryLoadData(&k->lib, k->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
        if (e == cudaSuccess) e = cudaLibraryGetKernel(&k->kern, k->lib, "lsm_expr_fill");
        if (e != cudaSuccess) {
            if (k->lib) cudaLibraryUnload(k->lib);
            k->lib = nullptr; k->kern = nullptr;
            *err = std::string("loading the compiled expression kernel failed: ") + cudaGetErrorString(e);
            return e == cudaErrorMemoryAllocation ? LSM_ERR_OOM : LSM_ERR_CUDA;
        }
    }
    *out = k;
    return LSM_OK;
}

bool expr_uses_t(const ExprKernel* k) { return k->uses_t; }

cudaError_t launch_expr_fill(const ExprKernel* k, const ExprArgs& A, int sm_count, cudaStream_t s) {
    const long total = (long)A.n[0] * A.n[1] * A.n[2];
    const int block = 256;
    long grid = (total + block - 1) / block;
    const long cap = (long)sm_count * 8;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    ExprArgs a = A;
    void* args[] = {&a};
    return cudaLaunchKernel(reinterpret_cast<const void*>(k->kern), dim3((unsigned)grid), dim3(block), args, 0, s);
}

}  // namespace lsm
