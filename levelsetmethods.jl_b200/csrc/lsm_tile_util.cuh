// lsm_tile_util.cuh — device / host helpers shared by the shared-memory stage kernels (lsm_tiled.cu, lsm_pair3d.cu):
// cp.async, TMA + mbarrier wrappers, the restructured WENO5 evaluation, ghost index maps, tensor-map encoding.
#pragma once
#include <type_traits>
#include <cstdint>
#include <cstdlib>
#include <mutex>
#include <cuda.h>          // CUtensorMap + enums only; cuTensorMapEncodeTiled is looked up at run time (no libcuda link)
#include "lsm_dev.cuh"
#include "lsm_bc.cuh"
#include "lsm_kernels.h"

namespace lsm {
namespace {

constexpr int HAL = 3;           // WENO5 reach; every term's stencil fits in it

enum : int { M_ADV_WENO = 1, M_ADV_UPWIND = 2, M_NORMAL = 4, M_CURV = 8, M_EIK = 16, M_ALL = 31 };

__device__ __forceinline__ void cp_async(void* smem_dst, const void* gsrc, int bytes8) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    if (bytes8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
    else        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_pending() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- TMA (cp.async.bulk.tensor) + mbarrier: one elected thread copies a whole (tile + halo) plane -----------
struct TmaMaps {
    int enabled;                       // tensor maps below are valid
    int _pad[15];
    alignas(64) CUtensorMap phi;       // stage input incl. its ghost planes: dims (n0, n1, halo + n2 + halo)
    alignas(64) CUtensorMap aux[8];    // staged coefficient components and phi^n: dims (n0, n1, n2)
};
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LSM_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LSM_DONE_%=;\n"
        "bra LSM_WAIT_%=;\n"
        "LSM_DONE_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned long long* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2),
                   "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

// 1/x for a positive normal x: MUFU.RCP64H seed (uses the top 32 bits of x: relative error ~2^-20) + Newton steps.
// STEPS = 2 gives ~1e-16; STEPS = 1 gives ~1e-12, enough where the quotient is a small correction term
// (WENO5: W = d2 + num/den with |num/den| <= max|e_k| << |d|; see DESIGN.md §4.1).
template <int STEPS>
__device__ __forceinline__ double fast_rcp(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
#pragma unroll
    for (int k = 0; k < STEPS; ++k) {
        const double t = fma(-x, y, 1.0);
        y = fma(y, t, y);
    }
    return y;
}

// The element of largest magnitude among a..e (exact; only its square is used).  A plain compare-select is
// DSETP + 2 SEL (~1 DP slot, measured 60 lane-ops/clk/SM for compare-select + add in tools/fp64_peak.cu), whereas
// fmax() carries NaN-handling code (~3.7 slots).  NaN inputs poison the smoothness indicators anyway.
__device__ __forceinline__ double absmax5(double a, double b, double c, double d, double e) {
    double m = a;
    m = fabs(b) > fabs(m) ? b : m;
    m = fabs(c) > fabs(m) ? c : m;
    m = fabs(d) > fabs(m) ? d : m;
    m = fabs(e) > fabs(m) ? e : m;
    return m;
}

// max|a..e| to 20 significant bits in 2-3 instructions instead of 4 DSETP + 8 FSEL (16 issue slots): the HIGH words of the five
// doubles are compared as Float32 bit patterns with the |.| operand modifier (FMNMX / FMNMX3: sign-cleared IEEE patterns of either
// width order like their magnitudes; a double high word is a finite Float32 pattern for |x| < 2^1017), and the result keeps the
// low word of `a`, which is dead afterwards — so no register move is needed to build the pair.  Only eps = 1e-6 max(v^2) + floor
// uses it (derivatives.jl:71): a relative error < 2^-20 in the maximum changes eps by < 2e-6 relative, which moves the C3 128^3
// result after 100 RK3 steps from 5.5e-15 to ~1e-13 of the oracle (bar 1e-10; tests/test_gpu_parity.py::
// test_config_parity_survey_sizes prints the observed value).  NaN / Inf inputs drop out of the maximum but still poison the
// smoothness indicators, like in the reference.  Used by the x-pair kernel (pure advection) only: with the curvature term on
// kinked data (C2 at 512^2) rounding-level differences are amplified ~1e4-fold over 100 steps (the strict kernel itself is
// 4.6e-12 from the oracle there), so the general tiled kernels keep the exact maximum.
__device__ __forceinline__ double absmax5_hi(double a, double b, double c, double d, double e) {
    const float fa = __int_as_float(__double2hiint(a)), fb = __int_as_float(__double2hiint(b)), fc = __int_as_float(__double2hiint(c)),
                fd = __int_as_float(__double2hiint(d)), fe = __int_as_float(__double2hiint(e));
    const float m = fmaxf(fmaxf(fmaxf(fabsf(fa), fabsf(fb)), fabsf(fc)), fmaxf(fabsf(fd), fabsf(fe)));
    return __hiloint2double(__float_as_int(m), __double2loint(a));
}

// Undivided upwind WENO5: given six samples in upwind order (q3 is the node, q0 the far upwind
// end), returns h * weno5 of the reference (derivatives.jl:61-121), i.e. the reference value is
// this divided by h and multiplied by s = sign of the sampling direction.
//   d_k  = q_{k+1} - q_k            (v_k * h of the reference, up to the global sign s)
//   e_k  = d_k - d_{k-1}
//   4*S1 = 13/3 (e2-e1)^2 + (3e2-e1)^2 ; 4*S2 = 13/3 (e3-e2)^2 + (e2+e3)^2 ; 4*S3 = 13/3 (e4-e3)^2 + (e4-3e3)^2
//   b_k  = 4 h^2 (S_k + eps) = 4*S_k(d) + 4e-6 max(d^2) + floor
//   w_k  ~ {1,6,3} / b_k^2  ->  result = d2 + (q1 G1 + q2 G2 + q3 G3) / (q1 + 6 q2 + 3 q3),  q1 = (b2 b3)^2 ...
//   G1 = 5/6 e2 - 1/3 e1 ; G2 = 2 e3 + e2 ; G3 = 2 e3 - 1/2 e4     (6 and 3 folded in)
// The floor 1e-70 replaces 4e-99*h^2 (which would underflow in the product form).  It only matters
// where every |d| < ~1e-26, i.e. on numerically flat data, where the result is O(|d|) either way.
// The five Float64 constants of the evaluation that do not fit an instruction immediate.  They travel in the kernel
// parameters (constant bank): as literals the compiler re-materialises them with 10 UMOV per node, from the constant bank
// it takes 3 uniform loads.

// weno5_up_f64: first differences in the storage type, everything after in Float64 — Julia's promotion for Float32 fields
// (all literals of derivatives.jl:61-81 are Float64).  weno5_up<T> below is this for T = double and the all-FP32 evaluation for
// T = float.
template <class T>
__device__ __forceinline__ double weno5_up_f64(const WenoK& K, T q0, T q1, T q2, T q3, T q4, T q5) {
    const double d0 = double(T(q1 - q0)), d1 = double(T(q2 - q1)), d2 = double(T(q3 - q2)),
                 d3 = double(T(q4 - q3)), d4 = double(T(q5 - q4));
    const double e1 = d1 - d0, e2 = d2 - d1, e3 = d3 - d2, e4 = d4 - d3;
    const double m = absmax5(d0, d1, d2, d3, d4);
    const double eps = fma(K.e6, m * m, K.fl);
    const double c133 = K.c133;
    const double t1a = e2 - e1, t1b = e3 - e2, t1c = e4 - e3;
    const double t2a = fma(3.0, e2, -e1), t2b = e2 + e3, t2c = fma(-3.0, e3, e4);
    const double b1 = fma(t2a, t2a, fma(c133, t1a * t1a, eps));
    const double b2 = fma(t2b, t2b, fma(c133, t1b * t1b, eps));
    const double b3 = fma(t2c, t2c, fma(c133, t1c * t1c, eps));
    const double p12 = b1 * b2, p13 = b1 * b3, p23 = b2 * b3;
    const double w1 = p23 * p23, w2 = p13 * p13, w3 = p12 * p12;
    const double den = fma(3.0, w3, fma(6.0, w2, w1));
    const double G1 = fma(K.c56, e2, K.cm13 * e1);
    const double G2 = fma(2.0, e3, e2);
    const double G3 = fma(2.0, e3, -0.5 * e4);
    const double num = fma(w3, G3, fma(w2, G2, w1 * G1));
    return fma(num, fast_rcp<1>(den), d2);
}

template <class T>
__device__ __forceinline__ double weno5_up(const WenoK& K, T q0, T q1, T q2, T q3, T q4, T q5) { return weno5_up_f64<T>(K, q0, q1, q2, q3, q4, q5); }

// Float32 fields: the same evaluation entirely in FP32 (FFMA issues at <= 1 slot, FP64 at 2; BASELINE tolerance for
// Float32 is 1e-4 against the oracle, which follows Julia's promotion to Float64 after the first difference).
// Range safety in FP32: the differences are normalised by 1/max|d| before squaring, so b_k = 4(S_k + eps)/max(d^2)
// lies in [4e-6, ~1e2], the weights in [1e-22, 1e8], and eps = 1e-6*max(v^2) becomes the exact constant 4e-6
// (flat data: max|d| = 0 -> all b_k equal -> result d2 = 0, finite).
template <>
__device__ __forceinline__ double weno5_up<float>(const WenoK&, float q0, float q1, float q2, float q3, float q4, float q5) {
    const float d0 = q1 - q0, d1 = q2 - q1, d2 = q3 - q2, d3 = q4 - q3, d4 = q5 - q4;
    const float e1 = d1 - d0, e2 = d2 - d1, e3 = d3 - d2, e4 = d4 - d3;
    const float m = fmaxf(fmaxf(fmaxf(fabsf(d0), fabsf(d1)), fmaxf(fabsf(d2), fabsf(d3))), fabsf(d4));
    const float im = m > 0.f ? __frcp_rn(m) : 0.f;
    const float s1 = e1 * im, s2 = e2 * im, s3 = e3 * im, s4 = e4 * im;
    const float c133 = 13.0f / 3.0f;
    const float t1a = s2 - s1, t1b = s3 - s2, t1c = s4 - s3;
    const float t2a = fmaf(3.0f, s2, -s1), t2b = s2 + s3, t2c = fmaf(-3.0f, s3, s4);
    const float b1 = fmaf(t2a, t2a, fmaf(c133, t1a * t1a, 4.0e-6f));
    const float b2 = fmaf(t2b, t2b, fmaf(c133, t1b * t1b, 4.0e-6f));
    const float b3 = fmaf(t2c, t2c, fmaf(c133, t1c * t1c, 4.0e-6f));
    const float p12 = b1 * b2, p13 = b1 * b3, p23 = b2 * b3;
    const float w1 = p23 * p23, w2 = p13 * p13, w3 = p12 * p12;
    const float den = fmaf(3.0f, w3, fmaf(6.0f, w2, w1));
    const float G1 = fmaf(5.0f / 6.0f, e2, (-1.0f / 3.0f) * e1);
    const float G2 = fmaf(2.0f, e3, e2);
    const float G3 = fmaf(2.0f, e3, -0.5f * e4);
    const float num = fmaf(w3, G3, fmaf(w2, G2, w1 * G1));
    return double(fmaf(num, __frcp_rn(den), d2));
}

// x / 3 correctly rounded without the generic division sequence (timestepping.jl:194 divides by 3 in the storage type):
// q0 = RN(x * RN(1/3)), r = x - 3 q0 (exact in an FMA), q = RN(q0 + r * RN(1/3)) is the correctly rounded quotient when the
// reciprocal is correctly rounded and q0 is within one ulp (Markstein's theorem; 3 has no all-ones significand).
__device__ __forceinline__ double div3(double x) {
    const double q = x * (1.0 / 3.0);
    return fma(fma(-3.0, q, x), 1.0 / 3.0, q);
}
__device__ __forceinline__ float div3(float x) {
    const float q = x * (1.0f / 3.0f);
    return fmaf(fmaf(-3.0f, q, x), 1.0f / 3.0f, q);
}

// Static term signature of the multi-term instantiations: TK packs the kind of term k in bits [3k, 3k+3)
// (SK_* below; TK < 0: kinds are runtime data), COEFK packs its coefficient kind in bits [2k, 2k+2) (COEFK < 0: runtime).
// static base modes of a launch (template parameter SB; -1 = runtime): BASE_* of lsm_dev.cuh plus the presence of out2
enum : int { SB_IN = 0, SB_S2 = 1, SB_S3 = 2, SB_IN_OUT2 = 3, SB_P0 = 4 };
enum : int { SK_ADV_WENO = 0, SK_ADV_UPWIND = 1, SK_NORMAL = 2, SK_CURV = 3, SK_EIK = 4 };
__host__ __device__ constexpr int sig_kind(int TK, int k) { return TK < 0 || k < 0 ? -1 : ((TK >> (3 * k)) & 7); }
__host__ __device__ constexpr int sig_coef(int COEFK, int k) { return COEFK < 0 || k < 0 ? -1 : ((COEFK >> (2 * k)) & 3); }
// first staged aux tile of term k when every FIELD coefficient before it is staged (the launcher checks)
__host__ __device__ constexpr int sig_first(int TK, int COEFK, int k, int ndim) {
    int f = 0;
    for (int j = 0; j < k; ++j)
        if (sig_coef(COEFK, j) == COEF_FIELD) f += (sig_kind(TK, j) == SK_ADV_WENO || sig_kind(TK, j) == SK_ADV_UPWIND) ? ndim : 1;
    return f;
}

// The static base mode of a launch whose kernel expects phi^n / corr (when staged) in aux slot p0_slot, or -1 when none fits.
template <class T>
int static_base(const StageParams<T>& P, const AuxList& A, int p0_slot) {
    if (A.p0 >= 0 && A.p0 != p0_slot) return -1;
    if (P.base == BASE_IN && !P.p0) return P.out2 ? SB_IN_OUT2 : SB_IN;
    if (!P.p0 || P.out2) return -1;
    if (P.base == BASE_RK3_S2) return SB_S2;
    if (P.base == BASE_RK3_S3) return SB_S3;
    if (P.base == BASE_P0) return SB_P0;
    return -1;
}
// launch(std::integral_constant<int, SB>{}) for a static base mode sb >= 0; cudaErrorNotSupported for sb = -1
template <class F>
cudaError_t with_static_base(int sb, F launch) {
    switch (sb) {
        case SB_IN:      return launch(std::integral_constant<int, SB_IN>{});
        case SB_S2:      return launch(std::integral_constant<int, SB_S2>{});
        case SB_S3:      return launch(std::integral_constant<int, SB_S3>{});
        case SB_IN_OUT2: return launch(std::integral_constant<int, SB_IN_OUT2>{});
        case SB_P0:      return launch(std::integral_constant<int, SB_P0>{});
        default:         return cudaErrorNotSupported;
    }
}

// levelsetterms.jl:184-187
// Same-sign test on the sign bits (LOP3 + ISETP instead of DMUL + DSETP): identical to `x*y > 0` except where the product
// underflows (|x||y| < 5e-324), where the reference returns 0 and this returns min(|x|,|y|) < 1e-150 — far below any tolerance.
// x == 0 or y == 0 selects the zero operand, as the reference's 0 result.
__device__ __forceinline__ double minmod(double x, double y) {
    const double m = fabs(x) <= fabs(y) ? x : y;
    return (__double2hiint(x) ^ __double2hiint(y)) < 0 ? 0.0 : m;
}



// Ghost index -> stored index for the boundary conditions that are pure index maps with weight 1
// (boundaryconditions.jl:107-119 periodic wrap, :134-144 with P = 0 i.e. NeumannBC, :146-153 symmetry).
// Applied independently per dimension this equals the reference's dimension-by-dimension recursion
// (meshfield.jl:248-260).  BC_HALO sides keep the index (stored ghost plane).  Needs n >= 4.
__device__ __forceinline__ int remap_index(int i, int n, int kind_lo, int kind_hi) {
    if (i < 0) {
        if (kind_lo == BC_PERIODIC) return i + n - 1;
        if (kind_lo == BC_EXTRAP) return 0;
        if (kind_lo == BC_SYMMETRY) return -i;
        return i;
    }
    if (i >= n) {
        if (kind_hi == BC_PERIODIC) return i - n + 1;
        if (kind_hi == BC_EXTRAP) return n - 1;
        if (kind_hi == BC_SYMMETRY) return 2 * (n - 1) - i;
        return i;
    }
    return i;
}

// cuTensorMapEncodeTiled through the runtime's driver-entry-point lookup (liblsm_b200 does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    // looked up once per translation unit (thread-safe static initialisation: contexts of one process may launch from several threads)
    static const EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            return reinterpret_cast<EncodeTiledFn>(p);
        return static_cast<EncodeTiledFn>(nullptr);
    }();
    return fn;
}

template <class T>
bool encode_map3(CUtensorMap* m, const void* base, long n0, long n1, long nplanes, int b0, int b1) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)n0, (cuuint64_t)n1, (cuuint64_t)nplanes};
    const cuuint64_t strides[2] = {(cuuint64_t)n0 * sizeof(T), (cuuint64_t)n0 * n1 * sizeof(T)};
    const cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, 1u};
    const cuuint32_t es[3] = {1u, 1u, 1u};
    return enc(m, sizeof(T) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims,
               strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Tensor maps are a pure function of (base, shape, box, dtype): encode each distinct one once per process and reuse it on every
// later launch (an RK loop cycles through a handful of buffers).  Thread-safe; bounded, evicting round-robin.
struct MapKey { const void* base; long n0, n1, np; int b0, b1, es; };
template <class T>
bool cached_map3(CUtensorMap* out, const void* base, long n0, long n1, long nplanes, int b0, int b1) {
    struct Entry { MapKey k; CUtensorMap m; };
    constexpr int CAP = 64;
    static Entry* tab = nullptr;
    static int used = 0, next = 0;
    static std::mutex mu;
    const MapKey k{base, n0, n1, nplanes, b0, b1, (int)sizeof(T)};
    std::lock_guard<std::mutex> lock(mu);
    if (!tab) tab = static_cast<Entry*>(aligned_alloc(64, sizeof(Entry) * CAP));
    if (!tab) return false;
    for (int i = 0; i < used; ++i) {
        const MapKey& q = tab[i].k;
        if (q.base == k.base && q.n0 == k.n0 && q.n1 == k.n1 && q.np == k.np && q.b0 == k.b0 && q.b1 == k.b1 && q.es == k.es) { *out = tab[i].m; return true; }
    }
    CUtensorMap m;
    if (!encode_map3<T>(&m, base, n0, n1, nplanes, b0, b1)) return false;
    const int slot = used < CAP ? used++ : (next = (next + 1) % CAP);
    tab[slot].k = k; tab[slot].m = m;
    *out = m;
    return true;
}

// environment switches are read once per process
inline bool env_flag(const char* name) { const char* v = getenv(name); return v && *v && *v != '0'; }
inline bool tma_disabled() { static const bool v = env_flag("LSM_B200_NO_TMA"); return v; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: remember the opt-in per (kernel instantiation, device)
template <class K>
cudaError_t ensure_dyn_smem(K kern, size_t smem, size_t (&granted)[16]) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const int slot = dev & 15;
    if (dev < 16 && smem <= granted[slot]) return cudaSuccess;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && dev < 16) granted[slot] = smem;
    return e;
}

}  // namespace
}  // namespace lsm
