// lsm_pair_common.cuh — device helpers shared by the x-pair kernels (lsm_pair3d.cu, lsm_pair2d.cu): pair loads from shared memory,
// the WENO5 evaluation on first differences and the two-node evaluation with the upwind side resolved by branch.
#pragma once
#include "lsm_tile_util.cuh"

namespace lsm {
namespace {

template <class T> struct Vec2;
template <> struct Vec2<double> { using type = double2; };
template <> struct Vec2<float> { using type = float2; };

// 128-bit (Float64 pair) / 64-bit (Float32 pair) shared-memory load from a 32-bit shared-window address.  Explicit addresses keep
// the per-thread base in ONE register for the whole plane loop (the compiler otherwise re-derives element offsets -> byte
// addresses in every evaluation block: ~19 integer instructions per node, measured with tools/ncu_opmix.py).
__device__ __forceinline__ double2 lds_pair(unsigned addr, double) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds_pair(unsigned addr, float) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}

// The WENO constants as the x-pair kernels hold them in registers.  Those that do not fit an instruction immediate are made
// opaque to ptxas (threadIdx.z is always 0, which the compiler cannot know): as plain kernel parameters it re-materialises them
// from the constant bank with ~12 moves in every one of the six evaluation blocks of a plane (36 issue slots per node, measured
// in SASS).  The default form (!XMAX) evaluates the smoothness indicators scaled by 3/16 (weno_core_de), so its eps constants
// are scaled with them; it reads neither c133 nor c56, and the compiler drops their registers.
template <bool XMAX>
__device__ __forceinline__ WenoK weno_regs(const WenoK& K) {
    const double zopq = __longlong_as_double((long long)threadIdx.z);
    const double s = XMAX ? 1.0 : 0.1875;
    WenoK R;
    R.c133 = K.c133 + zopq; R.c56 = K.c56 + zopq; R.cm13 = K.cm13 + zopq; R.e6 = K.e6 * s + zopq; R.fl = K.fl * s + zopq; R.pad = 0.0;
    return R;
}

// The reference's _weno5(v1..v5) (derivatives.jl:61-81) on UNDIVIDED first differences d0..d4 and their differences e1..e4,
// restructured like weno5_up of lsm_tile_util.cuh (second differences, one reciprocal); returns h * weno.  The function is
// odd: core(-v5..-v1 reversed) == -core(...) bit for bit, which is what makes the physical-order evaluation below identical to
// the upwind-ordered one of lsm_tiled.cu.  K comes from weno_regs<XMAX>.
// XMAX: exact max|d| for eps and the operations of weno5_up (bit-identical to lsm_tiled.cu).  Otherwise the 20-bit maximum
// (absmax5_hi) and the smoothness indicators as completed squares: the weights depend only on ratios of the b_k, so
//   (3/16) b1 = (e1 - 11/8 e2)^2 + 39/64 e2^2 + eps',  (3/16) b2 = (e2 - 5/8 e3)^2 + 39/64 e3^2 + eps',
//   (3/16) b3 = (e4 - 11/8 e3)^2 + 39/64 e3^2 + eps',  eps' = (3/16) eps
// give the same result with dyadic coefficients (instruction immediates) in 10 FP64 instructions instead of 15; every term is
// non-negative, so nothing cancels.  G1 = 5/6 e2 - 1/3 e1 = 3/8 e2 - 1/3 (e1 - 11/8 e2) reuses the first square's base.
template <bool XMAX>
__device__ __forceinline__ double weno_core_de(const WenoK& K, double d0, double d1, double d2, double d3, double d4,
                                               double e1, double e2, double e3, double e4) {
    const double m = XMAX ? absmax5(d0, d1, d2, d3, d4) : absmax5_hi(d0, d1, d2, d3, d4);
    const double eps = fma(K.e6, m * m, K.fl);
    double b1, b2, b3, X1 = 0.0;
    if constexpr (XMAX) {
        const double c133 = K.c133;
        const double t1a = e2 - e1, t1b = e3 - e2, t1c = e4 - e3;
        const double t2a = fma(3.0, e2, -e1), t2b = e2 + e3, t2c = fma(-3.0, e3, e4);
        b1 = fma(t2a, t2a, fma(c133, t1a * t1a, eps));
        b2 = fma(t2b, t2b, fma(c133, t1b * t1b, eps));
        b3 = fma(t2c, t2c, fma(c133, t1c * t1c, eps));
    } else {
        X1 = fma(-1.375, e2, e1);
        const double X2 = fma(-0.625, e3, e2), X3 = fma(-1.375, e3, e4);
        const double F2 = fma(0.609375, e2 * e2, eps), F3 = fma(0.609375, e3 * e3, eps);
        b1 = fma(X1, X1, F2);
        b2 = fma(X2, X2, F3);
        b3 = fma(X3, X3, F3);
    }
    const double p12 = b1 * b2, p13 = b1 * b3, p23 = b2 * b3;
    const double w1 = p23 * p23, w2 = p13 * p13, w3 = p12 * p12;
    const double den = fma(3.0, w3, fma(6.0, w2, w1));
    const double G1 = XMAX ? fma(K.c56, e2, K.cm13 * e1) : fma(0.375, e2, K.cm13 * X1);
    const double G2 = fma(2.0, e3, e2);
    const double G3 = fma(2.0, e3, -0.5 * e4);
    const double num = fma(w3, G3, fma(w2, G2, w1 * G1));
    return fma(num, fast_rcp<1>(den), d2);
}

template <bool XMAX>
__device__ __forceinline__ double weno_core(const WenoK& K, double d0, double d1, double d2, double d3, double d4) {
    return weno_core_de<XMAX>(K, d0, d1, d2, d3, d4, d1 - d0, d2 - d1, d3 - d2, d4 - d3);
}

// Float32 fields: all-FP32 evaluation with the differences normalised by 1/max|d| (see weno5_up<float>)
template <bool XMAX>
__device__ __forceinline__ double weno_core(const WenoK&, float d0, float d1, float d2, float d3, float d4) {
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

// The Float32 evaluation for TWO nodes at once with Blackwell's packed FP32 instructions (FFMA2 / FADD2 / FMUL2: one issue slot
// for both nodes; .x = node A, .y = node B).  Lane-wise IEEE, same operation order as the scalar version above, so the results
// are bit-identical to it; max|d| and the two reciprocals stay scalar (no packed FMNMX / MUFU).
#ifndef LSM_NO_F32X2
__device__ __forceinline__ float2 f2(float x, float y) { return make_float2(x, y); }
__device__ __forceinline__ float2 f2(float x) { return make_float2(x, x); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ void weno_core2(float2 d0, float2 d1, float2 d2, float2 d3, float2 d4, double& WA, double& WB) {
    const float2 e1 = sub2(d1, d0), e2 = sub2(d2, d1), e3 = sub2(d3, d2), e4 = sub2(d4, d3);
    const float ma = fmaxf(fmaxf(fmaxf(fabsf(d0.x), fabsf(d1.x)), fmaxf(fabsf(d2.x), fabsf(d3.x))), fabsf(d4.x));
    const float mb = fmaxf(fmaxf(fmaxf(fabsf(d0.y), fabsf(d1.y)), fmaxf(fabsf(d2.y), fabsf(d3.y))), fabsf(d4.y));
    const float2 im = f2(ma > 0.f ? __frcp_rn(ma) : 0.f, mb > 0.f ? __frcp_rn(mb) : 0.f);
    const float2 s1 = __fmul2_rn(e1, im), s2 = __fmul2_rn(e2, im), s3 = __fmul2_rn(e3, im), s4 = __fmul2_rn(e4, im);
    const float2 c133 = f2(13.0f / 3.0f), epsf = f2(4.0e-6f);
    const float2 t1a = sub2(s2, s1), t1b = sub2(s3, s2), t1c = sub2(s4, s3);
    const float2 t2a = __ffma2_rn(f2(3.0f), s2, f2(-s1.x, -s1.y)), t2b = __fadd2_rn(s2, s3), t2c = __ffma2_rn(f2(-3.0f), s3, s4);
    const float2 b1 = __ffma2_rn(t2a, t2a, __ffma2_rn(c133, __fmul2_rn(t1a, t1a), epsf));
    const float2 b2 = __ffma2_rn(t2b, t2b, __ffma2_rn(c133, __fmul2_rn(t1b, t1b), epsf));
    const float2 b3 = __ffma2_rn(t2c, t2c, __ffma2_rn(c133, __fmul2_rn(t1c, t1c), epsf));
    const float2 p12 = __fmul2_rn(b1, b2), p13 = __fmul2_rn(b1, b3), p23 = __fmul2_rn(b2, b3);
    const float2 w1 = __fmul2_rn(p23, p23), w2 = __fmul2_rn(p13, p13), w3 = __fmul2_rn(p12, p12);
    const float2 den = __ffma2_rn(f2(3.0f), w3, __ffma2_rn(f2(6.0f), w2, w1));
    const float2 G1 = __ffma2_rn(f2(5.0f / 6.0f), e2, __fmul2_rn(f2(-1.0f / 3.0f), e1));
    const float2 G2 = __ffma2_rn(f2(2.0f), e3, e2);
    const float2 G3 = __ffma2_rn(f2(2.0f), e3, __fmul2_rn(f2(-0.5f), e4));
    const float2 num = __ffma2_rn(w3, G3, __ffma2_rn(w2, G2, __fmul2_rn(w1, G1)));
    const float2 r = __ffma2_rn(num, f2(__frcp_rn(den.x), __frcp_rn(den.y)), d2);
    WA = double(r.x); WB = double(r.y);
}
#endif

// h * (the upwind-biased WENO5 derivative) at two nodes A and B along one dimension.  a[k] / b[k] is phi at offset k - 3 from
// node A / B; xa / xb carries sign(u * g) of the node in bit 31 (set: plus-biased stencil, derivatives.jl:109-121; clear:
// minus-biased, :89-101).  When B is A's neighbour along the dimension the caller passes b[k] = a[k + 1] and the common
// differences are shared by the compiler's value numbering.
template <class T, bool XMAX>
__device__ __forceinline__ void pair_eval(const WenoK& K, const T (&a)[7], const T (&b)[7], int xa, int xb, double& WA, double& WB) {
#ifndef LSM_NO_F32X2
    if constexpr (sizeof(T) == 4) {
        // Float32: both nodes in one packed evaluation (uniform directions); differences lane-wise, shared ones by value numbering
        if ((xa | xb) >= 0) {
            weno_core2(f2(a[1] - a[0], b[1] - b[0]), f2(a[2] - a[1], b[2] - b[1]), f2(a[3] - a[2], b[3] - b[2]), f2(a[4] - a[3], b[4] - b[3]),
                       f2(a[5] - a[4], b[5] - b[4]), WA, WB);
            return;
        }
        if ((xa & xb) < 0) {
            weno_core2(f2(a[6] - a[5], b[6] - b[5]), f2(a[5] - a[4], b[5] - b[4]), f2(a[4] - a[3], b[4] - b[3]), f2(a[3] - a[2], b[3] - b[2]),
                       f2(a[2] - a[1], b[2] - b[1]), WA, WB);
            return;
        }
    }
#endif
    if ((xa | xb) >= 0) {                 // both minus-biased: D-(I-2 .. I+2) = first differences -3 .. 1
        WA = weno_core<XMAX>(K, T(a[1] - a[0]), T(a[2] - a[1]), T(a[3] - a[2]), T(a[4] - a[3]), T(a[5] - a[4]));
        WB = weno_core<XMAX>(K, T(b[1] - b[0]), T(b[2] - b[1]), T(b[3] - b[2]), T(b[4] - b[3]), T(b[5] - b[4]));
    } else if ((xa & xb) < 0) {           // both plus-biased: D+(I+2), D+(I+1), D+(I), D+(I-1), D+(I-2)
        WA = weno_core<XMAX>(K, T(a[6] - a[5]), T(a[5] - a[4]), T(a[4] - a[3]), T(a[3] - a[2]), T(a[2] - a[1]));
        WB = weno_core<XMAX>(K, T(b[6] - b[5]), T(b[5] - b[4]), T(b[4] - b[3]), T(b[3] - b[2]), T(b[2] - b[1]));
    } else {                              // a sign change inside the pair: upwind-ordered samples per node (odd symmetry of the evaluation)
        const bool ma = xa >= 0, mb = xb >= 0;
        T qa[6], qb[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) { qa[k] = ma ? a[k] : a[6 - k]; qb[k] = mb ? b[k] : b[6 - k]; }
        const double wa = weno_core<XMAX>(K, T(qa[1] - qa[0]), T(qa[2] - qa[1]), T(qa[3] - qa[2]), T(qa[4] - qa[3]), T(qa[5] - qa[4]));
        const double wb = weno_core<XMAX>(K, T(qb[1] - qb[0]), T(qb[2] - qb[1]), T(qb[3] - qb[2]), T(qb[4] - qb[3]), T(qb[5] - qb[4]));
        WA = ma ? wa : -wa;
        WB = mb ? wb : -wb;
    }
}


}  // namespace
}  // namespace lsm
