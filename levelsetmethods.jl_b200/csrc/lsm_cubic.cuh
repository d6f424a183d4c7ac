// lsm_cubic.cuh — the tensor-product cubic interpolant of a scalar field (include/lsm_b200.h, "cubic interpolant"): value,
// gradient and Hessian at a point, in the contract's operation order.  Included by -fmad=false translation units only
// (lsm_redistance.cu), so that tests/cubic_ref.py restates it bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include "lsm_kernels.h"

namespace lsm {
namespace cubic {

// Lagrange weights on the nodes 0..3 at xi (a = xi - 1, b = xi - 2, c = xi - 3): w[0][k] = L_k, w[1][k] = L_k', w[2][k] = L_k''
__device__ __forceinline__ void weights(double xi, double (*w)[4], int order) {
    const double a = xi - 1.0, b = xi - 2.0, c = xi - 3.0;
    w[0][0] = ((a * b) * c) / (-6.0);
    w[0][1] = ((xi * b) * c) / 2.0;
    w[0][2] = ((xi * a) * c) / (-2.0);
    w[0][3] = ((xi * a) * b) / 6.0;
    if (order < 1) return;
    w[1][0] = ((a * b + a * c) + b * c) / (-6.0);
    w[1][1] = ((xi * b + xi * c) + b * c) / 2.0;
    w[1][2] = ((xi * a + xi * c) + a * c) / (-2.0);
    w[1][3] = ((xi * a + xi * b) + a * b) / 6.0;
    if (order < 2) return;
    w[2][0] = ((a + b) + c) / (-3.0);
    w[2][1] = (xi + b) + c;
    w[2][2] = -((xi + a) + c);
    w[2][3] = ((xi + a) + b) / 3.0;
}

__device__ __forceinline__ double sum4(const double* w, const double* f) {
    return ((w[0] * f[0] + w[1] * f[1]) + w[2] * f[2]) + w[3] * f[3];
}

// The interpolant of phi (the box of A: A.m nodes, A.lc, A.h, strides A.s1 / A.s2) at y.  ORDER 0: P; 1: P and g = grad P;
// 2: P, g and H (H[d][e] = H[e][d], computed once for d <= e).  Returns false, with every requested output NaN, when y is
// outside the box.  Derivative weights go on the differentiated axes; the contraction runs over axis 1, then 2, then 3.
template <class T, int N, int ORDER>
__device__ __forceinline__ bool eval(const IfaceArgs& A, const double* y, double& P, double* g, double (*H)[3]) {
    const T* phi = static_cast<const T*>(A.phi);
    double w[3][3][4];
    long long base = 0;
    bool inside = true;
    for (int d = 0; d < N; ++d) {
        const double u = (y[d] - A.lc[d]) / A.h[d];
        inside = inside && u >= 0.0 && u <= double(A.m[d] - 1);
        if (!inside) break;
        int c = (int)floor(u);
        c = c < A.m[d] - 2 ? c : A.m[d] - 2;
        int s = c - 1 > 0 ? c - 1 : 0;
        s = s < A.m[d] - 4 ? s : A.m[d] - 4;
        weights(u - double(s), w[d], ORDER);
        base += (long long)s * (d == 0 ? 1ll : d == 1 ? A.s1 : A.s2);
    }
    if (!inside) {
        P = CUDART_NAN;
        if constexpr (ORDER >= 1) for (int d = 0; d < N; ++d) g[d] = CUDART_NAN;
        if constexpr (ORDER >= 2) for (int d = 0; d < N; ++d) for (int e = 0; e < N; ++e) H[d][e] = CUDART_NAN;
        return false;
    }
    if constexpr (N == 1) {
        double f[4];
        for (int k = 0; k < 4; ++k) f[k] = double(phi[base + k]);
        P = sum4(w[0][0], f);
        if constexpr (ORDER >= 1) g[0] = sum4(w[0][1], f) / A.h[0];
        if constexpr (ORDER >= 2) H[0][0] = (sum4(w[0][2], f) / A.h[0]) / A.h[0];
    } else {
        // r2[q][k3]: the axis-1 and axis-2 contractions with derivative orders (a1, a2) = Q[q], for each plane k3 of the stencil
        constexpr int NQ = ORDER == 0 ? 1 : ORDER == 1 ? 3 : 6;
        constexpr int QA[6] = {0, 1, 0, 2, 1, 0}, QB[6] = {0, 0, 1, 0, 1, 2};
        constexpr int K3 = N == 3 ? 4 : 1;
        double r2[NQ][K3];
#pragma unroll
        for (int k3 = 0; k3 < K3; ++k3) {
            double r1[ORDER + 1][4];
#pragma unroll
            for (int k2 = 0; k2 < 4; ++k2) {
                double f[4];
                const long long row = base + k2 * A.s1 + k3 * A.s2;
                for (int k = 0; k < 4; ++k) f[k] = double(phi[row + k]);
                for (int a = 0; a <= ORDER; ++a) r1[a][k2] = sum4(w[0][a], f);
            }
#pragma unroll
            for (int q = 0; q < NQ; ++q) r2[q][k3] = sum4(w[1][QB[q]], r1[QA[q]]);
        }
        if constexpr (N == 2) {
            P = r2[0][0];
            if constexpr (ORDER >= 1) { g[0] = r2[1][0] / A.h[0]; g[1] = r2[2][0] / A.h[1]; }
            if constexpr (ORDER >= 2) {
                H[0][0] = (r2[3][0] / A.h[0]) / A.h[0];
                H[0][1] = H[1][0] = (r2[4][0] / A.h[0]) / A.h[1];
                H[1][1] = (r2[5][0] / A.h[1]) / A.h[1];
            }
        } else {
            P = sum4(w[2][0], r2[0]);
            if constexpr (ORDER >= 1) {
                g[0] = sum4(w[2][0], r2[1]) / A.h[0];
                g[1] = sum4(w[2][0], r2[2]) / A.h[1];
                g[2] = sum4(w[2][1], r2[0]) / A.h[2];
            }
            if constexpr (ORDER >= 2) {
                H[0][0] = (sum4(w[2][0], r2[3]) / A.h[0]) / A.h[0];
                H[0][1] = H[1][0] = (sum4(w[2][0], r2[4]) / A.h[0]) / A.h[1];
                H[1][1] = (sum4(w[2][0], r2[5]) / A.h[1]) / A.h[1];
                H[0][2] = H[2][0] = (sum4(w[2][1], r2[1]) / A.h[0]) / A.h[2];
                H[1][2] = H[2][1] = (sum4(w[2][1], r2[2]) / A.h[1]) / A.h[2];
                H[2][2] = (sum4(w[2][2], r2[0]) / A.h[2]) / A.h[2];
            }
        }
    }
    return true;
}

}  // namespace cubic
}  // namespace lsm
