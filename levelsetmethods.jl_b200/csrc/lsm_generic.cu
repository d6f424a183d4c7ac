// lsm_generic.cu — the STRICT generic kernels (compiled with -fmad=false).
//
// One thread per node, any N in {1,2,3}, any term set, any boundary condition.  Arithmetic is
// written in the reference's own operation order (true divisions by h, left-to-right sums, one
// rounding to the storage type per term), so results agree with the CPU oracle to the last
// bit wherever IEEE arithmetic is all that is involved.  This is the correctness anchor on the
// device and the path for everything the tiled kernels (lsm_tiled.cu) do not cover.
//
// Reference functions restated here (paths relative to the reference repo):
//   meshfield.jl:213-260 getindex/_getindexbc, boundaryconditions.jl:90-153 bc_stencil,
//   derivatives.jl:28-175, levelsetops.jl:197-244 curvature, levelsetterms.jl:73-265 terms,
//   timestepping.jl:128-202 stage combinations.
#include <algorithm>
#include "lsm_dev.cuh"
#include "lsm_bc.cuh"
#include "lsm_kernels.h"

namespace lsm {

template <class T> struct EpsV;
template <> struct EpsV<float>  { static constexpr double v = 1.1920928955078125e-07; };
template <> struct EpsV<double> { static constexpr double v = 2.220446049250313e-16; };

__device__ __forceinline__ double positive(double x) { return x > 0.0 ? x : 0.0; }
__device__ __forceinline__ double negative(double x) { return x < 0.0 ? x : 0.0; }
// levelsetterms.jl:184-187
__device__ __forceinline__ double limiter(double x, double y) {
    if (!(x * y > 0.0)) return 0.0;
    return fabs(x) <= fabs(y) ? x : y;
}
// Julia max(): NaN-propagating
__device__ __forceinline__ double jl_max(double a, double b) {
    return (isnan(a) || isnan(b)) ? __longlong_as_double(0x7FF8000000000000LL) : (b > a ? b : a);
}

template <int N, class T>
struct Reader {
    const View<T>& v;
    const T* c;          // centre node
    int i0, i1, i2;
    bool interior;       // every stencil read (|offset| <= 3 per dim) is a stored element
    __device__ __forceinline__ long stride(int d) const { return d == 0 ? 1L : (d == 1 ? v.s1 : v.s2); }
    __device__ __forceinline__ T at(int d, int o) const {
        if (interior) return c[(long)o * stride(d)];
        return getindex_slow<N, T>(v, i0 + (d == 0 ? o : 0), i1 + (d == 1 ? o : 0), i2 + (d == 2 ? o : 0));
    }
    __device__ __forceinline__ T at2(int d1, int o1, int d2, int o2) const {
        if (interior) return c[(long)o1 * stride(d1) + (long)o2 * stride(d2)];
        return getindex_slow<N, T>(v, i0 + (d1 == 0 ? o1 : 0) + (d2 == 0 ? o2 : 0),
                                   i1 + (d1 == 1 ? o1 : 0) + (d2 == 1 ? o2 : 0),
                                   i2 + (d1 == 2 ? o1 : 0) + (d2 == 2 ? o2 : 0));
    }
};

// derivatives.jl:28-57 evaluated at I + s*e_d
template <int N, class T> __device__ __forceinline__ double Dm(const Reader<N, T>& r, int d, int s, double h) {
    T df = r.at(d, s) - r.at(d, s - 1);
    return double(df) / h;
}
template <int N, class T> __device__ __forceinline__ double Dp(const Reader<N, T>& r, int d, int s, double h) {
    T df = r.at(d, s + 1) - r.at(d, s);
    return double(df) / h;
}
template <int N, class T> __device__ __forceinline__ double D0(const Reader<N, T>& r, int d, double h) {
    T df = r.at(d, 1) - r.at(d, -1);
    return double(df) / (2 * h);
}
// derivatives.jl:129-175
template <int N, class T> __device__ __forceinline__ double D20(const Reader<N, T>& r, int d, double h) {
    T df = r.at(d, 1) - T(2) * r.at(d, 0) + r.at(d, -1);
    return double(df) / (h * h);
}
template <int N, class T> __device__ __forceinline__ double D2pp(const Reader<N, T>& r, int d, double h) {
    T df = r.at(d, 0) - T(2) * r.at(d, 1) + r.at(d, 2);
    return double(df) / (h * h);
}
template <int N, class T> __device__ __forceinline__ double D2mm(const Reader<N, T>& r, int d, double h) {
    T df = r.at(d, -2) - T(2) * r.at(d, -1) + r.at(d, 0);
    return double(df) / (h * h);
}
template <int N, class T>
__device__ __forceinline__ double D2mixed(const Reader<N, T>& r, int d1, int d2, double h1, double h2) {
    T a = r.at2(d1, 1, d2, 1) - r.at2(d1, 1, d2, -1);
    T b = r.at2(d1, -1, d2, 1) - r.at2(d1, -1, d2, -1);
    return (double(a) / (2 * h2) - double(b) / (2 * h2)) / (2 * h1);
}

// derivatives.jl:61-81
__device__ __forceinline__ double weno5_strict(double v1, double v2, double v3, double v4, double v5) {
    const double c13 = 1.0 / 3.0, c76 = 7.0 / 6.0, c116 = 11.0 / 6.0, c16 = 1.0 / 6.0, c56 = 5.0 / 6.0;
    const double c1312 = 13.0 / 12.0, c14 = 1.0 / 4.0;
    double d1 = c13 * v1 - c76 * v2 + c116 * v3;
    double d2 = -c16 * v2 + c56 * v3 + c13 * v4;
    double d3 = c13 * v3 + c56 * v4 - c16 * v5;
    double a, b;
    a = v1 - 2 * v2 + v3;  b = v1 - 4 * v2 + 3 * v3;
    double S1 = c1312 * (a * a) + c14 * (b * b);
    a = v2 - 2 * v3 + v4;  b = v2 - v4;
    double S2 = c1312 * (a * a) + c14 * (b * b);
    a = v3 - 2 * v4 + v5;  b = 3 * v3 - 4 * v4 + v5;
    double S3 = c1312 * (a * a) + c14 * (b * b);
    double m = jl_max(jl_max(jl_max(jl_max(v1 * v1, v2 * v2), v3 * v3), v4 * v4), v5 * v5);
    double eps = 1.0e-6 * m + 1.0e-99;
    double t;
    t = S1 + eps; double a1 = 0.1 / (t * t);
    t = S2 + eps; double a2 = 0.6 / (t * t);
    t = S3 + eps; double a3 = 0.3 / (t * t);
    double w1 = a1 / (a1 + a2 + a3);
    double w2 = a2 / (a1 + a2 + a3);
    double w3 = a3 / (a1 + a2 + a3);
    return w1 * d1 + w2 * d2 + w3 * d3;
}

// levelsetterms.jl:156-170 / 252-265 : second-order ENO one-sided pair along dim d
template <int N, class T>
__device__ __forceinline__ void eno2_pair(const Reader<N, T>& r, int d, double h, double& neg, double& pos) {
    const double d20 = D20(r, d, h);
    neg = Dm(r, d, 0, h) + (0.5 * h) * limiter(D2mm(r, d, h), d20);
    pos = Dp(r, d, 0, h) - (0.5 * h) * limiter(D2pp(r, d, h), d20);
}

// levelsetops.jl:197-205
template <int N, class T>
__device__ inline double curvature(const Reader<N, T>& r, const double* h) {
    double g[3] = {0, 0, 0};
#pragma unroll
    for (int d = 0; d < N; ++d) g[d] = D0(r, d, h[d]);
    double nrmsq = 0.0;
#pragma unroll
    for (int d = 0; d < N; ++d) nrmsq += g[d] * g[d];
    if (nrmsq < EpsV<T>::v) return 0.0;
    double H[3][3];
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
        for (int i = 0; i <= j; ++i) {
            H[i][j] = (i == j) ? D20(r, i, h[i]) : D2mixed(r, i, j, h[i], h[j]);
            H[j][i] = H[i][j];
        }
    double tr = H[0][0];
#pragma unroll
    for (int d = 1; d < N; ++d) tr += H[d][d];
    double quad = 0.0;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        double w = g[0] * H[0][j];
#pragma unroll
        for (int i = 1; i < N; ++i) w += g[i] * H[i][j];
        quad = (j == 0) ? w * g[j] : quad + w * g[j];
    }
    return (tr * nrmsq - quad) / pow(nrmsq, 1.5);
}

template <int N, class T>
__device__ inline double godunov_norm(const Reader<N, T>& r, const double* h, bool vpos) {
    double sa = 0, sb = 0;
#pragma unroll
    for (int d = 0; d < N; ++d) {
        double A, B;
        eno2_pair(r, d, h[d], A, B);
        double a, b;
        if (vpos) { a = positive(A) * positive(A); b = negative(B) * negative(B); }
        else      { a = negative(A) * negative(A); b = positive(B) * positive(B); }
        sa = (d == 0) ? a : sa + a;
        sb = (d == 0) ? b : sb + b;
    }
    return sqrt(sa + sb);
}

template <int N, class T>
__device__ inline double compute_term(const Reader<N, T>& r, const TermDev& t, long node, const double* h, double dxmin, int skip_zero_u = 0) {
    switch (t.kind) {
        case TERM_ADVECTION: {   // levelsetterms.jl:73-82
            double s = 0.0;
#pragma unroll
            for (int d = 0; d < N; ++d) {
                const double v = coef_comp<T>(t, node, d, r.i0, r.i1, r.i2, N);
                double der;
                if (t.scheme == SCHEME_WENO5) {
                    if (v > 0) der = weno5_strict(Dm(r, d, -2, h[d]), Dm(r, d, -1, h[d]), Dm(r, d, 0, h[d]), Dm(r, d, 1, h[d]), Dm(r, d, 2, h[d]));
                    else       der = weno5_strict(Dp(r, d, 2, h[d]), Dp(r, d, 1, h[d]), Dp(r, d, 0, h[d]), Dp(r, d, -1, h[d]), Dp(r, d, -2, h[d]));
                } else {
                    der = (v > 0) ? Dm(r, d, 0, h[d]) : Dp(r, d, 0, h[d]);
                    if (skip_zero_u && v == 0.0) der = 0.0;
                }
                const double p = v * der;
                s = (d == 0) ? p : s + p;
            }
            return s;
        }
        case TERM_NORMAL: {      // levelsetterms.jl:156-170
            const double v = coef_comp<T>(t, node, 0, r.i0, r.i1, r.i2, N);
            double gp = 0, gm = 0;
#pragma unroll
            for (int d = 0; d < N; ++d) {
                double neg, pos;
                eno2_pair(r, d, h[d], neg, pos);
                const double a = positive(neg) * positive(neg) + negative(pos) * negative(pos);
                const double b = negative(neg) * negative(neg) + positive(pos) * positive(pos);
                gp = (d == 0) ? a : gp + a;
                gm = (d == 0) ? b : gm + b;
            }
            return positive(v) * sqrt(gp) + negative(v) * sqrt(gm);
        }
        case TERM_CURVATURE: {   // levelsetterms.jl:111-121
            const double kappa = curvature(r, h);
            const double b = coef_comp<T>(t, node, 0, r.i0, r.i1, r.i2, N);
            double p2 = 0;
#pragma unroll
            for (int d = 0; d < N; ++d) {
                const double q = D0(r, d, h[d]);
                p2 = (d == 0) ? q * q : p2 + q * q;
            }
            return b * kappa * sqrt(p2);
        }
        default: {               // levelsetterms.jl:234-248
            if (t.coef_kind == COEF_NONE) {
                const T p = r.at(0, 0);
                const double nrm = godunov_norm(r, h, p > T(0));
                const double den = sqrt(double(T(p * p)) + (nrm * nrm) * (dxmin * dxmin));
                const double S = (den == 0.0) ? 0.0 : double(p) / den;
                return S * (nrm - 1);
            }
            const double S0 = coef_comp<T>(t, node, 0, r.i0, r.i1, r.i2, N);
            const double nrm = godunov_norm(r, h, S0 > 0);
            return S0 * (nrm - 1);
        }
    }
}

template <int N, class T>
__global__ void __launch_bounds__(256) stage_generic_kernel(const __grid_constant__ StageParams<T> P) {
    const View<T>& v = P.in;
    const int n0 = v.n[0], n1 = v.n[1];
    int i0, i1 = 0, i2 = 0;
    if (N > 1 && P.bricks) {
        // narrow band: the blocks of list entry e cover the nodes of brick P.bricks[1 + e] (x fastest); entries past the count exit
        constexpr int BN = BRICK_X * BRICK_Y * (N == 3 ? BRICK_Z : 1);
        const long local = (long)blockIdx.x * blockDim.x + threadIdx.x;
        const int e = (int)(local / BN), q = (int)(local % BN);
        if (e >= P.bricks[0]) return;
        const int b = P.bricks[1 + e];
        const int nbx = (n0 + BRICK_X - 1) / BRICK_X, nby = (n1 + BRICK_Y - 1) / BRICK_Y;
        i0 = (b % nbx) * BRICK_X + q % BRICK_X;
        i1 = ((b / nbx) % nby) * BRICK_Y + (q / BRICK_X) % BRICK_Y;
        if (N == 3) i2 = (b / (nbx * nby)) * BRICK_Z + q / (BRICK_X * BRICK_Y);
        if (i0 >= n0 || i1 >= n1 || (N == 3 && i2 >= v.n[2])) return;
    } else {
        const int nr = P.r1 - P.r0;
        const long total = (N == 1) ? (long)nr : (N == 2) ? (long)n0 * nr : (long)n0 * n1 * nr;
        const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
        if (idx >= total) return;
        if (N == 1) { i0 = P.r0 + (int)idx; }
        else if (N == 2) { i0 = (int)(idx % n0); i1 = P.r0 + (int)(idx / n0); }
        else { i0 = (int)(idx % n0); long q = idx / n0; i1 = (int)(q % n1); i2 = P.r0 + (int)(q / n1); }
    }

    const long lin = (long)i0 + (long)i1 * v.s1 + (long)i2 * v.s2;
    const long node = (long)i0 + (long)n0 * ((long)i1 + (long)n1 * i2);   // coefficient boxes carry no ghosts

    bool interior = true;
    {
        const int R = 3;
        const int ii[3] = {i0, i1, i2};
#pragma unroll
        for (int d = 0; d < N; ++d) {
            if (ii[d] - R < 0 && v.bc[d][0].kind != BC_HALO) interior = false;
            if (ii[d] + R >= v.n[d] && v.bc[d][1].kind != BC_HALO) interior = false;
        }
    }
    Reader<N, T> r{v, v.p + lin, i0, i1, i2, interior};

    const T inc = v.p[lin];
    T x;
    switch (P.base) {
        case BASE_IN:     x = inc; break;
        case BASE_RK3_S2: x = T(0.75 * double(P.p0[lin]) + 0.25 * double(inc)); break;   // timestepping.jl:183
        case BASE_RK3_S3: x = T((P.p0[lin] + T(2) * inc) / T(3)); break;                  // timestepping.jl:194
        default:          x = P.p0[lin]; break;
    }
    T x2 = inc;
    for (int k = 0; k < P.nterms; ++k) {
        const double H = compute_term<N, T>(r, P.terms[k], node, P.h, P.dxmin, P.skip_zero_u);
        x = T(double(x) - P.c * H);
        if (P.out2) x2 = T(double(x2) - P.c2 * H);
    }
    P.out[lin] = x;
    if (P.out2) P.out2[lin] = x2;
}

template <class T>
cudaError_t launch_stage_generic(int ndim, const StageParams<T>& P, cudaStream_t s) {
    const View<T>& v = P.in;
    const long nr = P.r1 - P.r0;
    if (nr <= 0) return cudaSuccess;
    long total = ndim == 1 ? nr : ndim == 2 ? (long)v.n[0] * nr : (long)v.n[0] * v.n[1] * nr;
    if (P.bricks) {        // every brick of the box: the list's count stays on the device
        if (ndim == 1) return cudaErrorNotSupported;
        const long nb = (long)((v.n[0] + BRICK_X - 1) / BRICK_X) * ((v.n[1] + BRICK_Y - 1) / BRICK_Y) * (ndim == 3 ? (v.n[2] + BRICK_Z - 1) / BRICK_Z : 1);
        total = nb * BRICK_X * BRICK_Y * (ndim == 3 ? BRICK_Z : 1);
    }
    const int block = 256;
    const long grid = (total + block - 1) / block;
    if (grid > 2147483647L) return cudaErrorInvalidConfiguration;
    if (ndim == 1) stage_generic_kernel<1, T><<<(unsigned)grid, block, 0, s>>>(P);
    else if (ndim == 2) stage_generic_kernel<2, T><<<(unsigned)grid, block, 0, s>>>(P);
    else stage_generic_kernel<3, T><<<(unsigned)grid, block, 0, s>>>(P);
    return cudaGetLastError();
}
template cudaError_t launch_stage_generic<float>(int, const StageParams<float>&, cudaStream_t);
template cudaError_t launch_stage_generic<double>(int, const StageParams<double>&, cudaStream_t);

// ---------------------------------------------------------------------------------------------
// K3: CFL reduction (levelsetterms.jl:22-38, 90-96, 123-127, 172-178).
// The reference takes min over nodes of 1/sum_d(|u_d|/h_d) (advection), 1/sum_d(|v|/h_d) (normal),
// dx^2/(2|b|) (curvature).  x -> 1/x and the other two maps are monotone under correct rounding, so
// the min equals the map applied to the MAX of sum_d(|u_d|/h_d), |v|, |b| — bit for bit.  The
// kernel reduces that max (warp shuffle + block shared-memory + one atomicMax per block) on the
// IEEE bit pattern: non-negative doubles order like unsigned integers, and a (sign-cleared) NaN
// compares above +Inf, so a NaN anywhere wins the max and reaches the host, which then fails
// `dt > 0` exactly like the reference.
// ---------------------------------------------------------------------------------------------
template <int N, class T>
__global__ void __launch_bounds__(256) cfl_kernel(const __grid_constant__ CflParams P) {
    const TermDev& t = P.term;
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    const long stride = (long)gridDim.x * blockDim.x;
    unsigned long long best = 0ULL;
    auto fold = [&](double s) {
        const unsigned long long bits = isnan(s) ? 0x7FF8000000000000ULL : (unsigned long long)__double_as_longlong(s);
        best = bits > best ? bits : best;
    };
    if (t.coef_kind == COEF_FIELD && !t.coef_f64) {
        // stored coefficient: a pure streaming pass, no index decode; 4 independent loads in flight per thread
        const T* __restrict__ c = static_cast<const T*>(t.coef);
        const double g = t.scaled ? t.g : 1.0;
        long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
        for (; idx + 3 * stride < total; idx += 4 * stride) {
            // issue all loads before the first division: the IEEE-division slow-path branch would otherwise
            // fence every load behind the previous quotient and expose DRAM latency 4*N times per iteration
            double v[4][N];
#pragma unroll
            for (int k = 0; k < 4; ++k)
#pragma unroll
                for (int d = 0; d < N; ++d)
                    v[k][d] = t.kind == TERM_ADVECTION ? double(c[(long)d * t.cstride + idx + k * stride])
                                                       : (d == 0 ? double(c[idx + k * stride]) : 0.0);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (t.kind == TERM_ADVECTION) {
                    double acc = 0.0;
#pragma unroll
                    for (int d = 0; d < N; ++d) {
                        double w = v[k][d];
                        if (t.scaled) w = w * g;
                        const double q = fabs(w) / P.h[d];
                        acc = (d == 0) ? q : acc + q;
                    }
                    fold(acc);
                } else {
                    double w = v[k][0];
                    if (t.scaled) w = w * g;
                    fold(fabs(w));
                }
            }
        }
        for (; idx < total; idx += stride) {
            double acc;
            if (t.kind == TERM_ADVECTION) {
                acc = 0.0;
#pragma unroll
                for (int d = 0; d < N; ++d) {
                    double v = double(c[(long)d * t.cstride + idx]);
                    if (t.scaled) v = v * g;
                    const double q = fabs(v) / P.h[d];
                    acc = (d == 0) ? q : acc + q;
                }
            } else {
                double v = double(c[idx]);
                if (t.scaled) v = v * g;
                acc = fabs(v);
            }
            fold(acc);
        }
    } else {
        for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
            const int i0 = (int)(idx % P.n[0]);
            const long q = idx / P.n[0];
            const int i1 = (int)(q % P.n[1]);
            const int i2 = (int)(q / P.n[1]);
            double s;
            if (t.kind == TERM_ADVECTION) {
                s = 0.0;
#pragma unroll
                for (int d = 0; d < N; ++d) {
                    const double v = coef_comp<T>(t, idx, d, i0, i1, i2, N);
                    const double q2 = fabs(v) / P.h[d];
                    s = (d == 0) ? q2 : s + q2;
                }
            } else {
                s = fabs(coef_comp<T>(t, idx, 0, i0, i1, i2, N));
            }
            fold(s);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
    }
    __shared__ unsigned long long wbest[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) wbest[w] = best;
    __syncthreads();
    if (w == 0) {
        best = lane < (int)(blockDim.x >> 5) ? wbest[lane] : 0ULL;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other > best ? other : best;
        }
        if (lane == 0) atomicMax(P.out, best);
    }
}

cudaError_t launch_cfl(int ndim, int dtype_f64, const CflParams& P, int sm_count, cudaStream_t s) {
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    const int block = 256;
    long grid = (total + block - 1) / block;
    const long cap = (long)sm_count * 8;     // persistent-style: 8 CTAs of 256 threads per SM
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
#define LSM_CFL(NN) do { if (dtype_f64) cfl_kernel<NN, double><<<(unsigned)grid, block, 0, s>>>(P); \
                         else cfl_kernel<NN, float><<<(unsigned)grid, block, 0, s>>>(P); } while (0)
    if (ndim == 1) LSM_CFL(1); else if (ndim == 2) LSM_CFL(2); else LSM_CFL(3);
#undef LSM_CFL
    return cudaGetLastError();
}

// Candidate nodes of the CFL maximum (lsm_api.cu, cfl_candidates): the unscaled quantity s = sum_d |u_d| / h_d (advection) or
// |v| (normal motion, curvature), formed exactly like cfl_kernel does with g = 1; nodes with !(s < thr) — NaN included —
// append their raw coefficient tuple.
template <int N, class T>
__global__ void __launch_bounds__(256) cfl_candidates_kernel(const __grid_constant__ CandParams P) {
    const TermDev& t = P.term;
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    const long stride = (long)gridDim.x * blockDim.x;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
        const int i0 = (int)(idx % P.n[0]);
        const long q = idx / P.n[0];
        const int i1 = (int)(q % P.n[1]);
        const int i2 = (int)(q / P.n[1]);
        double v[3] = {0.0, 0.0, 0.0};
        double s;
        if (t.kind == TERM_ADVECTION) {
            s = 0.0;
#pragma unroll
            for (int d = 0; d < N; ++d) {
                v[d] = coef_comp<T>(t, idx, d, i0, i1, i2, N);
                const double q2 = fabs(v[d]) / P.h[d];
                s = (d == 0) ? q2 : s + q2;
            }
        } else {
            v[0] = coef_comp<T>(t, idx, 0, i0, i1, i2, N);
            s = fabs(v[0]);
        }
        if (!(s < P.thr)) {
            const unsigned k = atomicAdd(P.count, 1u);
            if (k < (unsigned)P.cap)
                for (int d = 0; d < P.ncomp; ++d) P.out[(long)k * P.ncomp + d] = v[d];
        }
    }
}

cudaError_t launch_cfl_candidates(int ndim, int dtype_f64, const CandParams& P, int sm_count, cudaStream_t s) {
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    const int block = 256;
    long grid = (total + block - 1) / block;
    const long cap = (long)sm_count * 8;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
#define LSM_CAND(NN) do { if (dtype_f64) cfl_candidates_kernel<NN, double><<<(unsigned)grid, block, 0, s>>>(P); \
                          else cfl_candidates_kernel<NN, float><<<(unsigned)grid, block, 0, s>>>(P); } while (0)
    if (ndim == 1) LSM_CAND(1); else if (ndim == 2) LSM_CAND(2); else LSM_CAND(3);
#undef LSM_CAND
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// analytic initial conditions / coefficients generated on the device.  MeshField(f, grid) (meshfield.jl:208-211) evaluates
// f at x = lc + (I - 1) h (meshes.jl:115-117); these kernels do the same for a small family of f, in the operation order
// stated in include/lsm_b200.h (this file is compiled without FMA contraction, so a NumPy restatement is bit-identical).
// ---------------------------------------------------------------------------------------------
template <class T>
__global__ void fill_shape_kernel(T* __restrict__ dst, const __grid_constant__ ShapeParams P) {
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        int I[3];
        I[0] = (int)(idx % P.n[0]);
        const long q = idx / P.n[0];
        I[1] = (int)(q % P.n[1]);
        I[2] = (int)(q / P.n[1]);
        I[P.ndim - 1] += P.first_last;
        double x[3];
        for (int d = 0; d < 3; ++d) x[d] = P.lc[d] + double(I[d]) * P.h[d];
        if (P.shape == 3) {                                   // CONST: one value per component
            for (int c = 0; c < P.ncomp; ++c) dst[(long)c * P.cstride + idx] = T(P.p[c]);
            continue;
        }
        double v = 0.0;
        if (P.shape == 0) {                                   // SPHERE: sqrt(sum_d (x_d - c_d)^2) - r
            double s = 0.0;
            for (int d = 0; d < P.ndim; ++d) { const double t = x[d] - P.p[d]; s = d == 0 ? t * t : s + t * t; }
            v = sqrt(s) - P.p[P.ndim];
        } else if (P.shape == 1) {                            // BOX: max_d (|x_d - c_d| - w_d / 2)
            for (int d = 0; d < P.ndim; ++d) {
                const double t = fabs(x[d] - P.p[d]) - P.p[P.ndim + d] / 2.0;
                v = d == 0 ? t : (t > v ? t : v);
            }
        } else {                                              // PLANE: sum_d n_d x_d - offset
            double s = 0.0;
            for (int d = 0; d < P.ndim; ++d) { const double t = P.p[d] * x[d]; s = d == 0 ? t : s + t; }
            v = s - P.p[P.ndim];
        }
        dst[idx] = T(v);
    }
}

cudaError_t launch_fill_shape(int f64, void* dst, const ShapeParams& P, cudaStream_t s) {
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    const int block = 256;
    const long grid = std::min<long>((total + block - 1) / block, 148L * 16);
    if (f64) fill_shape_kernel<double><<<(unsigned)std::max<long>(grid, 1), block, 0, s>>>(static_cast<double*>(dst), P);
    else fill_shape_kernel<float><<<(unsigned)std::max<long>(grid, 1), block, 0, s>>>(static_cast<float*>(dst), P);
    return cudaGetLastError();
}

struct SepParams { int n[3]; int ndim; long cstride; double scale[3]; const double* tab[3][3]; };

// component d of a separable vector field, materialised in SoA storage: ((scale_d * X_d[i]) * Y_d[j]) * Z_d[k]
template <class T>
__global__ void fill_separable_kernel(T* __restrict__ dst, const __grid_constant__ SepParams P) {
    const long total = (long)P.n[0] * P.n[1] * P.n[2];
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i0 = (int)(idx % P.n[0]);
        const long q = idx / P.n[0];
        const int i1 = (int)(q % P.n[1]);
        const int i2 = (int)(q / P.n[1]);
        for (int d = 0; d < P.ndim; ++d) {
            double v = P.scale[d] * P.tab[d][0][i0];
            if (P.ndim > 1) v = v * P.tab[d][1][i1];
            if (P.ndim > 2) v = v * P.tab[d][2][i2];
            dst[(long)d * P.cstride + idx] = T(v);
        }
    }
}

cudaError_t launch_fill_separable(int f64, void* dst, long cstride, const int* n, int ndim, const double* scale, const double* const (*tab)[3], cudaStream_t s) {
    SepParams P{};
    for (int d = 0; d < 3; ++d) { P.n[d] = n[d]; P.scale[d] = scale[d]; for (int a = 0; a < 3; ++a) P.tab[d][a] = tab[d][a]; }
    P.ndim = ndim; P.cstride = cstride;
    const long total = (long)n[0] * n[1] * n[2];
    const int block = 256;
    const long grid = std::max<long>(1, std::min<long>((total + block - 1) / block, 148L * 16));
    if (f64) fill_separable_kernel<double><<<(unsigned)grid, block, 0, s>>>(static_cast<double*>(dst), P);
    else fill_separable_kernel<float><<<(unsigned)grid, block, 0, s>>>(static_cast<float*>(dst), P);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// small elementwise kernels
// ---------------------------------------------------------------------------------------------
// EikonalReinitializationTerm(phi0): S0 = v / sqrt(v^2 + dx^2)   (levelsetterms.jl:217-221)
template <class T, class TO>
__global__ void eikonal_s0_kernel(const T* __restrict__ phi, TO* __restrict__ out, long n, double dx) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const T v = phi[i];
        out[i] = TO(double(v) / sqrt(double(T(v * v)) + dx * dx));
    }
}

cudaError_t launch_eikonal_s0(int src_f64, int dst_f64, const void* phi, void* out, long n, double dx, cudaStream_t s) {
    const int block = 256;
    long grid = (n + block - 1) / block; if (grid > 148L * 16) grid = 148L * 16; if (grid < 1) grid = 1;
    if (src_f64 && dst_f64) eikonal_s0_kernel<double, double><<<(unsigned)grid, block, 0, s>>>((const double*)phi, (double*)out, n, dx);
    else if (src_f64) eikonal_s0_kernel<double, float><<<(unsigned)grid, block, 0, s>>>((const double*)phi, (float*)out, n, dx);
    else if (dst_f64) eikonal_s0_kernel<float, double><<<(unsigned)grid, block, 0, s>>>((const float*)phi, (double*)out, n, dx);
    else eikonal_s0_kernel<float, float><<<(unsigned)grid, block, 0, s>>>((const float*)phi, (float*)out, n, dx);
    return cudaGetLastError();
}

// AoS (host layout, component fastest) <-> SoA (device layout) for vector coefficient fields
template <class T>
__global__ void aos_to_soa_kernel(const T* __restrict__ aos, T* __restrict__ soa, long n, int ncomp, long cstride) {
    const long tot = n * ncomp;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long)gridDim.x * blockDim.x) {
        const long node = i / ncomp; const int d = (int)(i % ncomp);
        soa[(long)d * cstride + node] = aos[i];
    }
}
template <class T>
__global__ void soa_to_aos_kernel(const T* __restrict__ soa, T* __restrict__ aos, long n, int ncomp, long cstride) {
    const long tot = n * ncomp;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long)gridDim.x * blockDim.x) {
        const long node = i / ncomp; const int d = (int)(i % ncomp);
        aos[i] = soa[(long)d * cstride + node];
    }
}
cudaError_t launch_transpose(int f64, bool to_soa, const void* src, void* dst, long n, int ncomp, long cstride, cudaStream_t s) {
    const int block = 256;
    long grid = (n * ncomp + block - 1) / block; if (grid > 148L * 16) grid = 148L * 16; if (grid < 1) grid = 1;
    if (f64) { if (to_soa) aos_to_soa_kernel<double><<<(unsigned)grid, block, 0, s>>>((const double*)src, (double*)dst, n, ncomp, cstride);
               else soa_to_aos_kernel<double><<<(unsigned)grid, block, 0, s>>>((const double*)src, (double*)dst, n, ncomp, cstride); }
    else     { if (to_soa) aos_to_soa_kernel<float><<<(unsigned)grid, block, 0, s>>>((const float*)src, (float*)dst, n, ncomp, cstride);
               else soa_to_aos_kernel<float><<<(unsigned)grid, block, 0, s>>>((const float*)src, (float*)dst, n, ncomp, cstride); }
    return cudaGetLastError();
}

// phi[I] for arbitrary (possibly out-of-grid) 1-based indices: meshfield.jl:213-217
template <int N, class T>
__global__ void getindex_kernel(const __grid_constant__ View<T> v, const int* __restrict__ idx, int count, double* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const int i0 = idx[t * N] - 1;
    const int i1 = N > 1 ? idx[t * N + 1] - 1 : 0;
    const int i2 = N > 2 ? idx[t * N + 2] - 1 : 0;
    out[t] = double(getindex_slow<N, T>(v, i0, i1, i2));
}
template <class T>
cudaError_t launch_getindex(int ndim, const View<T>& v, const int* d_idx, int count, double* d_out, cudaStream_t s) {
    const int block = 128, grid = (count + block - 1) / block;
    if (ndim == 1) getindex_kernel<1, T><<<grid, block, 0, s>>>(v, d_idx, count, d_out);
    else if (ndim == 2) getindex_kernel<2, T><<<grid, block, 0, s>>>(v, d_idx, count, d_out);
    else getindex_kernel<3, T><<<grid, block, 0, s>>>(v, d_idx, count, d_out);
    return cudaGetLastError();
}
template cudaError_t launch_getindex<float>(int, const View<float>&, const int*, int, double*, cudaStream_t);
template cudaError_t launch_getindex<double>(int, const View<double>&, const int*, int, double*, cudaStream_t);

// ---------------------------------------------------------------------------------------------
// volume / perimeter (levelsetops.jl:27-33, 139-149, smooth_heaviside / smooth_delta :186-195).  Deterministic two-stage
// sum: per-block partials in a fixed tree, then one block adds the partials in a fixed order.
// ---------------------------------------------------------------------------------------------
template <int N, class T, bool PERIM>
__global__ void __launch_bounds__(256) measure_kernel(const __grid_constant__ View<T> v, const double h0, const double h1, const double h2,
                                                      const double dmin, double* __restrict__ partials) {
    const double h[3] = {h0, h1, h2};
    const long total = (long)v.n[0] * v.n[1] * v.n[2];
    double acc = 0.0;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i0 = (int)(idx % v.n[0]);
        const long q = idx / v.n[0];
        const int i1 = (int)(q % v.n[1]), i2 = (int)(q / v.n[1]);
        const double x = double(v.p[(long)i0 + (long)i1 * v.s1 + (long)i2 * v.s2]);
        if (!PERIM) {
            const double y = -x;
            double hv;
            if (y > dmin) hv = 1.0;
            else if (y < -dmin) hv = 0.0;
            else hv = 0.5 * (1.0 + y / dmin + 1.0 / M_PI * sin(M_PI * y / dmin));
            acc += hv;
        } else if (!(fabs(x) > dmin)) {
            const double delta = 0.5 / dmin * (1.0 + cos(M_PI * x / dmin));
            double g2 = 0.0;
#pragma unroll
            for (int d = 0; d < N; ++d) {
                const T p = getindex_slow<N, T>(v, i0 + (d == 0), i1 + (d == 1), i2 + (d == 2));
                const T m = getindex_slow<N, T>(v, i0 - (d == 0), i1 - (d == 1), i2 - (d == 2));
                const double gd = double(T(p - m)) / (2 * h[d]);
                g2 = d == 0 ? gd * gd : g2 + gd * gd;
            }
            acc += delta * sqrt(g2);
        }
    }
    __shared__ double sh[256];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(256) measure_final_kernel(const double* __restrict__ partials, int n, double scale, double* out) {
    __shared__ double sh[256];
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) acc += partials[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0] * scale;
}
template <class T>
cudaError_t launch_measure(int ndim, bool perimeter, const View<T>& v, const double* h, double* d_partials, int nblocks, double* d_out, cudaStream_t s) {
    double dmin = h[0], vol = h[0];
    for (int d = 1; d < ndim; ++d) { dmin = h[d] < dmin ? h[d] : dmin; vol *= h[d]; }
#define LSM_MEAS(NN) do { if (perimeter) measure_kernel<NN, T, true><<<nblocks, 256, 0, s>>>(v, h[0], h[1], h[2], dmin, d_partials); \
                          else measure_kernel<NN, T, false><<<nblocks, 256, 0, s>>>(v, h[0], h[1], h[2], dmin, d_partials); } while (0)
    if (ndim == 1) LSM_MEAS(1); else if (ndim == 2) LSM_MEAS(2); else LSM_MEAS(3);
#undef LSM_MEAS
    measure_final_kernel<<<1, 256, 0, s>>>(d_partials, nblocks, vol, d_out);
    return cudaGetLastError();
}
template cudaError_t launch_measure<float>(int, bool, const View<float>&, const double*, double*, int, double*, cudaStream_t);
template cudaError_t launch_measure<double>(int, bool, const View<double>&, const double*, double*, int, double*, cudaStream_t);

// velocityextension.jl:95-116 (_signed_normal_components) + :82-93 (frozen mask): a_d = S * grad_d / |grad|, S = phi/sqrt(phi^2+dx^2),
// written SoA; zero where |grad|^2 <= min_norm^2 (reference) and on frozen nodes (so that the advection step leaves them untouched).
template <int N, class T>
__global__ void __launch_bounds__(256) signed_normals_kernel(const __grid_constant__ View<T> v, const double h0, const double h1, const double h2,
                                                             const double dx, const double min2, const unsigned char* __restrict__ frozen,
                                                             const double band_dx, T* __restrict__ a, const long cstride) {
    const double h[3] = {h0, h1, h2};
    const long total = (long)v.n[0] * v.n[1] * v.n[2];
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i0 = (int)(idx % v.n[0]);
        const long q = idx / v.n[0];
        const int i1 = (int)(q % v.n[1]), i2 = (int)(q / v.n[1]);
        const T p = v.p[(long)i0 + (long)i1 * v.s1 + (long)i2 * v.s2];
        const bool fr = frozen ? frozen[idx] != 0 : (fabs(double(p)) <= band_dx);
        T g[3] = {T(0), T(0), T(0)};
        T nrm2 = T(0);
#pragma unroll
        for (int d = 0; d < N; ++d) {
            const T pp = getindex_slow<N, T>(v, i0 + (d == 0), i1 + (d == 1), i2 + (d == 2));
            const T pm = getindex_slow<N, T>(v, i0 - (d == 0), i1 - (d == 1), i2 - (d == 2));
            g[d] = T(double(T(pp - pm)) / (2 * h[d]));
            nrm2 = d == 0 ? T(g[d] * g[d]) : T(nrm2 + T(g[d] * g[d]));
        }
        const bool zero = fr || double(nrm2) <= min2;
        const T invn = T(1) / T(sqrt(nrm2));
        const double S = double(p) / sqrt(double(T(p * p)) + dx * dx);
#pragma unroll
        for (int d = 0; d < N; ++d) a[(long)d * cstride + idx] = zero ? T(0) : T((S * double(g[d])) * double(invn));
    }
}
template <class T>
cudaError_t launch_signed_normals(int ndim, const View<T>& v, const double* h, double min_norm, const unsigned char* d_frozen, double band, T* a, long cstride, cudaStream_t s) {
    double dx = h[0];
    for (int d = 1; d < ndim; ++d) dx = h[d] < dx ? h[d] : dx;
    const long total = (long)v.n[0] * v.n[1] * v.n[2];
    long grid = (total + 255) / 256; if (grid > 148L * 16) grid = 148L * 16; if (grid < 1) grid = 1;
    if (ndim == 1) signed_normals_kernel<1, T><<<(unsigned)grid, 256, 0, s>>>(v, h[0], h[1], h[2], dx, min_norm * min_norm, d_frozen, band * dx, a, cstride);
    else if (ndim == 2) signed_normals_kernel<2, T><<<(unsigned)grid, 256, 0, s>>>(v, h[0], h[1], h[2], dx, min_norm * min_norm, d_frozen, band * dx, a, cstride);
    else signed_normals_kernel<3, T><<<(unsigned)grid, 256, 0, s>>>(v, h[0], h[1], h[2], dx, min_norm * min_norm, d_frozen, band * dx, a, cstride);
    return cudaGetLastError();
}
template cudaError_t launch_signed_normals<float>(int, const View<float>&, const double*, double, const unsigned char*, double, float*, long, cudaStream_t);
template cudaError_t launch_signed_normals<double>(int, const View<double>&, const double*, double, const unsigned char*, double, double*, long, cudaStream_t);

// levelsetops.jl:253-325: union! / intersect! / setdiff! / complement! as one pointwise pass.  Julia's min/max: NaN if either
// operand is NaN; equal operands (signed zeros) resolve to -0.0 for min and +0.0 for max.
template <class T> __device__ __forceinline__ T jl_min(T a, T b) {
    if (a != a || b != b) return a + b;
    if (a == b) return signbit(a) ? a : b;
    return a < b ? a : b;
}
template <class T> __device__ __forceinline__ T jl_max(T a, T b) {
    if (a != a || b != b) return a + b;
    if (a == b) return signbit(a) ? b : a;
    return a > b ? a : b;
}
template <class T>
__global__ void __launch_bounds__(256) csg_kernel(T* __restrict__ dst, const T* __restrict__ src, const long n, const int op) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const T a = dst[i];
        T r;
        if (op == 3) r = -a;
        else {
            const T b = src[i];
            r = op == 0 ? jl_min<T>(a, b) : (op == 1 ? jl_max<T>(a, b) : jl_max<T>(a, -b));
        }
        dst[i] = r;
    }
}
cudaError_t launch_csg(int f64, void* dst, const void* src, long n, int op, cudaStream_t s) {
    long grid = (n + 255) / 256; if (grid > 148L * 32) grid = 148L * 32; if (grid < 1) grid = 1;
    if (f64) csg_kernel<double><<<(unsigned)grid, 256, 0, s>>>(static_cast<double*>(dst), static_cast<const double*>(src), n, op);
    else csg_kernel<float><<<(unsigned)grid, 256, 0, s>>>(static_cast<float*>(dst), static_cast<const float*>(src), n, op);
    return cudaGetLastError();
}

// K6: max |a - b| (bit-pattern max, NaN wins)
template <class T>
__global__ void __launch_bounds__(256) max_abs_diff_kernel(const T* __restrict__ a, const T* __restrict__ b, long n, unsigned long long* out) {
    unsigned long long best = 0ULL;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const double d = fabs(double(a[i]) - double(b[i]));
        const unsigned long long bits = isnan(d) ? 0x7FF8000000000000ULL : (unsigned long long)__double_as_longlong(d);
        best = bits > best ? bits : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
    }
    if ((threadIdx.x & 31) == 0 && best) atomicMax(out, best);
}
cudaError_t launch_max_abs_diff(int f64, const void* a, const void* b, long n, unsigned long long* out, cudaStream_t s) {
    const int block = 256;
    long grid = (n + block - 1) / block; if (grid > 148L * 8) grid = 148L * 8; if (grid < 1) grid = 1;
    if (f64) max_abs_diff_kernel<double><<<(unsigned)grid, block, 0, s>>>((const double*)a, (const double*)b, n, out);
    else max_abs_diff_kernel<float><<<(unsigned)grid, block, 0, s>>>((const float*)a, (const float*)b, n, out);
    return cudaGetLastError();
}

}  // namespace lsm
