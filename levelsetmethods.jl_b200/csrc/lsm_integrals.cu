// lsm_integrals.cu — measures of the region {s <= 0} and of the zero level set {s = 0}, and the integrals of a field F over them
// (lsm_level_set_integrals), on the piecewise-linear geometry of lsm_interface_extract.
//
// Two kernels:
//   planes : one block per plane of cells (cells sharing the index of the last axis; one thread per cell in 1-D).  Each thread reads
//            the 2^N corners of its cells (phi, and F when given) once; a cell whose corners are all valid and inside adds the cell
//            volume (and the P1 integral of F over it) directly, a valid cell with every corner outside adds nothing, and only the
//            other cells walk their simplices: the inside part of a cut simplex from the crossing parameters of its cut edges, and
//            the primitives of the extraction (lsm_simplex.cuh: simplex_vertices) with their measures.  The block reduces its threads'
//            sums in a fixed tree and writes one partial per output and plane (32 bytes per plane);
//   sum    : one block; the plane partials in increasing plane order, into the four outputs.
// The order of every sum depends only on the shape of a plane, so the result does not depend on the slab decomposition: a rank
// writes the partials of the planes it owns into a buffer of all planes, zero elsewhere, the buffer is all-reduced (each entry has
// one non-zero contributor, so the sum is exact), and every rank then sums the planes as one GPU does.  The operation order of every
// contribution is the one include/lsm_b200.h states; tests/integrals_ref.py restates it in NumPy (compiled with -fmad=false).
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>
#include "lsm_kernels.h"
#include "lsm_simplex.cuh"

namespace lsm {
namespace {

constexpr int TPB = 256;         // threads of a plane block (and of the 1-D kernel)
constexpr int SUM_TPB = 256;     // threads of the sum block
constexpr int SUM_CHUNK = 1024;  // planes staged in shared memory per step of the sum

// the four running sums of a thread: |{s <= 0}|, |{s = 0}|, the integral of F over each
struct Acc { double vol, area, fvol, farea; };

// measure of a primitive from its vertex coordinates (the operation order of the header)
template <int N> __device__ __forceinline__ double prim_measure(const double (*V)[3]) {
    if constexpr (N == 1) return 1.0;
    else if constexpr (N == 2) {
        const double dx = V[1][0] - V[0][0], dy = V[1][1] - V[0][1];
        return sqrt(dx * dx + dy * dy);
    } else {
        double u[3], v[3];
        for (int d = 0; d < 3; ++d) { u[d] = V[1][d] - V[0][d]; v[d] = V[2][d] - V[0][d]; }
        const double cx = u[1] * v[2] - u[2] * v[1], cy = u[2] * v[0] - u[0] * v[2], cz = u[0] * v[1] - u[1] * v[0];
        return sqrt((cx * cx + cy * cy) + cz * cz) / 2.0;
    }
}

template <int N> __device__ __forceinline__ double prim_mean(const double* Fv) {
    if constexpr (N == 1) return Fv[0];
    else if constexpr (N == 2) return (Fv[0] + Fv[1]) / 2.0;
    else return ((Fv[0] + Fv[1]) + Fv[2]) / 3.0;
}

// The contributions of cell c (global coordinates c, box index cidx) to the thread's sums.  V = prod |h|, Vs = V / N!.  A cell that
// takes the simplex walk first copies its corner values to the thread's slots ss / sf in shared memory, where the walk indexes them
// with run-time corner numbers (in registers that would need a stack frame).
template <class T, class TF, int N>
__device__ __forceinline__ void cell_integrals(const IntegArgs& I, const int* c, long long cidx, double* ss, double* sf, Acc& acc) {
    constexpr bool WITH_F = !std::is_void_v<TF>;
    constexpr unsigned full = (1u << (1 << N)) - 1u;
    const IfaceArgs& A = I.g;
    double s[1 << N];
    const Masks M = cell_corners<T, N>(A, cidx, s);
    if (!M.nan && !M.in) return;                                      // every corner outside: nothing
    [[maybe_unused]] double f[1 << N];
    if constexpr (WITH_F) {
        const TF* F = static_cast<const TF*>(I.F);
#pragma unroll
        for (int k = 0; k < (1 << N); ++k) f[k] = double(F[cidx + corner_off(A, k)]);
    }
    if (!M.nan && M.in == full) {                                     // every corner inside: the whole cell
        acc.vol += I.V;
        if constexpr (WITH_F) {
            double mean;
            if constexpr (N == 1) mean = (f[0] + f[1]) / 2.0;
            else if constexpr (N == 2) mean = (f[0] + f[3]) / 3.0 + (f[1] + f[2]) / 6.0;
            else mean = (f[0] + f[7]) / 4.0 + (((((f[1] + f[2]) + f[3]) + f[4]) + f[5]) + f[6]) / 12.0;
            acc.fvol += I.V * mean;
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < (1 << N); ++k) {
        ss[k] = s[k];
        if constexpr (WITH_F) sf[k] = f[k];
    }
    const double Vs = I.Vs;
    for (int p = 0; p < nsimplices<N>(); ++p) {
        if (chain_mask<N>(p) & M.nan) continue;
        int inside = 0;
#pragma unroll
        for (int x = 0; x <= N; ++x) inside |= ((M.in >> chain<N>(p, x)) & 1) << x;
        const int k = __popc(inside);
        if (k == 0) continue;
        auto S = [&](int x) { return ss[chain<N>(p, x)]; };           // s and F at chain position x
        [[maybe_unused]] auto Fw = [&](int x) { return sf[chain<N>(p, x)]; };
        // F at the crossing of the simplex edge (x, y): the extraction's t, from the lower chain position
        [[maybe_unused]] auto Fc = [&](int x, int y) {
            const int a = x < y ? x : y, b = x < y ? y : x;
            const double sa = S(a), fa = Fw(a);
            const double t = sa / (sa - S(b));
            return fa + t * (Fw(b) - fa);
        };
        if (k == N + 1) {
            acc.vol += Vs;
            if constexpr (WITH_F) {
                double sum = Fw(0);
#pragma unroll
                for (int x = 1; x <= N; ++x) sum += Fw(x);
                acc.fvol += Vs * (sum / double(N + 1));
            }
        } else if (k == 1 || k == N) {
            // lone vertex q: the only inside one (k = 1, and always in 1-D), else the only outside one; the others o_0 < o_1 < ...
            // in chain order, u_j = s_q / (s_q - s_(o_j))
            const int q = __ffs(k == 1 ? inside : (~inside & ((1 << (N + 1)) - 1))) - 1;
            const double sq = S(q);
            int o[N];
            double u[N];
#pragma unroll
            for (int j = 0; j < N; ++j) { o[j] = j + (j >= q ? 1 : 0); u[j] = sq / (sq - S(o[j])); }
            double corner = u[0];
#pragma unroll
            for (int j = 1; j < N; ++j) corner = corner * u[j];
            if (k == 1) {                                             // the corner simplex at q
                acc.vol += Vs * corner;
                if constexpr (WITH_F) {
                    double sum = Fw(q);
#pragma unroll
                    for (int j = 0; j < N; ++j) sum += Fc(q, o[j]);
                    acc.fvol += (Vs * corner) * (sum / double(N + 1));
                }
            } else if constexpr (N == 2) {                            // the quad (r, s, P_qs, P_qr) as (r, s, P_qs), (r, P_qs, P_qr)
                const double va = Vs * (1.0 - u[1]), vb = Vs * (u[1] * (1.0 - u[0]));
                acc.vol += va;
                acc.vol += vb;
                if constexpr (WITH_F) {
                    const double Fr = Fc(q, o[0]), Fs = Fc(q, o[1]), fr = Fw(o[0]);
                    acc.fvol += va * (((fr + Fw(o[1])) + Fs) / 3.0);
                    acc.fvol += vb * (((fr + Fs) + Fr) / 3.0);
                }
            } else if constexpr (N == 3) {                            // the simplex minus the corner simplex at q
                acc.vol += Vs * (1.0 - corner);
                if constexpr (WITH_F) {
                    const double whole = Vs * ((((Fw(0) + Fw(1)) + Fw(2)) + Fw(3)) / 4.0);
                    const double cut = (Vs * corner) * ((((Fw(q) + Fc(q, o[0])) + Fc(q, o[1])) + Fc(q, o[2])) / 4.0);
                    acc.fvol += whole - cut;
                }
            }
        } else if constexpr (N == 3) {
            // inside {a < b}, outside {c < d}: the prism as (a, P_ac, P_ad, P_bd), (a, P_ac, P_bc, P_bd), (a, b, P_bc, P_bd),
            // with tau_xy = s_x / (s_x - s_y) measured from the inside end
            const int outside = ~inside & 15;
            const int a = __ffs(inside) - 1, b = __ffs(inside & (inside - 1)) - 1;
            const int cc = __ffs(outside) - 1, d = __ffs(outside & (outside - 1)) - 1;
            const double sa = S(a), sb = S(b), sc = S(cc), sd = S(d);
            const double tac = sa / (sa - sc), tad = sa / (sa - sd), tbc = sb / (sb - sc), tbd = sb / (sb - sd);
            const double v1 = Vs * ((tac * tad) * (1.0 - tbd)), v2 = Vs * ((tac * (1.0 - tbc)) * tbd), v3 = Vs * (tbc * tbd);
            acc.vol += v1;
            acc.vol += v2;
            acc.vol += v3;
            if constexpr (WITH_F) {
                const double Fac = Fc(a, cc), Fad = Fc(a, d), Fbc = Fc(b, cc), Fbd = Fc(b, d), fa = Fw(a);
                acc.fvol += v1 * ((((fa + Fac) + Fad) + Fbd) / 4.0);
                acc.fvol += v2 * ((((fa + Fac) + Fbc) + Fbd) / 4.0);
                acc.fvol += v3 * ((((fa + Fw(b)) + Fbc) + Fbd) / 4.0);
            }
        }
        if (k == N + 1) continue;
        // the primitives of the cut simplex, with the extraction's vertex coordinates
        if constexpr (WITH_F) {
            simplex_vertices<N>(A, c, ss, M, p, [&](const double (*V)[3], const double* Fv) {
                const double m = prim_measure<N>(V);
                acc.area += m;
                acc.farea += m * prim_mean<N>(Fv);
            }, [&](int kk) { return sf[kk]; });
        } else {
            simplex_vertices<N>(A, c, ss, M, p, [&](const double (*V)[3]) { acc.area += prim_measure<N>(V); });
        }
    }
}

// block-wide sum of one double over TPB threads, in a fixed tree; the result is valid in thread 0
__device__ __forceinline__ double block_sum(double v, double* sh) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) sh[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < TPB / 32 ? sh[lane] : 0.0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    }
    __syncthreads();
    return v;
}

// 2-D and 3-D: block b sums cell plane b of the box; thread t takes the plane's cells t, t + TPB, ... in column-major order
template <class T, class TF, int N>
__global__ void __launch_bounds__(TPB) integ_planes_kernel(const __grid_constant__ IntegArgs I) {
    constexpr int SLOT = (1 << N) + 1;                               // padded: fewer bank conflicts between the threads' slots
    __shared__ double sh[TPB / 32], cs[TPB * SLOT], cf[std::is_void_v<TF> ? 1 : TPB * SLOT];
    double* ss = cs + threadIdx.x * SLOT;
    double* sf = std::is_void_v<TF> ? nullptr : cf + threadIdx.x * SLOT;
    const IfaceArgs& A = I.g;
    const int cl = blockIdx.x;                                       // the plane's index in the box
    const int W = A.m[0] - 1, R = N == 3 ? A.m[1] - 1 : 1;
    const long long total = (long long)W * R;
    const long long plane_off = (long long)cl * (N == 3 ? A.s2 : A.s1);
    int c[3] = {0, 0, 0};
    c[N - 1] = cl + A.first_last;
    int i = threadIdx.x % W, j = threadIdx.x / W;
    const int di = TPB % W, dj = TPB / W;
    Acc acc{0.0, 0.0, 0.0, 0.0};
    for (long long l = threadIdx.x; l < total; l += TPB) {
        c[0] = i;
        if (N == 3) c[1] = j;
        cell_integrals<T, TF, N>(I, c, plane_off + i + (long long)j * A.s1, ss, sf, acc);
        i += di; j += dj;
        if (i >= W) { i -= W; ++j; }
    }
    const double vol = block_sum(acc.vol, sh), area = block_sum(acc.area, sh);
    double fvol = 0.0, farea = 0.0;
    if constexpr (!std::is_void_v<TF>) { fvol = block_sum(acc.fvol, sh); farea = block_sum(acc.farea, sh); }
    if (threadIdx.x == 0) {
        double* out = I.part + 4 * (I.plane0 + cl);
        out[0] = vol; out[1] = area; out[2] = fvol; out[3] = farea;
    }
}

// 1-D: a plane is one cell
template <class T, class TF>
__global__ void __launch_bounds__(TPB) integ_cells_1d_kernel(const __grid_constant__ IntegArgs I) {
    __shared__ double cs[TPB * 3], cf[std::is_void_v<TF> ? 1 : TPB * 3];
    const long long cl = (long long)blockIdx.x * TPB + threadIdx.x;
    if (cl >= I.planes) return;
    const int c[3] = {(int)cl + I.g.first_last, 0, 0};
    Acc acc{0.0, 0.0, 0.0, 0.0};
    cell_integrals<T, TF, 1>(I, c, cl, cs + threadIdx.x * 3, std::is_void_v<TF> ? nullptr : cf + threadIdx.x * 3, acc);
    double* out = I.part + 4 * (I.plane0 + cl);
    out[0] = acc.vol; out[1] = acc.area; out[2] = acc.fvol; out[3] = acc.farea;
}

// one block: out[q] = sum over planes, in increasing order, of part[4 plane + q]
__global__ void __launch_bounds__(SUM_TPB) integ_sum_kernel(const double* __restrict__ part, long long nplanes, double* __restrict__ out) {
    __shared__ double sh[4 * SUM_CHUNK];
    double acc = 0.0;
    for (long long b = 0; b < nplanes; b += SUM_CHUNK) {
        const int cnt = (int)(nplanes - b < SUM_CHUNK ? nplanes - b : SUM_CHUNK);
        for (int e = threadIdx.x; e < 4 * cnt; e += SUM_TPB) sh[e] = part[4 * b + e];
        __syncthreads();
        if (threadIdx.x < 4)
            for (int k = 0; k < cnt; ++k) acc += sh[4 * k + threadIdx.x];
        __syncthreads();
    }
    if (threadIdx.x < 4) out[threadIdx.x] = acc;
}

template <class T, class TF>
cudaError_t launch_tf(const IntegArgs& I, cudaStream_t s) {
    switch (I.g.ndim) {
        case 1: integ_cells_1d_kernel<T, TF><<<(unsigned)((I.planes + TPB - 1) / TPB), TPB, 0, s>>>(I); break;
        case 2: integ_planes_kernel<T, TF, 2><<<(unsigned)I.planes, TPB, 0, s>>>(I); break;
        default: integ_planes_kernel<T, TF, 3><<<(unsigned)I.planes, TPB, 0, s>>>(I); break;
    }
    return cudaGetLastError();
}

template <class T>
cudaError_t launch_t(const IntegArgs& I, cudaStream_t s) {
    if (!I.F) return launch_tf<T, void>(I, s);
    return I.F_f64 ? launch_tf<T, double>(I, s) : launch_tf<T, float>(I, s);
}

}  // namespace

cudaError_t launch_integral_planes(const IntegArgs& I, cudaStream_t s) {
    return I.g.f64 ? launch_t<double>(I, s) : launch_t<float>(I, s);
}

cudaError_t launch_integral_sum(const double* part, long long nplanes, double* out, cudaStream_t s) {
    integ_sum_kernel<<<1, SUM_TPB, 0, s>>>(part, nplanes, out);
    return cudaGetLastError();
}

}  // namespace lsm
