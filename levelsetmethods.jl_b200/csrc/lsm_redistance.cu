// lsm_redistance.cu — closest-point redistancing (lsm_redistance): phi <- the signed distance to the piecewise-linear mesh that
// lsm_interface_extract(phi, 0) returns, without building that mesh.
//
// Kernels:
//   flag  : one thread per node; classifies the node's cell (lsm_simplex.cuh) and appends it to a list when it holds a primitive;
//   cells : one block per listed cell, twice; the cell's primitives are rebuilt from phi exactly as the extraction builds them, then
//           every node whose window holds the cell evaluates them: pass 0 takes the atomic minimum of the distance bits, pass 1 the
//           atomic minimum of the (cell, primitive) order key among the candidates at that distance.  Together that is the first
//           strictly closest primitive of the node's column-major scan, independent of the list order.  (A node-centric scan of the
//           window, the direct form of the contract, leaves most lanes of a warp idle: along x only one or two of 32 nodes' cells
//           are cut at a time.)
//   pick  : one thread per node; the closest point of the winning primitive (NaN when there is none);
//   flood : jump flooding over closest points, launched once per step k (2^(L-1), ..., 2, 1, then 1 again), reading one point
//           buffer and writing the other; candidates are the node's own point, then its 3^N - 1 neighbours at +-k in column-major
//           order of the offset, and the strictly closest one wins;
//   write : phi = -d inside, +d outside (at least the smallest positive subnormal of the dtype), NaN nodes and nodes without a
//           point unchanged.
// The closest-point extension (lsm_extend_closest_point) is a compile-time variant of pick / flood / write (TF, the dtype of F, not
// void; EXT in the flood): pick also interpolates F at the winning closest point, the flood carries that value with the point (as
// an (N+1)-th component of the point buffers), and write stores it into F, and the signed distance into phi when asked.  flag and
// the cell passes are shared as they are, so the points are the ones lsm_redistance computes.
// Cubic redistancing (lsm_redistance_cubic) runs lsm_redistance's kernels unchanged with one more between the last flood and the
// write:
//   refine: one thread per node; Newton on the KKT system of the closest point on the cubic interpolant (lsm_cubic.cuh), from the
//           node's linear closest point, into the spare point buffer; a node that falls back keeps the linear point and is counted.
// One launcher, launch_closest_points, enqueues all three: the extension's variant when RedistArgs::F is set, the refinement when
// RedistArgs::fallbacks is.  cubic_interp_kernel evaluates the same interpolant at arbitrary points for lsm_interpolate_cubic.
// The operation order of every distance, closest point and value is the one include/lsm_b200.h states; tests/redistance_ref.py and
// tests/extension_ref.py (and tests/cubic_ref.py for the cubic kernels) restate it in NumPy and agree with this file bit for bit (it
// is compiled with -fmad=false).
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>
#include <math_constants.h>
#include "lsm_kernels.h"
#include "lsm_simplex.cuh"
#include "lsm_cubic.cuh"

namespace lsm {
namespace {

constexpr int TPB = 256;
constexpr int CTPB = 128;      // threads of a cell block (redist_cells_kernel)

template <int N> __device__ __forceinline__ double dot(const double* a, const double* b) {
    double r = a[0] * b[0];
    for (int d = 1; d < N; ++d) r = r + a[d] * b[d];
    return r;
}

// sqrt(((x1 - p1)^2 + (x2 - p2)^2) + (x3 - p3)^2)
template <int N> __device__ __forceinline__ double dist(const double* x, const double* p) {
    double r = (x[0] - p[0]) * (x[0] - p[0]);
    for (int d = 1; d < N; ++d) r = r + (x[d] - p[d]) * (x[d] - p[d]);
    return sqrt(r);
}

// Where a closest point lies on its primitive, for the value of F there: vertex a, b or c; edge ab, ac or bc at parameter t from its
// first vertex; or the face at Ericson's (v, w) = (t, w).  Only the WHERE variants of the routines below report it.
enum : int { AT_A, AT_B, AT_C, ON_AB, ON_AC, ON_BC, ON_FACE };
struct Where { int at; double t, w; };

// closest point of segment [a, b] to x: t = clamp(dot(x - a, b - a) / dot(b - a, b - a), 0, 1); a when a == b.  WHERE: *W = (at_a)
// when a == b, else (on_ab, t).
template <int N, bool WHERE = false>
__device__ __forceinline__ void closest_seg(const double* x, const double* a, const double* b, double* q, Where* W = nullptr,
                                            int at_a = AT_A, int on_ab = ON_AB) {
    double ab[N], ax[N];
    bool same = true;
    for (int d = 0; d < N; ++d) { ab[d] = b[d] - a[d]; ax[d] = x[d] - a[d]; same = same && a[d] == b[d]; }
    if (same) {
        for (int d = 0; d < N; ++d) q[d] = a[d];
        if constexpr (WHERE) W->at = at_a;
        return;
    }
    double t = dot<N>(ax, ab) / dot<N>(ab, ab);
    t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t);
    for (int d = 0; d < N; ++d) q[d] = a[d] + t * ab[d];
    if constexpr (WHERE) { W->at = on_ab; W->t = t; }
}

// Ericson, Real-Time Collision Detection 5.1.5, ClosestPtPointTriangle, in its operation order.  Where the region's divisor is 0
// (a triangle made degenerate by exact zeros at nodes), the closest of the projections on ab, ac, bc, in that order.  WHERE: *W is
// the region and its parameters (for the fallback, those of the segment it picked).
template <bool WHERE = false>
__device__ __forceinline__ void closest_tri(const double* p, const double* a, const double* b, const double* c, double* q,
                                            Where* W = nullptr) {
    double ab[3], ac[3], ap[3], bp[3], cp[3];
    for (int d = 0; d < 3; ++d) { ab[d] = b[d] - a[d]; ac[d] = c[d] - a[d]; ap[d] = p[d] - a[d]; }
    const double d1 = dot<3>(ab, ap), d2 = dot<3>(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) {
        for (int d = 0; d < 3; ++d) q[d] = a[d];
        if constexpr (WHERE) W->at = AT_A;
        return;
    }
    for (int d = 0; d < 3; ++d) bp[d] = p[d] - b[d];
    const double d3 = dot<3>(ab, bp), d4 = dot<3>(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) {
        for (int d = 0; d < 3; ++d) q[d] = b[d];
        if constexpr (WHERE) W->at = AT_B;
        return;
    }
    const double vc = d1 * d4 - d3 * d2;
    bool degenerate = false;
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
        const double den = d1 - d3;
        if (den != 0.0) {
            const double v = d1 / den;
            for (int d = 0; d < 3; ++d) q[d] = a[d] + v * ab[d];
            if constexpr (WHERE) { W->at = ON_AB; W->t = v; }
            return;
        }
        degenerate = true;
    }
    if (!degenerate) {
        for (int d = 0; d < 3; ++d) cp[d] = p[d] - c[d];
        const double d5 = dot<3>(ab, cp), d6 = dot<3>(ac, cp);
        if (d6 >= 0.0 && d5 <= d6) {
            for (int d = 0; d < 3; ++d) q[d] = c[d];
            if constexpr (WHERE) W->at = AT_C;
            return;
        }
        const double vb = d5 * d2 - d1 * d6;
        if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
            const double den = d2 - d6;
            if (den != 0.0) {
                const double w = d2 / den;
                for (int d = 0; d < 3; ++d) q[d] = a[d] + w * ac[d];
                if constexpr (WHERE) { W->at = ON_AC; W->t = w; }
                return;
            }
            degenerate = true;
        }
        if (!degenerate) {
            const double va = d3 * d6 - d5 * d4;
            if (va <= 0.0 && (d4 - d3) >= 0.0 && (d5 - d6) >= 0.0) {
                const double den = (d4 - d3) + (d5 - d6);
                if (den != 0.0) {
                    const double w = (d4 - d3) / den;
                    for (int d = 0; d < 3; ++d) q[d] = b[d] + w * (c[d] - b[d]);
                    if constexpr (WHERE) { W->at = ON_BC; W->t = w; }
                    return;
                }
                degenerate = true;
            }
            if (!degenerate) {
                const double den = (va + vb) + vc;
                if (den != 0.0) {
                    const double denom = 1.0 / den, v = vb * denom, w = vc * denom;
                    for (int d = 0; d < 3; ++d) q[d] = (a[d] + ab[d] * v) + ac[d] * w;
                    if constexpr (WHERE) { W->at = ON_FACE; W->t = v; W->w = w; }
                    return;
                }
            }
        }
    }
    double s[3], best;
    Where Ws;
    closest_seg<3, WHERE>(p, a, b, q, W, AT_A, ON_AB);
    best = dist<3>(p, q);
    closest_seg<3, WHERE>(p, a, c, s, &Ws, AT_A, ON_AC);
    double ds = dist<3>(p, s);
    if (ds < best) {
        best = ds;
        for (int d = 0; d < 3; ++d) q[d] = s[d];
        if constexpr (WHERE) *W = Ws;
    }
    closest_seg<3, WHERE>(p, b, c, s, &Ws, AT_B, ON_BC);
    ds = dist<3>(p, s);
    if (ds < best) {
        for (int d = 0; d < 3; ++d) q[d] = s[d];
        if constexpr (WHERE) *W = Ws;
    }
}

// F at a closest point from the values f[j] at the primitive's vertices, in the form of its region (a constant F comes back exactly)
template <int N> __device__ __forceinline__ double value_at(const Where& W, const double* f) {
    if constexpr (N == 1) return f[0];
    else if constexpr (N == 2) return W.at == AT_A ? f[0] : f[0] + W.t * (f[1] - f[0]);
    else {
        switch (W.at) {
            case AT_A: return f[0];
            case AT_B: return f[1];
            case AT_C: return f[2];
            case ON_AB: return f[0] + W.t * (f[1] - f[0]);
            case ON_AC: return f[0] + W.t * (f[2] - f[0]);
            case ON_BC: return f[1] + W.t * (f[2] - f[1]);
            default: return (f[0] + (f[1] - f[0]) * W.t) + (f[2] - f[0]) * W.w;
        }
    }
}

__device__ __forceinline__ void node_coords(const IfaceArgs& A, const int* i, double* x) {
    for (int d = 0; d < 3; ++d) x[d] = A.lc[d] + double(i[d]) * A.h[d];
}

template <int N, bool WHERE = false>
__device__ __forceinline__ void closest(const double* x, const double (*V)[3], double* q, Where* W = nullptr) {
    if constexpr (N == 1) {
        q[0] = V[0][0];
        if constexpr (WHERE) W->at = AT_A;
    }
    else if constexpr (N == 2) closest_seg<2, WHERE>(x, V[0], V[1], q, W);
    else closest_tri<WHERE>(x, V[0], V[1], V[2], q, W);
}

constexpr unsigned long long NONE = ~0ull;                    // dmin / ord of a node outside every window
constexpr unsigned long long INF_BITS = 0x7ff0000000000000ull; // dmin of a band node whose candidates are all NaN

// every node: dmin = ord = NONE; a node whose cell holds a primitive appends the cell to the list
template <class T, int N>
__global__ void __launch_bounds__(TPB) redist_flag_kernel(const __grid_constant__ RedistArgs R) {
    const IfaceArgs& A = R.g;
    const long long idx = (long long)blockIdx.x * TPB + threadIdx.x;
    bool cut = false;
    if (idx < A.nodes) {
        int i[3];
        node_index(A, idx, i);
        cut = cell_prims<N>(classify<T, N>(A, idx, i)) > 0;
        R.dmin[idx] = NONE;
        R.ord[idx] = NONE;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, cut);
    if (!bal) return;
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(R.ncells, (unsigned long long)__popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (cut) R.list[base + __popc(bal & ((1u << lane) - 1u))] = idx;
}

// One block per cut cell (grid-stride over the list): the cell's primitives go to shared memory, then every node whose window holds
// the cell evaluates them.  pass 0: dmin = min over the node's candidates of the IEEE bits of dist (NaN as +inf);  pass 1: ord = the
// smallest (cell, primitive) order key among the candidates whose distance equals dmin.  Both are atomicMin, so the result does not
// depend on the order of the list: it is the first strictly closest candidate of the column-major scan the contract states.
template <class T, int N>
__global__ void __launch_bounds__(CTPB) redist_cells_kernel(const __grid_constant__ RedistArgs R, int pass) {
    constexpr int MAXP = N == 3 ? 12 : N == 2 ? 2 : 1;
    __shared__ double sV[MAXP][N][3];
    const IfaceArgs& A = R.g;
    const long long ncells = (long long)*R.ncells;
    const int W = 2 * R.band;
    int nwin = W;
    for (int d = 1; d < N; ++d) nwin *= W;
    for (long long t = blockIdx.x; t < ncells; t += gridDim.x) {
        const long long cidx = R.list[t];
        int c[3];
        node_index(A, cidx, c);
        double s[1 << N];
        const Masks M = cell_corners<T, N>(A, cidx, s);
        if (threadIdx.x < nsimplices<N>() && prims_of_simplex<N>(M, threadIdx.x)) {
            int off = 0;
            for (int q = 0; q < (int)threadIdx.x; ++q) off += prims_of_simplex<N>(M, q);
            simplex_vertices<N>(A, c, s, M, threadIdx.x, [&](const double (*V)[3]) {
                for (int j = 0; j < N; ++j) for (int d = 0; d < N; ++d) sV[off][j][d] = V[j][d];
                ++off;
            });
        }
        const int P = cell_prims<N>(M);
        __syncthreads();
        for (int r = threadIdx.x; r < nwin; r += CTPB) {
            int j[3] = {0, 0, 0}, rr = r;
            bool inbox = true;
            for (int d = 0; d < N; ++d) {
                j[d] = c[d] + (rr % W) - R.band + 1;
                rr /= W;
                inbox = inbox && j[d] >= 0 && j[d] < A.m[d];
            }
            if (!inbox) continue;
            const long long jdx = j[0] + j[1] * A.s1 + j[2] * A.s2;
            double x[3];
            node_coords(A, j, x);
            if (pass == 0) {
                unsigned long long best = INF_BITS;
                for (int k = 0; k < P; ++k) {
                    double q[3];
                    closest<N>(x, sV[k], q);
                    const double dq = dist<N>(x, q);
                    if (dq < CUDART_INF) { const unsigned long long b = __double_as_longlong(dq); best = b < best ? b : best; }
                }
                atomicMin(&R.dmin[jdx], best);
            } else {
                const unsigned long long dm = R.dmin[jdx];
                if (dm == INF_BITS) continue;
                for (int k = 0; k < P; ++k) {
                    double q[3];
                    closest<N>(x, sV[k], q);
                    const double dq = dist<N>(x, q);
                    if (dq < CUDART_INF && (unsigned long long)__double_as_longlong(dq) == dm) {
                        atomicMin(&R.ord[jdx], (unsigned long long)cidx * 16ull + (unsigned long long)k);
                        break;
                    }
                }
            }
        }
        __syncthreads();
    }
}

// every node: the closest point of the winning primitive (NaN when there is none) into pa, with the extension also the value of F
// there; counts the band nodes
template <class T, int N, class TF = void>
__global__ void __launch_bounds__(TPB) redist_pick_kernel(const __grid_constant__ RedistArgs R) {
    const IfaceArgs& A = R.g;
    const long long idx = (long long)blockIdx.x * TPB + threadIdx.x;
    bool band = false;
    if (idx < A.nodes) {
        band = R.dmin[idx] != NONE;
        const unsigned long long o = R.ord[idx];
        double P[3] = {CUDART_NAN, CUDART_NAN, CUDART_NAN};
        [[maybe_unused]] double val = CUDART_NAN;
        if (o != NONE) {
            const long long cidx = (long long)(o >> 4);
            int want = (int)(o & 15ull), c[3], i[3];
            node_index(A, cidx, c);
            node_index(A, idx, i);
            double s[1 << N], x[3];
            node_coords(A, i, x);
            const Masks M = cell_corners<T, N>(A, cidx, s);
            for (int p = 0; p < nsimplices<N>() && want >= 0; ++p) {
                if (!prims_of_simplex<N>(M, p)) continue;
                if constexpr (std::is_void_v<TF>) {
                    simplex_vertices<N>(A, c, s, M, p, [&](const double (*V)[3]) {
                        if (want-- == 0) closest<N>(x, V, P);
                    });
                } else {
                    const TF* F = static_cast<const TF*>(R.F);
                    simplex_vertices<N>(A, c, s, M, p, [&](const double (*V)[3], const double* Fv) {
                        if (want-- == 0) {
                            Where W;
                            closest<N, true>(x, V, P, &W);
                            val = value_at<N>(W, Fv);
                        }
                    }, [&](int k) { return double(F[cidx + corner_off(A, k)]); });
                }
            }
        }
        for (int d = 0; d < N; ++d) R.pa[d * A.nodes + idx] = P[d];
        if constexpr (!std::is_void_v<TF>) R.pa[N * A.nodes + idx] = val;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, band);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(R.count, (unsigned long long)__popc(bal));
}

// EXT: the value at the point (component N) goes with it; it is read once, from the winning candidate
template <int N, bool EXT = false>
__global__ void __launch_bounds__(TPB) redist_flood_kernel(const __grid_constant__ RedistArgs R, int k, const double* __restrict__ src,
                                                           double* __restrict__ dst) {
    const IfaceArgs& A = R.g;
    const long long idx = (long long)blockIdx.x * TPB + threadIdx.x;
    if (idx >= A.nodes) return;
    int i[3];
    node_index(A, idx, i);
    double x[3], P[3] = {CUDART_NAN, CUDART_NAN, CUDART_NAN}, best = CUDART_INF;
    [[maybe_unused]] long long from = -1;
    node_coords(A, i, x);
    auto consider = [&](long long j) {
        double q[3];
        q[0] = src[j];
        if (q[0] != q[0]) return;                 // no point
        for (int d = 1; d < N; ++d) q[d] = src[d * A.nodes + j];
        const double dq = dist<N>(x, q);
        if (dq < best) {
            best = dq;
            for (int d = 0; d < N; ++d) P[d] = q[d];
            if constexpr (EXT) from = j;
        }
    };
    consider(idx);
    const int r2 = N > 2 ? 1 : 0, r1 = N > 1 ? 1 : 0;
    for (int o2 = -r2; o2 <= r2; ++o2) {
        const int j2 = i[2] + o2 * k;
        if (j2 < 0 || j2 >= A.m[2]) continue;
        for (int o1 = -r1; o1 <= r1; ++o1) {
            const int j1 = i[1] + o1 * k;
            if (j1 < 0 || j1 >= A.m[1]) continue;
            for (int o0 = -1; o0 <= 1; ++o0) {
                const int j0 = i[0] + o0 * k;
                if ((o0 | o1 | o2) == 0 || j0 < 0 || j0 >= A.m[0]) continue;
                consider(j0 + j1 * A.s1 + j2 * A.s2);
            }
        }
    }
    for (int d = 0; d < N; ++d) dst[d * A.nodes + idx] = P[d];
    if constexpr (EXT) dst[N * A.nodes + idx] = from >= 0 ? src[N * A.nodes + from] : CUDART_NAN;
}

template <class T> __device__ __forceinline__ T smallest_subnormal();
template <> __device__ __forceinline__ float smallest_subnormal<float>() { return 1.40129846e-45f; }
template <> __device__ __forceinline__ double smallest_subnormal<double>() { return 4.9406564584124654e-324; }

// with the extension (TF not void) F = the value at the point, rounded to TF, on the same nodes; phi only when R.write_phi
template <class T, int N, class TF = void>
__global__ void __launch_bounds__(TPB) redist_write_kernel(const __grid_constant__ RedistArgs R,
                                                           const double* __restrict__ pts) {
    const IfaceArgs& A = R.g;
    const long long idx = (long long)blockIdx.x * TPB + threadIdx.x;
    if (idx >= A.nodes) return;
    T* phi = static_cast<T*>(const_cast<void*>(A.phi));
    const double s = double(phi[idx]);
    double q[3];
    q[0] = pts[idx];
    if (s != s || q[0] != q[0]) return;           // NaN node, or no interface at all
    if constexpr (!std::is_void_v<TF>) {
        static_cast<TF*>(R.F)[idx] = TF(pts[N * A.nodes + idx]);
        if (!R.write_phi) return;
    }
    for (int d = 1; d < N; ++d) q[d] = pts[d * A.nodes + idx];
    int i[3];
    node_index(A, idx, i);
    double x[3];
    node_coords(A, i, x);
    const double dq = dist<N>(x, q);
    if (s <= 0.0) { phi[idx] = T(-dq); return; }
    T v = T(dq);
    if (v == T(0)) v = smallest_subnormal<T>();   // an outside node stays outside
    phi[idx] = v;
}

// ---- lsm_redistance_cubic: Newton refinement of the closest points on the cubic interpolant (lsm_cubic.cuh) -------------------
constexpr int NEWTON_ITERS = 20;

__device__ __forceinline__ bool finite(double v) { return fabs(v) < CUDART_INF; }

// Solves M z = r, M (K x K), by Gaussian elimination with partial pivoting (the first row of largest |entry| wins; columns left to
// right; then back substitution).  Rows are swapped with compile-time indices only, so M stays in registers.  false on a zero pivot.
template <int K> __device__ __forceinline__ bool solve(double (*M)[K], double* r, double* z) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
        int p = k;
        double big = fabs(M[k][k]);
#pragma unroll
        for (int i = k + 1; i < K; ++i) if (fabs(M[i][k]) > big) { big = fabs(M[i][k]); p = i; }
        if (big == 0.0) return false;
#pragma unroll
        for (int i = k + 1; i < K; ++i) {
            if (i == p) {
#pragma unroll
                for (int j = k; j < K; ++j) { const double t = M[k][j]; M[k][j] = M[i][j]; M[i][j] = t; }
                const double t = r[k]; r[k] = r[i]; r[i] = t;
            }
        }
#pragma unroll
        for (int i = k + 1; i < K; ++i) {
            const double f = M[i][k] / M[k][k];
#pragma unroll
            for (int j = k + 1; j < K; ++j) M[i][j] = M[i][j] - f * M[k][j];
            r[i] = r[i] - f * r[k];
        }
    }
#pragma unroll
    for (int i = K - 1; i >= 0; --i) {
        double s = r[i];
#pragma unroll
        for (int j = i + 1; j < K; ++j) s = s - M[i][j] * z[j];
        z[i] = s / M[i][i];
    }
    return true;
}

// Newton on the KKT system of min |y - x| subject to P(y) = 0, from the linear closest point y0 (include/lsm_b200.h states the
// iteration).  Returns true with the refined point in y, or false (fall back to y0).
template <class T, int N>
__device__ __forceinline__ bool newton(const IfaceArgs& A, const double* x, const double* y0, double* y) {
    double P, g[N], H[3][3];
    cubic::eval<T, N, 1>(A, y0, P, g, H);
    const double gg = dot<N>(g, g);
    if (!finite(gg) || gg == 0.0) return false;
    double xy[N];
    for (int d = 0; d < N; ++d) { xy[d] = x[d] - y0[d]; y[d] = y0[d]; }
    double lam = dot<N>(xy, g) / gg;
    if (!finite(lam)) return false;
    double hmin = fabs(A.h[0]), hmax = fabs(A.h[0]);
    for (int d = 1; d < N; ++d) { hmin = fmin(hmin, fabs(A.h[d])); hmax = fmax(hmax, fabs(A.h[d])); }
    const double tol = 1e-10 * hmin, reach = 2.0 * hmax;
    for (int it = 0; it < NEWTON_ITERS; ++it) {
        if (!cubic::eval<T, N, 2>(A, y, P, g, H)) return false;
        bool fin = finite(P);
        double M[N + 1][N + 1], r[N + 1], z[N + 1];
#pragma unroll
        for (int i = 0; i < N; ++i) {
#pragma unroll
            for (int j = 0; j < N; ++j) { M[i][j] = i == j ? 1.0 + lam * H[i][j] : lam * H[i][j]; fin = fin && finite(H[i][j]); }
            M[i][N] = g[i];
            M[N][i] = g[i];
            r[i] = -((y[i] - x[i]) + lam * g[i]);
            fin = fin && finite(g[i]);
        }
        M[N][N] = 0.0;
        r[N] = -P;
        if (!fin) return false;
        if (!solve<N + 1>(M, r, z)) return false;
        bool zf = true;
        for (int d = 0; d <= N; ++d) zf = zf && finite(z[d]);
        if (!zf) return false;
        for (int d = 0; d < N; ++d) y[d] = y[d] + z[d];
        lam = lam + z[N];
        bool ok = finite(lam);
        for (int d = 0; d < N; ++d) {
            const double u = (y[d] - A.lc[d]) / A.h[d];
            ok = ok && finite(y[d]) && u >= 0.0 && u <= double(A.m[d] - 1);
        }
        if (!ok || dist<N>(y, y0) > reach) return false;
        const double zero[N] = {};
        if (dist<N>(z, zero) <= tol) return true;
    }
    return false;
}

// every node: the refined closest point from the linear one in src (NaN = no point) into dst; a NaN node keeps its point (the write
// pass leaves it alone).  Counts the nodes that fall back to the linear point.
template <class T, int N>
__global__ void __launch_bounds__(TPB) redist_refine_kernel(const __grid_constant__ RedistArgs R, const double* __restrict__ src,
                                                            double* __restrict__ dst, unsigned long long* fallbacks) {
    const IfaceArgs& A = R.g;
    const long long idx = (long long)blockIdx.x * TPB + threadIdx.x;
    bool fell = false;
    if (idx < A.nodes) {
        double y0[N], y[N];
        for (int d = 0; d < N; ++d) y0[d] = src[d * A.nodes + idx];
        const double s = double(static_cast<const T*>(A.phi)[idx]);
        if (y0[0] == y0[0] && s == s) {
            int i[3];
            node_index(A, idx, i);
            double x[3];
            node_coords(A, i, x);
            fell = !newton<T, N>(A, x, y0, y);
            if (fell) for (int d = 0; d < N; ++d) y[d] = y0[d];
        } else {
            for (int d = 0; d < N; ++d) y[d] = y0[d];
        }
        for (int d = 0; d < N; ++d) dst[d * A.nodes + idx] = y[d];
    }
    const unsigned bal = __ballot_sync(0xffffffffu, fell);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(fallbacks, (unsigned long long)__popc(bal));
}

// lsm_interpolate_cubic: one thread per point; pts AoS (npts x N), outputs AoS and optional
template <class T, int N>
__global__ void __launch_bounds__(TPB) cubic_interp_kernel(const __grid_constant__ IfaceArgs A, long long npts,
                                                           const double* __restrict__ pts, double* val, double* grad, double* hess) {
    const long long p = (long long)blockIdx.x * TPB + threadIdx.x;
    if (p >= npts) return;
    double y[N], P, g[N], H[3][3];
    for (int d = 0; d < N; ++d) y[d] = pts[p * N + d];
    cubic::eval<T, N, 2>(A, y, P, g, H);
    if (val) val[p] = P;
    if (grad) for (int d = 0; d < N; ++d) grad[p * N + d] = g[d];
    if (hess) for (int d = 0; d < N; ++d) for (int e = 0; e < N; ++e) hess[(p * N + d) * N + e] = H[d][e];
}

template <class T, int N, class TF>
cudaError_t launch_n(const RedistArgs& R, int cell_blocks, cudaStream_t s, int* launches) {
    constexpr bool EXT = !std::is_void_v<TF>;
    const unsigned grid = (unsigned)((R.g.nodes + TPB - 1) / TPB);
    redist_flag_kernel<T, N><<<grid, TPB, 0, s>>>(R);
    for (int pass = 0; pass < 2; ++pass) redist_cells_kernel<T, N><<<cell_blocks, CTPB, 0, s>>>(R, pass);
    redist_pick_kernel<T, N, TF><<<grid, TPB, 0, s>>>(R);
    *launches = 4;
    int maxn = 1, L = 0;
    for (int d = 0; d < N; ++d) maxn = R.g.m[d] > maxn ? R.g.m[d] : maxn;
    while ((1 << L) < maxn) ++L;
    double *src = R.pa, *dst = R.pb;
    for (int k = 1 << (L - 1); ; k >>= 1) {
        const int kk = k > 0 ? k : 1;             // k = 2^(L-1), ..., 2, 1, then one more pass with k = 1
        redist_flood_kernel<N, EXT><<<grid, TPB, 0, s>>>(R, kk, src, dst);
        ++*launches;
        double* t = src; src = dst; dst = t;
        if (k == 0) break;
    }
    if constexpr (!EXT) {
        if (R.fallbacks) {                        // the cubic refinement: the spare point buffer takes the refined points
            redist_refine_kernel<T, N><<<grid, TPB, 0, s>>>(R, src, dst, R.fallbacks);
            ++*launches;
            src = dst;
        }
    }
    redist_write_kernel<T, N, TF><<<grid, TPB, 0, s>>>(R, src);
    ++*launches;
    return cudaGetLastError();
}

template <class T, class TF>
cudaError_t launch_t(const RedistArgs& R, int cell_blocks, cudaStream_t s, int* launches) {
    switch (R.g.ndim) {
        case 1: return launch_n<T, 1, TF>(R, cell_blocks, s, launches);
        case 2: return launch_n<T, 2, TF>(R, cell_blocks, s, launches);
        default: return launch_n<T, 3, TF>(R, cell_blocks, s, launches);
    }
}

template <class TF>
cudaError_t launch_tf(const RedistArgs& R, int cell_blocks, cudaStream_t s, int* launches) {
    return R.g.f64 ? launch_t<double, TF>(R, cell_blocks, s, launches) : launch_t<float, TF>(R, cell_blocks, s, launches);
}

template <class T>
cudaError_t launch_interp_t(const IfaceArgs& A, long long npts, const double* pts, double* val, double* grad, double* hess,
                            cudaStream_t s) {
    const unsigned grid = (unsigned)((npts + TPB - 1) / TPB);
    switch (A.ndim) {
        case 1: cubic_interp_kernel<T, 1><<<grid, TPB, 0, s>>>(A, npts, pts, val, grad, hess); break;
        case 2: cubic_interp_kernel<T, 2><<<grid, TPB, 0, s>>>(A, npts, pts, val, grad, hess); break;
        default: cubic_interp_kernel<T, 3><<<grid, TPB, 0, s>>>(A, npts, pts, val, grad, hess); break;
    }
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_closest_points(const RedistArgs& R, int sm_count, cudaStream_t s, int* launches) {
    if (!R.F) return launch_tf<void>(R, sm_count * 16, s, launches);
    return R.F_f64 ? launch_tf<double>(R, sm_count * 16, s, launches) : launch_tf<float>(R, sm_count * 16, s, launches);
}

cudaError_t launch_interp_cubic(const IfaceArgs& A, long long npts, const double* pts, double* val, double* grad, double* hess,
                                cudaStream_t s) {
    if (npts <= 0) return cudaSuccess;
    return A.f64 ? launch_interp_t<double>(A, npts, pts, val, grad, hess, s) : launch_interp_t<float>(A, npts, pts, val, grad, hess, s);
}

}  // namespace lsm
