// lsm_semi_implicit.cu — the inflow-implicit / outflow-explicit step of one AdvectionTerm (LSM_SEMI_IMPLICIT), compiled with
// -fmad=false so that the temporally blocked sweeps and the one-sweep-per-launch reference form agree bit for bit.
//
// The scheme (phi_t + u.grad phi = 0 at the nodes, step dt from tc; DESIGN.md §4.6).  The velocity is taken at t* = tc + dt/2.
// For each node I and dimension d:  c_d = dt u_d(I, t*) / h_d,  a_d = |c_d| / 2,  s_d = +1 if c_d > 0 else -1 (a zero or NaN
// velocity takes the -1 branch).  The inflow half is implicit, the outflow half explicit:
//     (1 + sum_d a_d) x_I - sum_d a_d x_{I - s_d e_d}  =  r_I  =  phi_I - sum_d a_d (phi_{I + s_d e_d} - phi_I)
// sums left to right over d.  Off-grid reads on both sides go through the boundary condition's index map (periodic with the
// reference's n == 1 wrap, Neumann = ExtrapolationBC{0}, symmetry): every ghost weight is 1, so the matrix is a diagonally dominant
// M-matrix.  It is solved by Jacobi sweeps from x = r:
//     x_I <- (r_I + sum_d a_d x_{I - s_d e_d}) / (1 + sum_d a_d)
// Each sweep contracts the max-norm error by q = (C/2) / (1 + C/2), C = max_I sum_d |c_d|; the host fixes the number of sweeps
// from q in advance (lsm_semi_implicit_sweeps), so a step has no reduction, no copy to the host and no synchronisation.
// Float32 states: differences of stored values in float, everything else in double, rounded to float on every store (r and
// every iterate), the same in both sweep forms.
#include <algorithm>
#include "lsm_dev.cuh"
#include "lsm_kernels.h"

namespace lsm {
namespace {

// the in-grid node that stands for index j (j = -1 .. n) along an axis of n >= 2 nodes
__device__ __forceinline__ int si_map(int j, int n, const BCDev* bc) {
    if (j >= 0 && j < n) return j;
    const int k = bc[j < 0 ? 0 : 1].kind;
    if (k == BC_PERIODIC) return j < 0 ? (n - 1) + j : 1 + j - n;      // boundaryconditions.jl:107-119: node n duplicates node 1
    if (k == BC_SYMMETRY) return j < 0 ? -j : 2 * (n - 1) - j;         // boundaryconditions.jl:146-153
    return j < 0 ? 0 : n - 1;                                           // ExtrapolationBC{0}
}

// b_d = c_d / 2, so that a_d = |b_d| and s_d = b_d > 0 ? +1 : -1
template <class T, int N>
__device__ __forceinline__ void si_half_courant(const SemiArgs<T>& A, long node, const int* i, double* b) {
#pragma unroll
    for (int d = 0; d < N; ++d) b[d] = ((A.dt * coef_comp<T>(A.u, node, d, i[0], i[1], i[2], N)) / A.h[d]) * 0.5;
}

// one Jacobi update of a node from the iterate values xn of its inflow neighbours
template <int N>
__device__ __forceinline__ double si_update(double r, const double* b, const double* xn) {
    double s = fabs(b[0]) * xn[0], a = fabs(b[0]);
#pragma unroll
    for (int d = 1; d < N; ++d) { s = s + fabs(b[d]) * xn[d]; a = a + fabs(b[d]); }
    return (r + s) / (1.0 + a);
}

__device__ __forceinline__ void si_coords(long l, const int* n, int* i) {
    i[0] = (int)(l % n[0]);
    const long q = l / n[0];
    i[1] = (int)(q % n[1]);
    i[2] = (int)(q / n[1]);
}

template <class T> __device__ __forceinline__ long si_stride(const View<T>& v, int d) { return d == 0 ? 1L : (d == 1 ? v.s1 : v.s2); }

template <class T, int N>
__global__ void si_rhs_kernel(SemiArgs<T> A, T* r) {
    const long total = (long)A.x.n[0] * A.x.n[1] * A.x.n[2];
    for (long l = blockIdx.x * (long)blockDim.x + threadIdx.x; l < total; l += (long)gridDim.x * blockDim.x) {
        int i[3];
        si_coords(l, A.x.n, i);
        const T p = A.phi[l];
        double s = 0.0;
#pragma unroll
        for (int d = 0; d < N; ++d) {      // b_d one dimension at a time: an array of all N kept 3-D spilling 32 bytes
            const double b = ((A.dt * coef_comp<T>(A.u, l, d, i[0], i[1], i[2], N)) / A.h[d]) * 0.5;     // as si_half_courant
            const int j = si_map(i[d] + (b > 0 ? 1 : -1), A.x.n[d], A.x.bc[d]);
            const T df = A.phi[l + (long)(j - i[d]) * si_stride(A.x, d)] - p;
            const double t = fabs(b) * double(df);
            s = d == 0 ? t : s + t;
        }
        r[l] = T(double(p) - s);
    }
}

// one sweep per launch, every read from global memory (the default: faster than the blocked form on a B200, DESIGN.md §4.6)
template <class T, int N>
__global__ void __launch_bounds__(256) si_sweep_kernel(SemiArgs<T> A, const T* x, T* out) {
    const long total = (long)A.x.n[0] * A.x.n[1] * A.x.n[2];
    for (long l = blockIdx.x * (long)blockDim.x + threadIdx.x; l < total; l += (long)gridDim.x * blockDim.x) {
        int i[3];
        si_coords(l, A.x.n, i);
        double b[N], xn[N];
        si_half_courant<T, N>(A, l, i, b);
#pragma unroll
        for (int d = 0; d < N; ++d) {
            const int j = si_map(i[d] - (b[d] > 0 ? 1 : -1), A.x.n[d], A.x.bc[d]);
            xn[d] = double(x[l + (long)(j - i[d]) * si_stride(A.x, d)]);
        }
        out[l] = T(si_update<N>(double(A.r[l]), b, xn));
    }
}

// ---- temporally blocked sweeps (LSM_OPT_KERNEL = 2) ----------------------------------------------------------------------
// A block owns a tile of B_d nodes per axis and runs up to M sweeps on a region around it in shared memory.  A node's value after
// k sweeps depends only on nodes within k inflow hops, so the region holds, per axis, every node within M hops of the tile:
//   * the main interval [t0 - M, t0 + B + M) clipped to the grid;
//   * on a periodic axis whose main interval was clipped, the nodes the wrap reaches: [n - 1 - M, n) at the low end, [0, M + 1)
//     at the high end;
//   * the whole axis when it is short (n <= B + 3M: then the two parts would overlap).
// A region node whose inflow neighbour lies outside the region reads its own value instead, so it is wrong from the first sweep on.
// The missing neighbour is at least M + 1 hops from the tile (the edge node itself can be exactly M hops away), and a wrong value
// moves one hop per sweep, so within M sweeps it never reaches the tile.  After the sweeps the tile's nodes are exactly the
// one-sweep form's.
struct SiAxis { int a, b, w0, w1, len; };

__device__ __forceinline__ SiAxis si_axis(int t0, int B, int M, int n, const BCDev* bc) {
    SiAxis X{0, n, 0, 0, n};
    if (n <= B + 3 * M) return X;
    X.a = max(0, t0 - M); X.b = min(n, t0 + B + M);
    if (bc[0].kind == BC_PERIODIC) {
        if (t0 - M < 0) { X.w0 = n - 1 - M; X.w1 = n; }
        else if (t0 + B + M > n) { X.w0 = 0; X.w1 = M + 1; }
    }
    X.len = (X.b - X.a) + (X.w1 - X.w0);
    return X;
}
__device__ __forceinline__ int si_node(const SiAxis& X, int q) { return q < X.b - X.a ? X.a + q : X.w0 + (q - (X.b - X.a)); }
__device__ __forceinline__ int si_pos(const SiAxis& X, int j) {
    if (j >= X.a && j < X.b) return j - X.a;
    if (j >= X.w0 && j < X.w1) return (X.b - X.a) + (j - X.w0);
    return -1;
}

template <int N, int B0, int B1, int B2, int M> struct SiTile {
    static constexpr int L0 = B0 + 3 * M, L1 = N > 1 ? B1 + 3 * M : 1, L2 = N > 2 ? B2 + 3 * M : 1;
    static constexpr int P = L0 * L1 * L2;      // region nodes at most
};

template <class T, int N, int B0, int B1, int B2, int M, int THREADS>
__global__ void __launch_bounds__(THREADS) si_block_kernel(SemiArgs<T> A, const T* x, T* out, int sweeps) {
    using Tile = SiTile<N, B0, B1, B2, M>;
    constexpr int PPT = (Tile::P + THREADS - 1) / THREADS;
    extern __shared__ __align__(16) unsigned char si_smem[];
    T* buf = reinterpret_cast<T*>(si_smem);      // two region-sized iterate buffers
    const int Bd[3] = {B0, B1, B2};
    const int t0[3] = {(int)blockIdx.x * B0, (int)blockIdx.y * B1, (int)blockIdx.z * B2};
    SiAxis X[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) X[d] = d < N ? si_axis(t0[d], Bd[d], M, A.x.n[d], A.x.bc[d]) : SiAxis{0, 1, 0, 0, 1};
    const int P = X[0].len * X[1].len * X[2].len;
    const int Ls[3] = {1, X[0].len, X[0].len * X[1].len};

    double rr[PPT], bb[PPT][N];
    int nb[PPT][N];
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        const int p = threadIdx.x + k * THREADS;
        if (p >= P) continue;
        const int q[3] = {p % X[0].len, (p / X[0].len) % X[1].len, p / Ls[2]};
        int i[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) i[d] = si_node(X[d], q[d]);
        const long l = i[0] + i[1] * A.x.s1 + i[2] * A.x.s2;
        si_half_courant<T, N>(A, l, i, bb[k]);
        rr[k] = double(A.r[l]);
        buf[p] = x[l];
#pragma unroll
        for (int d = 0; d < N; ++d) {
            const int qd = si_pos(X[d], si_map(i[d] - (bb[k][d] > 0 ? 1 : -1), A.x.n[d], A.x.bc[d]));
            nb[k][d] = qd < 0 ? p : p + (qd - q[d]) * Ls[d];
        }
    }
    for (int it = 0; it < sweeps; ++it) {
        __syncthreads();
        const T* src = buf + (it & 1) * Tile::P;
        T* dst = buf + ((it + 1) & 1) * Tile::P;
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            const int p = threadIdx.x + k * THREADS;
            if (p >= P) continue;
            double xn[N];
#pragma unroll
            for (int d = 0; d < N; ++d) xn[d] = double(src[nb[k][d]]);
            dst[p] = T(si_update<N>(rr[k], bb[k], xn));
        }
    }
    __syncthreads();
    const T* fin = buf + (sweeps & 1) * Tile::P;
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        const int p = threadIdx.x + k * THREADS;
        if (p >= P) continue;
        const int q[3] = {p % X[0].len, (p / X[0].len) % X[1].len, p / Ls[2]};
        bool inner = true;
        int i[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            i[d] = si_node(X[d], q[d]);
            inner = inner && q[d] < X[d].b - X[d].a && (d >= N || (i[d] >= t0[d] && i[d] < t0[d] + Bd[d]));
        }
        if (inner) out[i[0] + i[1] * A.x.s1 + i[2] * A.x.s2] = fin[p];
    }
}

// tile shapes and sweeps per launch: 1-D 2048 nodes / 16 sweeps, 2-D 32 x 32 / 8, 3-D 8 x 8 x 8 / 2
template <int N> struct SiShape;
template <> struct SiShape<1> { static constexpr int B0 = 2048, B1 = 1, B2 = 1, M = 16, THREADS = 512; };
template <> struct SiShape<2> { static constexpr int B0 = 32, B1 = 32, B2 = 1, M = 8, THREADS = 512; };
template <> struct SiShape<3> { static constexpr int B0 = 8, B1 = 8, B2 = 8, M = 2, THREADS = 512; };

int si_grid(long total) { return (int)std::min<long>((total + 255) / 256, 148L * 16); }

template <class T, int N>
cudaError_t si_sweeps_n(const SemiArgs<T>& A, int k, bool blocked, T* xa, T* xb, cudaStream_t s, int* launches) {
    using S = SiShape<N>;
    using Tile = SiTile<N, S::B0, S::B1, S::B2, S::M>;
    const long total = (long)A.x.n[0] * A.x.n[1] * A.x.n[2];
    const int per = blocked ? S::M : 1;
    const int L = (k + per - 1) / per;
    const size_t smem = 2 * sizeof(T) * Tile::P;
    auto kern = si_block_kernel<T, N, S::B0, S::B1, S::B2, S::M, S::THREADS>;
    if (blocked) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const dim3 grid((A.x.n[0] + S::B0 - 1) / S::B0, N > 1 ? (A.x.n[1] + S::B1 - 1) / S::B1 : 1, N > 2 ? (A.x.n[2] + S::B2 - 1) / S::B2 : 1);
    const T* in = A.r;                             // x^0 = r
    for (int j = 0; j < L; ++j) {
        T* o = (L - 1 - j) % 2 == 0 ? xa : xb;    // the last launch writes xa
        if (blocked) kern<<<grid, S::THREADS, smem, s>>>(A, in, o, std::min(per, k - j * per));
        else si_sweep_kernel<T, N><<<si_grid(total), 256, 0, s>>>(A, in, o);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        ++*launches;
        in = o;
    }
    return cudaSuccess;
}

}  // namespace

template <class T>
cudaError_t launch_si_rhs(int ndim, const SemiArgs<T>& A, T* r, cudaStream_t s) {
    const long total = (long)A.x.n[0] * A.x.n[1] * A.x.n[2];
    const int g = si_grid(total);
    if (ndim == 1) si_rhs_kernel<T, 1><<<g, 256, 0, s>>>(A, r);
    else if (ndim == 2) si_rhs_kernel<T, 2><<<g, 256, 0, s>>>(A, r);
    else si_rhs_kernel<T, 3><<<g, 256, 0, s>>>(A, r);
    return cudaGetLastError();
}

template <class T>
cudaError_t launch_si_sweeps(int ndim, const SemiArgs<T>& A, int k, bool blocked, T* xa, T* xb, cudaStream_t s, int* launches) {
    *launches = 0;
    if (ndim == 1) return si_sweeps_n<T, 1>(A, k, blocked, xa, xb, s, launches);
    if (ndim == 2) return si_sweeps_n<T, 2>(A, k, blocked, xa, xb, s, launches);
    return si_sweeps_n<T, 3>(A, k, blocked, xa, xb, s, launches);
}

template cudaError_t launch_si_rhs<float>(int, const SemiArgs<float>&, float*, cudaStream_t);
template cudaError_t launch_si_rhs<double>(int, const SemiArgs<double>&, double*, cudaStream_t);
template cudaError_t launch_si_sweeps<float>(int, const SemiArgs<float>&, int, bool, float*, float*, cudaStream_t, int*);
template cudaError_t launch_si_sweeps<double>(int, const SemiArgs<double>&, int, bool, double*, double*, cudaStream_t, int*);

}  // namespace lsm
