// lsm_semi_implicit.cu — the inflow-implicit / outflow-explicit step of one AdvectionTerm (LSM_SEMI_IMPLICIT), compiled with
// -fmad=false: every product and sum is rounded on its own, as in the SciPy restatement the step is checked against
// (tests/semi_implicit_ref.py), so that contracting them into FMAs cannot change the checked results.
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
// every iterate).
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

// one sweep per launch, every read from global memory (faster on a B200 than sweeps blocked in shared memory, DESIGN.md §4.6)
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

int si_grid(long total) { return (int)std::min<long>((total + 255) / 256, 148L * 16); }

template <class T, int N>
cudaError_t si_sweeps_n(const SemiArgs<T>& A, int k, T* xa, T* xb, cudaStream_t s, int* launches) {
    const long total = (long)A.x.n[0] * A.x.n[1] * A.x.n[2];
    const T* in = A.r;                             // x^0 = r
    for (int j = 0; j < k; ++j) {
        T* o = (k - 1 - j) % 2 == 0 ? xa : xb;    // the last launch writes xa
        si_sweep_kernel<T, N><<<si_grid(total), 256, 0, s>>>(A, in, o);
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
cudaError_t launch_si_sweeps(int ndim, const SemiArgs<T>& A, int k, T* xa, T* xb, cudaStream_t s, int* launches) {
    *launches = 0;
    if (ndim == 1) return si_sweeps_n<T, 1>(A, k, xa, xb, s, launches);
    if (ndim == 2) return si_sweeps_n<T, 2>(A, k, xa, xb, s, launches);
    return si_sweeps_n<T, 3>(A, k, xa, xb, s, launches);
}

template cudaError_t launch_si_rhs<float>(int, const SemiArgs<float>&, float*, cudaStream_t);
template cudaError_t launch_si_rhs<double>(int, const SemiArgs<double>&, double*, cudaStream_t);
template cudaError_t launch_si_sweeps<float>(int, const SemiArgs<float>&, int, float*, float*, cudaStream_t, int*);
template cudaError_t launch_si_sweeps<double>(int, const SemiArgs<double>&, int, double*, double*, cudaStream_t, int*);

}  // namespace lsm
