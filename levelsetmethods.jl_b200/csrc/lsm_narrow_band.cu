// lsm_narrow_band.cu — the brick band of lsm_field_set_band (include/lsm_b200.h, DESIGN.md §4.7).
//
// A field is cut into bricks of BRICK_X x BRICK_Y x BRICK_Z nodes (2-D: BRICK_X x BRICK_Y), numbered column-major.  A brick is
// CORE when it holds a node with !(|phi| > gamma); ACTIVE when a core brick lies in its neighbourhood N(b); SHELL when it lies in
// N(a) of an active brick a without being active.  N(b) is the product over axes of R_d(b_d) = {b-1, b, b+1} in range, plus on a
// periodic axis the wrap partners of the reference's periodic rule (node n duplicates node 1, boundaryconditions.jl:107-119):
// the brick holding nodes 0..2 adds the bricks holding nodes n-4..n-2, a brick holding one of nodes n-3..n-1 adds the brick
// holding nodes 1..3.  Every brick is at least 16 nodes wide, so no stencil read (reach 3) of a brick's nodes leaves N(b).
//
// Everything stays on the device: the core flags (a full pass, or a pass over the previous active list), the dilation into one
// state byte per brick, an ordered compaction into the active and shell lists ({count, brick, ...}, ascending) and the copies of
// listed bricks between fields.  Kernels over a list are launched for every brick of the box and the surplus blocks exit at once,
// so the host never reads a count.
#include "lsm_kernels.h"

namespace lsm {

namespace {

constexpr int CB = 256;          // threads per block of the per-brick kernels
constexpr int CT = 1024;         // threads of the one-block compaction

struct BrickGeom {
    int n[3], nb[3], B[3];
    __device__ void origin(int b, int* o) const {
        o[0] = (b % nb[0]) * B[0]; o[1] = ((b / nb[0]) % nb[1]) * B[1]; o[2] = (b / (nb[0] * nb[1])) * B[2];
    }
    __device__ int nodes() const { return B[0] * B[1] * B[2]; }
};

BrickGeom geom(const BandArgs& A) {
    BrickGeom g;
    const int B[3] = {BRICK_X, BRICK_Y, A.ndim == 3 ? BRICK_Z : 1};
    for (int d = 0; d < 3; ++d) { g.n[d] = A.n[d]; g.B[d] = B[d]; g.nb[d] = (A.n[d] + B[d] - 1) / B[d]; }
    return g;
}

// R_d(b) (inverse = false) or {b' : b in R_d(b')} (inverse = true) on an axis of n nodes, nb bricks of B nodes; returns the count
__device__ int axis_set(int b, int n, int nb, int B, bool periodic, bool inverse, int* out) {
    int c = 0;
    auto add = [&](int k) {
        for (int i = 0; i < c; ++i) if (out[i] == k) return;
        out[c++] = k;
    };
    for (int k = b - 1; k <= b + 1; ++k) if (k >= 0 && k < nb) add(k);
    if (periodic) {
        const int lo_a = max(n - 4, 0) / B, lo_b = max(n - 2, 0) / B;     // the bricks holding nodes n-4..n-2
        const int hi_a = max(n - 3, 0) / B, hi_b = (n - 1) / B;           // the bricks holding nodes n-3..n-1
        // brick 0 holds nodes 0..2 and 1..3
        if (!inverse) {
            if (b == 0) { add(lo_a); add(lo_b); }
            if (b == hi_a || b == hi_b) add(0);
        } else {
            if (b == lo_a || b == lo_b) add(0);
            if (b == 0) { add(hi_a); add(hi_b); }
        }
    }
    return c;
}

template <class T>
__global__ void __launch_bounds__(CB) band_core_kernel(const T* __restrict__ phi, const BrickGeom g, const double gamma,
                                                       const int* __restrict__ list, uint8_t* __restrict__ core) {
    int b = blockIdx.x;
    if (list) {
        if ((int)blockIdx.x >= list[0]) return;
        b = list[1 + blockIdx.x];
    }
    int o[3];
    g.origin(b, o);
    bool hit = false;
    for (int q = threadIdx.x; q < g.nodes(); q += CB) {
        const int i0 = o[0] + q % g.B[0], i1 = o[1] + (q / g.B[0]) % g.B[1], i2 = o[2] + q / (g.B[0] * g.B[1]);
        if (i0 < g.n[0] && i1 < g.n[1] && i2 < g.n[2])
            hit |= !(fabs(double(phi[(long)i0 + (long)g.n[0] * ((long)i1 + (long)g.n[1] * i2)])) > gamma);
    }
    hit = __syncthreads_or(hit);
    if (threadIdx.x == 0) core[b] = hit ? 1 : 0;
}

// state = 2 | core when a core brick lies in N(b), else 0
__global__ void band_active_kernel(const BrickGeom g, const int3 per, const uint8_t* __restrict__ core, uint8_t* __restrict__ state) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= g.nb[0] * g.nb[1] * g.nb[2]) return;
    const int c[3] = {b % g.nb[0], (b / g.nb[0]) % g.nb[1], b / (g.nb[0] * g.nb[1])};
    const int pd[3] = {per.x, per.y, per.z};
    int r[3][5], m[3];
    for (int d = 0; d < 3; ++d) m[d] = axis_set(c[d], g.n[d], g.nb[d], g.B[d], pd[d], false, r[d]);
    bool act = false;
    for (int z = 0; z < m[2] && !act; ++z)
        for (int y = 0; y < m[1] && !act; ++y)
            for (int x = 0; x < m[0] && !act; ++x) act = core[r[0][x] + g.nb[0] * (r[1][y] + g.nb[1] * r[2][z])] != 0;
    state[b] = act ? (uint8_t)(2 | core[b]) : (uint8_t)0;
}

// state = 1 for a brick that is not active but lies in N(a) of an active brick a.  Other threads may turn a state 0 into 1 while
// this one reads it; only bit 1 (active) is read, and no thread of this kernel changes it.
__global__ void band_shell_kernel(const BrickGeom g, const int3 per, uint8_t* state) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= g.nb[0] * g.nb[1] * g.nb[2] || state[b] >= 2) return;
    const int c[3] = {b % g.nb[0], (b / g.nb[0]) % g.nb[1], b / (g.nb[0] * g.nb[1])};
    const int pd[3] = {per.x, per.y, per.z};
    int r[3][5], m[3];
    for (int d = 0; d < 3; ++d) m[d] = axis_set(c[d], g.n[d], g.nb[d], g.B[d], pd[d], true, r[d]);
    bool sh = false;
    for (int z = 0; z < m[2] && !sh; ++z)
        for (int y = 0; y < m[1] && !sh; ++y)
            for (int x = 0; x < m[0] && !sh; ++x) sh = (state[r[0][x] + g.nb[0] * (r[1][y] + g.nb[1] * r[2][z])] & 2) != 0;
    if (sh) state[b] = 1;
}

// One block: the active and shell lists in ascending brick order, and the (core, active, shell) counts
__global__ void __launch_bounds__(CT) band_compact_kernel(const uint8_t* __restrict__ state, const int nb, int* __restrict__ active,
                                                          int* __restrict__ shell, long long* __restrict__ counts) {
    __shared__ int sc[3][CT];
    const int t = threadIdx.x, per = (nb + CT - 1) / CT, lo = min(nb, t * per), hi = min(nb, lo + per);
    int ca = 0, cs = 0, cc = 0;
    for (int b = lo; b < hi; ++b) { const int s = state[b]; ca += s >= 2; cs += s == 1; cc += s == 3; }
    sc[0][t] = ca; sc[1][t] = cs; sc[2][t] = cc;
    __syncthreads();
    for (int off = 1; off < CT; off <<= 1) {          // inclusive Hillis-Steele scan of the three counts
        int v[3];
        for (int k = 0; k < 3; ++k) v[k] = t >= off ? sc[k][t - off] : 0;
        __syncthreads();
        for (int k = 0; k < 3; ++k) sc[k][t] += v[k];
        __syncthreads();
    }
    int pa = sc[0][t] - ca, ps = sc[1][t] - cs;
    for (int b = lo; b < hi; ++b) {
        const int s = state[b];
        if (s >= 2) active[1 + pa++] = b;
        else if (s == 1) shell[1 + ps++] = b;
    }
    if (t == CT - 1) {
        active[0] = sc[0][t]; shell[0] = sc[1][t];
        counts[0] = sc[2][t]; counts[1] = sc[0][t]; counts[2] = sc[1][t];
    }
}

template <class T>
__global__ void __launch_bounds__(CB) band_copy_kernel(const BrickGeom g, const int* __restrict__ list, const T* __restrict__ src,
                                                       T* __restrict__ d0, T* __restrict__ d1) {
    if ((int)blockIdx.x >= list[0]) return;
    int o[3];
    g.origin(list[1 + blockIdx.x], o);
    for (int q = threadIdx.x; q < g.nodes(); q += CB) {
        const int i0 = o[0] + q % g.B[0], i1 = o[1] + (q / g.B[0]) % g.B[1], i2 = o[2] + q / (g.B[0] * g.B[1]);
        if (i0 < g.n[0] && i1 < g.n[1] && i2 < g.n[2]) {
            const long l = (long)i0 + (long)g.n[0] * ((long)i1 + (long)g.n[1] * i2);
            const T v = src[l];
            d0[l] = v;
            if (d1) d1[l] = v;
        }
    }
}

}  // namespace

int band_bricks(int ndim, const int* n) {
    long nb = (long)((n[0] + BRICK_X - 1) / BRICK_X) * ((n[1] + BRICK_Y - 1) / BRICK_Y);
    if (ndim == 3) nb *= (n[2] + BRICK_Z - 1) / BRICK_Z;
    return nb > 0x3FFFFFFFL ? -1 : (int)nb;
}

cudaError_t launch_band_rebuild(const BandArgs& A, bool from_active, cudaStream_t s, int* launches) {
    const BrickGeom g = geom(A);
    const int nb = A.nbricks;
    const int3 per = make_int3(A.periodic[0], A.periodic[1], A.periodic[2]);
    const int* list = from_active ? A.active : nullptr;
    if (A.f64) band_core_kernel<double><<<nb, CB, 0, s>>>(static_cast<const double*>(A.phi), g, A.gamma, list, A.core);
    else band_core_kernel<float><<<nb, CB, 0, s>>>(static_cast<const float*>(A.phi), g, A.gamma, list, A.core);
    const int tb = 256, gb = (nb + tb - 1) / tb;
    band_active_kernel<<<gb, tb, 0, s>>>(g, per, A.core, A.state);
    band_shell_kernel<<<gb, tb, 0, s>>>(g, per, A.state);
    band_compact_kernel<<<1, CT, 0, s>>>(A.state, nb, A.active, A.shell, A.counts);
    *launches = 4;
    return cudaGetLastError();
}

cudaError_t launch_band_copy(const BandArgs& A, const int* list, const void* src, void* d0, void* d1, cudaStream_t s) {
    const BrickGeom g = geom(A);
    if (A.f64) band_copy_kernel<double><<<A.nbricks, CB, 0, s>>>(g, list, static_cast<const double*>(src), static_cast<double*>(d0), static_cast<double*>(d1));
    else band_copy_kernel<float><<<A.nbricks, CB, 0, s>>>(g, list, static_cast<const float*>(src), static_cast<float*>(d0), static_cast<float*>(d1));
    return cudaGetLastError();
}

}  // namespace lsm
