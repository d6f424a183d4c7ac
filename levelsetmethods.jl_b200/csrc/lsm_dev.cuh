// lsm_dev.cuh — device-side data layout shared by all kernels of liblsm_b200.
//
// HBM layout (DESIGN.md §3):
//   * a scalar node field is a dense column-major box n1 x n2 x n3 (dim 1 contiguous), preceded
//     and followed by `halo` ghost planes of the LAST dimension when the field is slab-decomposed
//     (nranks > 1).  View::p points at the first OWNED node, so ghost planes sit at negative /
//     beyond-the-end offsets along the last dimension and a plane is always contiguous.
//   * a vector coefficient (velocity) is stored SoA: component d is a scalar box at p + d*cstride.
//     (The host API speaks AoS like Array{SVector{N,T},N}; upload/download transpose on device.)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lsm {

enum : int { BC_NONE = -1, BC_PERIODIC = 0, BC_EXTRAP = 1, BC_SYMMETRY = 2, BC_HALO = 3 };
enum : int { TERM_ADVECTION = 0, TERM_NORMAL = 1, TERM_CURVATURE = 2, TERM_EIKONAL = 3 };
enum : int { SCHEME_UPWIND = 0, SCHEME_WENO5 = 1 };
enum : int { COEF_CONST = 0, COEF_FIELD = 1, COEF_SEPARABLE = 2, COEF_NONE = 3 };
// stage base: how the accumulator is seeded before the terms are subtracted (timestepping.jl:128-202)
enum : int {
    BASE_IN = 0,        // x = in[I]                              FE, RK2 S1 (pred & corr), RK3 S1
    BASE_RK3_S2 = 1,    // x = 0.75*p0[I] + 0.25*in[I]            RK3 S2 (p0 = phi^n)
    BASE_RK3_S3 = 2,    // x = (p0[I] + 2*in[I]) / 3  (in V)      RK3 S3
    BASE_P0 = 3         // x = p0[I]                              RK2 S2 (p0 = corr)
};

struct BCDev { int kind, P; };

// Narrow-band bricks (lsm_narrow_band.cu): the tiled stage kernel's x-y tile times 16 planes; 2-D fields use BRICK_X x BRICK_Y
enum : int { BRICK_X = 32, BRICK_Y = 16, BRICK_Z = 16 };

// Is a boundary side (kind, extrapolation order P) a pure index map with weight 1: periodic, symmetry, ExtrapolationBC{0}, or
// the stored ghost planes of the decomposed axis?  ExtrapolationBC{P >= 1} is a weighted stencil.  Takes the BC_* kinds of a
// View and the LSM_BC_* kinds of a field alike (they share 0..2; BC_HALO appears only on the last axis, see make_view).
__host__ __device__ inline bool bc_index_map(int kind, int P) {
    return kind == BC_PERIODIC || kind == BC_SYMMETRY || kind == BC_HALO || (kind == BC_EXTRAP && P == 0);
}

template <class T>
struct View {
    const T* p;          // first owned node
    int n[3];            // owned nodes per dim (1 for unused dims)
    long s1, s2;         // element strides of dim 2 and dim 3 (dim 1 is contiguous)
    BCDev bc[3][2];      // BC_HALO on a side whose ghost planes are stored
    int halo;            // ghost planes of the last dimension stored before the first owned node (0 or 3)
    int _pad;
};

struct TermDev {
    int kind, scheme, coef_kind, scaled;   // scaled: multiply coefficient by g (tscale_kind != NONE)
    double g;
    double cval[3];
    const void* coef;    // SoA coefficient data (dtype T unless coef_f64)
    long cstride;        // component stride (elements)
    int coef_f64;        // coefficient stored as double although T == float (S0)
    int _pad;
    const double* tab[3][3];   // SEPARABLE: tab[d][axis] -> this rank's slice
};

template <class T>
struct StageParams {
    View<T> in;          // stencil input (stage field)
    const T* p0;         // pointwise second input (phi^n or corr); same box layout as in.p
    T* out;              // stage output (may alias p0: written pointwise by the thread that read it)
    T* out2;             // RK2 S1 second accumulator (corr) or nullptr
    int base;            // BASE_*
    int nterms;
    double c, c2;        // x -= c * H ; x2 -= c2 * H
    double h[3];         // meshsize per dim
    double dxmin;        // minimum(meshsize)
    int r0, r1;          // range [r0, r1) of the LAST dimension to update (interior/boundary split)
    int skip_zero_u;     // upwind advection: a component with u_d == 0 contributes exactly 0 even when its one-sided difference is
    int _pad1;           // NaN / Inf (extend_along_normals!: frozen nodes keep their value, velocityextension.jl:53-56)
    const int* bricks;   // narrow band: device list {count, brick, brick, ...} of the bricks to update (BRICK_X x BRICK_Y x BRICK_Z,
                         // column-major numbering), or nullptr for the whole box.  Its 8 bytes keep terms[] 8 bytes past a 16-byte
                         // boundary: that alignment decides which of its fields the stage kernels fetch in pairs with 128-bit
                         // constant loads, and so the code they compile to
    TermDev terms[4];
};

// component d of a term's coefficient at node (i0, i1, i2), linear index `node`, times its time factor
template <class T>
__device__ __forceinline__ double coef_comp(const TermDev& t, long node, int d, int i0, int i1, int i2, int N) {
    double v;
    if (t.coef_kind == COEF_CONST) {
        v = t.cval[d];
    } else if (t.coef_kind == COEF_FIELD) {
        const long l = (long)d * t.cstride + node;
        v = t.coef_f64 ? static_cast<const double*>(t.coef)[l] : double(static_cast<const T*>(t.coef)[l]);
    } else if (t.coef_kind == COEF_SEPARABLE) {
        v = t.cval[d];
        v = v * t.tab[d][0][i0];
        if (N > 1) v = v * t.tab[d][1][i1];
        if (N > 2) v = v * t.tab[d][2][i2];
    } else {
        v = 0.0;
    }
    if (t.scaled) v = v * t.g;
    return v;
}

// coefficient box without ghost planes: linear node index of (i0,i1,i2)
struct CoefBox { int n0, n1; };

}  // namespace lsm
