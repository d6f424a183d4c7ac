// lsm_kernels.h — launchers implemented by the .cu translation units, called by lsm_api.cu.
#pragma once
#include <string>
#include "lsm_dev.cuh"

namespace lsm {

struct CflParams {
    TermDev term;
    int n[3];                  // owned nodes (1 for unused dims)
    double h[3];
    unsigned long long* out;   // device scalar, zeroed by the caller
};

// CFL candidate extraction (see lsm_api.cu, cfl_candidates): every node whose unscaled CFL quantity reaches `thr` appends its
// raw coefficient tuple (ncomp doubles) to `out`; `count` keeps counting past `cap` so that the host can tell an overflow.
struct CandParams {
    TermDev term;              // scaled == 0
    int n[3];
    double h[3];
    double thr;
    int cap, ncomp;
    unsigned* count;           // device counter, zeroed by the caller
    double* out;               // cap x ncomp
};

// lsm_generic.cu (strict arithmetic, -fmad=false)
template <class T> cudaError_t launch_stage_generic(int ndim, const StageParams<T>& P, cudaStream_t s);
cudaError_t launch_cfl(int ndim, int dtype_f64, const CflParams& P, int sm_count, cudaStream_t s);
cudaError_t launch_cfl_candidates(int ndim, int dtype_f64, const CandParams& P, int sm_count, cudaStream_t s);
cudaError_t launch_eikonal_s0(int src_f64, int dst_f64, const void* phi, void* out, long n, double dx, cudaStream_t s);
cudaError_t launch_transpose(int f64, bool to_soa, const void* src, void* dst, long n, int ncomp, long cstride, cudaStream_t s);
template <class T> cudaError_t launch_getindex(int ndim, const View<T>& v, const int* d_idx, int count, double* d_out, cudaStream_t s);
template <class T> cudaError_t launch_measure(int ndim, bool perimeter, const View<T>& v, const double* h, double* d_partials, int nblocks, double* d_out, cudaStream_t s);
template <class T> cudaError_t launch_signed_normals(int ndim, const View<T>& v, const double* h, double min_norm, const unsigned char* d_frozen, double band, T* a, long cstride, cudaStream_t s);
// analytic generators (meshfield.jl:208-211 evaluated on the device): see lsm_field_fill_shape / lsm_field_fill_separable
struct ShapeParams {
    int shape, ndim, ncomp;
    int n[3];                  // owned nodes
    int first_last;            // global index of the first owned plane of the last dimension
    double lc[3], h[3];
    double p[8];               // shape parameters
    long cstride;
};
cudaError_t launch_fill_shape(int f64, void* dst, const ShapeParams& P, cudaStream_t s);
cudaError_t launch_fill_separable(int f64, void* dst, long cstride, const int* n, int ndim, const double* scale, const double* const (*tab)[3], cudaStream_t s);
cudaError_t launch_csg(int f64, void* dst, const void* src, long n, int op, cudaStream_t s);

// lsm_expr.cu: coefficients given as CUDA C++ expressions in x1..xN and t, compiled at run time with NVRTC (lsm_field_set_expr)
struct ExprKernel;             // one compiled pointwise kernel of the process-wide cache (never freed)
struct ExprArgs {              // the generated kernel's parameter (its device twin is generated in lsm_expr.cu)
    void* dst;                 // first owned node of component 0 (SoA, components cstride apart)
    unsigned long long* cfl;   // CFL maximum of the rounded values (IEEE bits, atomicMax), zeroed by the caller; unused when cfl_kind == 0
    long long cstride;
    int n[3];                  // owned nodes
    int first_last;            // global index of the first owned plane of the last dimension
    int f64;                   // dtype of dst
    int cfl_kind;              // 0 none, 1 advection (sum_d |u_d| / h_d), 2 normal motion / curvature (|v|)
    double lc[3], h[3];
    double t;
};
// Validates, generates and compiles (or finds in the cache) the kernel of `exprs` (ncomp pointers, then NULL); load != 0 also
// loads it for launching (needs a device).  On failure returns an LSM_ERR_* status and the reason in *err.
int32_t expr_get(int ndim, int ncomp, const char* const* exprs, bool load, const ExprKernel** out, std::string* err);
bool expr_uses_t(const ExprKernel* k);
cudaError_t launch_expr_fill(const ExprKernel* k, const ExprArgs& A, int sm_count, cudaStream_t s);
cudaError_t launch_max_abs_diff(int f64, const void* a, const void* b, long n, unsigned long long* out, cudaStream_t s);

// lsm_interface.cu: zero-level-set extraction (lsm_interface_extract).  The node box is this rank's owned nodes plus, below the
// last rank, the first plane of the next rank (the upper ghost plane), so that every cell whose lower corner the rank owns is whole.
struct IfaceArgs {
    const void* phi;           // first node of the box (dense column-major, dim 1 contiguous)
    int f64, ndim;
    int m[3];                  // box nodes per dim (1 for unused dims)
    int first_last;            // global index of the box's first plane of the last dimension
    int hsign;                 // sign of prod_d h_d: a mirrored grid mirrors every simplex
    long long s1, s2;          // element strides of dims 2 and 3
    long long nodes, ntiles;   // nodes in the box, tiles of the passes
    long long lin0;            // global column-major index of the box's first node
    double level;
    double lc[3], h[3];
};
long long iface_tiles(long long nodes);
size_t iface_scratch_bytes(long long ntiles);
long long* iface_totals(const IfaceArgs& A, void* scratch);     // device address of (nverts, nprims) after pass 0
// pass 0: count + scan (totals at iface_totals); pass 1: vertices and keys; pass 2: primitives (needs the keys of pass 1)
cudaError_t launch_iface(const IfaceArgs& A, int pass, void* scratch, double* verts, long long* keys, int* prims, cudaStream_t s);

// lsm_redistance.cu: closest-point redistancing (lsm_redistance), its closest-point extension (lsm_extend_closest_point) and its
// cubic refinement (lsm_redistance_cubic), single-rank fields.  The box is the whole field.
struct RedistArgs {
    IfaceArgs g;               // the field (level 0; ntiles and lin0 unused); the write pass stores through g.phi
    int band;                  // cell window half-width
    double* pa;                // point buffers: N components of g.nodes doubles each (SoA), N + 1 with F (the value at the point
    double* pb;                // last); NaN = no point
    long long* list;           // cut cells (up to g.nodes entries; aliases pa until the pick pass writes it)
    unsigned long long* dmin;  // per node: smallest candidate distance (IEEE bits) of the band scan
    unsigned long long* ord;   // per node: order key (cell * 16 + primitive) of the first candidate at that distance
    unsigned long long* ncells;// listed cells, zeroed by the caller
    unsigned long long* count; // band nodes, zeroed by the caller
    void* F;                   // the extension: scalar field on g's grid, read by the pick pass and written by the write pass; null
                               // for redistancing
    bool F_f64;                // F's dtype
    int write_phi;             // with F: the write pass also stores the signed distance through g.phi, as it does without F
    unsigned long long* fallbacks; // the cubic refinement (null: none): nodes that keep their linear closest point, zeroed by the caller
};
// enqueues flag, the two cell passes, pick, the jump-flooding passes, with fallbacks set the Newton refinement on the cubic
// interpolant (lsm_cubic.cuh), and the write pass on s; *launches = kernels enqueued
cudaError_t launch_closest_points(const RedistArgs& R, int sm_count, cudaStream_t s, int* launches);
// lsm_interpolate_cubic: the interpolant of A's field at npts points (pts AoS, npts x ndim); val (npts), grad (npts x ndim) and
// hess (npts x ndim x ndim) may each be null
cudaError_t launch_interp_cubic(const IfaceArgs& A, long long npts, const double* pts, double* val, double* grad, double* hess,
                                cudaStream_t s);

// lsm_integrals.cu: measures of {s <= 0} and {s = 0} and the integrals of F over them (lsm_level_set_integrals).  The box is
// field_box's (with the upper ghost plane below the last rank); partials are 4 doubles per cell plane of the whole grid.
struct IntegArgs {
    IfaceArgs g;               // the box and the level (ntiles and lin0 unused)
    const void* F;             // scalar field on g's grid, same box layout, or null
    int F_f64;                 // F's dtype
    long long planes;          // cell planes of the box (m_last - 1)
    long long plane0;          // global index of the box's first cell plane
    double V, Vs;              // prod_d |h_d| and V / N!
    double* part;              // partials: part[4 plane + q], q = region, interface, F over the region, F over the interface
};
// one block per cell plane (one thread per cell in 1-D): writes the partials of the box's planes
cudaError_t launch_integral_planes(const IntegArgs& I, cudaStream_t s);
// one block: out[q] = sum of part[4 plane + q] over the planes in increasing order
cudaError_t launch_integral_sum(const double* part, long long nplanes, double* out, cudaStream_t s);

// The five Float64 constants of the WENO5 evaluation that do not fit an instruction immediate travel in the kernel parameters
// (constant bank): as literals the compiler re-materialises them with 10 UMOV per node, from the constant bank it takes 3 uniform loads.
// The 3-D x-pair kernel's default form scales e6 and fl by 3/16 once per thread (lsm_pair_common.cuh: weno_regs).
struct WenoK { double c133, c56, cm13, e6, fl, pad; };
inline WenoK weno_constants() { return {13.0 / 3.0, 5.0 / 6.0, -1.0 / 3.0, 4.0e-6, 1.0e-70, 0.0}; }

// stored coefficient components and phi^n staged in shared memory next to the phi ring
struct AuxList {
    int n;                 // number of staged scalar tiles per plane
    int first[4];          // first aux index of term k (-1: not staged)
    int p0;                // aux index of phi^n / corr (-1: none)
    const void* src[8];    // box pointers (no ghost planes before the first owned node; same strides as the state)
    WenoK wk;              // see WenoK
};

// lsm_pair3d.cu (3-D single-term WENO5 advection, x-pair threads).  cudaErrorNotSupported -> use the general tiled kernel.
template <class T> cudaError_t launch_stage_pair3d(const StageParams<T>& P, const AuxList& A, cudaStream_t s, bool exact_eps);
// lsm_pair2d.cu (2-D WENO5 advection [+ constant-b curvature], x-pair threads marching along y)
template <class T> cudaError_t launch_stage_pair2d(const StageParams<T>& P, const AuxList& A, cudaStream_t s, bool force, int sm_count);

// lsm_resident2d.cu (small 2-D grids: the whole time loop of one stored-velocity WENO5 advection term in one cluster kernel)
template <class T>
struct ResidentArgs {
    const T* phi;          // state, read once
    T* out;                // state, written once (may alias phi)
    const T* u[2];         // velocity components (same box as the state)
    int n[2];
    long s1;               // row stride (elements)
    int bc[2][2];          // BC_* kinds (index maps only)
    double h[2];
    int nstages;           // 1 ForwardEuler, 2 RK2, 3 TVD-RK3
    int nruns;             // run-length encoded step sizes: count[r] steps of dt[r]
    double dt[4];
    long count[4];
    WenoK wk;
    unsigned long long* status;   // device word, zeroed by the caller: != 0 after the run = internal protocol failure (never expected)
};
template <class T> bool resident2d_supported(int n0, int n1);
template <class T> cudaError_t launch_resident2d(const ResidentArgs<T>& R, cudaStream_t s);

// lsm_tiled.cu (performance kernels).  Returns cudaErrorNotSupported when the configuration is
// not covered, in which case the caller uses the generic kernel.
template <class T> cudaError_t launch_stage_tiled(int ndim, const StageParams<T>& P, int sm_count, cudaStream_t s, int pair_mode = 1, int* used_pair = nullptr);   // pair_mode: 0 never, 1 x-pair kernels (3-D: 20-bit eps max), 2 3-D x-pair kernel with the exact eps max, 3 x-pair kernels forced on small 2-D grids too
template <class T> bool stage_tiled_supported(int ndim, const StageParams<T>& P);

}  // namespace lsm
