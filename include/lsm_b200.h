/*
 * lsm_b200.h — C ABI of liblsm_b200.so, a B200 (sm_100a) engine for the dense-grid explicit
 * time-integration path of LevelSetMethods.jl (reference v0.2.0).
 *
 * The reference has no FFI: its seam is Julia dispatch on four internal generics plus the
 * AbstractMeshField interface (SURVEY.md §8b).  Each entry point below names the reference
 * function(s) it replaces (paths relative to the reference repo root).  Julia binds these with
 * `ccall` (julia/LSMB200.jl, shown in INTEGRATION.md); Python binds them with ctypes
 * (levelsetmethods.jl_b200/_lib.py).
 *
 * Conventions
 *  - plain C types only; every function returns an int32 status (LSM_OK == 0); C++ exceptions
 *    never cross the boundary; lsm_last_error() gives the message of the last failure.
 *  - host arrays are column-major (dim 1 contiguous) exactly like a Julia Array{V,N}; vector
 *    fields are AoS like Array{SVector{N,T},N} (shape (N, n1, .., nN)).  Host pointers are
 *    never retained after a call returns.
 *  - one context == one process == one GPU.  With nranks > 1 every field is slab-partitioned
 *    along its LAST dimension and each rank uploads / downloads only its own slab.
 *  - handles are not thread-safe; distinct contexts are independent.
 *  - there is no CPU fallback: every compute entry point fails with LSM_ERR_CUDA when no
 *    sm_100 device is usable.
 */
#ifndef LSM_B200_H
#define LSM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSM_ABI_VERSION 1

/* ---- status codes -------------------------------------------------------------------------- */
enum {
    LSM_OK = 0,
    LSM_ERR_ARG = 1,          /* bad argument (null handle, bad enum, shape mismatch)                     */
    LSM_ERR_CFL = 2,          /* levelsetterms.jl:26  ArgumentError("invalid time-step based on CFL ...") */
    LSM_ERR_TIME = 3,         /* levelsetequation.jl:196  ArgumentError("final time ... must be >= ...")  */
    LSM_ERR_BC = 4,           /* boundaryconditions.jl:184-186 periodic mixed; levelsetequation.jl:69-70  */
    LSM_ERR_CUDA = 5,
    LSM_ERR_NCCL = 6,
    LSM_ERR_OOM = 7,
    LSM_ERR_UNSUPPORTED = 8
};

enum { LSM_F32 = 0, LSM_F64 = 1 };

/* boundaryconditions.jl:27-74.  NeumannBC == EXTRAP with P = 0, LinearExtrapolationBC == P = 1. */
enum { LSM_BC_NONE = -1, LSM_BC_PERIODIC = 0, LSM_BC_EXTRAP = 1, LSM_BC_SYMMETRY = 2 };
#define LSM_MAX_EXTRAP_P 5
typedef struct { int32_t kind; int32_t P; } lsm_bc;

/* levelsetterms.jl:45-49,104-106,139-142,211-213 */
enum { LSM_TERM_ADVECTION = 0, LSM_TERM_NORMAL = 1, LSM_TERM_CURVATURE = 2, LSM_TERM_EIKONAL = 3 };
/* derivatives.jl:11,20 */
enum { LSM_UPWIND = 0, LSM_WENO5 = 1 };
/* how a term's coefficient (velocity / speed / b / S0) is given; replaces _eval_field (levelsetterms.jl:42-43) */
enum {
    LSM_COEF_CONST = 0,       /* cval[0..N-1] (velocity) or cval[0]                                        */
    LSM_COEF_FIELD = 1,       /* device field (ncomp = N for a velocity, 1 otherwise)                      */
    LSM_COEF_SEPARABLE = 2,   /* field made by lsm_field_create_separable: u_d = s_d X_d[i1] Y_d[i2] Z_d[i3] */
    LSM_COEF_NONE = 3,        /* EikonalReinitializationTerm() — live sign (levelsetterms.jl:222)           */
    LSM_COEF_EXPR = 4         /* field with expressions attached (lsm_field_set_expr): f(x, t) of levelsetterms.jl:42-43,
                                 materialised on the device at every time a term needs it; no time factor (t is in the expression) */
};
/* time factor g(t) multiplying the coefficient (device-side stand-in for update_func / f(x,t)) */
enum { LSM_TS_NONE = 0, LSM_TS_COS = 1 /* cos(pi t / tparam) */, LSM_TS_HOST = 2 /* caller passes g per call */ };

/* timestepping.jl:26-28,46-48,65-67 */
enum { LSM_FORWARD_EULER = 0, LSM_RK2 = 1, LSM_RK3 = 2 };

typedef struct lsm_ctx lsm_ctx;
typedef struct lsm_field lsm_field;

#define LSM_MAX_TERMS 4
typedef struct {
    int32_t kind;             /* LSM_TERM_*   */
    int32_t scheme;           /* LSM_UPWIND / LSM_WENO5 (advection only) */
    int32_t coef_kind;        /* LSM_COEF_*   */
    int32_t tscale_kind;      /* LSM_TS_*     */
    double  cval[3];
    double  tparam;
    lsm_field* field;         /* coefficient field for FIELD / SEPARABLE, else NULL */
} lsm_term;

typedef struct {
    int64_t kernel_launches;  /* kernels of this library launched since ctx creation */
    int64_t stage_launches;   /* of which fused stage kernels                         */
    int64_t cfl_passes;       /* CFL reduction passes actually run (cache misses)     */
    int64_t h2d_bytes, d2h_bytes;
    int64_t halo_bytes_sent;  /* NCCL send bytes (multi-rank)                          */
    double  last_stage_ms;    /* CUDA-event time of the last timed stage (see LSM_OPT_TIME_STAGES) */
    double  sum_stage_ms;     /* accumulated over timed stages since lsm_reset_counters */
    int64_t timed_stages;
    int64_t pair_launches;    /* stage launches that took the x-pair kernel (3-D single-term WENO5 advection)  */
    int64_t resident_steps;   /* time steps taken inside the resident cluster kernel (small 2-D grids; one launch per lsm_integrate) */
} lsm_counters;

/* options for lsm_set_option */
enum {
    LSM_OPT_KERNEL = 0,       /* 0 auto (x-pair / tiled where available), 1 force generic strict kernel, 2 force tiled / x-pair, 3 tiled without the x-pair kernel,
                                 4 x-pair kernel with the exact WENO epsilon maximum (bit-identical to 3; default is a 20-bit maximum) */
    LSM_OPT_TIME_STAGES = 1,  /* 1: bracket every stage launch with CUDA events, resolved at the next sync  */
    LSM_OPT_CFL_CACHE = 2,    /* 1 (default): reuse the CFL reduction while coefficient data/scale unchanged  */
    LSM_OPT_OVERLAP = 3,      /* 1 (default): overlap halo exchange with interior compute (multi-rank)        */
    /* 4 is retired and not reused: lsm_set_option rejects it with LSM_ERR_ARG */
    LSM_OPT_GRAPH = 5,        /* 1 (default): lsm_integrate replays a captured CUDA graph of one step's stage launches on small grids (launch-bound regime) */
    LSM_OPT_CFL_CANDIDATES = 6, /* 1 (default): the CFL maximum of a TIME-SCALED static coefficient field is evaluated on the host over the few nodes that
                                  can attain it for any scale (exact, see lsm_api.cu) - no reduction pass, D2H or host sync per step */
    LSM_OPT_RESIDENT = 7      /* 1 (default): lsm_integrate runs the whole time loop of a small 2-D grid (<= 2^15 nodes, one stored-velocity WENO5
                                 advection term without a time factor, index-map BCs) in ONE cluster kernel that keeps the state in distributed
                                 shared memory (lsm_resident2d.cu); bit-identical to the per-stage kernels */
};

/* ---- lifecycle ------------------------------------------------------------------------------ */
int32_t lsm_abi_version(void);
/* Thread-local message of the last failing call (ctx may be NULL). */
const char* lsm_last_error(void);
int32_t lsm_device_count(int32_t* n_out);

/* Single-GPU context on `device`. */
int32_t lsm_ctx_create(int32_t device, lsm_ctx** out);
/* Multi-GPU: rank 0 calls lsm_nccl_unique_id and the host broadcasts the 128 bytes (MPI.jl,
 * torch.distributed, a file ...); then every rank creates its context. */
int32_t lsm_nccl_unique_id(void* id128);
int32_t lsm_ctx_create_rank(int32_t device, int32_t rank, int32_t nranks, const void* id128, lsm_ctx** out);
/* Multi-GPU from ONE process (one Julia task / one Python thread driving a whole box): n_gpus contexts, rank r on
 * device_ids[r], whose NCCL communicators come from ncclCommInitAll.  `out` receives n_gpus handles.  Per-rank calls without
 * an exchange (lsm_field_create / upload / download / set_bc / fill / destroy) are made one context after the other; the
 * collective ones (everything that exchanges halos or all-reduces: compute_cfl, stage, advance, integrate) must run on all
 * ranks concurrently — the lsm_multi_* entry points below do that on one host thread per GPU and return the first error. */
int32_t lsm_ctx_create_multi(int32_t n_gpus, const int32_t* device_ids, lsm_ctx** out);
int32_t lsm_multi_compute_cfl(int32_t n_gpus, lsm_ctx* const* ctx, lsm_field* const* phi, const lsm_term* const* terms, int32_t nterms,
                              double t, const double* gscale, double* dt_out);
int32_t lsm_multi_integrate(int32_t n_gpus, lsm_ctx* const* ctx, int32_t integrator, double cfl, lsm_field* const* phi,
                            const lsm_term* const* terms, int32_t nterms, double t0, double tf, double dt_max, int64_t max_steps,
                            double* t_out, int64_t* steps_out);
int32_t lsm_ctx_destroy(lsm_ctx* ctx);
int32_t lsm_sync(lsm_ctx* ctx);
int32_t lsm_set_option(lsm_ctx* ctx, int32_t option, int32_t value);
int32_t lsm_get_counters(lsm_ctx* ctx, lsm_counters* out);
int32_t lsm_reset_counters(lsm_ctx* ctx);

/* CUDA-event timing on the context's compute stream (the stream every kernel of this library is
 * launched on): record into slot 0..7, then read the elapsed milliseconds between two slots
 * (synchronises on the later event). */
int32_t lsm_event_record(lsm_ctx* ctx, int32_t slot);
int32_t lsm_event_elapsed_ms(lsm_ctx* ctx, int32_t slot_start, int32_t slot_stop, double* ms_out);

/* Pin / unpin a host array (e.g. the memory of a Julia Array) so uploads/downloads run at full
 * PCIe speed.  Optional. */
int32_t lsm_host_register(void* ptr, int64_t bytes);
int32_t lsm_host_unregister(void* ptr);

/* Pure host function (no GPU needed): which planes of the last dimension rank `rank` owns.
 * first_out is 0-based. */
int32_t lsm_slab_plan(int32_t n_last, int32_t nranks, int32_t rank, int32_t* first_out, int32_t* count_out);

/* Pure host function (no GPU needed): the step sizes the time loop takes when the CFL step dt_cfl is CONSTANT (static coefficients), i.e.
 * the loop of _integrate! (timestepping.jl:104-118) replayed with its own arithmetic: while t <= tf - eps(t): dt = min(dt_max, cfl * dt_cfl,
 * tf - t); t += dt — at most max_steps steps (< 0: no limit).  The sequence is run-length encoded into dt_out / count_out (capacity cap;
 * cap = 0 only counts): normally two runs, n full steps and one shorter final step.  This is what lsm_integrate hands to the resident
 * cluster kernel of small 2-D grids (LSM_OPT_RESIDENT); t_out / steps_out are the time and step count that loop reaches. */
int32_t lsm_step_plan(double t0, double tf, double dt_max, double cfl, double dt_cfl, int64_t max_steps, int32_t cap,
                      double* dt_out, int64_t* count_out, int32_t* nruns_out, int64_t* steps_out, double* t_out);

/* ---- grid + field : CartesianGrid (meshes.jl:1-5,34-42) + MeshField (meshfield.jl:51-55) ------ */
/* n = GLOBAL node counts.  ncomp = 1 (scalar) or ndim (velocity).  The field owns its device
 * memory (and, for a state field, the RK stage buffers of _alloc_buffers, timestepping.jl:126,141,168). */
int32_t lsm_field_create(lsm_ctx* ctx, int32_t ndim, const int32_t* n, int32_t dtype, int32_t ncomp,
                         const double* lc, const double* hc, lsm_field** out);
/* Rank-1 separable vector coefficient: component d at node (i1,i2,i3) is
 * scale[d] * tab[d][0][i1] * tab[d][1][i2] * tab[d][2][i3].  `tabs` is the concatenation, for
 * d = 0..ndim-1 and axis a = 0..ndim-1, of n[a] doubles (GLOBAL extents, host memory, copied). */
int32_t lsm_field_create_separable(lsm_ctx* ctx, int32_t ndim, const int32_t* n, const double* lc, const double* hc,
                                   const double* scale, const double* tabs, lsm_field** out);
int32_t lsm_field_destroy(lsm_field* f);
/* _normalize_bc'd boundary conditions: bc[2*d + side], side 0 = left, 1 = right
 * (boundaryconditions.jl:166-188; periodic on one side only -> LSM_ERR_BC). */
int32_t lsm_field_set_bc(lsm_field* f, const lsm_bc* bc);
/* Local (this rank's) extents: n_local[ndim], and the 0-based global index of the first owned
 * plane of the last dimension. */
int32_t lsm_field_local_extent(const lsm_field* f, int32_t* n_local, int32_t* first_last);
/* values(phi) <- host / host <- values(phi): this rank's slab, column-major, AoS for ncomp > 1. Blocking. */
int32_t lsm_field_upload(lsm_field* f, const void* host);
int32_t lsm_field_download(lsm_field* f, void* host);
/* copy!(dst, src) (meshfield.jl:275-278) */
int32_t lsm_field_copy(lsm_field* dst, const lsm_field* src);
/* meshsize(phi) (meshes.jl:109-110) */
int32_t lsm_field_meshsize(const lsm_field* f, double* h_out);
/* phi[I] (meshfield.jl:213-260): BC-aware read evaluated ON THE DEVICE by the same ghost-cell
 * code the stencil kernels use.  I is 1-based like the reference and may lie outside the grid
 * (single-rank contexts only).  count indices of ndim int32 each -> count doubles. */
int32_t lsm_field_getindex(lsm_field* f, const int32_t* I, int32_t count, double* out);
/* Borrowed handle to RK stage buffer `which` (1 or 2) of a state field (the tuple returned by
 * _alloc_buffers, timestepping.jl:126,141,168), so host update_func callbacks can be handed the
 * stage field like the reference does.  Owned by `phi`; do not destroy. */
int32_t lsm_field_stage_buffer(lsm_field* phi, int32_t which, lsm_field** out);

/* ---- the hot path ----------------------------------------------------------------------------- */
/* compute_cfl(terms, phi, t) (levelsetterms.jl:22-38): minimum over terms and nodes, all-reduced
 * over ranks.  gscale: per-term g for LSM_TS_HOST terms (may be NULL).  LSM_ERR_CFL unless dt > 0. */
int32_t lsm_compute_cfl(lsm_ctx* ctx, lsm_field* phi, const lsm_term* terms, int32_t nterms, double t,
                        const double* gscale, double* dt_out);
/* Number of stages of an integrator (1, 2, 3). */
int32_t lsm_nstages(int32_t integrator);
/* One stage (1-based) of _advance! (timestepping.jl:128-137,143-164,170-202), so that a host can
 * run update_term! callbacks between stages like the reference does.  Asynchronous. */
int32_t lsm_stage(lsm_ctx* ctx, int32_t integrator, int32_t stage, lsm_field* phi, const lsm_term* terms,
                  int32_t nterms, double tc, double dt, const double* gscale);
/* _advance!(integrator, phi, buffers, terms, tc, dt): all stages.  Asynchronous. */
int32_t lsm_advance(lsm_ctx* ctx, int32_t integrator, lsm_field* phi, const lsm_term* terms, int32_t nterms,
                    double tc, double dt);
/* integrate!(eq, tf, dt_max) with default hooks: the whole step loop of _integrate!
 * (timestepping.jl:101-122) — dt = min(dt_max, cfl*compute_cfl, tf - tc), loop while
 * tc <= tf - eps(tc), land exactly on tf.  max_steps < 0 = unlimited.  Blocking. */
int32_t lsm_integrate(lsm_ctx* ctx, int32_t integrator, double cfl, lsm_field* phi, const lsm_term* terms,
                      int32_t nterms, double t0, double tf, double dt_max, int64_t max_steps,
                      double* t_out, int64_t* steps_out);

/* EikonalReinitializationTerm(phi0) constructor (levelsetterms.jl:217-221): dst = phi0/sqrt(phi0^2+min(h)^2). */
int32_t lsm_eikonal_s0(lsm_field* dst, const lsm_field* phi0);

/* ---- level-set measures (SURVEY.md §8f "next" row 1): the usual posthook / update_func payload, reduced on the device ---- */
/* volume(phi) (levelsetops.jl:27-33): prod(h) * sum smooth_heaviside(-phi, min h), all-reduced over ranks. */
int32_t lsm_volume(lsm_ctx* ctx, lsm_field* phi, double* out);
/* perimeter(phi) (levelsetops.jl:139-149): prod(h) * sum smooth_delta(phi, min h) * |grad phi| with centred differences; a field
 * without boundary conditions is given LinearExtrapolationBC like the reference does.  Single-rank contexts, or multi-rank
 * fields whose ghost planes are current. */
int32_t lsm_perimeter(lsm_ctx* ctx, lsm_field* phi, double* out);

/* extend_along_normals!(F, phi; nb_iters, cfl, frozen, interface_band, min_norm) (velocityextension.jl:20-116, "next" row 2):
 * nb_iters first-order upwind pseudo-time steps of F_tau + sign(phi) n.grad F = 0 with tau = cfl * min(h).  Runs as ForwardEuler
 * stages of an upwind AdvectionTerm whose velocity is the signed normal S grad(phi)/|grad(phi)|, zeroed on frozen nodes (which
 * reproduces the reference's Dirichlet constraint exactly).  frozen: host uint8 mask of this rank's slab (1 = frozen) or NULL
 * for the band |phi| <= interface_band * min(h).  F and phi must share grid and dtype. */
int32_t lsm_extend_along_normals(lsm_ctx* ctx, lsm_field* F, lsm_field* phi, int32_t nb_iters, double cfl, const uint8_t* frozen,
                                 double interface_band, double min_norm);

/* Set operations on level sets, in place on the device (levelsetops.jl:253-325, "next" row 3):
 *   LSM_CSG_UNION      dst = min(dst, src)   union!      LSM_CSG_INTERSECT  dst = max(dst, src)   intersect!
 *   LSM_CSG_SETDIFF    dst = max(dst, -src)  setdiff!    LSM_CSG_COMPLEMENT dst = -dst (src NULL) complement!
 * min/max follow Julia: NaN if either operand is NaN, min(0.0,-0.0) = -0.0, max(0.0,-0.0) = 0.0. */
enum { LSM_CSG_UNION = 0, LSM_CSG_INTERSECT = 1, LSM_CSG_SETDIFF = 2, LSM_CSG_COMPLEMENT = 3 };
int32_t lsm_field_csg(lsm_ctx* ctx, lsm_field* dst, const lsm_field* src, int32_t op);

/* Analytic initial conditions and coefficients generated ON THE DEVICE ("next" row 3): the reference builds them with
 * MeshField(f, grid) (meshfield.jl:208-211: f evaluated at x = lc + (I-1) h, meshes.jl:115-117) and combines them with the set
 * operations above (docs/src/example-zalesak.md:21-40).  A 1024^3 configuration is 60 GB of fields: generating them in HBM avoids
 * building and uploading them from the host.  Operation order (no FMA), so that a NumPy restatement is bit-identical:
 *   LSM_SHAPE_SPHERE  params = c[ndim], r        sqrt(((x1-c1)^2 + (x2-c2)^2) + (x3-c3)^2) - r
 *   LSM_SHAPE_BOX     params = c[ndim], w[ndim]  max_d (|x_d - c_d| - w_d / 2)           (the notch of the Zalesak disk)
 *   LSM_SHAPE_PLANE   params = n[ndim], offset   ((n1 x1 + n2 x2) + n3 x3) - offset
 *   LSM_SHAPE_CONST   params = v[ncomp]          every node of component c = v[c]        (scalar or vector fields)
 * with x_d = lc_d + i_d * h_d, i_d the 0-based GLOBAL node index.  Values are rounded to the field's dtype at the end. */
enum { LSM_SHAPE_SPHERE = 0, LSM_SHAPE_BOX = 1, LSM_SHAPE_PLANE = 2, LSM_SHAPE_CONST = 3 };
int32_t lsm_field_fill_shape(lsm_field* f, int32_t shape, const double* params, int32_t nparams);
/* Materialise a separable velocity (lsm_field_create_separable) into a stored vector field:
 * u_d[i,j,k] = ((scale_d * X_d[i]) * Y_d[j]) * Z_d[k] — rigid rotation, shear, the Enright field ... from 3 x ndim small tables. */
int32_t lsm_field_fill_separable(lsm_field* dst, const lsm_field* sep);

/* Function-valued coefficients f(x, t) (_eval_field, levelsetterms.jl:42-43) on the device.  One CUDA C++ expression per component
 * (ncomp = 1 for a speed or b, ndim for a velocity), evaluated in double with these names in scope: x1 .. xN (the node coordinate
 * lc_d + i_d h_d, i_d the 0-based global index), t (the evaluation time), pi (the double nearest pi, numpy.pi) and CUDA's
 * double-precision math functions.  The list `exprs` holds ncomp pointers followed by a NULL pointer.  Rejected with LSM_ERR_ARG
 * and a message naming the reason: an empty expression, the characters ; { } # " ' \ and the backtick, identifiers starting with
 * lsm_ or __, an integer-literal division such as 1/3 (0 in C++, 0.333... in Julia and Python), an expression count other than
 * ncomp, ncomp not in {1, ndim}; an expression NVRTC does not compile (lsm_last_error holds NVRTC's log).  The expressions are
 * compiled once per process for sm_100a with --fmad=false and without fast-math, so + - * / sqrt fabs fmin fmax give results
 * bit-identical to the same formula in NumPy float64; values are rounded to the field's dtype on store.  NVRTC is loaded at run
 * time: without it these entry points fail with LSM_ERR_UNSUPPORTED and the rest of the library is unaffected.
 * Pure host function (no GPU needed): validate and compile. */
int32_t lsm_expr_check(int32_t ndim, int32_t ncomp, const char* const* exprs);
/* Attach f->ncomp expressions to a stored field (compiled, or taken from the process-wide cache).  The field is then usable as an
 * LSM_COEF_EXPR coefficient: lsm_compute_cfl, lsm_stage, lsm_advance and lsm_integrate materialise it at the time the reference
 * calls f (the CFL at tc; the stage times tc / tc + dt / tc + dt/2), and the same pass reduces the CFL maximum of the values, so
 * no separate reduction runs.  An expression set that does not use `t` is materialised once and then behaves exactly like
 * LSM_COEF_FIELD.  A field whose data was overwritten (upload, copy) is materialised again when a term next needs it. */
int32_t lsm_field_set_expr(lsm_field* f, const char* const* exprs);
/* Materialise the attached expressions at time t: MeshField(f, grid) (meshfield.jl:208-211) for any f, the general form of
 * lsm_field_fill_shape. */
int32_t lsm_field_fill_expr(lsm_field* f, double t);

/* ---- zero-level-set extraction: the interface {phi = level} as a compact mesh, so that only the mesh leaves the device ------
 * The reference draws the interface from values(phi) on the host (ext/MakieExt.jl); these entry points replace that download.
 * Marching simplices on the Freudenthal–Kuhn triangulation of the node lattice (no case tables, no ambiguous cases, watertight):
 *  - s = double(phi) - level; a node is inside if s <= 0, outside if s > 0, invalid if s is NaN.  level must be finite and every
 *    n_d >= 2 (else LSM_ERR_ARG).
 *  - cells are the global lower corners c, 0 <= c_d <= n_d - 2, in column-major order; cell c is split into N! simplices, one per
 *    permutation pi of the axes in lexicographic order: w_0 = c, w_k = w_{k-1} + e_pi(k).  A simplex with an invalid vertex emits
 *    nothing.
 *  - vertices: the edge (a, b) = (w_i, w_j), i < j, e = b - a in {0,1}^N, is cut when one end is inside and the other outside.  Its
 *    key is lin(a) (2^N - 1) + sum_d e_d 2^(d-1) - 1 (lin: global 0-based column-major node index, d = 1..N).  With
 *    t = s_a / (s_a - s_b):  x_d = lc_d + (a_d + t) h_d where e_d = 1,  x_d = lc_d + a_d h_d where e_d = 0 (double, each operation
 *    rounded, no FMA).  Vertices are sorted by key, one per cut lattice edge of the grid.
 *  - primitives, N vertex indices each (0-based int32), in cell order, then simplex order, then as listed:
 *      1-D: a point;  2-D: one segment per cut triangle, with the inside on its left;
 *      3-D: a lone inside or outside vertex q: one triangle (qr, qs, qu), r < s < u in chain order, last two swapped if needed;
 *           inside {a < b}, outside {c < d}: the quad (ac, ad, bd, bc) as (ac, ad, bd), (ac, bd, bc), or (ac, bd, ad), (ac, bc, bd);
 *      every triangle is oriented so that (v1 - v0) x (v2 - v0) points toward s > 0, by a rule on pi, the inside mask and the signs
 *      of h only, so triangles made degenerate by exact zeros at nodes are oriented consistently too.
 *    This makes about 9 triangles per h^2 of interface against about 2 for marching cubes: the price of having no ambiguity.
 *  - periodic axes: node n duplicates node 1, so no cell wraps; boundary conditions play no role.
 * More than 2^31 - 1 vertices: LSM_ERR_UNSUPPORTED.  Scalar, non-separable fields only.
 * With nranks > 1 rank r extracts the cells whose lower corner it owns (the call exchanges the ghost planes first when they are
 * stale, so it is collective); a piece's vertices are the cut edges of its cells, so edges in a slab-boundary plane appear in two
 * pieces with the same global key: welding the pieces by key gives the single-GPU mesh bit for bit.
 * Blocking: one synchronisation and a 16-byte copy of the two counts; the mesh stays on the device in the context's persistent
 * scratch (grown on demand) until the next extraction on this context replaces it. */
int32_t lsm_interface_extract(lsm_ctx* ctx, lsm_field* phi, double level, int64_t* nverts_out, int64_t* nprims_out);
/* Copy the last extraction of this context to the host: verts (nverts x ndim doubles, AoS), keys (nverts, may be NULL) and prims
 * (nprims x ndim int32).  An array may be NULL when its count is 0.  LSM_ERR_ARG if nothing has been extracted on this context. */
int32_t lsm_interface_fetch(lsm_ctx* ctx, double* verts, int64_t* keys, int32_t* prims);
/* lsm_interface_extract on every rank of a lsm_ctx_create_multi box, on one host thread per GPU; counts per rank (n entries each). */
int32_t lsm_multi_interface_extract(int32_t n, lsm_ctx* const* ctx, lsm_field* const* phi, double level, int64_t* nverts_out, int64_t* nprims_out);

/* ---- closest-point redistancing: phi <- the signed distance to its own zero-level-set mesh, on the device ----------------------
 * The reference reinitialises phi between steps with reinitialize! (reinitializer.jl:12-42: Newton on Bernstein patches found with
 * a KD-tree, on the host, after downloading values(phi)).  lsm_redistance does the same on the device with the linear interface:
 * it replaces phi in place by the signed distance to the mesh that lsm_interface_extract(ctx, phi, 0.0, ...) would return, without
 * building or fetching that mesh and without touching the context's last extraction.  lsm_redistance_cubic (below) adds the
 * reference's Newton step on the cubic interpolant, seeded with these closest points.
 *  - s = double(phi); inside s <= 0, outside s > 0, invalid s NaN (the extraction's rules); node coordinates x_d = lc_d + i_d h_d.
 *  - primitives are the extraction's, rebuilt from phi with the same crossing formula and quad split, so their vertices are
 *    bit-identical to lsm_interface_extract's.  All arithmetic in double, each operation rounded, no FMA; dot(u, v) =
 *    (u1 v1 + u2 v2) + u3 v3 and dist(x, p) = sqrt(((x1 - p1)^2 + (x2 - p2)^2) + (x3 - p3)^2) (fewer terms in 1-D / 2-D).
 *  - closest point p of a primitive to x: 1-D the vertex; 2-D the segment projection a + t (b - a), t = clamp(dot(x - a, b - a) /
 *    dot(b - a, b - a), 0, 1), or a if a == b; 3-D Ericson's ClosestPtPointTriangle (Real-Time Collision Detection 5.1.5) in its
 *    operation order, on the triangle's vertices in the extraction's order.  Where the divisor of the region it reaches is 0
 *    (d1 - d3, d2 - d6, (d4 - d3) + (d5 - d6), or (va + vb) + vc: a triangle made degenerate by exact zeros at nodes), p is the
 *    closest of the segment projections on ab, ac, bc, in that order (a later one only if strictly closer).
 *  1. band: node i scans the cells c with max(0, i_d - band) <= c_d <= min(n_d - 2, i_d + band - 1) in increasing column-major order
 *     and, within a cell, the primitives in the extraction's order; a candidate replaces the current point only if dist(x, p) is
 *     strictly smaller.  A node whose window holds at least one primitive is a band node; every other node has no point yet.
 *  2. propagation: jump flooding over the whole box with k = 2^(ceil(log2 max_d n_d) - 1), ..., 2, 1, then once more k = 1.  Each
 *     pass reads one point buffer and writes the other; a node's candidates are its own point, then the points of the nodes
 *     i + k o, o in {-1,0,1}^N \ {0} in column-major order of o, inside the box (no wrap on any axis); nodes without a point are
 *     skipped and the strictly closest candidate wins, so a tie keeps the node's own point.
 *  3. write: with d = dist(x, p), an inside node gets -d, an outside node +d, raised to the smallest positive subnormal of the
 *     field's dtype if it rounds to 0, so that every node keeps its classification; values are rounded to the dtype on store.  NaN
 *     nodes keep NaN; a node without a point keeps its value, which happens only when there is no interface, and then nothing
 *     changes.
 * Guarantee: a band node with d < band * min_d |h_d| holds the minimum over the whole mesh (any primitive outside its window is at
 * least band |h_d| away along some axis); propagation can only replace it by a point whose computed distance is smaller in the last
 * bits.  Elsewhere |phi| is the distance to a point on the mesh, never less than the true distance up to rounding.  band >= 1
 * (3 in the Python and Julia wrappers: WENO5 reads 3 nodes on each side, so every value a stage reads near the interface is
 * exact), else LSM_ERR_ARG.  Scalar, non-separable fields with every n_d >= 2, else LSM_ERR_ARG; nranks > 1: LSM_ERR_UNSUPPORTED
 * (slab decomposition is not supported).  Boundary conditions play no role and are not required; on a periodic axis nodes 1 and
 * n can therefore get different values.
 * Asynchronous when band_nodes_out is NULL (no synchronisation, no copy: cheap in a prehook); otherwise one synchronisation and
 * an 8-byte copy of the number of band nodes.  Bumps the field's version like every other write, so CFL caches, halos and
 * expression fills see the new data.  Scratch: 16 N + 16 bytes per node (two point buffers of N doubles, two 8-byte keys of the band
 * scan), persistent in the context and grown on demand (8.6 GB for a 512^3 3-D field). */
int32_t lsm_redistance(lsm_ctx* ctx, lsm_field* phi, int32_t band, int64_t* band_nodes_out);

/* ---- closest-point extension: F(x) <- F at the closest point of x on phi's zero-level-set mesh, on the device -----------------
 * The reference extends a speed off the interface with extend_along_normals! (velocityextension.jl:20-78, upwind pseudo-time steps;
 * lsm_extend_along_normals here), usually next to reinitialize! in the loop.  lsm_extend_closest_point gives each node the value of
 * F, interpolated linearly on the mesh, at the closest point lsm_redistance(ctx, phi, band, ...) finds for it, in one call.
 *  - geometry: exactly lsm_redistance's (the same primitives, band scan and winning primitive, closest point, jump-flooding passes
 *    and tie rule), so every node ends up with the point lsm_redistance uses, bit for bit.  Arithmetic in double, each operation
 *    rounded, no FMA.
 *  - vertex value: a mesh vertex lies on the lattice edge (a, b), a = w_i, b = w_j, i < j, as the extraction defines them, at
 *    t = s_a / (s_a - s_b), the t of its coordinates; its value is F_v = Fa + t (Fb - Fa), Fa = double(F[a]), Fb = double(F[b]).
 *  - value at the closest point, following the branch the closest-point routine took, with F0, F1, F2 the values of the
 *    primitive's vertices in the extraction's order: 1-D F_v; 2-D F0 + t (F1 - F0) with the clamped t of the projection, or F0 when
 *    a == b; 3-D, Ericson's regions: vertex a / b / c F0 / F1 / F2, edge ab F0 + v (F1 - F0), edge ac F0 + w (F2 - F0), edge bc
 *    F1 + w (F2 - F1), the interior (F0 + (F1 - F0) v) + (F2 - F0) w, with the routine's own v and w; the degenerate fallback
 *    uses the segment it picked with that segment's t (its first vertex's value when the segment is a point).  These forms return
 *    a constant F exactly, which barycentric u F0 + v F1 + w F2 would not.  A NaN in F gives NaN wherever it enters.
 *  - propagation: each jump-flooding pass carries the value with the point; the winning candidate's value wins.
 *  - write: every node that has a point and a non-NaN phi gets F = value, rounded to F's dtype.  NaN-phi nodes keep their F, and
 *    so does every node when there is no interface.  With redistance_phi != 0 the same call also writes phi exactly as
 *    lsm_redistance(ctx, phi, band, ...) would (bit for bit): one scan for the usual reinitialise-and-extend prehook.
 * F and phi are scalar, non-separable fields of this context on the same grid (n, lc, h), F is not phi, band >= 1 and every
 * n_d >= 2, else LSM_ERR_ARG; F's dtype may differ from phi's.  nranks > 1: LSM_ERR_UNSUPPORTED (slab decomposition is not
 * supported).  No boundary conditions are needed.  Asynchronous when band_nodes_out is NULL; otherwise one synchronisation and an
 * 8-byte copy of the number of band nodes.  Bumps F's version, and phi's when phi is written, so CFL caches and expression fills
 * see the new data.  Scratch: lsm_redistance's plus two value buffers, 16 N + 32 bytes per node in the same context buffer
 * (10.7 GB for a 512^3 3-D field). */
int32_t lsm_extend_closest_point(lsm_ctx* ctx, lsm_field* F, lsm_field* phi, int32_t band, int32_t redistance_phi, int64_t* band_nodes_out);

/* ---- cubic interpolant: phi between the nodes, as a degree-3 polynomial per cell, on the device --------------------------------
 * The reference's reinitialize! (interpolation.jl, bernstein.jl) interpolates phi cell by cell with a tensor-product Bernstein patch
 * of degree 3 fitted to the 4^N surrounding nodes.  With 4 nodes per axis that fit interpolates exactly, so the patch is the same
 * polynomial as the tensor-product Lagrange interpolant below; the two agree as polynomials, not bit for bit (the reference solves
 * with a pseudo-inverse of the Kronecker matrix).  In double, each operation rounded, no FMA:
 *  - u_d = (y_d - lc_d) / h_d; y is inside the box when 0 <= u_d <= n_d - 1 for every d (mirrored grids, h_d < 0, included).
 *  - cell c_d = min(floor(u_d), n_d - 2); stencil start s_d = min(max(c_d - 1, 0), n_d - 4): the 4 nodes s_d .. s_d + 3, one-sided
 *    at the box faces, so no boundary conditions are used (needs n_d >= 4); xi = u_d - s_d, a = xi - 1, b = xi - 2, c = xi - 3.
 *  - weights  L0 = ((a b) c) / -6, L1 = ((xi b) c) / 2, L2 = ((xi a) c) / -2, L3 = ((xi a) b) / 6;
 *             L0' = ((a b + a c) + b c) / -6, L1' = ((xi b + xi c) + b c) / 2, L2' = ((xi a + xi c) + a c) / -2,
 *             L3' = ((xi a + xi b) + a b) / 6;
 *             L0'' = ((a + b) + c) / -3, L1'' = (xi + b) + c, L2'' = -((xi + a) + c), L3'' = ((xi + a) + b) / 3.
 *    At integer xi the L are exactly 0 or 1, so the interpolant reproduces the node values.
 *  - contraction over axis 1, then 2, then 3, each sum ((t0 + t1) + t2) + t3 with t_k = w_k * double(phi[s + k]).  The value uses L
 *    on every axis; d/dy_d uses L' on axis d and is divided by h_d after the contraction; d2/dy_d dy_e uses L'' on axis d (d = e) or
 *    L' on both axes (d < e) and is divided as (S / h_d) / h_e; the Hessian is symmetric (entry (e, d) = entry (d, e)).
 *  - a NaN node in the stencil gives NaN.
 * lsm_interpolate_cubic evaluates it at npts points: pts is npts x ndim (AoS, host), val npts, grad npts x ndim, hess
 * npts x ndim x ndim (host); any output may be NULL.  A point outside the box gets NaN in every output.  Blocking: one host-to-
 * device copy of the points, one kernel, device-to-host copies of the requested outputs, through the context's persistent scratch.
 * Scalar, non-separable fields of this context with every n_d >= 4, npts >= 0 and pts not NULL when npts > 0, else LSM_ERR_ARG;
 * nranks > 1: LSM_ERR_UNSUPPORTED (slab decomposition is not supported). */
int32_t lsm_interpolate_cubic(lsm_ctx* ctx, lsm_field* phi, int64_t npts, const double* pts, double* val, double* grad, double* hess);

/* ---- cubic closest-point redistancing: phi <- the signed distance to the zero set of its cubic interpolant, on the device --------
 * lsm_redistance's passes, then a Newton refinement of every closest point on the interpolant P above, as the reference's
 * reinitialize! refines its KD-tree seeds (reinitializer.jl:12-42, sdf.jl).  Here the seed of node x is the linear closest point y0
 * lsm_redistance finds (an O(h^2)-accurate seed), so classification, NaN nodes and the no-interface case are lsm_redistance's.  In
 * double, each operation rounded, no FMA, with lsm_redistance's dot and dist; P, g = grad P and H = the Hessian of P at y are the
 * interpolant at y (the patch of the cell containing y):
 *  - g = grad P(y0); lambda = dot(x - y0, g) / dot(g, g); y = y0.
 *  - up to 20 iterations: evaluate P, g, H at y; solve the (N+1) x (N+1) system M z = r of the KKT conditions of min |y - x| on
 *    P = 0, M = [[I + lambda H, g], [g^T, 0]] (diagonal 1 + lambda H_dd, off-diagonal lambda H_de), r = (-((y_d - x_d) + lambda g_d),
 *    -P), by Gaussian elimination with partial pivoting (for column k the first row i >= k of largest |M_ik| is swapped into row k;
 *    f = M_ik / M_kk, M_ij = M_ij - f M_kj for j > k, r_i = r_i - f r_k; then z_i = (((r_i - M_i,i+1 z_i+1) - ...) - M_iN z_N) / M_ii
 *    for i = N .. 0); y_d = y_d + z_d, lambda = lambda + z_N; converged when dist(z, 0) <= 1e-10 min_d |h_d| (z's first N entries).
 *  - fallback to y0 when: dot(g, g) is 0 or not finite at the start, or lambda is not finite; a value of P, g or H at y is not
 *    finite; a pivot is 0; z, y or lambda is not finite; y leaves the box; dist(y, y0) > 2 max_d |h_d|; or 20 iterations pass
 *    without convergence.  The node then gets exactly lsm_redistance's distance, so the call is never worse than lsm_redistance
 *    on a node.
 *  - NaN nodes and nodes without a point are not refined; lsm_redistance's write pass then stores -d / +d (raised to the smallest
 *    subnormal) with d = dist(x, y).
 * band >= 1, scalar non-separable fields of this context with every n_d >= 4, else LSM_ERR_ARG; nranks > 1: LSM_ERR_UNSUPPORTED
 * (slab decomposition is not supported).  No boundary conditions are needed.  Asynchronous when both out-pointers are NULL;
 * otherwise one synchronisation and a 16-byte copy of the number of band nodes (as lsm_redistance counts them) and of the nodes
 * that fell back.  Bumps the field's version.  Scratch: lsm_redistance's (the refined points go to its spare point buffer). */
int32_t lsm_redistance_cubic(lsm_ctx* ctx, lsm_field* phi, int32_t band, int64_t* band_nodes_out, int64_t* fallback_nodes_out);

/* ---- level-set integrals: how much region and interface the zero level set holds, and integrals of a field over them -----------
 * The reference integrates over implicit domains on the host (ext/ImplicitIntegrationExt.jl); lsm_volume and lsm_perimeter above
 * give its smoothed-Heaviside and smoothed-delta sums, whose values depend on the smoothing width.  lsm_level_set_integrals measures
 * the sharp piecewise-linear geometry of lsm_interface_extract instead, on the device, and returns
 *   out[0] = |{s <= 0}|,  out[1] = |{s = 0}|,  out[2] = integral of F over {s <= 0},  out[3] = integral of F over {s = 0}
 * (out[2] and out[3] are NaN when F is NULL).  In double, each operation rounded, no FMA:
 *  - geometry: s = double(phi) - level; a node is inside if s <= 0, outside if s > 0, invalid if s is NaN.  Cells, simplices, cut
 *    edges, vertex coordinates and primitives are exactly those of lsm_interface_extract; a simplex with an invalid vertex
 *    contributes nothing to any output.  The region is {P1(s) <= 0}, P1 the piecewise-linear interpolant on the triangulation.
 *  - F is the P1 interpolant of its node values f = double(F): at the crossing of the simplex edge (w_x, w_y), x < y, its value is
 *    Fa + t (Fb - Fa), t = s_a / (s_a - s_b), a = w_x, b = w_y (lsm_extend_closest_point's vertex value).  A sub-simplex contributes
 *    its volume times the mean of F over its N+1 vertices, (((v0 + v1) + v2) + v3) / (N + 1); a primitive its measure times the mean
 *    over its N vertices, (v0 + v1) / 2 or ((v0 + v1) + v2) / 3.  Both are exact for a linear F.  A NaN in F propagates.
 *  - region (out[0], out[2]), with V = (|h1| |h2|) |h3| and Vs = V / N!:
 *      a cell whose 2^N corners are all valid and inside contributes V, and V ((f0 + f7) / 4 + (((((f1 + f2) + f3) + f4) + f5) + f6) / 12)
 *      to the integral of F (2-D: V ((f0 + f3) / 3 + (f1 + f2) / 6); 1-D: V ((f0 + f1) / 2); corner k = c + sum_d bit_d(k) e_d):
 *      that is the sum over its simplices, and it makes a fully inside box exact;  a cell whose corners are all valid and outside
 *      contributes nothing;  every other cell contributes its simplices in order:
 *      a simplex whose vertices are all inside contributes Vs; a cut simplex the volume of its inside part, in fractions of Vs from
 *      the crossing parameters of its cut edges:
 *      - one lone vertex q (the only inside one; in 1-D always): with u_j = s_q / (s_q - s_oj) for the other vertices o_0 < o_1 < ..
 *        in chain order, the corner simplex (q, P_qo0, ..) of volume Vs ((u_0 u_1) u_2).  1-D: the segment; 2-D and 3-D: a corner.
 *      - 2-D, one lone outside vertex q, others r < s: the quad as the triangles (r, s, P_qs) of volume Vs (1 - u_s) and
 *        (r, P_qs, P_qr) of volume Vs (u_s (1 - u_r)).
 *      - 3-D, one lone outside vertex q: the tet minus the corner tet at q, volume Vs (1 - (u_0 u_1) u_2), integral of F
 *        Vs mean(f over the tet) - (Vs ((u_0 u_1) u_2)) mean(corner tet).
 *      - 3-D, inside {a < b}, outside {c < d} (the 2–2 prism), tau_xy = s_x / (s_x - s_y): the three tets (a, P_ac, P_ad, P_bd),
 *        (a, P_ac, P_bc, P_bd), (a, b, P_bc, P_bd) of volumes Vs ((tau_ac tau_ad) (1 - tau_bd)), Vs ((tau_ac (1 - tau_bc)) tau_bd),
 *        Vs (tau_bc tau_bd).
 *  - interface (out[1], out[3]): the sum of the primitive measures, from the extraction's vertex coordinates v0, v1, v2: 1-D one per
 *    point; 2-D sqrt(dx dx + dy dy), d = v1 - v0; 3-D sqrt((cx cx + cy cy) + cz cz) / 2, c = (v1 - v0) x (v2 - v0) with
 *    cx = uy wz - uz wy, cy = uz wx - ux wz, cz = ux wy - uy wx, u = v1 - v0, w = v2 - v0.  This is the measure of the mesh
 *    lsm_interface_extract returns, primitive by primitive; a lattice plane of exact zeros is counted once (from the cells on its
 *    outside), since the cells on its inside have no cut edge.
 *  - summation: each plane of cells (the cells sharing the index of the last axis) is summed to one partial per output, in a fixed
 *    order that depends only on the plane's shape; then the planes are summed in increasing order.  The result does not depend
 *    on the slab decomposition, bit for bit.
 * F, when given, is a scalar, non-separable field of this context on phi's grid (n, lc and h), of either dtype, and may be phi itself;
 * phi is a scalar, non-separable field of this context with every n_d >= 2; level is finite; out is not NULL; else LSM_ERR_ARG.
 * Boundary conditions play no role (periodic axes: node n duplicates node 1, so no cell wraps).  With nranks > 1 the call is
 * collective: rank r integrates the cell planes whose lower corner it owns (exchanging the ghost planes of phi, and of F, when they
 * are stale), writes its plane partials into a buffer of n_last - 1 planes that is zero elsewhere, all-reduces the buffer (every
 * entry has one non-zero contributor, so the sum is exact) and sums the planes as one GPU does: every rank returns the single-GPU
 * value bit for bit.  Blocking: one synchronisation and a 32-byte copy; the plane partials (32 bytes per plane) live in the
 * context's persistent reduction scratch, so the last extraction and the redistancing scratch are untouched.  Two kernel launches. */
int32_t lsm_level_set_integrals(lsm_ctx* ctx, lsm_field* phi, lsm_field* F, double level, double* out);
/* lsm_level_set_integrals on every rank of a lsm_ctx_create_multi box, on one host thread per GPU; F may be NULL (no F on any rank).
 * out receives the 4 results, which are identical on every rank. */
int32_t lsm_multi_level_set_integrals(int32_t n, lsm_ctx* const* ctx, lsm_field* const* phi, lsm_field* const* F,
                                      double level, double* out);

/* ---- diagnostics (test harness; SURVEY.md §2.2 K6) -------------------------------------------- */
/* max |a - b| over all owned nodes, all-reduced over ranks. */
int32_t lsm_max_abs_diff(lsm_ctx* ctx, const lsm_field* a, const lsm_field* b, double* out);

#ifdef __cplusplus
}
#endif
#endif /* LSM_B200_H */
