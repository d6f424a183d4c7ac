// lsm_api.cu — implementation of the C ABI declared in include/lsm_b200.h.
//
// Host-side runtime of the engine: contexts (one process == one GPU == one rank), device
// fields with ghost planes for slab decomposition, NCCL halo exchange overlapped with interior
// compute, the CFL cache, and the step loop of _integrate! (timestepping.jl:101-122).
// No CPU fallback exists: every compute entry point needs a CUDA device.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/lsm_b200.h"
#include "lsm_dev.cuh"
#include "lsm_kernels.h"
#include "nccl_dyn.h"
#include <nvtx3/nvToolsExt.h>     // header-only NVTX v3: ranges are no-ops unless a profiler injects itself

using namespace lsm;

namespace {

thread_local std::string g_err;

// NVTX ranges around the step loop, every RK stage and the halo exchange (SURVEY.md §5): visible in Nsight Systems timelines,
// free otherwise.  LSM_B200_NVTX=0 turns even the (tiny) call overhead off.
struct NvtxRange {
    static bool enabled() { static const bool on = [] { const char* e = getenv("LSM_B200_NVTX"); return !(e && *e == '0'); }(); return on; }
    bool on;
    explicit NvtxRange(const char* name) : on(enabled()) { if (on) nvtxRangePushA(name); }
    ~NvtxRange() { if (on) nvtxRangePop(); }
};

int32_t fail(int32_t code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
    return code;
}

#define CU(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) \
    return fail(e_ == cudaErrorMemoryAllocation ? LSM_ERR_OOM : LSM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
#define NC(expr) do { ncclResult_t r_ = (expr); if (r_ != ncclSuccess) \
    return fail(LSM_ERR_NCCL, "%s failed: %s (%s:%d)", #expr, nccl().GetErrorString ? nccl().GetErrorString(r_) : "?", __FILE__, __LINE__); } while (0)
#define TRY(expr) do { int32_t rc_ = (expr); if (rc_ != LSM_OK) return rc_; } while (0)

constexpr int HALO = 3;    // ghost planes per side of the decomposed axis (WENO5 reach)

inline double jl_min(double a, double b) {
    return (std::isnan(a) || std::isnan(b)) ? std::numeric_limits<double>::quiet_NaN() : (b < a ? b : a);
}
inline double jl_eps(double x) {    // Base.eps(::Float64)
    x = std::fabs(x);
    return std::nextafter(x, std::numeric_limits<double>::infinity()) - x;
}

// What is known about the CFL maximum of one (term kind, stored or separable coefficient field) at one version of the field's data.
//   * The last exact answer of a full reduction pass, for its scale g.
//   * The candidate set of a TIME-SCALED field, which answers every scale without touching the device again (no reduction pass,
//     no 8-byte D2H, no host sync per step).  The reference's per-node quantity is s_i(g) = sum_d fl(|fl(u_d g)| / h_d)
//     (levelsetterms.jl:90-96) = |g| S_i (1 + theta), |theta| <= 4.5e-16, with S_i = sum_d |u_d| / h_d.  A node with
//     S_i < (1 - 1e-12) max_j S_j can therefore never attain max_i s_i(g) for ANY g, so the maximum over the (few) candidate nodes
//     above that threshold, evaluated on the host with the same IEEE operations, is bit-identical to the full reduction.  For the
//     scalar coefficients (normal motion, curvature) |fl(v g)| is monotone in |v|, and the same argument holds with S_i = |v_i|.
struct CflMemo {
    int kind = 0; const void* field = nullptr; uint64_t version = 0;
    bool have_bits = false; int scaled = 0; double g = 0; unsigned long long bits = 0;     // last full pass
    int ncomp = 0, seen = 0;     // candidates: coefficient components, time-scaled requests seen
    bool built = false, overflow = false;
    std::vector<double> tup;     // distinct raw coefficient tuples of the candidate nodes (all ranks)
};
constexpr int CAND_CAP = 8192;   // per rank

}  // namespace

struct lsm_ctx {
    int device = 0, rank = 0, nranks = 1, sm_count = 148;
    cudaStream_t stream = nullptr, comm = nullptr, bstream = nullptr;     // compute, halo traffic, boundary slabs (high priority)
    cudaEvent_t ev_boundary = nullptr, ev_halo = nullptr, ev_main = nullptr;
    ncclComm_t nccl_comm = nullptr;
    unsigned long long* d_scalar = nullptr;     // device scalar for reductions
    unsigned long long* h_scalar = nullptr;     // pinned
    lsm_counters cnt{};
    int opt_kernel = 0, opt_time = 0, opt_cfl_cache = 1, opt_overlap = 1;
    int interior_first = 0;     // LSM_B200_INTERIOR_FIRST (experiments): round-2's original launch order of the overlapped stage
    std::vector<CflMemo> cfl_memo;
    int opt_cand = 1;           // LSM_OPT_CFL_CANDIDATES
    int opt_resident = 1;       // LSM_OPT_RESIDENT
    int stage_skip_zero_u = 0;  // transient: set by lsm_extend_along_normals around its stages (StageParams::skip_zero_u)
    unsigned* d_cand_count = nullptr; double* d_cand = nullptr; double* h_cand = nullptr;   // candidate staging (device / pinned)
    void* stage[2] = {nullptr, nullptr};        // AoS <-> SoA staging chunks of vector-field transfers (allocated on first use)
    cudaEvent_t ev_stage[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    void* d_work = nullptr; size_t d_work_bytes = 0;       // persistent scratch of the reductions / getindex (grown on demand)
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed;     // pending stage timings
    std::vector<cudaEvent_t> ev_pool;
    cudaEvent_t ev_user[8] = {};
    int opt_graph = 1;          // lsm_integrate replays a captured CUDA graph of the stage launches on small grids
    // the mesh of the last lsm_interface_extract (persistent, grown on demand): nverts x ndim doubles, nverts keys, nprims x ndim int32
    void* d_iface = nullptr; size_t d_iface_bytes = 0;
    bool iface_valid = false;
    int iface_ndim = 0;
    int64_t iface_nv = 0, iface_np = 0;
    // lsm_redistance scratch (persistent, grown on demand): two point buffers of ndim doubles per node (ndim + 1 for
    // lsm_extend_closest_point: the value at the point), the two 8-byte keys of the band scan per node, three counters (listed
    // cells, band nodes, lsm_redistance_cubic's fallbacks); lsm_interpolate_cubic's points and results use the same buffer
    void* d_redist = nullptr; size_t d_redist_bytes = 0;
};

struct lsm_field {
    lsm_ctx* ctx = nullptr;
    int ndim = 0, dtype = LSM_F64, ncomp = 1;
    int nglob[3] = {1, 1, 1}, n[3] = {1, 1, 1};
    int first_last = 0;          // global 0-based index of the first owned plane of the last dim
    int halo = 0;                // stored ghost planes per side (last dim)
    double lc[3] = {0, 0, 0}, hc[3] = {1, 1, 1}, h[3] = {1, 1, 1};
    lsm_bc bc[3][2];
    bool has_bc = false;
    void* base = nullptr;        // allocation start
    void* p = nullptr;           // first owned node
    long plane = 1;              // elements per plane of the last dim
    long owned = 1;              // owned elements per component
    long cstride = 0;            // component stride (SoA)
    uint64_t version = 1;
    bool halo_valid = false;
    lsm_field* buf1 = nullptr;   // RK stage buffers (timestepping.jl:126,141,168)
    lsm_field* buf2 = nullptr;
    // separable coefficient
    bool separable = false;
    double scale[3] = {1, 1, 1};
    double* d_tabs = nullptr;
    const double* tab[3][3] = {};
    // expressions attached by lsm_field_set_expr (LSM_COEF_EXPR)
    const ExprKernel* expr = nullptr;
    bool expr_filled = false;    // the data holds the expressions at expr_t, materialised at version expr_ver
    double expr_t = 0;
    uint64_t expr_ver = 0;
    int expr_cfl_kind = 0;       // CFL quantity the last fill reduced into d_expr_cfl (ExprArgs::cfl_kind)
    bool expr_cfl_read = false;  // expr_cfl_bits holds that maximum, all-reduced over ranks
    unsigned long long expr_cfl_bits = 0;
    unsigned long long* d_expr_cfl = nullptr;
};

namespace {

size_t esize(int dtype) { return dtype == LSM_F32 ? 4 : 8; }

int32_t ctx_common_init(lsm_ctx* c) {
    CU(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, c->device));
    if (prop.major < 10) return fail(LSM_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", c->device, prop.major, prop.minor);
    c->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    {   // the boundary-slab stream and the halo-exchange stream outrank the compute stream: their (small) grids are placed first
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(cudaStreamCreateWithPriority(&c->comm, cudaStreamNonBlocking, getenv("LSM_B200_INTERIOR_FIRST") ? lo : hi));
        CU(cudaStreamCreateWithPriority(&c->bstream, cudaStreamNonBlocking, hi));
    }
    CU(cudaEventCreateWithFlags(&c->ev_main, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_boundary, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_halo, cudaEventDisableTiming));
    CU(cudaMalloc(&c->d_scalar, 64));
    CU(cudaMallocHost(&c->h_scalar, 64));
    if (getenv("LSM_B200_NO_OVERLAP")) c->opt_overlap = 0;
    if (getenv("LSM_B200_INTERIOR_FIRST")) c->interior_first = 1;
    if (getenv("LSM_B200_NO_GRAPH")) c->opt_graph = 0;
    return LSM_OK;
}

void slab_plan(int n_last, int nranks, int rank, int* first, int* count) {
    const int base = n_last / nranks, rem = n_last % nranks;
    *count = base + (rank < rem ? 1 : 0);
    *first = rank * base + (rank < rem ? rank : rem);
}

int32_t field_alloc(lsm_ctx* ctx, int ndim, const int32_t* n, int dtype, int ncomp, const double* lc, const double* hc,
                    bool with_halo, lsm_field** out) {
    if (!ctx || !n || !out) return fail(LSM_ERR_ARG, "null argument");
    if (ndim < 1 || ndim > 3) return fail(LSM_ERR_ARG, "ndim must be 1, 2 or 3 (got %d)", ndim);
    if (dtype != LSM_F32 && dtype != LSM_F64) return fail(LSM_ERR_ARG, "bad dtype %d", dtype);
    if (ncomp != 1 && ncomp != ndim) return fail(LSM_ERR_ARG, "ncomp must be 1 or ndim");
    lsm_field* f = new (std::nothrow) lsm_field();
    if (!f) return fail(LSM_ERR_OOM, "host allocation failed");
    f->ctx = ctx; f->ndim = ndim; f->dtype = dtype; f->ncomp = ncomp;
    for (int d = 0; d < 3; ++d) {
        f->nglob[d] = d < ndim ? n[d] : 1;
        f->n[d] = f->nglob[d];
        f->lc[d] = (d < ndim && lc) ? lc[d] : 0.0;
        f->hc[d] = (d < ndim && hc) ? hc[d] : 1.0;
        if (d < ndim && n[d] < 1) { delete f; return fail(LSM_ERR_ARG, "n[%d] = %d", d, n[d]); }
        f->h[d] = d < ndim ? (f->hc[d] - f->lc[d]) / double(f->nglob[d] - 1) : 1.0;    // meshes.jl:109-110
        f->bc[d][0] = {LSM_BC_NONE, 0}; f->bc[d][1] = {LSM_BC_NONE, 0};
    }
    const int last = ndim - 1;
    int first = 0, count = f->nglob[last];
    if (ctx->nranks > 1) {
        slab_plan(f->nglob[last], ctx->nranks, ctx->rank, &first, &count);
        if (count < HALO + 1) { delete f; return fail(LSM_ERR_ARG, "slab of %d planes is thinner than %d; use fewer ranks", count, HALO + 1); }
    }
    f->first_last = first; f->n[last] = count;
    f->plane = 1; for (int d = 0; d < last; ++d) f->plane *= f->n[d];
    f->owned = f->plane * f->n[last];
    f->halo = (with_halo && ctx->nranks > 1 && ncomp == 1) ? HALO : 0;
    const long per_comp = f->owned + 2L * f->halo * f->plane;
    f->cstride = per_comp;
    cudaError_t e = cudaMalloc(&f->base, (size_t)per_comp * ncomp * esize(dtype));
    if (e != cudaSuccess) { delete f; return fail(e == cudaErrorMemoryAllocation ? LSM_ERR_OOM : LSM_ERR_CUDA, "cudaMalloc of %.1f MB failed: %s", per_comp * ncomp * esize(dtype) / 1e6, cudaGetErrorString(e)); }
    f->p = static_cast<char*>(f->base) + (size_t)f->halo * f->plane * esize(dtype);
    if (f->halo) cudaMemsetAsync(f->base, 0, (size_t)per_comp * esize(dtype), ctx->stream);
    *out = f;
    return LSM_OK;
}

void field_free(lsm_field* f) {
    if (!f) return;
    if (f->buf1) field_free(f->buf1);
    if (f->buf2) field_free(f->buf2);
    if (f->base) cudaFree(f->base);
    if (f->d_tabs) cudaFree(f->d_tabs);
    if (f->d_expr_cfl) cudaFree(f->d_expr_cfl);
    delete f;
}

// grows one of the context's persistent device buffers (*buf, *size bytes) to at least `need` bytes; the old buffer is freed once
// the context's stream has drained, so no work in flight still reads it
int32_t grow_scratch(lsm_ctx* c, void** buf, size_t* size, size_t need) {
    if (need > *size) {
        CU(cudaStreamSynchronize(c->stream));
        if (*buf) cudaFree(*buf);
        *buf = nullptr; *size = 0;
        CU(cudaMalloc(buf, need));
        *size = need;
    }
    return LSM_OK;
}

// persistent device scratch of the context (reductions, getindex): grown on demand, never freed per call
int32_t ctx_scratch(lsm_ctx* c, size_t bytes, void** out) {
    TRY(grow_scratch(c, &c->d_work, &c->d_work_bytes, std::max<size_t>(bytes, 1u << 16)));
    *out = c->d_work;
    return LSM_OK;
}

int32_t ensure_buffers(lsm_field* phi, int nbuf) {
    lsm_field** slots[2] = {&phi->buf1, &phi->buf2};
    for (int b = 0; b < nbuf; ++b) {
        if (*slots[b]) continue;
        lsm_field* nb = nullptr;
        TRY(field_alloc(phi->ctx, phi->ndim, phi->nglob, phi->dtype, 1, phi->lc, phi->hc, true, &nb));
        std::memcpy(nb->bc, phi->bc, sizeof phi->bc);
        nb->has_bc = phi->has_bc;
        *slots[b] = nb;
    }
    return LSM_OK;
}

template <class T>
View<T> make_view(const lsm_field* f) {
    View<T> v;
    v.p = static_cast<const T*>(f->p);
    for (int d = 0; d < 3; ++d) v.n[d] = f->n[d];
    v.s1 = f->ndim > 1 ? (long)f->n[0] : 0;
    v.s2 = f->ndim > 2 ? (long)f->n[0] * f->n[1] : 0;
    v.halo = f->halo; v._pad = 0;
    const lsm_ctx* c = f->ctx;
    const int last = f->ndim - 1;
    for (int d = 0; d < 3; ++d)
        for (int s = 0; s < 2; ++s) { v.bc[d][s].kind = f->bc[d][s].kind; v.bc[d][s].P = f->bc[d][s].P; }
    if (c->nranks > 1 && f->halo) {
        const bool periodic = f->bc[last][0].kind == LSM_BC_PERIODIC;
        if (c->rank > 0 || periodic) v.bc[last][0].kind = BC_HALO;
        if (c->rank < c->nranks - 1 || periodic) v.bc[last][1].kind = BC_HALO;
    }
    return v;
}

double term_scale(const lsm_term& t, double time, const double* gscale, int k) {
    switch (t.tscale_kind) {
        case LSM_TS_COS:  return std::cos(M_PI * time / t.tparam);
        case LSM_TS_HOST: return gscale ? gscale[k] : 1.0;
        default:          return 1.0;
    }
}

int32_t make_term_dev(const lsm_field* phi, const lsm_term& t, double g, TermDev* out) {
    TermDev d{};
    if (t.kind < LSM_TERM_ADVECTION || t.kind > LSM_TERM_EIKONAL) return fail(LSM_ERR_ARG, "bad term kind %d", t.kind);
    d.kind = t.kind; d.scheme = t.scheme; d.coef_kind = t.coef_kind;
    d.scaled = t.tscale_kind != LSM_TS_NONE; d.g = g;
    for (int i = 0; i < 3; ++i) d.cval[i] = t.cval[i];
    if (t.kind == LSM_TERM_ADVECTION && t.scheme != LSM_UPWIND && t.scheme != LSM_WENO5) return fail(LSM_ERR_ARG, "bad scheme %d", t.scheme);
    if (t.kind == LSM_TERM_EIKONAL && t.coef_kind != LSM_COEF_NONE && t.coef_kind != LSM_COEF_FIELD)
        return fail(LSM_ERR_ARG, "eikonal term takes a frozen S0 field or no coefficient");
    if (t.kind != LSM_TERM_EIKONAL && t.coef_kind == LSM_COEF_NONE) return fail(LSM_ERR_ARG, "term %d needs a coefficient", t.kind);
    if (t.coef_kind == LSM_COEF_FIELD || t.coef_kind == LSM_COEF_SEPARABLE || t.coef_kind == LSM_COEF_EXPR) {
        const lsm_field* cf = t.field;
        if (!cf) return fail(LSM_ERR_ARG, "coefficient field is NULL");
        if (cf->ctx != phi->ctx) return fail(LSM_ERR_ARG, "coefficient field belongs to another context");
        const int want = t.kind == LSM_TERM_ADVECTION ? phi->ndim : 1;
        if (cf->ndim != phi->ndim || cf->ncomp != want) return fail(LSM_ERR_ARG, "coefficient field has ndim=%d ncomp=%d, expected %d/%d", cf->ndim, cf->ncomp, phi->ndim, want);
        for (int a = 0; a < phi->ndim; ++a)
            if (cf->nglob[a] != phi->nglob[a]) return fail(LSM_ERR_ARG, "coefficient field shape mismatch along dim %d", a + 1);
        if (t.coef_kind == LSM_COEF_SEPARABLE) {
            if (!cf->separable) return fail(LSM_ERR_ARG, "LSM_COEF_SEPARABLE needs a field from lsm_field_create_separable");
            for (int c = 0; c < 3; ++c) { d.cval[c] = cf->scale[c]; for (int a = 0; a < 3; ++a) d.tab[c][a] = cf->tab[c][a]; }
        } else {
            if (cf->separable) return fail(LSM_ERR_ARG, "separable field passed as LSM_COEF_FIELD");
            if (cf->dtype != phi->dtype) {
                if (cf->dtype == LSM_F64 && phi->dtype == LSM_F32) d.coef_f64 = 1;
                else return fail(LSM_ERR_UNSUPPORTED, "Float32 coefficient with a Float64 state is not supported");
            }
            d.coef = cf->p; d.cstride = cf->cstride;
            d.coef_kind = COEF_FIELD;       // an expression field is read like a stored one once materialised
        }
    }
    *out = d;
    return LSM_OK;
}

// ---- expression coefficients (lsm_field_set_expr; the kernel is generated in lsm_expr.cu) ----------------------------------
// Materialise the expressions of f at time t; cfl_kind != 0 also reduces that CFL quantity of the rounded values into d_expr_cfl.
int32_t expr_fill(lsm_field* f, double t, int cfl_kind) {
    lsm_ctx* c = f->ctx;
    ExprArgs A{};
    A.dst = f->p; A.cfl = f->d_expr_cfl; A.cstride = f->cstride; A.first_last = f->first_last;
    A.f64 = f->dtype == LSM_F64; A.cfl_kind = cfl_kind; A.t = t;
    for (int d = 0; d < 3; ++d) { A.n[d] = f->n[d]; A.lc[d] = f->lc[d]; A.h[d] = d < f->ndim ? f->h[d] : 0.0; }
    if (cfl_kind) CU(cudaMemsetAsync(f->d_expr_cfl, 0, 8, c->stream));
    cudaError_t e = launch_expr_fill(f->expr, A, c->sm_count, c->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "expression kernel launch failed: %s", cudaGetErrorString(e));
    c->cnt.kernel_launches += 1;
    f->version++; f->halo_valid = false;
    f->expr_filled = true; f->expr_t = t; f->expr_ver = f->version;
    f->expr_cfl_kind = cfl_kind; f->expr_cfl_read = false;
    return LSM_OK;
}

// Make f hold its expressions' values at time t for a term of kind term_kind: nothing to do when it already holds them (same
// time, or no `t` in the expressions, and not overwritten since) and, with need_cfl, the last fill reduced this kind's CFL
// quantity.  Otherwise one fill, which also reduces that quantity for the next CFL request at t.
int32_t expr_ensure(lsm_field* f, double t, int term_kind, bool need_cfl) {
    const int kind = term_kind == LSM_TERM_ADVECTION ? 1 : 2;
    const bool fresh = f->expr_filled && f->version == f->expr_ver &&
                       (!expr_uses_t(f->expr) || std::memcmp(&f->expr_t, &t, sizeof t) == 0);
    if (fresh && (!need_cfl || f->expr_cfl_kind == kind)) return LSM_OK;
    return expr_fill(f, t, kind);
}

// LSM_COEF_EXPR terms are checked like stored fields.  An expression set without `t` is materialised once and from then on lowered
// to LSM_COEF_FIELD, so the CFL cache, graph replay, the resident and the x-pair kernels apply to it unchanged.  A time-dependent
// one stays LSM_COEF_EXPR: run_stage_t and cfl_term materialise it at the times they need.
int32_t prepare_terms(lsm_field* phi, const lsm_term* terms, int nterms, lsm_term* out) {
    for (int k = 0; k < nterms; ++k) {
        out[k] = terms[k];
        if (terms[k].coef_kind != LSM_COEF_EXPR) continue;
        if (terms[k].tscale_kind != LSM_TS_NONE) return fail(LSM_ERR_ARG, "an expression coefficient takes no time factor: t is already in the expression");
        TermDev td;
        TRY(make_term_dev(phi, terms[k], 1.0, &td));
        lsm_field* f = terms[k].field;
        if (!f->expr) return fail(LSM_ERR_ARG, "LSM_COEF_EXPR needs a field with attached expressions (lsm_field_set_expr)");
        if (!expr_uses_t(f->expr)) {
            TRY(expr_ensure(f, 0.0, terms[k].kind, false));
            out[k].coef_kind = LSM_COEF_FIELD;
        }
    }
    return LSM_OK;
}

// ---- halo exchange (SURVEY.md §8e): whole contiguous planes of the decomposed (last) axis -------
int32_t exchange_halo(lsm_field* f, cudaStream_t s) {
    lsm_ctx* c = f->ctx;
    if (c->nranks == 1 || !f->halo) { f->halo_valid = true; return LSM_OK; }
    NvtxRange nvtx("lsm halo exchange");
    const int last = f->ndim - 1;
    const bool periodic = f->bc[last][0].kind == LSM_BC_PERIODIC;
    const size_t es = esize(f->dtype);
    const size_t bytes = (size_t)HALO * f->plane * es;
    char* p = static_cast<char*>(f->p);
    const int nl = f->n[last], R = c->rank, G = c->nranks;
    auto plane_ptr = [&](int k) { return p + (ptrdiff_t)k * (ptrdiff_t)f->plane * (ptrdiff_t)es; };
    // Wrap-around neighbours honour the reference's periodic rule (boundaryconditions.jl:107-119): node n
    // duplicates node 1, so ghost(n+k) = node(1+k) and ghost(1-k) = node(n-k): the last rank ships its planes
    // nl-4..nl-2 (not its very last plane) upward to rank 0, rank 0 ships its planes 1..3 downward to the last rank.
    const int up = (R + 1 < G) ? R + 1 : (periodic ? 0 : -1);
    const int down = (R > 0) ? R - 1 : (periodic ? G - 1 : -1);
    const int top_first = (R + 1 < G) ? nl - HALO : nl - 1 - HALO;      // planes sent upward
    const int bottom_first = (R > 0) ? 0 : 1;                            // planes sent downward
    NC(nccl().GroupStart());
    // Every rank issues UPWARD traffic first, then DOWNWARD: NCCL matches the sends and receives of a pair of
    // ranks in issue order, and with 2 ranks and a periodic axis both directions join the same pair.
    // (a failing call still closes the group before the error is reported)
    ncclResult_t gr = ncclSuccess;
    auto keep = [&](ncclResult_t r) { if (gr == ncclSuccess) gr = r; };
    if (up >= 0)   { keep(nccl().Send(plane_ptr(top_first), bytes, ncclInt8, up, c->nccl_comm, s)); c->cnt.halo_bytes_sent += (int64_t)bytes; }
    if (down >= 0) { keep(nccl().Recv(plane_ptr(-HALO), bytes, ncclInt8, down, c->nccl_comm, s)); }
    if (down >= 0) { keep(nccl().Send(plane_ptr(bottom_first), bytes, ncclInt8, down, c->nccl_comm, s)); c->cnt.halo_bytes_sent += (int64_t)bytes; }
    if (up >= 0)   { keep(nccl().Recv(plane_ptr(nl), bytes, ncclInt8, up, c->nccl_comm, s)); }
    keep(nccl().GroupEnd());
    NC(gr);
    f->halo_valid = true;
    return LSM_OK;
}

cudaEvent_t pool_event(lsm_ctx* c) {
    if (!c->ev_pool.empty()) { cudaEvent_t e = c->ev_pool.back(); c->ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr; cudaEventCreate(&e); return e;
}

void resolve_timings(lsm_ctx* c) {
    if (c->timed.empty()) return;
    cudaStreamSynchronize(c->stream);
    for (auto& pr : c->timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
            c->cnt.last_stage_ms = ms; c->cnt.sum_stage_ms += ms; c->cnt.timed_stages += 1;
        }
        c->ev_pool.push_back(pr.first); c->ev_pool.push_back(pr.second);
    }
    c->timed.clear();
}

template <class T>
int32_t launch_stage_range(lsm_ctx* c, int ndim, StageParams<T>& P, int r0, int r1, cudaStream_t st = nullptr) {
    if (!st) st = c->stream;
    if (r1 <= r0) return LSM_OK;
    P.r0 = r0; P.r1 = r1;
    cudaError_t e = cudaErrorNotSupported;
    int used_pair = 0;
    if (c->opt_kernel != 1 && stage_tiled_supported<T>(ndim, P)) e = launch_stage_tiled<T>(ndim, P, c->sm_count, st, c->opt_kernel == 3 ? 0 : (c->opt_kernel == 4 ? 2 : (c->opt_kernel == 2 ? 3 : 1)), &used_pair);
    else if (c->opt_kernel == 2) return fail(LSM_ERR_UNSUPPORTED, "tiled kernel forced but this configuration is not covered");
    if (e == cudaErrorNotSupported) e = launch_stage_generic<T>(ndim, P, st);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "stage kernel launch failed: %s", cudaGetErrorString(e));
    c->cnt.kernel_launches += 1; c->cnt.stage_launches += 1; c->cnt.pair_launches += used_pair;
    return LSM_OK;
}

// One fused RK stage: out = base(in, p0) - c * sum_k H_k(in), written in the reference's rounding
// order, with the output's halo exchange overlapped with the interior update.
template <class T>
int32_t run_stage_t(lsm_ctx* c, lsm_field* in, lsm_field* p0, lsm_field* out, lsm_field* out2, int base, double cc, double c2,
                    const lsm_term* terms, int nterms, double tstage, const double* gscale, bool out_needs_halo) {
    NvtxRange nvtx("lsm RK stage");
    StageParams<T> P{};
    P.in = make_view<T>(in);
    P.p0 = p0 ? static_cast<const T*>(p0->p) : nullptr;
    P.out = static_cast<T*>(out->p);
    P.out2 = out2 ? static_cast<T*>(out2->p) : nullptr;
    P.base = base; P.nterms = nterms; P.c = cc; P.c2 = c2;
    double dxmin = in->h[0];
    for (int d = 0; d < 3; ++d) { P.h[d] = in->h[d]; if (d < in->ndim) dxmin = std::min(dxmin, in->h[d]); }
    P.dxmin = dxmin;
    for (int k = 0; k < nterms; ++k) TRY(make_term_dev(in, terms[k], term_scale(terms[k], tstage, gscale, k), &P.terms[k]));
    for (int k = 0; k < nterms; ++k)
        if (terms[k].coef_kind == LSM_COEF_EXPR) TRY(expr_ensure(terms[k].field, tstage, terms[k].kind, false));
    P.skip_zero_u = c->stage_skip_zero_u;

    const int last = in->ndim - 1, nl = in->n[last];
    if (c->nranks > 1 && !in->halo_valid) {        // e.g. right after an upload
        TRY(exchange_halo(in, c->stream));
    }
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    if (c->opt_time) { t0 = pool_event(c); t1 = pool_event(c); cudaEventRecord(t0, c->stream); }
    if (c->nranks > 1 && out_needs_halo && c->opt_overlap && nl >= 4 * HALO) {
        // The two thin boundary slabs run on a high-priority side stream CONCURRENTLY with the interior kernel (their
        // blocks fill SMs the interior leaves idle at its tail and vice versa); as soon as they are done the comm stream
        // ships them (NCCL send/recv) while the interior is still being computed.  The next stage waits for both.
        CU(cudaEventRecord(c->ev_main, c->stream));                 // everything enqueued so far (previous stage, halos, memsets)
        CU(cudaStreamWaitEvent(c->bstream, c->ev_main, 0));
        // the slabs hold exactly the planes exchange_halo ships: HALO planes per side, one more when the decomposed axis is periodic
        // (the wrap-around partner receives planes 1..3 / nl-4..nl-2, boundaryconditions.jl:107-119)
        const int sl = HALO + (in->bc[last][0].kind == LSM_BC_PERIODIC ? 1 : 0);
        TRY(launch_stage_range<T>(c, in->ndim, P, 0, sl, c->bstream));
        TRY(launch_stage_range<T>(c, in->ndim, P, nl - sl, nl, c->bstream));
        CU(cudaEventRecord(c->ev_boundary, c->bstream));
        CU(cudaStreamWaitEvent(c->comm, c->ev_boundary, 0));
        TRY(exchange_halo(out, c->comm));
        CU(cudaEventRecord(c->ev_halo, c->comm));
        // The interior launch waits for the slabs too: they fill the GPU anyway (thousands of blocks), and the exchange kernel
        // (a few blocks of NCCL's, more registers per block than an SM has left beside a resident interior block) then becomes
        // runnable TOGETHER with the interior grid and — on a higher-priority stream — is placed first; launched behind an
        // interior grid that already occupies every SM it would only run in that grid's tail, i.e. not overlapped at all.
        if (!c->interior_first) CU(cudaStreamWaitEvent(c->stream, c->ev_boundary, 0));
        TRY(launch_stage_range<T>(c, in->ndim, P, sl, nl - sl));
        CU(cudaStreamWaitEvent(c->stream, c->ev_boundary, 0));
        CU(cudaStreamWaitEvent(c->stream, c->ev_halo, 0));
    } else {
        TRY(launch_stage_range<T>(c, in->ndim, P, 0, nl));
        if (c->nranks > 1 && out_needs_halo) TRY(exchange_halo(out, c->stream));
    }
    if (c->opt_time) { cudaEventRecord(t1, c->stream); c->timed.emplace_back(t0, t1); }
    out->version++; out->halo_valid = (c->nranks == 1) || out_needs_halo;
    if (out2) { out2->version++; out2->halo_valid = (c->nranks == 1); }
    return LSM_OK;
}

int32_t run_stage(lsm_ctx* c, lsm_field* in, lsm_field* p0, lsm_field* out, lsm_field* out2, int base, double cc, double c2,
                  const lsm_term* terms, int nterms, double tstage, const double* gscale, bool out_needs_halo) {
    if (in->dtype == LSM_F64) return run_stage_t<double>(c, in, p0, out, out2, base, cc, c2, terms, nterms, tstage, gscale, out_needs_halo);
    return run_stage_t<float>(c, in, p0, out, out2, base, cc, c2, terms, nterms, tstage, gscale, out_needs_halo);
}

void swap_storage(lsm_field* a, lsm_field* b) {
    std::swap(a->base, b->base); std::swap(a->p, b->p);
    std::swap(a->halo_valid, b->halo_valid);
    a->version++; b->version++;
}

int32_t check_state(lsm_ctx* ctx, lsm_field* phi, const lsm_term* terms, int nterms) {
    if (!ctx || !phi || !terms) return fail(LSM_ERR_ARG, "null argument");
    if (phi->ctx != ctx) return fail(LSM_ERR_ARG, "field belongs to another context");
    if (nterms < 1 || nterms > LSM_MAX_TERMS) return fail(LSM_ERR_ARG, "nterms must be in 1..%d", LSM_MAX_TERMS);
    if (phi->ncomp != 1 || phi->separable) return fail(LSM_ERR_ARG, "the state must be a scalar field");
    if (!phi->has_bc) return fail(LSM_ERR_BC, "no boundary conditions: call lsm_field_set_bc on the state");   // levelsetequation.jl:69-70
    CU(cudaSetDevice(ctx->device));
    return LSM_OK;
}

int32_t stage_impl(lsm_ctx* ctx, int integ, int stage, lsm_field* phi, const lsm_term* terms, int nterms, double tc, double dt, const double* gs) {
    switch (integ) {
        case LSM_FORWARD_EULER:      // timestepping.jl:128-137
            if (stage != 1) return fail(LSM_ERR_ARG, "ForwardEuler has 1 stage");
            TRY(ensure_buffers(phi, 1));
            TRY(run_stage(ctx, phi, nullptr, phi->buf1, nullptr, BASE_IN, dt, 0, terms, nterms, tc, gs, true));
            swap_storage(phi, phi->buf1);          // copy!(phi, dst) without the copy
            return LSM_OK;
        case LSM_RK2:                // timestepping.jl:143-164
            TRY(ensure_buffers(phi, 2));
            if (stage == 1) return run_stage(ctx, phi, nullptr, phi->buf1, phi->buf2, BASE_IN, dt, 0.5 * dt, terms, nterms, tc, gs, true);
            if (stage == 2) return run_stage(ctx, phi->buf1, phi->buf2, phi, nullptr, BASE_P0, 0.5 * dt, 0, terms, nterms, tc + dt, gs, true);
            return fail(LSM_ERR_ARG, "RK2 has 2 stages");
        case LSM_RK3:                // timestepping.jl:170-202
            TRY(ensure_buffers(phi, 2));
            if (stage == 1) return run_stage(ctx, phi, nullptr, phi->buf1, nullptr, BASE_IN, dt, 0, terms, nterms, tc, gs, true);
            if (stage == 2) return run_stage(ctx, phi->buf1, phi, phi->buf2, nullptr, BASE_RK3_S2, 0.25 * dt, 0, terms, nterms, tc + dt, gs, true);
            if (stage == 3) return run_stage(ctx, phi->buf2, phi, phi, nullptr, BASE_RK3_S3, (2.0 / 3.0) * dt, 0, terms, nterms, tc + 0.5 * dt, gs, true);
            return fail(LSM_ERR_ARG, "RK3 has 3 stages");
        default: return fail(LSM_ERR_ARG, "bad integrator %d", integ);
    }
}

int nstages(int integ) { return integ == LSM_FORWARD_EULER ? 1 : integ == LSM_RK2 ? 2 : 3; }

// The step sizes of the time loop for a CONSTANT CFL step dt_cfl (static coefficients), replayed with the loop's own arithmetic
// (timestepping.jl:104-118): while t <= tf - eps(t): dt = min(dt_max, cfl * dt_cfl, tf - t); t += dt.  Run-length encoded; stops
// after `limit` steps (< 0: none).  Returns the time reached and the number of steps.
void plan_steps(double t0, double tf, double dt_max, double cfl, double dt_cfl, int64_t limit,
                std::vector<std::pair<double, long>>& runs, double* t_end, int64_t* nsteps) {
    const double D = jl_min(dt_max, cfl * dt_cfl);
    double t = t0; int64_t n = 0;
    while (t <= tf - jl_eps(t) && (limit < 0 || n < limit)) {
        const double dt = jl_min(D, tf - t);                       // timestepping.jl:111
        if (!runs.empty() && runs.back().first == dt) runs.back().second++; else runs.emplace_back(dt, 1L);
        t += dt; ++n;
    }
    *t_end = t; *nsteps = n;
}

// lsm_resident2d.cu covers: single rank, 2-D, ONE AdvectionTerm(stored velocity of the state's dtype, WENO5) without a time factor,
// index-map boundary conditions (periodic / Neumann / symmetry), automatic kernel selection, no per-stage timing
bool resident_eligible(const lsm_ctx* ctx, const lsm_field* phi, const lsm_term* terms, int nterms) {
    if (!ctx->opt_resident || ctx->nranks != 1 || ctx->opt_time || ctx->opt_kernel != 0) return false;
    if (phi->ndim != 2 || nterms != 1) return false;
    const lsm_term& t = terms[0];
    if (t.kind != LSM_TERM_ADVECTION || t.scheme != LSM_WENO5 || t.coef_kind != LSM_COEF_FIELD || t.tscale_kind != LSM_TS_NONE) return false;
    if (!t.field || t.field->separable || t.field->dtype != phi->dtype || t.field->ncomp != 2 || t.field->ctx != ctx) return false;
    for (int d = 0; d < 2; ++d) {
        if (t.field->nglob[d] != phi->nglob[d]) return false;
        for (int sd = 0; sd < 2; ++sd) {
            const int k = phi->bc[d][sd].kind;
            if (!(k == LSM_BC_PERIODIC || k == LSM_BC_SYMMETRY || (k == LSM_BC_EXTRAP && phi->bc[d][sd].P == 0))) return false;
        }
    }
    return phi->dtype == LSM_F64 ? resident2d_supported<double>(phi->n[0], phi->n[1]) : resident2d_supported<float>(phi->n[0], phi->n[1]);
}

template <class T>
int32_t run_resident(lsm_ctx* ctx, int integ, lsm_field* phi, const lsm_term& term, const std::vector<std::pair<double, long>>& runs) {
    NvtxRange nvtx("lsm resident time loop");
    ResidentArgs<T> R{};
    R.phi = static_cast<const T*>(phi->p);
    R.out = static_cast<T*>(phi->p);
    const lsm_field* u = term.field;
    for (int d = 0; d < 2; ++d) {
        R.u[d] = static_cast<const T*>(u->p) + (size_t)d * u->cstride;
        R.n[d] = phi->n[d]; R.h[d] = phi->h[d];
        for (int sd = 0; sd < 2; ++sd) R.bc[d][sd] = phi->bc[d][sd].kind;
    }
    R.s1 = phi->n[0];
    R.nstages = nstages(integ);
    R.wk = weno_constants();
    R.status = ctx->d_scalar + 2;
    CU(cudaMemsetAsync(R.status, 0, 8, ctx->stream));
    int64_t done = 0;
    for (size_t i = 0; i < runs.size(); i += 4) {
        R.nruns = (int)std::min<size_t>(4, runs.size() - i);
        int64_t here = 0;
        for (int k = 0; k < R.nruns; ++k) { R.dt[k] = runs[i + k].first; R.count[k] = runs[i + k].second; here += runs[i + k].second; }
        cudaError_t e = launch_resident2d<T>(R, ctx->stream);
        if (e == cudaErrorNotSupported && done == 0) return LSM_ERR_UNSUPPORTED;          // nothing has run: the caller takes the regular path
        if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "resident kernel launch failed: %s", cudaGetErrorString(e));
        done += here;
        ctx->cnt.kernel_launches += 1; ctx->cnt.resident_steps += here;
    }
    phi->version++; phi->halo_valid = true;
    CU(cudaMemcpyAsync(ctx->h_scalar + 2, R.status, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));                    // lsm_integrate returns synchronised anyway
    ctx->cnt.d2h_bytes += 8;
    if (ctx->h_scalar[2] != 0ULL) return fail(LSM_ERR_CUDA, "resident kernel: halo protocol failure (status %llu); the state is not valid", ctx->h_scalar[2]);
    return LSM_OK;
}

unsigned long long dbits(double s) {
    unsigned long long b;
    if (std::isnan(s)) return 0x7FF8000000000000ULL;
    std::memcpy(&b, &s, 8);
    return b;
}

// The reference's CFL quantity of one node with coefficient tuple v (ndim velocity components, or one scalar coefficient):
// sum_d fl(|fl(v_d g)| / h_d) for advection (levelsetterms.jl:90-96), |fl(v g)| otherwise; an unscaled term takes v as it is.
// The expression of cfl_kernel, operation for operation (this translation unit is compiled without FMA contraction).
double cfl_node(int kind, const double* v, int ndim, const double* h, bool scaled, double g) {
    if (kind != LSM_TERM_ADVECTION) return std::fabs(scaled ? v[0] * g : v[0]);
    double acc = 0.0;
    for (int d = 0; d < ndim; ++d) {
        const double w = scaled ? v[d] * g : v[d];
        const double q = std::fabs(w) / h[d];
        acc = d == 0 ? q : acc + q;
    }
    return acc;
}

// max over the candidate tuples of the CFL quantity at scale g
unsigned long long cand_eval(const CflMemo& e, const lsm_field* phi, double g) {
    unsigned long long best = 0ULL;
    const size_t n = e.tup.size() / e.ncomp;
    for (size_t k = 0; k < n; ++k) {
        const unsigned long long b = dbits(cfl_node(e.kind, &e.tup[k * e.ncomp], e.ncomp, phi->h, true, g));
        best = b > best ? b : best;
    }
    return best;
}

// the memo of (t.kind, t.field), created on first use and emptied when the field's data has changed since it was filled
CflMemo& cfl_memo(lsm_ctx* ctx, const lsm_term& t) {
    CflMemo* e = nullptr;
    for (auto& m : ctx->cfl_memo) if (m.kind == t.kind && m.field == t.field) { e = &m; break; }
    if (!e) { ctx->cfl_memo.emplace_back(); e = &ctx->cfl_memo.back(); }
    if (e->field != t.field || e->version != t.field->version) { *e = CflMemo{}; e->kind = t.kind; e->field = t.field; e->version = t.field->version; }
    return *e;
}

// one reduction pass over every owned node (all ranks), read back: the exact maximum as IEEE bits (see lsm_generic.cu K3)
int32_t full_cfl_pass(lsm_ctx* ctx, lsm_field* phi, const TermDev& td, unsigned long long* bits_out) {
    CflParams P{};
    P.term = td;
    for (int d = 0; d < 3; ++d) { P.n[d] = phi->n[d]; P.h[d] = phi->h[d]; }
    P.out = ctx->d_scalar;
    CU(cudaMemsetAsync(ctx->d_scalar, 0, 8, ctx->stream));
    cudaError_t e = launch_cfl(phi->ndim, phi->dtype == LSM_F64, P, ctx->sm_count, ctx->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "CFL kernel launch failed: %s", cudaGetErrorString(e));
    ctx->cnt.kernel_launches += 1; ctx->cnt.cfl_passes += 1;
    if (ctx->nranks > 1) NC(nccl().AllReduce(ctx->d_scalar, ctx->d_scalar, 1, ncclUint64, ncclMax, ctx->nccl_comm, ctx->stream));
    CU(cudaMemcpyAsync(ctx->h_scalar, ctx->d_scalar, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->cnt.d2h_bytes += 8;
    *bits_out = *ctx->h_scalar;
    return LSM_OK;
}

// Build the candidate set of a scaled coefficient field: one unscaled reduction (global maximum M), one extraction pass
// (nodes with S_i >= (1 - 1e-12) M), one gather.  Multi-rank: every rank contributes a fixed-size segment of a zero-filled
// buffer and the segments are concatenated with an all-reduce(sum) (x + 0 = x exactly), so all ranks hold the same set.
int32_t cand_build(lsm_ctx* ctx, lsm_field* phi, const lsm_term& t, const TermDev& td_scaled, CflMemo* e) {
    TermDev td = td_scaled;
    td.scaled = 0; td.g = 1.0;
    e->ncomp = t.kind == LSM_TERM_ADVECTION ? phi->ndim : 1;
    e->built = false; e->overflow = false; e->tup.clear();
    unsigned long long mb = 0;
    TRY(full_cfl_pass(ctx, phi, td, &mb));
    double M; std::memcpy(&M, &mb, 8);
    const int R = ctx->nranks;
    const size_t seg = 1 + (size_t)CAND_CAP * e->ncomp;          // [count, tuples...] per rank
    const size_t total = seg * R;
    if (!ctx->d_cand) {
        const size_t cap_bytes = (1 + (size_t)CAND_CAP * 3) * (size_t)R * sizeof(double);
        CU(cudaMalloc(&ctx->d_cand, cap_bytes));
        CU(cudaMalloc(&ctx->d_cand_count, 16));
        CU(cudaMallocHost(&ctx->h_cand, cap_bytes));
    }
    if (M == 0.0) {                                              // identically zero field: s_i(g) = 0 for every g
        e->tup.assign(e->ncomp, 0.0);
        e->built = true;
        return LSM_OK;
    }
    CandParams P{};
    P.term = td;
    for (int d = 0; d < 3; ++d) { P.n[d] = phi->n[d]; P.h[d] = phi->h[d]; }
    P.thr = M * (1.0 - 1e-12);                                    // NaN maximum -> every node qualifies -> overflow -> regular path
    P.cap = CAND_CAP; P.ncomp = e->ncomp;
    P.count = ctx->d_cand_count;
    P.out = ctx->d_cand + seg * ctx->rank + 1;
    CU(cudaMemsetAsync(ctx->d_cand, 0, total * sizeof(double), ctx->stream));
    CU(cudaMemsetAsync(ctx->d_cand_count, 0, 4, ctx->stream));
    cudaError_t ce = launch_cfl_candidates(phi->ndim, phi->dtype == LSM_F64, P, ctx->sm_count, ctx->stream);
    if (ce != cudaSuccess) return fail(LSM_ERR_CUDA, "CFL candidate kernel launch failed: %s", cudaGetErrorString(ce));
    ctx->cnt.kernel_launches += 1;
    unsigned cnt = 0;
    CU(cudaMemcpyAsync(&cnt, ctx->d_cand_count, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const double cntd = (double)cnt;
    CU(cudaMemcpyAsync(ctx->d_cand + seg * ctx->rank, &cntd, 8, cudaMemcpyHostToDevice, ctx->stream));
    if (R > 1) NC(nccl().AllReduce(ctx->d_cand, ctx->d_cand, total, ncclDouble, ncclSum, ctx->nccl_comm, ctx->stream));
    // single rank: only the filled part of the segment travels
    const size_t take = R > 1 ? total : 1 + (size_t)std::min<unsigned>(cnt, (unsigned)CAND_CAP) * e->ncomp;
    CU(cudaMemcpyAsync(ctx->h_cand, ctx->d_cand, take * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->cnt.d2h_bytes += (int64_t)(take * sizeof(double)) + 4;
    std::vector<std::vector<double>> rows;
    for (int r = 0; r < R; ++r) {
        const double* sg = ctx->h_cand + seg * r;
        const double c = sg[0];
        if (!(c <= (double)CAND_CAP)) { e->overflow = true; return LSM_OK; }      // too many ties (e.g. a constant field): regular path
        for (int k = 0; k < (int)c; ++k) rows.emplace_back(sg + 1 + (size_t)k * e->ncomp, sg + 1 + (size_t)(k + 1) * e->ncomp);
    }
    if (rows.empty()) { e->overflow = true; return LSM_OK; }                       // cannot happen (the maximum itself qualifies)
    // distinct tuples only (NaN-safe: compare bit patterns)
    auto key = [](const std::vector<double>& a, const std::vector<double>& b) {
        for (size_t i = 0; i < a.size(); ++i) {
            unsigned long long x, y; std::memcpy(&x, &a[i], 8); std::memcpy(&y, &b[i], 8);
            if (x != y) return x < y;
        }
        return false;
    };
    std::sort(rows.begin(), rows.end(), key);
    for (size_t i = 0; i < rows.size(); ++i)
        if (i == 0 || key(rows[i - 1], rows[i])) e->tup.insert(e->tup.end(), rows[i].begin(), rows[i].end());
    e->built = true;
    return LSM_OK;
}

// max over owned nodes of the CFL quantity of one term, as IEEE bits (see lsm_generic.cu K3)
int32_t cfl_bits(lsm_ctx* ctx, lsm_field* phi, const lsm_term& t, double g, unsigned long long* bits_out) {
    TermDev td;
    TRY(make_term_dev(phi, t, g, &td));
    CflMemo* e = nullptr;
    if (ctx->opt_cfl_cache && (t.coef_kind == LSM_COEF_FIELD || t.coef_kind == LSM_COEF_SEPARABLE)) {
        e = &cfl_memo(ctx, t);
        if (e->have_bits && e->scaled == td.scaled && (!td.scaled || e->g == g)) { *bits_out = e->bits; return LSM_OK; }
        if (ctx->opt_cand && td.scaled) {
            // time-scaled static coefficient: the second request for the same data builds the candidate set, every later one is
            // answered on the host (no kernel, no D2H, no sync)
            e->seen++;
            if (!e->built && !e->overflow && e->seen >= 2) TRY(cand_build(ctx, phi, t, td, e));
            if (e->built && !e->overflow) { *bits_out = cand_eval(*e, phi, g); return LSM_OK; }
        }
    }
    TRY(full_cfl_pass(ctx, phi, td, bits_out));
    if (e) { e->have_bits = true; e->scaled = td.scaled; e->g = g; e->bits = *bits_out; }
    return LSM_OK;
}

double bits_to_double(unsigned long long b) { double d; std::memcpy(&d, &b, 8); return d; }

// CFL maximum of a time-dependent expression coefficient at time t: reduced by the fill that materialised it (at this CFL request,
// or earlier by a stage at the same time), read once (one 8-byte D2H and a sync, like any coefficient that changes between steps)
int32_t expr_cfl_bits(lsm_ctx* ctx, lsm_field* f, double t, int term_kind, unsigned long long* bits_out) {
    TRY(expr_ensure(f, t, term_kind, true));
    if (!f->expr_cfl_read) {
        if (ctx->nranks > 1) NC(nccl().AllReduce(f->d_expr_cfl, f->d_expr_cfl, 1, ncclUint64, ncclMax, ctx->nccl_comm, ctx->stream));
        CU(cudaMemcpyAsync(ctx->h_scalar + 3, f->d_expr_cfl, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        ctx->cnt.d2h_bytes += 8;
        f->expr_cfl_bits = ctx->h_scalar[3];
        f->expr_cfl_read = true;
    }
    *bits_out = f->expr_cfl_bits;
    return LSM_OK;
}

// _compute_cfl(term, phi, t) for one term (levelsetterms.jl:30-37 + per-node rules)
int32_t cfl_term(lsm_ctx* ctx, lsm_field* phi, const lsm_term& t, double time, double g, double* dt_out) {
    const int N = phi->ndim;
    double dxmin = phi->h[0];
    for (int d = 1; d < N; ++d) dxmin = std::min(dxmin, phi->h[d]);
    const double inf = std::numeric_limits<double>::infinity();
    if (t.kind == LSM_TERM_EIKONAL) { *dt_out = jl_min(inf, dxmin); return LSM_OK; }    // levelsetterms.jl:250
    const bool scaled = t.tscale_kind != LSM_TS_NONE;
    double m;     // max over nodes of sum_d |u_d|/h_d (advection) or of |coefficient| (normal, curvature)
    if (t.coef_kind == LSM_COEF_CONST) {
        m = cfl_node(t.kind, t.cval, N, phi->h, scaled, g);
    } else if (t.coef_kind == LSM_COEF_EXPR) {
        unsigned long long bits = 0;
        TRY(expr_cfl_bits(ctx, t.field, time, t.kind, &bits));
        m = bits_to_double(bits);
    } else {
        unsigned long long bits = 0;
        TRY(cfl_bits(ctx, phi, t, g, &bits));
        m = bits_to_double(bits);
    }
    double r;
    if (t.kind == LSM_TERM_ADVECTION) r = 1 / m;                                  // levelsetterms.jl:90-96
    else if (t.kind == LSM_TERM_NORMAL) {                                         // levelsetterms.jl:172-178
        double s = 0;
        for (int d = 0; d < N; ++d) { const double q = m / phi->h[d]; s = d == 0 ? q : s + q; }
        r = 1 / s;
    } else r = (dxmin * dxmin) / (2 * m);                                         // levelsetterms.jl:123-127
    *dt_out = jl_min(inf, r);
    return LSM_OK;
}

int32_t compute_cfl_impl(lsm_ctx* ctx, lsm_field* phi, const lsm_term* terms, int nterms, double t, const double* gs, double* dt_out) {
    double dt = std::numeric_limits<double>::infinity();
    for (int k = 0; k < nterms; ++k) {
        double d;
        TRY(cfl_term(ctx, phi, terms[k], t, term_scale(terms[k], t, gs, k), &d));
        dt = k == 0 ? d : jl_min(dt, d);
    }
    *dt_out = dt;
    if (!(dt > 0)) return fail(LSM_ERR_CFL, "invalid time-step based on CFL condition: dt = %g (check for NaN/Inf in velocity or speed)", dt);
    return LSM_OK;
}

// ---- zero-level-set operations (lsm_interface.cu, lsm_redistance.cu) ------------------------------
// The checks every operation on a level set makes: a real-valued field of this context with at least min_n nodes along every
// dimension and, for the operations that have no multi-rank form, a context of one rank.  `what` names the operation.
int32_t check_level_set(lsm_ctx* ctx, const lsm_field* phi, const char* what, int min_n, bool single_rank) {
    if (!ctx || !phi) return fail(LSM_ERR_ARG, "null argument");
    if (phi->ctx != ctx || phi->ncomp != 1 || phi->separable) return fail(LSM_ERR_ARG, "%s needs a real-valued field of this context", what);
    for (int d = 0; d < phi->ndim; ++d)
        if (phi->nglob[d] < min_n)
            return fail(LSM_ERR_ARG, "%s needs at least %d nodes along every dimension (n[%d] = %d)", what, min_n, d, phi->nglob[d]);
    if (single_rank && ctx->nranks > 1)
        return fail(LSM_ERR_UNSUPPORTED, "%s: slab decomposition is not supported (nranks = %d)", what, ctx->nranks);
    return LSM_OK;
}

// A second field F of an operation on phi (checked by check_level_set too) must lie on phi's grid: same node counts, same owned
// slab, same lower corner and spacing.
int32_t check_same_grid(const lsm_field* F, const lsm_field* phi) {
    bool same = F->ndim == phi->ndim;
    for (int d = 0; same && d < phi->ndim; ++d)
        same = F->nglob[d] == phi->nglob[d] && F->n[d] == phi->n[d] && F->lc[d] == phi->lc[d] && F->h[d] == phi->h[d];
    if (!same) return fail(LSM_ERR_ARG, "F and phi must be on the same grid (n, lc and h)");
    return LSM_OK;
}

// The node box of phi for the kernels: this rank's owned nodes and, with `ghost`, the first plane of the next rank.  Level 0,
// ntiles unset.
IfaceArgs field_box(const lsm_field* phi, bool ghost) {
    IfaceArgs A{};
    A.phi = phi->p; A.f64 = phi->dtype == LSM_F64; A.ndim = phi->ndim;
    A.first_last = phi->first_last;
    A.hsign = 1;
    for (int d = 0; d < 3; ++d) {
        A.m[d] = phi->n[d] + (d == phi->ndim - 1 && ghost ? 1 : 0);
        A.lc[d] = phi->lc[d]; A.h[d] = d < phi->ndim ? phi->h[d] : 0.0;
        if (d < phi->ndim && phi->h[d] < 0) A.hsign = -A.hsign;
    }
    A.s1 = A.m[0]; A.s2 = (long long)A.m[0] * A.m[1];
    A.nodes = (long long)A.m[0] * A.m[1] * A.m[2];
    A.lin0 = (long long)phi->first_last * phi->plane;
    return A;
}

// one synchronisation and one copy of n adjacent 8-byte device counters into ctx->h_scalar[0 .. n-1]
int32_t read_counts(lsm_ctx* ctx, const void* d_counts, int n) {
    CU(cudaMemcpyAsync(ctx->h_scalar, d_counts, 8 * n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->cnt.d2h_bytes += 8 * n;
    return LSM_OK;
}

// The closest-point passes on phi (checked by the caller): the extension of F unless F is null, redistancing of phi when write_phi
// (the caller sets it when F is null), with `cubic` the Newton refinement before the write.  Scratch: two point buffers of N doubles
// per node (N + 1 with F: the value at the point), the two 8-byte keys of the band scan per node, and three counters (listed
// cells, band nodes, fallbacks).  Asynchronous unless an out-pointer is given; then one synchronisation and one copy of the band-node
// count, and with `cubic` of the fallback count next to it.
int32_t closest_points(lsm_ctx* ctx, lsm_field* phi, int32_t band, lsm_field* F, bool write_phi, bool cubic,
                       int64_t* band_nodes_out, int64_t* fallback_nodes_out) {
    CU(cudaSetDevice(ctx->device));
    RedistArgs R{};
    R.g = field_box(phi, false);
    R.band = band;
    R.F = F ? F->p : nullptr; R.F_f64 = F && F->dtype == LSM_F64; R.write_phi = write_phi;
    const long long nodes = R.g.nodes;
    const size_t pbytes = (size_t)nodes * (phi->ndim + (F ? 1 : 0)) * sizeof(double), kbytes = (size_t)nodes * sizeof(unsigned long long);
    TRY(grow_scratch(ctx, &ctx->d_redist, &ctx->d_redist_bytes, 2 * pbytes + 2 * kbytes + 3 * sizeof(unsigned long long)));
    char* base = static_cast<char*>(ctx->d_redist);
    R.pa = reinterpret_cast<double*>(base);
    R.pb = reinterpret_cast<double*>(base + pbytes);
    R.list = reinterpret_cast<long long*>(R.pa);
    R.dmin = reinterpret_cast<unsigned long long*>(base + 2 * pbytes);
    R.ord = R.dmin + nodes;
    R.ncells = R.ord + nodes;
    R.count = R.ncells + 1;
    R.fallbacks = cubic ? R.count + 1 : nullptr;
    CU(cudaMemsetAsync(R.ncells, 0, 3 * sizeof(unsigned long long), ctx->stream));
    int launches = 0;
    CU(launch_closest_points(R, ctx->sm_count, ctx->stream, &launches));
    ctx->cnt.kernel_launches += launches;
    if (F) { F->version++; F->halo_valid = false; }
    if (R.write_phi) { phi->version++; phi->halo_valid = false; }
    if (band_nodes_out || fallback_nodes_out) {
        TRY(read_counts(ctx, R.count, cubic ? 2 : 1));
        if (band_nodes_out) *band_nodes_out = (int64_t)ctx->h_scalar[0];
        if (fallback_nodes_out) *fallback_nodes_out = (int64_t)ctx->h_scalar[1];
    }
    return LSM_OK;
}

}  // namespace

// =================================================================================================
namespace {
// run f(r) for every rank on its own host thread (NCCL collectives of the ranks must be in flight together); the first failing
// rank's status and message are handed back to the calling thread
template <class F>
int32_t fan_out(int n, F f) {
    std::vector<int32_t> rcs(n, LSM_OK);
    std::vector<std::string> msgs(n);
    std::vector<std::thread> th;
    th.reserve(n);
    for (int r = 0; r < n; ++r) th.emplace_back([&, r] { rcs[r] = f(r); if (rcs[r] != LSM_OK) msgs[r] = g_err; });
    for (auto& t : th) t.join();
    for (int r = 0; r < n; ++r) if (rcs[r] != LSM_OK) { g_err = msgs[r]; return rcs[r]; }
    return LSM_OK;
}

}  // namespace

extern "C" {

int32_t lsm_abi_version(void) { return LSM_ABI_VERSION; }
const char* lsm_last_error(void) { return g_err.c_str(); }

int32_t lsm_device_count(int32_t* n_out) {
    if (!n_out) return fail(LSM_ERR_ARG, "null argument");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *n_out = 0; return fail(LSM_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *n_out = n;
    return LSM_OK;
}

int32_t lsm_ctx_create(int32_t device, lsm_ctx** out) {
    if (!out) return fail(LSM_ERR_ARG, "null argument");
    lsm_ctx* c = new (std::nothrow) lsm_ctx();
    if (!c) return fail(LSM_ERR_OOM, "host allocation failed");
    c->device = device;
    int32_t rc = ctx_common_init(c);
    if (rc != LSM_OK) { lsm_ctx_destroy(c); return rc; }      // releases whatever was created; the error text is already set
    *out = c;
    return LSM_OK;
}

int32_t lsm_nccl_unique_id(void* id128) {
    if (!id128) return fail(LSM_ERR_ARG, "null argument");
    const char* why = "";
    if (!nccl().load(&why)) return fail(LSM_ERR_NCCL, "cannot load NCCL: %s", why);
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NC(nccl().GetUniqueId(&id));
    std::memcpy(id128, &id, 128);
    return LSM_OK;
}

int32_t lsm_ctx_create_rank(int32_t device, int32_t rank, int32_t nranks, const void* id128, lsm_ctx** out) {
    if (!out) return fail(LSM_ERR_ARG, "null argument");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(LSM_ERR_ARG, "bad rank %d of %d", rank, nranks);
    if (nranks == 1) return lsm_ctx_create(device, out);
    if (!id128) return fail(LSM_ERR_ARG, "null NCCL id");
    const char* why = "";
    if (!nccl().load(&why)) return fail(LSM_ERR_NCCL, "cannot load NCCL: %s", why);
    lsm_ctx* c = new (std::nothrow) lsm_ctx();
    if (!c) return fail(LSM_ERR_OOM, "host allocation failed");
    c->device = device; c->rank = rank; c->nranks = nranks;
    int32_t rc = ctx_common_init(c);
    if (rc != LSM_OK) { lsm_ctx_destroy(c); return rc; }
    ncclUniqueId id;
    std::memcpy(&id, id128, 128);
    ncclResult_t r = nccl().CommInitRank(&c->nccl_comm, nranks, id, rank);
    if (r != ncclSuccess) { c->nccl_comm = nullptr; lsm_ctx_destroy(c); return fail(LSM_ERR_NCCL, "ncclCommInitRank failed: %s", nccl().GetErrorString(r)); }
    *out = c;
    return LSM_OK;
}

int32_t lsm_ctx_create_multi(int32_t n, const int32_t* devs, lsm_ctx** out) {
    if (!devs || !out || n < 1 || n > 64) return fail(LSM_ERR_ARG, "bad argument");
    if (n == 1) return lsm_ctx_create(devs[0], out);
    const char* why = "";
    if (!nccl().load(&why)) return fail(LSM_ERR_NCCL, "cannot load NCCL: %s", why);
    for (int r = 0; r < n; ++r) out[r] = nullptr;
    int32_t rc = LSM_OK;
    for (int r = 0; r < n && rc == LSM_OK; ++r) {
        lsm_ctx* c = new (std::nothrow) lsm_ctx();
        if (!c) { rc = fail(LSM_ERR_OOM, "host allocation failed"); break; }
        c->device = devs[r]; c->rank = r; c->nranks = n;
        out[r] = c;
        rc = ctx_common_init(c);
    }
    if (rc == LSM_OK) {
        std::vector<ncclComm_t> comms(n);
        std::vector<int> ids(devs, devs + n);
        ncclResult_t r = nccl().CommInitAll(comms.data(), n, ids.data());
        if (r != ncclSuccess) rc = fail(LSM_ERR_NCCL, "ncclCommInitAll failed: %s", nccl().GetErrorString(r));
        else for (int k = 0; k < n; ++k) out[k]->nccl_comm = comms[k];
    }
    if (rc != LSM_OK) {
        const std::string msg = g_err;
        for (int r = 0; r < n; ++r) if (out[r]) { lsm_ctx_destroy(out[r]); out[r] = nullptr; }
        g_err = msg;
    }
    return rc;
}

int32_t lsm_multi_compute_cfl(int32_t n, lsm_ctx* const* ctx, lsm_field* const* phi, const lsm_term* const* terms, int32_t nterms,
                              double t, const double* gscale, double* dt_out) {
    if (!ctx || !phi || !terms || !dt_out || n < 1) return fail(LSM_ERR_ARG, "bad argument");
    std::vector<double> dts(n, 0.0);
    TRY(fan_out(n, [&](int r) { return lsm_compute_cfl(ctx[r], phi[r], terms[r], nterms, t, gscale, &dts[r]); }));
    *dt_out = dts[0];        // all-reduced: identical on every rank
    return LSM_OK;
}

int32_t lsm_multi_integrate(int32_t n, lsm_ctx* const* ctx, int32_t integrator, double cfl, lsm_field* const* phi,
                            const lsm_term* const* terms, int32_t nterms, double t0, double tf, double dt_max, int64_t max_steps,
                            double* t_out, int64_t* steps_out) {
    if (!ctx || !phi || !terms || n < 1) return fail(LSM_ERR_ARG, "bad argument");
    std::vector<double> ts(n, t0);
    std::vector<int64_t> st(n, 0);
    TRY(fan_out(n, [&](int r) { return lsm_integrate(ctx[r], integrator, cfl, phi[r], terms[r], nterms, t0, tf, dt_max, max_steps, &ts[r], &st[r]); }));
    if (t_out) *t_out = ts[0];
    if (steps_out) *steps_out = st[0];
    return LSM_OK;
}

int32_t lsm_multi_interface_extract(int32_t n, lsm_ctx* const* ctx, lsm_field* const* phi, double level, int64_t* nverts_out, int64_t* nprims_out) {
    if (!ctx || !phi || !nverts_out || !nprims_out || n < 1) return fail(LSM_ERR_ARG, "bad argument");
    return fan_out(n, [&](int r) { return lsm_interface_extract(ctx[r], phi[r], level, &nverts_out[r], &nprims_out[r]); });
}

int32_t lsm_ctx_destroy(lsm_ctx* c) {
    if (!c) return LSM_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    resolve_timings(c);
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    for (auto e : c->ev_user) if (e) cudaEventDestroy(e);
    if (c->nccl_comm) nccl().CommDestroy(c->nccl_comm);
    if (c->d_scalar) cudaFree(c->d_scalar);
    if (c->h_scalar) cudaFreeHost(c->h_scalar);
    for (int b = 0; b < 2; ++b) { if (c->stage[b]) cudaFree(c->stage[b]); if (c->ev_stage[b]) cudaEventDestroy(c->ev_stage[b]); if (c->ev_free[b]) cudaEventDestroy(c->ev_free[b]); }
    if (c->d_work) cudaFree(c->d_work);
    if (c->d_iface) cudaFree(c->d_iface);
    if (c->d_redist) cudaFree(c->d_redist);
    if (c->d_cand) cudaFree(c->d_cand);
    if (c->d_cand_count) cudaFree(c->d_cand_count);
    if (c->h_cand) cudaFreeHost(c->h_cand);
    if (c->ev_boundary) cudaEventDestroy(c->ev_boundary);
    if (c->ev_halo) cudaEventDestroy(c->ev_halo);
    if (c->ev_main) cudaEventDestroy(c->ev_main);
    if (c->bstream) cudaStreamDestroy(c->bstream);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->comm) cudaStreamDestroy(c->comm);
    delete c;
    return LSM_OK;
}

int32_t lsm_sync(lsm_ctx* c) {
    if (!c) return fail(LSM_ERR_ARG, "null context");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->comm));
    CU(cudaStreamSynchronize(c->stream));
    return LSM_OK;
}

int32_t lsm_set_option(lsm_ctx* c, int32_t option, int32_t value) {
    if (!c) return fail(LSM_ERR_ARG, "null context");
    switch (option) {
        case LSM_OPT_KERNEL: if (value < 0 || value > 4) return fail(LSM_ERR_ARG, "LSM_OPT_KERNEL takes 0..4"); c->opt_kernel = value; break;
        case LSM_OPT_TIME_STAGES: c->opt_time = value != 0; break;
        case LSM_OPT_CFL_CACHE: c->opt_cfl_cache = value != 0; c->cfl_memo.clear(); break;
        case LSM_OPT_CFL_CANDIDATES:
            c->opt_cand = value != 0;
            for (auto& e : c->cfl_memo) { e.ncomp = 0; e.seen = 0; e.built = false; e.overflow = false; e.tup.clear(); }
            break;
        case LSM_OPT_RESIDENT: c->opt_resident = value != 0; break;
        case LSM_OPT_OVERLAP: c->opt_overlap = value != 0; break;
        case LSM_OPT_GRAPH: c->opt_graph = value != 0; break;
        default: return fail(LSM_ERR_ARG, "unknown option %d", option);
    }
    return LSM_OK;
}

int32_t lsm_get_counters(lsm_ctx* c, lsm_counters* out) {
    if (!c || !out) return fail(LSM_ERR_ARG, "null argument");
    resolve_timings(c);
    *out = c->cnt;
    return LSM_OK;
}

int32_t lsm_reset_counters(lsm_ctx* c) {
    if (!c) return fail(LSM_ERR_ARG, "null context");
    resolve_timings(c);
    c->cnt = lsm_counters{};
    return LSM_OK;
}

int32_t lsm_event_record(lsm_ctx* c, int32_t slot) {
    if (!c || slot < 0 || slot >= 8) return fail(LSM_ERR_ARG, "bad event slot");
    CU(cudaSetDevice(c->device));
    if (!c->ev_user[slot]) CU(cudaEventCreate(&c->ev_user[slot]));
    CU(cudaStreamWaitEvent(c->stream, c->ev_halo, 0));     // fold in outstanding halo traffic
    CU(cudaEventRecord(c->ev_user[slot], c->stream));
    return LSM_OK;
}
int32_t lsm_event_elapsed_ms(lsm_ctx* c, int32_t a, int32_t b, double* ms_out) {
    if (!c || !ms_out || a < 0 || a >= 8 || b < 0 || b >= 8 || !c->ev_user[a] || !c->ev_user[b]) return fail(LSM_ERR_ARG, "bad event slot");
    CU(cudaSetDevice(c->device));
    CU(cudaEventSynchronize(c->ev_user[b]));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, c->ev_user[a], c->ev_user[b]));
    *ms_out = ms;
    return LSM_OK;
}

int32_t lsm_host_register(void* ptr, int64_t bytes) {
    if (!ptr || bytes <= 0) return fail(LSM_ERR_ARG, "bad host range");
    CU(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault));
    return LSM_OK;
}
int32_t lsm_host_unregister(void* ptr) {
    if (!ptr) return fail(LSM_ERR_ARG, "null pointer");
    CU(cudaHostUnregister(ptr));
    return LSM_OK;
}

int32_t lsm_slab_plan(int32_t n_last, int32_t nranks, int32_t rank, int32_t* first_out, int32_t* count_out) {
    if (!first_out || !count_out || nranks < 1 || rank < 0 || rank >= nranks || n_last < 1) return fail(LSM_ERR_ARG, "bad slab plan arguments");
    int f, c;
    slab_plan(n_last, nranks, rank, &f, &c);
    *first_out = f; *count_out = c;
    return LSM_OK;
}

int32_t lsm_step_plan(double t0, double tf, double dt_max, double cfl, double dt_cfl, int64_t max_steps, int32_t cap,
                      double* dt_out, int64_t* count_out, int32_t* nruns_out, int64_t* steps_out, double* t_out) {
    if (!nruns_out || !steps_out || !t_out || cap < 0 || (cap > 0 && (!dt_out || !count_out))) return fail(LSM_ERR_ARG, "bad step plan arguments");
    if (!(tf >= t0)) return fail(LSM_ERR_TIME, "final time %g must be >= initial time %g: the level-set equation cannot be solved back in time", tf, t0);
    const double D = jl_min(dt_max, cfl * dt_cfl);
    if (!(std::isfinite(D) && D > 0.0) && t0 <= tf - jl_eps(t0)) return fail(LSM_ERR_ARG, "step plan needs a finite positive step (got %g)", D);
    std::vector<std::pair<double, long>> runs;
    double t = t0; int64_t n = 0;
    constexpr int64_t PLAN_CAP = 1LL << 26;                        // a step that does not advance t must not loop for ever
    plan_steps(t0, tf, dt_max, cfl, dt_cfl, max_steps < 0 ? PLAN_CAP : max_steps, runs, &t, &n);
    if (max_steps < 0 && n >= PLAN_CAP) return fail(LSM_ERR_ARG, "step plan exceeds %lld steps", (long long)PLAN_CAP);
    *nruns_out = (int32_t)runs.size(); *steps_out = n; *t_out = t;
    if ((int64_t)runs.size() > cap) return cap == 0 ? LSM_OK : fail(LSM_ERR_ARG, "step plan has %zu runs, capacity %d", runs.size(), cap);
    for (size_t i = 0; i < runs.size(); ++i) { dt_out[i] = runs[i].first; count_out[i] = runs[i].second; }
    return LSM_OK;
}

int32_t lsm_field_create(lsm_ctx* ctx, int32_t ndim, const int32_t* n, int32_t dtype, int32_t ncomp,
                         const double* lc, const double* hc, lsm_field** out) {
    if (!ctx) return fail(LSM_ERR_ARG, "null context");
    CU(cudaSetDevice(ctx->device));
    return field_alloc(ctx, ndim, n, dtype, ncomp, lc, hc, true, out);
}

int32_t lsm_field_create_separable(lsm_ctx* ctx, int32_t ndim, const int32_t* n, const double* lc, const double* hc,
                                   const double* scale, const double* tabs, lsm_field** out) {
    if (!ctx || !n || !scale || !tabs || !out) return fail(LSM_ERR_ARG, "null argument");
    if (ndim < 1 || ndim > 3) return fail(LSM_ERR_ARG, "ndim must be 1, 2 or 3");
    CU(cudaSetDevice(ctx->device));
    lsm_field* f = new (std::nothrow) lsm_field();
    if (!f) return fail(LSM_ERR_OOM, "host allocation failed");
    f->ctx = ctx; f->ndim = ndim; f->dtype = LSM_F64; f->ncomp = ndim; f->separable = true;
    long tot = 0;
    for (int d = 0; d < 3; ++d) {
        f->nglob[d] = d < ndim ? n[d] : 1; f->n[d] = f->nglob[d];
        f->lc[d] = (d < ndim && lc) ? lc[d] : 0; f->hc[d] = (d < ndim && hc) ? hc[d] : 1;
        f->h[d] = d < ndim ? (f->hc[d] - f->lc[d]) / double(f->nglob[d] - 1) : 1.0;
        f->scale[d] = d < ndim ? scale[d] : 0.0;
        if (d < ndim) tot += n[d];
    }
    const int last = ndim - 1;
    int first = 0, count = f->nglob[last];
    if (ctx->nranks > 1) slab_plan(f->nglob[last], ctx->nranks, ctx->rank, &first, &count);
    f->first_last = first; f->n[last] = count;
    const size_t bytes = (size_t)tot * ndim * sizeof(double);
    cudaError_t e = cudaMalloc(&f->d_tabs, bytes);
    if (e != cudaSuccess) { delete f; return fail(LSM_ERR_OOM, "cudaMalloc failed: %s", cudaGetErrorString(e)); }
    e = cudaMemcpy(f->d_tabs, tabs, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(f->d_tabs); delete f; return fail(LSM_ERR_CUDA, "cudaMemcpy failed: %s", cudaGetErrorString(e)); }
    ctx->cnt.h2d_bytes += (int64_t)bytes;
    long off = 0;
    for (int d = 0; d < ndim; ++d)
        for (int a = 0; a < ndim; ++a) {
            f->tab[d][a] = f->d_tabs + off + (a == last ? first : 0);
            off += n[a];
        }
    *out = f;
    return LSM_OK;
}

int32_t lsm_field_destroy(lsm_field* f) {
    if (!f) return LSM_OK;
    cudaSetDevice(f->ctx->device);
    cudaStreamSynchronize(f->ctx->stream);
    cudaStreamSynchronize(f->ctx->comm);
    // drop the CFL memos of this field: a new field at the same address must not find them
    auto& cm = f->ctx->cfl_memo;
    for (size_t i = 0; i < cm.size();) { if (cm[i].field == f) cm.erase(cm.begin() + i); else ++i; }
    field_free(f);
    return LSM_OK;
}

int32_t lsm_field_set_bc(lsm_field* f, const lsm_bc* bc) {
    if (!f || !bc) return fail(LSM_ERR_ARG, "null argument");
    for (int d = 0; d < f->ndim; ++d) {
        const lsm_bc l = bc[2 * d], r = bc[2 * d + 1];
        for (const lsm_bc& b : {l, r}) {
            if (b.kind < LSM_BC_PERIODIC || b.kind > LSM_BC_SYMMETRY) return fail(LSM_ERR_BC, "invalid boundary condition kind %d for dimension %d", b.kind, d + 1);
            if (b.kind == LSM_BC_EXTRAP && (b.P < 0 || b.P > LSM_MAX_EXTRAP_P)) return fail(LSM_ERR_BC, "extrapolation order P must be in 0..%d", LSM_MAX_EXTRAP_P);
        }
        if ((l.kind == LSM_BC_PERIODIC) != (r.kind == LSM_BC_PERIODIC))     // boundaryconditions.jl:184-186
            return fail(LSM_ERR_BC, "periodic boundary conditions cannot be mixed with others in dimension %d", d + 1);
    }
    for (int d = 0; d < f->ndim; ++d) { f->bc[d][0] = bc[2 * d]; f->bc[d][1] = bc[2 * d + 1]; }
    f->has_bc = true;
    f->halo_valid = false;
    for (lsm_field* b : {f->buf1, f->buf2}) if (b) { std::memcpy(b->bc, f->bc, sizeof f->bc); b->has_bc = true; b->halo_valid = false; }
    return LSM_OK;
}

int32_t lsm_field_local_extent(const lsm_field* f, int32_t* n_local, int32_t* first_last) {
    if (!f || !n_local) return fail(LSM_ERR_ARG, "null argument");
    for (int d = 0; d < f->ndim; ++d) n_local[d] = f->n[d];
    if (first_last) *first_last = f->first_last;
    return LSM_OK;
}

int32_t lsm_field_meshsize(const lsm_field* f, double* h_out) {
    if (!f || !h_out) return fail(LSM_ERR_ARG, "null argument");
    for (int d = 0; d < f->ndim; ++d) h_out[d] = f->h[d];
    return LSM_OK;
}

int32_t lsm_field_getindex(lsm_field* f, const int32_t* I, int32_t count, double* out) {
    if (!f || !I || !out || count < 1) return fail(LSM_ERR_ARG, "bad argument");
    if (f->separable || f->ncomp != 1) return fail(LSM_ERR_ARG, "getindex needs a scalar dense field");
    lsm_ctx* c = f->ctx;
    if (c->nranks > 1) return fail(LSM_ERR_UNSUPPORTED, "lsm_field_getindex is single-rank only");
    CU(cudaSetDevice(c->device));
    // in-grid reads need no BC; out-of-grid reads without BCs throw in the reference (meshfield.jl:222-232)
    for (int t = 0; t < count; ++t)
        for (int d = 0; d < f->ndim; ++d)
            if ((I[t * f->ndim + d] < 1 || I[t * f->ndim + d] > f->n[d]) && !f->has_bc)
                return fail(LSM_ERR_BC, "index lies outside the grid, but the field has no boundary conditions to resolve it");
    void* work = nullptr;
    TRY(ctx_scratch(c, sizeof(double) * (size_t)count + sizeof(int) * (size_t)count * f->ndim, &work));
    double* d_out = static_cast<double*>(work);
    int* d_idx = reinterpret_cast<int*>(d_out + count);
    cudaError_t e = cudaMemcpyAsync(d_idx, I, sizeof(int) * (size_t)count * f->ndim, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = f->dtype == LSM_F64 ? launch_getindex<double>(f->ndim, make_view<double>(f), d_idx, count, d_out, c->stream)
                                                  : launch_getindex<float>(f->ndim, make_view<float>(f), d_idx, count, d_out, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "getindex failed: %s", cudaGetErrorString(e));
    c->cnt.kernel_launches += 1;
    return LSM_OK;
}

int32_t lsm_field_stage_buffer(lsm_field* phi, int32_t which, lsm_field** out) {
    if (!phi || !out || (which != 1 && which != 2)) return fail(LSM_ERR_ARG, "bad argument");
    if (phi->ncomp != 1 || phi->separable) return fail(LSM_ERR_ARG, "not a state field");
    CU(cudaSetDevice(phi->ctx->device));
    TRY(ensure_buffers(phi, which));
    *out = which == 1 ? phi->buf1 : phi->buf2;
    return LSM_OK;
}

// Vector fields are AoS on the host (Array{SVector{N,T},N}) and SoA on the device.  The transfer runs in chunks through two
// persistent 32 MB staging buffers: the copy engine moves chunk k+1 on the comm stream while the transpose kernel handles chunk k
// on the compute stream — no second full-size allocation (a 1024^3 Float64 velocity is 25.8 GB) and no cudaMalloc per call.
constexpr size_t STAGE_BYTES = 32u << 20;

int32_t staged_vector_transfer(lsm_field* f, void* host, bool upload) {
    lsm_ctx* c = f->ctx;
    const size_t es = esize(f->dtype);
    for (int b = 0; b < 2; ++b) {
        if (!c->stage[b]) CU(cudaMalloc(&c->stage[b], STAGE_BYTES));
        if (!c->ev_stage[b]) CU(cudaEventCreateWithFlags(&c->ev_stage[b], cudaEventDisableTiming));
        if (!c->ev_free[b]) CU(cudaEventCreateWithFlags(&c->ev_free[b], cudaEventDisableTiming));
    }
    const long chunk = (long)(STAGE_BYTES / (es * f->ncomp));
    char* hp = static_cast<char*>(host);
    char* dp = static_cast<char*>(f->p);
    int k = 0;
    for (long a = 0; a < f->owned; a += chunk, ++k) {
        const int b = k & 1;
        const long n = std::min(chunk, f->owned - a);
        const size_t hb = (size_t)n * f->ncomp * es;
        cudaError_t e;
        if (upload) {
            CU(cudaStreamWaitEvent(c->comm, c->ev_free[b], 0));                  // the transpose of chunk k-2 has drained this buffer
            CU(cudaMemcpyAsync(c->stage[b], hp + (size_t)a * f->ncomp * es, hb, cudaMemcpyHostToDevice, c->comm));
            CU(cudaEventRecord(c->ev_stage[b], c->comm));
            CU(cudaStreamWaitEvent(c->stream, c->ev_stage[b], 0));
            e = launch_transpose(f->dtype == LSM_F64, true, c->stage[b], dp + (size_t)a * es, n, f->ncomp, f->cstride, c->stream);
            CU(cudaEventRecord(c->ev_free[b], c->stream));
        } else {
            CU(cudaStreamWaitEvent(c->stream, c->ev_free[b], 0));                // the D2H of chunk k-2 has drained this buffer
            e = launch_transpose(f->dtype == LSM_F64, false, dp + (size_t)a * es, c->stage[b], n, f->ncomp, f->cstride, c->stream);
            CU(cudaEventRecord(c->ev_stage[b], c->stream));
            CU(cudaStreamWaitEvent(c->comm, c->ev_stage[b], 0));
            CU(cudaMemcpyAsync(hp + (size_t)a * f->ncomp * es, c->stage[b], hb, cudaMemcpyDeviceToHost, c->comm));
            CU(cudaEventRecord(c->ev_free[b], c->comm));
        }
        if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "transpose kernel launch failed: %s", cudaGetErrorString(e));
        c->cnt.kernel_launches += 1;
    }
    CU(cudaStreamSynchronize(c->comm));
    CU(cudaStreamSynchronize(c->stream));
    return LSM_OK;
}

int32_t lsm_field_upload(lsm_field* f, const void* host) {
    if (!f || !host) return fail(LSM_ERR_ARG, "null argument");
    if (f->separable) return fail(LSM_ERR_ARG, "separable fields have no dense storage");
    lsm_ctx* c = f->ctx;
    CU(cudaSetDevice(c->device));
    const size_t bytes = (size_t)f->owned * f->ncomp * esize(f->dtype);
    if (f->ncomp == 1) {
        CU(cudaMemcpyAsync(f->p, host, bytes, cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    } else {
        CU(cudaStreamSynchronize(c->comm));
        TRY(staged_vector_transfer(f, const_cast<void*>(host), true));
    }
    c->cnt.h2d_bytes += (int64_t)bytes;
    f->version++; f->halo_valid = false;
    return LSM_OK;
}

int32_t lsm_field_download(lsm_field* f, void* host) {
    if (!f || !host) return fail(LSM_ERR_ARG, "null argument");
    if (f->separable) return fail(LSM_ERR_ARG, "separable fields have no dense storage");
    lsm_ctx* c = f->ctx;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->comm));
    const size_t bytes = (size_t)f->owned * f->ncomp * esize(f->dtype);
    if (f->ncomp == 1) {
        CU(cudaMemcpyAsync(host, f->p, bytes, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    } else {
        TRY(staged_vector_transfer(f, host, false));
    }
    c->cnt.d2h_bytes += (int64_t)bytes;
    return LSM_OK;
}

int32_t lsm_field_copy(lsm_field* dst, const lsm_field* src) {
    if (!dst || !src) return fail(LSM_ERR_ARG, "null argument");
    if (dst->separable || src->separable) return fail(LSM_ERR_ARG, "separable fields cannot be copied");
    if (dst->ctx != src->ctx || dst->ndim != src->ndim || dst->dtype != src->dtype || dst->ncomp != src->ncomp)
        return fail(LSM_ERR_ARG, "copy between incompatible fields");
    for (int d = 0; d < dst->ndim; ++d) if (dst->nglob[d] != src->nglob[d]) return fail(LSM_ERR_ARG, "copy between fields of different shape");
    lsm_ctx* c = dst->ctx;
    CU(cudaSetDevice(c->device));
    for (int k = 0; k < dst->ncomp; ++k) {
        const char* s = static_cast<const char*>(src->p) + (size_t)k * src->cstride * esize(src->dtype);
        char* d = static_cast<char*>(dst->p) + (size_t)k * dst->cstride * esize(dst->dtype);
        CU(cudaMemcpyAsync(d, s, (size_t)dst->owned * esize(dst->dtype), cudaMemcpyDeviceToDevice, c->stream));
    }
    dst->version++; dst->halo_valid = false;
    return LSM_OK;
}

int32_t lsm_compute_cfl(lsm_ctx* ctx, lsm_field* phi, const lsm_term* terms, int32_t nterms, double t,
                        const double* gscale, double* dt_out) {
    if (!dt_out) return fail(LSM_ERR_ARG, "null argument");
    TRY(check_state(ctx, phi, terms, nterms));
    lsm_term tl[LSM_MAX_TERMS];
    TRY(prepare_terms(phi, terms, nterms, tl));
    return compute_cfl_impl(ctx, phi, tl, nterms, t, gscale, dt_out);
}

int32_t lsm_nstages(int32_t integrator) { return nstages(integrator); }

int32_t lsm_stage(lsm_ctx* ctx, int32_t integrator, int32_t stage, lsm_field* phi, const lsm_term* terms,
                  int32_t nterms, double tc, double dt, const double* gscale) {
    TRY(check_state(ctx, phi, terms, nterms));
    lsm_term tl[LSM_MAX_TERMS];
    TRY(prepare_terms(phi, terms, nterms, tl));
    return stage_impl(ctx, integrator, stage, phi, tl, nterms, tc, dt, gscale);
}

int32_t lsm_advance(lsm_ctx* ctx, int32_t integrator, lsm_field* phi, const lsm_term* terms, int32_t nterms,
                    double tc, double dt) {
    TRY(check_state(ctx, phi, terms, nterms));
    if (integrator < LSM_FORWARD_EULER || integrator > LSM_RK3) return fail(LSM_ERR_ARG, "bad integrator %d", integrator);
    lsm_term tl[LSM_MAX_TERMS];
    TRY(prepare_terms(phi, terms, nterms, tl));
    for (int s = 1; s <= nstages(integrator); ++s) TRY(stage_impl(ctx, integrator, s, phi, tl, nterms, tc, dt, nullptr));
    return LSM_OK;
}

int32_t lsm_integrate(lsm_ctx* ctx, int32_t integrator, double cfl, lsm_field* phi, const lsm_term* terms,
                      int32_t nterms, double t0, double tf, double dt_max, int64_t max_steps,
                      double* t_out, int64_t* steps_out) {
    TRY(check_state(ctx, phi, terms, nterms));
    NvtxRange nvtx("lsm_integrate");
    if (integrator < LSM_FORWARD_EULER || integrator > LSM_RK3) return fail(LSM_ERR_ARG, "bad integrator %d", integrator);
    if (!(tf >= t0))     // levelsetequation.jl:196
        return fail(LSM_ERR_TIME, "final time %g must be >= initial time %g: the level-set equation cannot be solved back in time", tf, t0);
    lsm_term tl[LSM_MAX_TERMS];
    TRY(prepare_terms(phi, terms, nterms, tl));
    terms = tl;
    double tc = t0;
    int64_t steps = 0;
    bool finished = true;
    int32_t rc = LSM_OK;
    // Launch-bound regime (small grids: a stage kernel lasts a few microseconds, comparable to its launch): when nothing but the
    // state changes from step to step — single rank, RK2/RK3 (whose buffers do not rotate), terms without a time factor, no
    // per-stage timing — the stage launches of one step are captured once into a CUDA graph and every later step with the same
    // dt replays it (one graph launch instead of 2-3 kernel launches plus their host-side setup).
    bool graph_ok = ctx->opt_graph && ctx->nranks == 1 && integrator != LSM_FORWARD_EULER && !ctx->opt_time &&
                    phi->owned <= (1L << 22);
    // (a time-dependent expression coefficient is materialised at each stage time: a captured fill would freeze t)
    for (int k = 0; k < nterms && graph_ok; ++k) if (terms[k].tscale_kind != LSM_TS_NONE || terms[k].coef_kind == LSM_COEF_EXPR) graph_ok = false;
    cudaGraphExec_t gexec = nullptr;
    double gdt = 0.0;
    lsm_counters gdelta{};          // counters of one captured step
    uint64_t gver[3] = {0, 0, 0};   // version bumps of phi / buf1 / buf2 per step
    // Small 2-D grids (the reference's CPU-sized cases): the whole time loop runs in ONE cluster kernel that keeps the state, the
    // stage buffers and the velocity in distributed shared memory (lsm_resident2d.cu).  The step sizes of a static velocity are
    // known in advance: dt = min(dt_max, cfl * dt_cfl, tf - tc) with a constant dt_cfl (timestepping.jl:104-118), so the host replays
    // the loop's arithmetic and hands the kernel the run-length encoded sequence.  Whatever is left (max_steps, more than
    // RES_STEP_CAP steps, a launch that is not possible) is done by the regular loop below.
    if (resident_eligible(ctx, phi, terms, nterms) && tc <= tf - jl_eps(tc) && (max_steps < 0 || max_steps > 0)) {
        double dt_cfl;
        rc = compute_cfl_impl(ctx, phi, terms, nterms, tc, nullptr, &dt_cfl);
        if (rc != LSM_OK) { if (t_out) *t_out = tc; if (steps_out) *steps_out = 0; return rc; }
        const double D = jl_min(dt_max, cfl * dt_cfl);
        if (std::isfinite(D) && D > 0.0) {
            constexpr int64_t RES_STEP_CAP = 1 << 22;
            std::vector<std::pair<double, long>> runs;
            double t = tc; int64_t n = 0;
            plan_steps(tc, tf, dt_max, cfl, dt_cfl, max_steps < 0 ? RES_STEP_CAP : std::min<int64_t>(max_steps, RES_STEP_CAP), runs, &t, &n);
            int32_t rr = phi->dtype == LSM_F64 ? run_resident<double>(ctx, integrator, phi, terms[0], runs)
                                               : run_resident<float>(ctx, integrator, phi, terms[0], runs);
            if (rr == LSM_OK) { tc = t; steps = n; }
            else if (rr != LSM_ERR_UNSUPPORTED) { if (t_out) *t_out = tc; if (steps_out) *steps_out = 0; return rr; }
        }
    }
    while (tc <= tf - jl_eps(tc)) {                                   // timestepping.jl:104
        if (max_steps >= 0 && steps >= max_steps) { finished = false; break; }
        double dt_cfl;
        rc = compute_cfl_impl(ctx, phi, terms, nterms, tc, nullptr, &dt_cfl);
        if (rc != LSM_OK) { finished = false; break; }
        const double dt = jl_min(jl_min(dt_max, cfl * dt_cfl), tf - tc);   // timestepping.jl:111
        if (gexec && dt == gdt) {
            cudaError_t ge = cudaGraphLaunch(gexec, ctx->stream);
            if (ge != cudaSuccess) { rc = fail(LSM_ERR_CUDA, "cudaGraphLaunch failed: %s", cudaGetErrorString(ge)); finished = false; break; }
            ctx->cnt.kernel_launches += gdelta.kernel_launches; ctx->cnt.stage_launches += gdelta.stage_launches;
            phi->version += gver[0]; if (phi->buf1) phi->buf1->version += gver[1]; if (phi->buf2) phi->buf2->version += gver[2];
            tc += dt;
            ++steps;
            continue;
        }
        // capture on the second step of the call (the first one has set every launch attribute and filled the CFL cache)
        const bool capture = graph_ok && !gexec && steps >= 1;
        lsm_counters before = ctx->cnt;
        uint64_t vb[3] = {phi->version, phi->buf1 ? phi->buf1->version : 0, phi->buf2 ? phi->buf2->version : 0};
        if (capture && cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); graph_ok = false; }
        const bool capturing = capture && graph_ok;
        for (int s = 1; s <= nstages(integrator) && rc == LSM_OK; ++s) rc = stage_impl(ctx, integrator, s, phi, terms, nterms, tc, dt, nullptr);
        if (capturing) {
            cudaGraph_t graph = nullptr;
            cudaError_t ge = cudaStreamEndCapture(ctx->stream, &graph);
            if (ge == cudaSuccess && graph && rc == LSM_OK) ge = cudaGraphInstantiate(&gexec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (rc == LSM_OK && ge == cudaSuccess && gexec && cudaGraphLaunch(gexec, ctx->stream) == cudaSuccess) {
                gdt = dt;
                gdelta.kernel_launches = ctx->cnt.kernel_launches - before.kernel_launches;
                gdelta.stage_launches = ctx->cnt.stage_launches - before.stage_launches;
                gver[0] = phi->version - vb[0]; gver[1] = phi->buf1 ? phi->buf1->version - vb[1] : 0; gver[2] = phi->buf2 ? phi->buf2->version - vb[2] : 0;
            } else {
                // capture not possible here: nothing of this step has run yet — drop graph mode and run the step directly
                // (an error raised while capturing is treated as "cannot capture": a real one recurs in the direct run)
                cudaGetLastError();
                if (gexec) { cudaGraphExecDestroy(gexec); gexec = nullptr; }
                graph_ok = false;
                ctx->cnt = before;
                rc = LSM_OK;
                for (int s = 1; s <= nstages(integrator) && rc == LSM_OK; ++s) rc = stage_impl(ctx, integrator, s, phi, terms, nterms, tc, dt, nullptr);
            }
        }
        if (rc != LSM_OK) { finished = false; break; }
        tc += dt;
        ++steps;
    }
    if (gexec) { cudaStreamSynchronize(ctx->stream); cudaGraphExecDestroy(gexec); }
    cudaStreamSynchronize(ctx->comm);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (t_out) *t_out = finished ? tf : tc;                           // timestepping.jl:120
    if (steps_out) *steps_out = steps;
    if (rc != LSM_OK) return rc;
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "device error during integration: %s", cudaGetErrorString(e));
    return LSM_OK;
}

int32_t lsm_eikonal_s0(lsm_field* dst, const lsm_field* phi0) {
    if (!dst || !phi0) return fail(LSM_ERR_ARG, "null argument");
    if (dst->ctx != phi0->ctx || dst->ndim != phi0->ndim || dst->ncomp != 1 || phi0->ncomp != 1 || dst->separable || phi0->separable)
        return fail(LSM_ERR_ARG, "incompatible fields");
    for (int d = 0; d < dst->ndim; ++d) if (dst->nglob[d] != phi0->nglob[d]) return fail(LSM_ERR_ARG, "shape mismatch");
    lsm_ctx* c = dst->ctx;
    CU(cudaSetDevice(c->device));
    double dx = phi0->h[0];
    for (int d = 1; d < phi0->ndim; ++d) dx = std::min(dx, phi0->h[d]);
    cudaError_t e = launch_eikonal_s0(phi0->dtype == LSM_F64, dst->dtype == LSM_F64, phi0->p, dst->p, phi0->owned, dx, c->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    c->cnt.kernel_launches += 1;
    dst->version++; dst->halo_valid = false;
    return LSM_OK;
}

static int32_t measure_impl(lsm_ctx* ctx, lsm_field* phi, bool perimeter, double* out) {
    if (!ctx || !phi || !out) return fail(LSM_ERR_ARG, "null argument");
    if (phi->ctx != ctx || phi->ncomp != 1 || phi->separable) return fail(LSM_ERR_ARG, "volume/perimeter need a real-valued field of this context");
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->comm));
    const int nblocks = ctx->sm_count * 8;
    void* work = nullptr;
    TRY(ctx_scratch(ctx, sizeof(double) * (size_t)(nblocks + 1), &work));      // persistent: a posthook payload must not cudaMalloc per call
    double* d_part = static_cast<double*>(work);
    cudaError_t e;
    // perimeter reaches off-grid at the border: a field without BCs gets LinearExtrapolationBC (levelsetops.jl:142)
    lsm_bc saved[3][2];
    std::memcpy(saved, phi->bc, sizeof saved);
    const bool had_bc = phi->has_bc;
    if (perimeter && !had_bc) for (int d = 0; d < phi->ndim; ++d) { phi->bc[d][0] = {LSM_BC_EXTRAP, 1}; phi->bc[d][1] = {LSM_BC_EXTRAP, 1}; }
    if (perimeter && ctx->nranks > 1 && !phi->halo_valid) {
        int32_t rc = exchange_halo(phi, ctx->stream);
        if (rc != LSM_OK) return rc;
    }
    if (phi->dtype == LSM_F64) e = launch_measure<double>(phi->ndim, perimeter, make_view<double>(phi), phi->h, d_part, nblocks, d_part + nblocks, ctx->stream);
    else e = launch_measure<float>(phi->ndim, perimeter, make_view<float>(phi), phi->h, d_part, nblocks, d_part + nblocks, ctx->stream);
    std::memcpy(phi->bc, saved, sizeof saved);
    if (e == cudaSuccess && ctx->nranks > 1) {
        ncclResult_t r = nccl().AllReduce(d_part + nblocks, d_part + nblocks, 1, ncclDouble, ncclSum, ctx->nccl_comm, ctx->stream);
        if (r != ncclSuccess) return fail(LSM_ERR_NCCL, "ncclAllReduce failed: %s", nccl().GetErrorString(r));
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_part + nblocks, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "measure kernel failed: %s", cudaGetErrorString(e));
    ctx->cnt.kernel_launches += 2; ctx->cnt.d2h_bytes += 8;
    return LSM_OK;
}
int32_t lsm_volume(lsm_ctx* ctx, lsm_field* phi, double* out) { return measure_impl(ctx, phi, false, out); }
int32_t lsm_perimeter(lsm_ctx* ctx, lsm_field* phi, double* out) { return measure_impl(ctx, phi, true, out); }

int32_t lsm_extend_along_normals(lsm_ctx* ctx, lsm_field* F, lsm_field* phi, int32_t nb_iters, double cfl, const uint8_t* frozen,
                                 double interface_band, double min_norm) {
    if (!ctx || !F || !phi) return fail(LSM_ERR_ARG, "null argument");
    if (F->ctx != ctx || phi->ctx != ctx || F == phi || F->ncomp != 1 || phi->ncomp != 1 || F->separable || phi->separable)
        return fail(LSM_ERR_ARG, "F and phi must be distinct scalar fields of this context");
    if (F->ndim != phi->ndim || F->dtype != phi->dtype) return fail(LSM_ERR_ARG, "F and phi must be defined on the same mesh with the same valtype");
    for (int d = 0; d < F->ndim; ++d) if (F->nglob[d] != phi->nglob[d]) return fail(LSM_ERR_ARG, "F and phi must have the same size");
    if (nb_iters < 0) return fail(LSM_ERR_ARG, "nb_iters must be non-negative");
    if (!(cfl > 0)) return fail(LSM_ERR_ARG, "cfl must be strictly positive");
    if (interface_band < 0 || min_norm < 0) return fail(LSM_ERR_ARG, "interface_band and min_norm must be non-negative");
    CU(cudaSetDevice(ctx->device));
    // boundary conditions: phi's, or LinearExtrapolationBC everywhere (velocityextension.jl:38-43); F gets the same
    lsm_bc savedP[3][2], savedF[3][2];
    std::memcpy(savedP, phi->bc, sizeof savedP); std::memcpy(savedF, F->bc, sizeof savedF);
    const bool hadP = phi->has_bc, hadF = F->has_bc;
    if (!hadP) for (int d = 0; d < phi->ndim; ++d) { phi->bc[d][0] = {LSM_BC_EXTRAP, 1}; phi->bc[d][1] = {LSM_BC_EXTRAP, 1}; }
    std::memcpy(F->bc, phi->bc, sizeof savedF);
    F->has_bc = true; F->halo_valid = false;
    for (lsm_field* b : {F->buf1, F->buf2}) if (b) { std::memcpy(b->bc, F->bc, sizeof savedF); b->has_bc = true; }
    auto restore = [&]() {
        std::memcpy(phi->bc, savedP, sizeof savedP);
        std::memcpy(F->bc, savedF, sizeof savedF); F->has_bc = hadF; F->halo_valid = false;
        for (lsm_field* b : {F->buf1, F->buf2}) if (b) { std::memcpy(b->bc, F->bc, sizeof savedF); b->has_bc = hadF; }
    };
    lsm_field* vel = nullptr;
    int32_t rc = field_alloc(ctx, phi->ndim, phi->nglob, phi->dtype, phi->ndim, phi->lc, phi->hc, false, &vel);
    if (rc != LSM_OK) { restore(); return rc; }
    unsigned char* d_frozen = nullptr;
    cudaError_t e = cudaSuccess;
    if (frozen) {
        e = cudaMalloc(&d_frozen, (size_t)phi->owned);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_frozen, frozen, (size_t)phi->owned, cudaMemcpyHostToDevice, ctx->stream);
        ctx->cnt.h2d_bytes += phi->owned;
    }
    if (e == cudaSuccess && ctx->nranks > 1 && !phi->halo_valid) { rc = exchange_halo(phi, ctx->stream); }
    if (e == cudaSuccess && rc == LSM_OK) {
        e = phi->dtype == LSM_F64
                ? launch_signed_normals<double>(phi->ndim, make_view<double>(phi), phi->h, min_norm, d_frozen, interface_band, static_cast<double*>(vel->p), vel->cstride, ctx->stream)
                : launch_signed_normals<float>(phi->ndim, make_view<float>(phi), phi->h, min_norm, d_frozen, interface_band, static_cast<float*>(vel->p), vel->cstride, ctx->stream);
        ctx->cnt.kernel_launches += 1;
    }
    if (e == cudaSuccess && rc == LSM_OK) {
        double dx = phi->h[0];
        for (int d = 1; d < phi->ndim; ++d) dx = std::min(dx, phi->h[d]);
        const double tau = cfl * dx;
        lsm_term term{};
        term.kind = LSM_TERM_ADVECTION; term.scheme = LSM_UPWIND; term.coef_kind = LSM_COEF_FIELD; term.tscale_kind = LSM_TS_NONE; term.field = vel;
        // frozen / degenerate nodes carry a zero velocity: with skip_zero_u they keep their value exactly even when a neighbour of
        // F is NaN / Inf (F is often undefined away from the interface) — the reference copies them untouched (velocityextension.jl:53-56)
        ctx->stage_skip_zero_u = 1;
        for (int it = 0; it < nb_iters && rc == LSM_OK; ++it) rc = stage_impl(ctx, LSM_FORWARD_EULER, 1, F, &term, 1, 0.0, tau, nullptr);
        ctx->stage_skip_zero_u = 0;
    }
    cudaStreamSynchronize(ctx->comm);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    if (d_frozen) cudaFree(d_frozen);
    field_free(vel);
    restore();
    if (rc != LSM_OK) return rc;
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(LSM_ERR_CUDA, "extend_along_normals failed: %s", cudaGetErrorString(e != cudaSuccess ? e : e2));
    F->version++;
    return LSM_OK;
}

int32_t lsm_interface_extract(lsm_ctx* ctx, lsm_field* phi, double level, int64_t* nverts_out, int64_t* nprims_out) {
    if (!ctx || !phi || !nverts_out || !nprims_out) return fail(LSM_ERR_ARG, "null argument");
    ctx->iface_valid = false;                   // a failed extraction leaves nothing to fetch
    TRY(check_level_set(ctx, phi, "interface extraction", 2, false));
    if (!std::isfinite(level)) return fail(LSM_ERR_ARG, "level must be finite (got %g)", level);
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_halo, 0));
    // the cells of the rank's last owned plane reach into the next rank's first plane (the upper ghost plane); the exchange is
    // collective, so every rank takes part
    if (ctx->nranks > 1 && !phi->halo_valid) TRY(exchange_halo(phi, ctx->stream));
    IfaceArgs A = field_box(phi, ctx->nranks > 1 && ctx->rank < ctx->nranks - 1);
    A.level = level;
    A.ntiles = iface_tiles(A.nodes);
    void* work = nullptr;
    TRY(ctx_scratch(ctx, iface_scratch_bytes(A.ntiles), &work));
    CU(launch_iface(A, 0, work, nullptr, nullptr, nullptr, ctx->stream));
    TRY(read_counts(ctx, iface_totals(A, work), 2));
    ctx->cnt.kernel_launches += 2;
    const int64_t nv = (int64_t)ctx->h_scalar[0], np = (int64_t)ctx->h_scalar[1];
    if (nv > (int64_t)std::numeric_limits<int32_t>::max())
        return fail(LSM_ERR_UNSUPPORTED, "the interface has %lld vertices; int32 vertex indices hold at most 2^31 - 1", (long long)nv);
    const int N = phi->ndim;
    const size_t vbytes = (size_t)nv * N * sizeof(double), kbytes = (size_t)nv * sizeof(int64_t), pbytes = (size_t)np * N * sizeof(int32_t);
    TRY(grow_scratch(ctx, &ctx->d_iface, &ctx->d_iface_bytes, vbytes + kbytes + pbytes));
    char* base = static_cast<char*>(ctx->d_iface);
    double* verts = reinterpret_cast<double*>(base);
    long long* keys = reinterpret_cast<long long*>(base + vbytes);
    int* prims = reinterpret_cast<int*>(base + vbytes + kbytes);
    if (nv > 0) { CU(launch_iface(A, 1, work, verts, keys, prims, ctx->stream)); ctx->cnt.kernel_launches += 1; }
    if (np > 0) { CU(launch_iface(A, 2, work, verts, keys, prims, ctx->stream)); ctx->cnt.kernel_launches += 1; }
    ctx->iface_valid = true; ctx->iface_ndim = N; ctx->iface_nv = nv; ctx->iface_np = np;
    *nverts_out = nv; *nprims_out = np;
    return LSM_OK;
}

int32_t lsm_interface_fetch(lsm_ctx* ctx, double* verts, int64_t* keys, int32_t* prims) {
    if (!ctx) return fail(LSM_ERR_ARG, "null context");
    if (!ctx->iface_valid) return fail(LSM_ERR_ARG, "no interface has been extracted on this context");
    const int64_t nv = ctx->iface_nv, np = ctx->iface_np;
    if ((nv > 0 && !verts) || (np > 0 && !prims)) return fail(LSM_ERR_ARG, "null output array");
    CU(cudaSetDevice(ctx->device));
    const size_t vbytes = (size_t)nv * ctx->iface_ndim * sizeof(double), kbytes = (size_t)nv * sizeof(int64_t);
    const size_t pbytes = (size_t)np * ctx->iface_ndim * sizeof(int32_t);
    const char* base = static_cast<const char*>(ctx->d_iface);
    if (vbytes) CU(cudaMemcpyAsync(verts, base, vbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (kbytes && keys) CU(cudaMemcpyAsync(keys, base + vbytes, kbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (pbytes) CU(cudaMemcpyAsync(prims, base + vbytes + kbytes, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->cnt.d2h_bytes += (int64_t)(vbytes + (keys ? kbytes : 0) + pbytes);
    return LSM_OK;
}

int32_t lsm_redistance(lsm_ctx* ctx, lsm_field* phi, int32_t band, int64_t* band_nodes_out) {
    if (band < 1) return fail(LSM_ERR_ARG, "band must be at least 1 (got %d)", band);
    TRY(check_level_set(ctx, phi, "redistancing", 2, true));
    return closest_points(ctx, phi, band, nullptr, true, false, band_nodes_out, nullptr);
}

int32_t lsm_extend_closest_point(lsm_ctx* ctx, lsm_field* F, lsm_field* phi, int32_t band, int32_t redistance_phi, int64_t* band_nodes_out) {
    if (band < 1) return fail(LSM_ERR_ARG, "band must be at least 1 (got %d)", band);
    if (F && F == phi) return fail(LSM_ERR_ARG, "the extended field F must not be phi");
    for (const lsm_field* f : {F, phi}) TRY(check_level_set(ctx, f, "the closest-point extension", 2, true));
    TRY(check_same_grid(F, phi));
    return closest_points(ctx, phi, band, F, redistance_phi != 0, false, band_nodes_out, nullptr);
}

int32_t lsm_interpolate_cubic(lsm_ctx* ctx, lsm_field* phi, int64_t npts, const double* pts, double* val, double* grad, double* hess) {
    TRY(check_level_set(ctx, phi, "cubic interpolation", 4, true));
    if (npts < 0) return fail(LSM_ERR_ARG, "npts must not be negative (got %lld)", (long long)npts);
    if (npts > 0 && !pts) return fail(LSM_ERR_ARG, "null points");
    if (npts == 0) return LSM_OK;
    CU(cudaSetDevice(ctx->device));
    const int N = phi->ndim;
    // scratch: points, then values, gradients and Hessians (only the requested ones)
    const size_t pb = (size_t)npts * N * sizeof(double), vb = val ? (size_t)npts * sizeof(double) : 0,
                 gb = grad ? pb : 0, hb = hess ? pb * N : 0;
    TRY(grow_scratch(ctx, &ctx->d_redist, &ctx->d_redist_bytes, pb + vb + gb + hb));
    char* base = static_cast<char*>(ctx->d_redist);
    double* dp = reinterpret_cast<double*>(base);
    double* dv = val ? reinterpret_cast<double*>(base + pb) : nullptr;
    double* dg = grad ? reinterpret_cast<double*>(base + pb + vb) : nullptr;
    double* dh = hess ? reinterpret_cast<double*>(base + pb + vb + gb) : nullptr;
    CU(cudaMemcpyAsync(dp, pts, pb, cudaMemcpyHostToDevice, ctx->stream));
    ctx->cnt.h2d_bytes += pb;
    CU(launch_interp_cubic(field_box(phi, false), npts, dp, dv, dg, dh, ctx->stream));
    ctx->cnt.kernel_launches += 1;
    if (val) CU(cudaMemcpyAsync(val, dv, vb, cudaMemcpyDeviceToHost, ctx->stream));
    if (grad) CU(cudaMemcpyAsync(grad, dg, gb, cudaMemcpyDeviceToHost, ctx->stream));
    if (hess) CU(cudaMemcpyAsync(hess, dh, hb, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->cnt.d2h_bytes += vb + gb + hb;
    CU(cudaStreamSynchronize(ctx->stream));
    return LSM_OK;
}

int32_t lsm_redistance_cubic(lsm_ctx* ctx, lsm_field* phi, int32_t band, int64_t* band_nodes_out, int64_t* fallback_nodes_out) {
    if (band < 1) return fail(LSM_ERR_ARG, "band must be at least 1 (got %d)", band);
    TRY(check_level_set(ctx, phi, "cubic redistancing", 4, true));
    return closest_points(ctx, phi, band, nullptr, true, true, band_nodes_out, fallback_nodes_out);
}

int32_t lsm_level_set_integrals(lsm_ctx* ctx, lsm_field* phi, lsm_field* F, double level, double* out) {
    TRY(check_level_set(ctx, phi, "level-set integrals", 2, false));
    if (F) {
        TRY(check_level_set(ctx, F, "level-set integrals", 2, false));
        TRY(check_same_grid(F, phi));
    }
    if (!std::isfinite(level)) return fail(LSM_ERR_ARG, "level must be finite (got %g)", level);
    if (!out) return fail(LSM_ERR_ARG, "null argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_halo, 0));
    // the cells of the rank's last owned plane reach into the next rank's first plane (the upper ghost plane); the exchanges are
    // collective, so every rank takes part
    if (ctx->nranks > 1 && !phi->halo_valid) TRY(exchange_halo(phi, ctx->stream));
    if (ctx->nranks > 1 && F && F != phi && !F->halo_valid) TRY(exchange_halo(F, ctx->stream));
    const int N = phi->ndim, last = N - 1;
    IntegArgs I{};
    I.g = field_box(phi, ctx->nranks > 1 && ctx->rank < ctx->nranks - 1);
    I.g.level = level;
    I.F = F ? F->p : nullptr; I.F_f64 = F && F->dtype == LSM_F64;
    I.planes = I.g.m[last] - 1;
    I.plane0 = phi->first_last;
    I.V = std::fabs(phi->h[0]);
    for (int d = 1; d < N; ++d) I.V = I.V * std::fabs(phi->h[d]);
    I.Vs = N == 3 ? I.V / 6.0 : N == 2 ? I.V / 2.0 : I.V;
    // the partials of every cell plane of the grid (32 bytes each), then the four results
    const long long nplanes = phi->nglob[last] - 1;
    void* work = nullptr;
    TRY(ctx_scratch(ctx, sizeof(double) * 4 * (size_t)(nplanes + 1), &work));
    I.part = static_cast<double*>(work);
    double* res = I.part + 4 * nplanes;
    if (ctx->nranks > 1) CU(cudaMemsetAsync(I.part, 0, sizeof(double) * 4 * (size_t)nplanes, ctx->stream));
    CU(launch_integral_planes(I, ctx->stream));
    if (ctx->nranks > 1) NC(nccl().AllReduce(I.part, I.part, (size_t)(4 * nplanes), ncclDouble, ncclSum, ctx->nccl_comm, ctx->stream));
    CU(launch_integral_sum(I.part, nplanes, res, ctx->stream));
    ctx->cnt.kernel_launches += 2;
    TRY(read_counts(ctx, res, 4));
    std::memcpy(out, ctx->h_scalar, 4 * sizeof(double));
    if (!F) out[2] = out[3] = std::numeric_limits<double>::quiet_NaN();
    return LSM_OK;
}

int32_t lsm_multi_level_set_integrals(int32_t n, lsm_ctx* const* ctx, lsm_field* const* phi, lsm_field* const* F, double level,
                                      double* out) {
    if (!ctx || !phi || !out || n < 1) return fail(LSM_ERR_ARG, "bad argument");
    std::vector<double> res(4 * (size_t)n, 0.0);
    TRY(fan_out(n, [&](int r) { return lsm_level_set_integrals(ctx[r], phi[r], F ? F[r] : nullptr, level, &res[4 * (size_t)r]); }));
    std::memcpy(out, res.data(), 4 * sizeof(double));       // identical on every rank
    return LSM_OK;
}

int32_t lsm_field_csg(lsm_ctx* ctx, lsm_field* dst, const lsm_field* src, int32_t op) {
    if (!ctx || !dst) return fail(LSM_ERR_ARG, "null argument");
    if (op < LSM_CSG_UNION || op > LSM_CSG_COMPLEMENT) return fail(LSM_ERR_ARG, "unknown set operation %d", op);
    if (dst->ctx != ctx || dst->ncomp != 1 || dst->separable) return fail(LSM_ERR_ARG, "set operations need a real-valued field of this context");
    if (op != LSM_CSG_COMPLEMENT) {
        if (!src) return fail(LSM_ERR_ARG, "null argument");
        if (src->ctx != ctx || src->ncomp != 1 || src->separable || src->ndim != dst->ndim || src->dtype != dst->dtype)
            return fail(LSM_ERR_ARG, "set operation between incompatible fields");
        for (int d = 0; d < dst->ndim; ++d) if (dst->nglob[d] != src->nglob[d]) return fail(LSM_ERR_ARG, "set operation between fields of different shape");
    }
    CU(cudaSetDevice(ctx->device));
    CU(launch_csg(dst->dtype == LSM_F64, dst->p, op == LSM_CSG_COMPLEMENT ? nullptr : src->p, dst->owned, op, ctx->stream));
    ctx->cnt.kernel_launches += 1;
    dst->version++; dst->halo_valid = false;
    return LSM_OK;
}

int32_t lsm_field_fill_shape(lsm_field* f, int32_t shape, const double* params, int32_t nparams) {
    if (!f || !params) return fail(LSM_ERR_ARG, "null argument");
    if (f->separable) return fail(LSM_ERR_ARG, "cannot fill a separable field");
    if (shape < LSM_SHAPE_SPHERE || shape > LSM_SHAPE_CONST) return fail(LSM_ERR_ARG, "unknown shape %d", shape);
    const int want = shape == LSM_SHAPE_SPHERE || shape == LSM_SHAPE_PLANE ? f->ndim + 1 : shape == LSM_SHAPE_BOX ? 2 * f->ndim : f->ncomp;
    if (nparams != want) return fail(LSM_ERR_ARG, "shape %d on a %d-D field takes %d parameters (got %d)", shape, f->ndim, want, nparams);
    if (shape != LSM_SHAPE_CONST && f->ncomp != 1) return fail(LSM_ERR_ARG, "shapes fill scalar fields");
    lsm_ctx* ctx = f->ctx;
    CU(cudaSetDevice(ctx->device));
    ShapeParams P{};
    P.shape = shape; P.ndim = f->ndim; P.ncomp = f->ncomp; P.first_last = f->first_last; P.cstride = f->cstride;
    for (int d = 0; d < 3; ++d) { P.n[d] = f->n[d]; P.lc[d] = f->lc[d]; P.h[d] = d < f->ndim ? f->h[d] : 0.0; }
    for (int k = 0; k < nparams; ++k) P.p[k] = params[k];
    cudaError_t e = launch_fill_shape(f->dtype == LSM_F64, f->p, P, ctx->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    ctx->cnt.kernel_launches += 1;
    f->version++; f->halo_valid = false;
    return LSM_OK;
}

int32_t lsm_field_fill_separable(lsm_field* dst, const lsm_field* sep) {
    if (!dst || !sep) return fail(LSM_ERR_ARG, "null argument");
    if (!sep->separable || dst->separable) return fail(LSM_ERR_ARG, "lsm_field_fill_separable(dst, sep): sep must come from lsm_field_create_separable, dst must be a stored field");
    if (dst->ctx != sep->ctx || dst->ndim != sep->ndim || dst->ncomp != sep->ndim) return fail(LSM_ERR_ARG, "destination must be a vector field of the same context and dimension");
    for (int d = 0; d < dst->ndim; ++d) if (dst->nglob[d] != sep->nglob[d]) return fail(LSM_ERR_ARG, "shape mismatch along dim %d", d + 1);
    lsm_ctx* ctx = dst->ctx;
    CU(cudaSetDevice(ctx->device));
    cudaError_t e = launch_fill_separable(dst->dtype == LSM_F64, dst->p, dst->cstride, dst->n, dst->ndim, sep->scale, sep->tab, ctx->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    ctx->cnt.kernel_launches += 1;
    dst->version++; dst->halo_valid = false;
    return LSM_OK;
}

int32_t lsm_expr_check(int32_t ndim, int32_t ncomp, const char* const* exprs) {
    const ExprKernel* k = nullptr;
    std::string err;
    const int32_t rc = expr_get(ndim, ncomp, exprs, false, &k, &err);
    if (rc != LSM_OK) g_err = err;
    return rc;
}

int32_t lsm_field_set_expr(lsm_field* f, const char* const* exprs) {
    if (!f) return fail(LSM_ERR_ARG, "null field");
    if (f->separable) return fail(LSM_ERR_ARG, "a separable field cannot carry expressions");
    CU(cudaSetDevice(f->ctx->device));
    const ExprKernel* k = nullptr;
    std::string err;
    const int32_t rc = expr_get(f->ndim, f->ncomp, exprs, true, &k, &err);
    if (rc != LSM_OK) { g_err = err; return rc; }
    if (!f->d_expr_cfl) CU(cudaMalloc(&f->d_expr_cfl, 8));
    f->expr = k;
    f->expr_filled = false;
    return LSM_OK;
}

int32_t lsm_field_fill_expr(lsm_field* f, double t) {
    if (!f) return fail(LSM_ERR_ARG, "null field");
    if (!f->expr) return fail(LSM_ERR_ARG, "no expressions attached: call lsm_field_set_expr first");
    CU(cudaSetDevice(f->ctx->device));
    return expr_fill(f, t, 0);
}

int32_t lsm_max_abs_diff(lsm_ctx* ctx, const lsm_field* a, const lsm_field* b, double* out) {
    if (!ctx || !a || !b || !out) return fail(LSM_ERR_ARG, "null argument");
    if (a->ctx != ctx || b->ctx != ctx || a->dtype != b->dtype || a->ncomp != 1 || b->ncomp != 1 || a->owned != b->owned)
        return fail(LSM_ERR_ARG, "incompatible fields");
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->comm));
    CU(cudaMemsetAsync(ctx->d_scalar, 0, 8, ctx->stream));
    cudaError_t e = launch_max_abs_diff(a->dtype == LSM_F64, a->p, b->p, a->owned, ctx->d_scalar, ctx->stream);
    if (e != cudaSuccess) return fail(LSM_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    ctx->cnt.kernel_launches += 1;
    if (ctx->nranks > 1) NC(nccl().AllReduce(ctx->d_scalar, ctx->d_scalar, 1, ncclUint64, ncclMax, ctx->nccl_comm, ctx->stream));
    CU(cudaMemcpyAsync(ctx->h_scalar, ctx->d_scalar, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->cnt.d2h_bytes += 8;
    *out = bits_to_double(*ctx->h_scalar);
    return LSM_OK;
}

}  // extern "C"
