// lsm_pair2d.cu — the x-pair design of lsm_pair3d.cu for 2-D grids (BASELINE configs 1 and 2): one fused RK stage of
// AdvectionTerm(stored velocity, WENO5) alone or followed by CurvatureTerm(constant b), pipelined along y.
//
// The round-1 2-D kernel processed ONE tile per block (load, wait, compute): no overlap of loads and arithmetic at all.  Here a
// block of 4 warps owns a strip of 256 columns and MARCHES along y over a chunk of rows, exactly like the 3-D kernel marches
// along z over planes:
//   * ring of 8 rows (strip + 4 columns of halo each side) filled by TMA (cp.async.bulk.tensor + mbarrier, one elected thread per
//     row) four rows ahead of their use; the velocity / phi^n rows of the next iteration arrive in a second double-buffered set;
//   * every thread owns two adjacent x nodes: 128-bit shared loads / global stores, shared x differences, upwind side by branch
//     (lsm_pair_common.cuh);
//   * ghost rows in y are remapped TMA row coordinates; the x ghost cells of row j+2 (needed one row early by the curvature
//     term's corner reads, levelsetops.jl:197-244) are fetched from their remapped global address while row j is computed;
//   * the curvature term b kappa |grad phi| = b (tr(H) q - g'Hg) / q is evaluated from the rows the advection term already holds
//     (4 extra shared loads per pair), with the operations of lsm_tiled.cu.
// Float32 fields evaluate WENO5 in Julia's promoted Float64 form (first differences in Float32): with the curvature term on the
// Zalesak disk the all-FP32 evaluation leaves the 1e-4 bar at 512^2 (DESIGN.md §2).
#include <algorithm>
#include "lsm_pair_common.cuh"

namespace lsm {

namespace {

template <class T, int NT>
struct Pair2Geom {
    static constexpr int NW = NT / 32;
    static constexpr int BX = 64 * NW;            // columns per strip
    static constexpr int XL = 4;
    static constexpr int W = BX + 2 * XL;
    static constexpr int WB = 136;                // a TMA box holds at most 256 elements per dimension: a row is NBOX boxes of 136
    static constexpr int NBOX = BX / 128;         // elements at columns 0, 128, ... of the slot (8 columns written twice, 128-byte aligned)
    static constexpr int ROW = ((W * (int)sizeof(T) + 127) / 128) * 128 / (int)sizeof(T);     // slot stride (elements), 128 B granules
    static constexpr int RING = 2 * HAL + 2;
    static size_t smem_bytes(int naux) { return ((size_t)RING * ROW + 2 * (size_t)naux * BX) * sizeof(T) + 128 + 16; }
};

// two-node WENO5 with Julia's promotion for Float32 fields: differences in T, evaluation in Float64
template <class T, bool XMAX>
__device__ __forceinline__ void pair_eval_promoted(const WenoK& K, const T (&a)[7], const T (&b)[7], int xa, int xb, double& WA, double& WB) {
    if constexpr (sizeof(T) == 8) {
        pair_eval<T, XMAX>(K, a, b, xa, xb, WA, WB);
    } else {
        auto D = [](T hi, T lo) -> double { return double(T(hi - lo)); };
        auto one = [&](const T (&q)[7], int x) -> double {
            return x >= 0 ? weno_core<XMAX>(K, D(q[1], q[0]), D(q[2], q[1]), D(q[3], q[2]), D(q[4], q[3]), D(q[5], q[4]))
                          : weno_core<XMAX>(K, D(q[6], q[5]), D(q[5], q[4]), D(q[4], q[3]), D(q[3], q[2]), D(q[2], q[1]));
        };
        WA = one(a, xa);
        WB = one(b, xb);
    }
}

// SB: static RK base mode.  CURV: the term list is (AdvectionTerm, CurvatureTerm(constant b)); else the advection term alone.
template <class T, int NT, int SB, bool XMAX, bool CURV>
__global__ void __launch_bounds__(NT, 512 / NT)
pair2d_kernel(const __grid_constant__ StageParams<T> P, const __grid_constant__ AuxList A, const __grid_constant__ TmaMaps M, const int cy) {
    using G = Pair2Geom<T, NT>;
    using V2 = typename Vec2<T>::type;
    constexpr int RING = G::RING, W = G::W, ROW = G::ROW, BX = G::BX;
    constexpr bool HAS_P0 = SB == SB_S2 || SB == SB_S3 || SB == SB_P0;
    constexpr bool HAS_OUT2 = SB == SB_IN_OUT2;
    constexpr int NAUX = 2 + (HAS_P0 ? 1 : 0);
    constexpr int ES = (int)sizeof(T);
    constexpr unsigned PHI_BYTES = (unsigned)(G::NBOX * G::WB * ES);
    constexpr unsigned AUX_BYTES = (unsigned)(NAUX * BX * ES);
    constexpr int ABUF = NAUX * BX * ES;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned char* const sm128 = smem_raw + ((128u - ((unsigned)__cvta_generic_to_shared(smem_raw) & 127u)) & 127u);
    T* const ring = reinterpret_cast<T*>(sm128);
    T* const aux = ring + (size_t)RING * ROW;
    unsigned long long* const bar = reinterpret_cast<unsigned long long*>(aux + 2 * (size_t)NAUX * BX);

    const int n0 = P.in.n[0], n1 = P.in.n[1];
    const long vs1 = P.in.s1;
    const T* __restrict__ const vp = P.in.p;
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * BX;
    const int jbeg = P.r0 + blockIdx.y * cy;
    const int jend = min(P.r1, jbeg + cy);
    if (jbeg >= jend) return;
    const int kyl = P.in.bc[1][0].kind, kyh = P.in.bc[1][1].kind;
    const bool leader = tid == 0;

    auto issue_phi = [&](int j, int off) {
        const int row = remap_index(j, n1, kyl, kyh) + P.in.halo;
#pragma unroll
        for (int b = 0; b < G::NBOX; ++b) tma_load_3d(reinterpret_cast<unsigned char*>(ring) + off + b * 128 * ES, &M.phi, x0 - G::XL + b * 128, row, 0, bar);
    };
    auto issue_aux = [&](int j, int boff) {
#pragma unroll
        for (int a = 0; a < NAUX; ++a)
#pragma unroll
            for (int b = 0; b < BX / 256; ++b) tma_load_3d(reinterpret_cast<unsigned char*>(aux) + boff + (a * BX + b * 256) * ES, &M.aux[a], x0 + b * 256, j, 0, bar);
    };

    if (leader) mbar_init(bar, 1);
    __syncthreads();
    if (leader) {
        mbar_expect_tx(bar, (2 * HAL + 1) * PHI_BYTES + AUX_BYTES);
        for (int p = 0; p <= 2 * HAL; ++p) issue_phi(jbeg - HAL + p, p * ROW * ES);
        issue_aux(jbeg, 0);
    }

    // x ghost cells of a strip that touches the boundary: thread t < 6 owns ghost column gx = -1-t (t < 3) or n0 + (t-3)
    const bool need_fix = (x0 == 0) || (x0 + BX + HAL > n0);
    int gsx = -1, gcol = 0;                 // remapped source column, destination column inside a row slot
    if (need_fix && tid < 2 * HAL) {
        const int gx = tid < HAL ? -1 - tid : n0 + (tid - HAL);
        const int col = gx - (x0 - G::XL);
        if (col >= 0 && col < W) {
            gsx = min(max(remap_index(gx, n0, P.in.bc[0][0].kind, P.in.bc[0][1].kind), 0), n0 - 1);
            gcol = col;
        }
    }
    auto ghost_row = [&](int j) -> long {   // stored row a ghost cell of row j is read from (rows outside the grid are remapped rows)
        return (long)remap_index(j, n1, kyl, kyh) * vs1;
    };

    const int lane = tid & 31, warp = tid >> 5;
    const int i = x0 + warp * 64 + 2 * lane;
    const int scx = G::XL + warp * 64 + 2 * lane;             // element offset of node i inside a row slot
    const bool act = i < n0;
    const double g = P.terms[0].scaled ? P.terms[0].g : 1.0;
    const int ghi = __double2hiint(g);
    const double ih0 = 1.0 / P.h[0], ih1 = 1.0 / P.h[1];
    const double gih[2] = {g * ih0, g * ih1};
    double bcurv = 0.0;
    if (CURV) { bcurv = P.terms[1].cval[0]; if (P.terms[1].scaled) bcurv = bcurv * P.terms[1].g; }
    const double zopq = __longlong_as_double((long long)threadIdx.z);
    WenoK KR;
    KR.c133 = A.wk.c133 + zopq; KR.c56 = A.wk.c56 + zopq; KR.cm13 = A.wk.cm13 + zopq; KR.e6 = A.wk.e6 + zopq; KR.fl = A.wk.fl + zopq; KR.pad = 0.0;
    long lin = (long)i + (long)jbeg * vs1;

    mbar_wait(bar, 0);
    unsigned phase = 1;
    if (gsx >= 0) {        // ghosts of rows jbeg-1, jbeg, jbeg+1 (slots HAL-1 .. HAL+1)
#pragma unroll
        for (int k = -1; k <= 1; ++k) ring[(HAL + k) * ROW + gcol] = vp[ghost_row(jbeg + k) + gsx];
    }
    __syncthreads();

    int zo[2 * HAL + 1];                                       // BYTE offsets of the slots of rows j-3 .. j+3
#pragma unroll
    for (int k = 0; k <= 2 * HAL; ++k) zo[k] = k * ROW * ES;
    int onew = (2 * HAL + 1) * ROW * ES;
    int ab = 0;
    const unsigned sc_a = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)(scx * ES);
    const unsigned st_a = (unsigned)__cvta_generic_to_shared(aux) + (unsigned)((warp * 64 + 2 * lane) * ES);

    for (int j = jbeg; j < jend; ++j) {
        const bool lp = j + HAL + 1 <= jend - 1 + HAL;
        const bool la = j + 1 < jend;
        if (leader && (lp || la)) {
            mbar_expect_tx(bar, (lp ? PHI_BYTES : 0u) + (la ? AUX_BYTES : 0u));
            if (lp) issue_phi(j + HAL + 1, onew);
            if (la) issue_aux(j + 1, ABUF - ab);
        }
        // x ghosts of row j+2 (resident since two iterations; its corner cells are read when row j+1 is computed)
        T gval = T(0);
        const bool fix = gsx >= 0 && la;
        if (fix) gval = __ldg(vp + ghost_row(j + 2) + gsx);

        if (act) {
            const unsigned cur = sc_a + (unsigned)zo[HAL];
            const unsigned auxz = st_a + (unsigned)ab;
            // ---- x
            const V2 m2 = lds_pair(cur - 4 * ES, T()), m1 = lds_pair(cur - 2 * ES, T()), c0 = lds_pair(cur, T()),
                     p1 = lds_pair(cur + 2 * ES, T()), p2 = lds_pair(cur + 4 * ES, T());
            const V2 u0 = lds_pair(auxz, T()), u1 = lds_pair(auxz + BX * ES, T());
            double H[2];
            {
                const T a[7] = {m2.y, m1.x, m1.y, c0.x, c0.y, p1.x, p1.y};
                const T b[7] = {m1.x, m1.y, c0.x, c0.y, p1.x, p1.y, p2.x};
                double wa, wb;
                pair_eval_promoted<T, XMAX>(KR, a, b, __double2hiint(double(u0.x)) ^ ghi, __double2hiint(double(u0.y)) ^ ghi, wa, wb);
                H[0] = (double(u0.x) * gih[0]) * wa;
                H[1] = (double(u0.y) * gih[0]) * wb;
            }
            // ---- y: the column of every node through the ring
            V2 yv[7];
#pragma unroll
            for (int k = 0; k < 7; ++k) yv[k] = k == HAL ? c0 : lds_pair(sc_a + (unsigned)zo[k], T());
            {
                const T a[7] = {yv[0].x, yv[1].x, yv[2].x, yv[3].x, yv[4].x, yv[5].x, yv[6].x};
                const T b[7] = {yv[0].y, yv[1].y, yv[2].y, yv[3].y, yv[4].y, yv[5].y, yv[6].y};
                double wa, wb;
                pair_eval_promoted<T, XMAX>(KR, a, b, __double2hiint(double(u1.x)) ^ ghi, __double2hiint(double(u1.y)) ^ ghi, wa, wb);
                H[0] = fma(double(u1.x) * gih[1], wa, H[0]);
                H[1] = fma(double(u1.y) * gih[1], wb, H[1]);
            }
            // ---- RK base, then the terms one after the other (timestepping.jl:128-202)
            T xb[2] = {c0.x, c0.y};
            if (HAS_P0) {
                const V2 pn = lds_pair(auxz + 2 * BX * ES, T());
                const T pv[2] = {pn.x, pn.y};
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    if (SB == SB_S2) xb[c] = T(fma(0.75, double(pv[c]), 0.25 * double(xb[c])));
                    else if (SB == SB_S3) xb[c] = div3(T(pv[c] + T(2) * xb[c]));
                    else xb[c] = pv[c];
                }
            }
            T x2[2] = {c0.x, c0.y};
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                xb[c] = T(fma(-P.c, H[c], double(xb[c])));
                if (HAS_OUT2) x2[c] = T(fma(-P.c2, H[c], double(x2[c])));
            }
            if (CURV) {
                // levelsetterms.jl:111-121 + levelsetops.jl:197-244:  b kappa |grad phi| = b (tr(H) q - g'Hg) / q  (no pow, no sqrt)
                const V2 dl = lds_pair(sc_a + (unsigned)zo[HAL - 1] - 2 * ES, T()), dr = lds_pair(sc_a + (unsigned)zo[HAL - 1] + 2 * ES, T());
                const V2 ul = lds_pair(sc_a + (unsigned)zo[HAL + 1] - 2 * ES, T()), ur = lds_pair(sc_a + (unsigned)zo[HAL + 1] + 2 * ES, T());
                // rows j-1 / j / j+1 at columns i-1 .. i+2
                const T rm[4] = {dl.y, yv[HAL - 1].x, yv[HAL - 1].y, dr.x};
                const T r0[4] = {m1.y, c0.x, c0.y, p1.x};
                const T rp[4] = {ul.y, yv[HAL + 1].x, yv[HAL + 1].y, ur.x};
                const double eps = sizeof(T) == 8 ? 2.220446049250313e-16 : 1.1920928955078125e-07;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const T qc = r0[c + 1];
                    const double g0 = double(T(r0[c + 2] - r0[c])) * (0.5 * ih0);
                    const double g1 = double(T(rp[c + 1] - rm[c + 1])) * (0.5 * ih1);
                    const double h00 = double(T(r0[c + 2] - T(2) * qc + r0[c])) * (ih0 * ih0);
                    const double h11 = double(T(rp[c + 1] - T(2) * qc + rm[c + 1])) * (ih1 * ih1);
                    const double ma = double(T(rp[c + 2] - rm[c + 2])), mb = double(T(rp[c] - rm[c]));
                    const double h01 = (ma - mb) * (0.25 * ih0 * ih1);
                    const double q = fma(g1, g1, g0 * g0);
                    const double tr = h00 + h11;
                    const double quad = fma(h11 * g1, g1, fma(h00 * g0, g0, 2.0 * (h01 * g0 * g1)));
                    const double Hc = q < eps ? bcurv * 0.0 : bcurv * (fma(tr, q, -quad) * fast_rcp<2>(q));
                    xb[c] = T(fma(-P.c, Hc, double(xb[c])));
                    if (HAS_OUT2) x2[c] = T(fma(-P.c2, Hc, double(x2[c])));
                }
            }
            V2 o; o.x = xb[0]; o.y = xb[1];
            *reinterpret_cast<V2*>(P.out + lin) = o;
            if (HAS_OUT2) { V2 o2; o2.x = x2[0]; o2.y = x2[1]; *reinterpret_cast<V2*>(P.out2 + lin) = o2; }
        }
        if (fix) reinterpret_cast<T*>(reinterpret_cast<unsigned char*>(ring) + zo[HAL + 2])[gcol] = gval;
        if (lp || la) { mbar_wait(bar, phase); phase ^= 1u; }
        __syncthreads();
        {
            const int freed = zo[0];
#pragma unroll
            for (int k = 0; k < 2 * HAL; ++k) zo[k] = zo[k + 1];
            zo[2 * HAL] = onew;
            onew = freed;
        }
        ab = ABUF - ab;
        lin += vs1;
    }
}

template <class T, int SB, bool XMAX, bool CURV>
cudaError_t launch_pair2(const StageParams<T>& P, const AuxList& A, cudaStream_t s, int sm_count) {
#ifndef LSM_PAIR2D_NT
#define LSM_PAIR2D_NT 128      // 4 warps per strip (8 warps measured 1.5 % slower on C2)
#endif
    constexpr int NT = LSM_PAIR2D_NT;
    using G = Pair2Geom<T, NT>;
    auto kern = pair2d_kernel<T, NT, SB, XMAX, CURV>;
    constexpr bool HAS_P0 = SB == SB_S2 || SB == SB_S3 || SB == SB_P0;
    constexpr int NAUX = 2 + (HAS_P0 ? 1 : 0);
    const size_t smem = G::smem_bytes(NAUX);
    static size_t attr_smem[16] = {};
    { cudaError_t e = ensure_dyn_smem(kern, smem, attr_smem); if (e != cudaSuccess) return e; }
    const View<T>& v = P.in;
    TmaMaps M;
    M.enabled = 1;
    const T* base = v.p - (long)v.halo * v.s1;
    if ((uintptr_t)base % 16 != 0 || !cached_map3<T>(&M.phi, base, v.n[0], (long)v.n[1] + 2L * v.halo, 1, G::WB, 1)) return cudaErrorNotSupported;
    for (int a = 0; a < NAUX; ++a)
        if ((uintptr_t)A.src[a] % 16 != 0 || !cached_map3<T>(&M.aux[a], A.src[a], v.n[0], v.n[1], 1, 256, 1)) return cudaErrorNotSupported;
    // y chunk per block: the grid should fill the SMs' block slots (4 per SM) about once or twice; at least 8 rows per chunk
    const int nr = P.r1 - P.r0;
    const int strips = (v.n[0] + G::BX - 1) / G::BX;
    const long slots = (512L / NT) * std::max(sm_count, 1);
    int nchunks = (int)std::max<long>(1, (slots + strips - 1) / strips);
    nchunks = std::min(nchunks, std::max(1, nr / 8));
    const int cy = (nr + nchunks - 1) / nchunks;
    dim3 block(NT), grid(strips, (nr + cy - 1) / cy);
    kern<<<grid, block, smem, s>>>(P, A, M, cy);
    return cudaGetLastError();
}

template <class T, bool XMAX, bool CURV>
cudaError_t launch_pair2_sb(const StageParams<T>& P, const AuxList& A, cudaStream_t s, int sm_count) {
    return with_static_base(static_base(P, A, 2), [&](auto SB) { return launch_pair2<T, decltype(SB)::value, XMAX, CURV>(P, A, s, sm_count); });
}

}  // namespace

// 2-D: AdvectionTerm(stored velocity, WENO5) [+ CurvatureTerm(constant b)] with index-map boundary conditions on a TMA-compatible
// box; anything else reports cudaErrorNotSupported and the caller takes the general tiled kernel.
template <class T>
cudaError_t launch_stage_pair2d(const StageParams<T>& P, const AuxList& A, cudaStream_t s, bool force, int sm_count) {
    if (tma_disabled() || !encode_tiled_fn()) return cudaErrorNotSupported;
    if (P.nterms != 1 && P.nterms != 2) return cudaErrorNotSupported;
    const TermDev& ta = P.terms[0];
    if (ta.kind != TERM_ADVECTION || ta.scheme != SCHEME_WENO5 || ta.coef_kind != COEF_FIELD || ta.coef_f64 || A.first[0] != 0) return cudaErrorNotSupported;
    const bool curv = P.nterms == 2;
    if (curv && (P.terms[1].kind != TERM_CURVATURE || P.terms[1].coef_kind != COEF_CONST)) return cudaErrorNotSupported;
    const View<T>& v = P.in;
    if ((v.n[0] * sizeof(T)) % 16 != 0 || v.n[0] < 16 || v.n[1] < 8) return cudaErrorNotSupported;
    // small grids (C1: 128^2) are launch / latency bound: a 7-row prologue per strip costs more than the single-tile kernel's one load
    // (measured 29.7 vs 11.1 us per RK3 step at 128^2); LSM_OPT_KERNEL = 2 forces this kernel for tests
    if (!force && (long)v.n[0] * v.n[1] < (1L << 18)) return cudaErrorNotSupported;
    for (int d = 0; d < 2; ++d)
        for (int sd = 0; sd < 2; ++sd)
            if (!bc_index_map(v.bc[d][sd].kind, v.bc[d][sd].P)) return cudaErrorNotSupported;
    // 2-D always evaluates eps from the EXACT maximum: with the curvature term on kinked data (C2) the 20-bit maximum of the 3-D
    // advection kernel is amplified past the 1e-10 bar at 512^2 (DESIGN.md §2)
    if (curv) return launch_pair2_sb<T, true, true>(P, A, s, sm_count);
    return launch_pair2_sb<T, true, false>(P, A, s, sm_count);
}

template cudaError_t launch_stage_pair2d<float>(const StageParams<float>&, const AuxList&, cudaStream_t, bool, int);
template cudaError_t launch_stage_pair2d<double>(const StageParams<double>&, const AuxList&, cudaStream_t, bool, int);

}  // namespace lsm
