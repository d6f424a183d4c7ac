// lsm_tiled.cu — performance kernels: fused RK-stage stencil kernels for 2-D and 3-D grids.
//
// K1 (SURVEY.md §2.2): one kernel per RK stage = ghost resolution + the finite differences of
// every term + each term's Hamiltonian + the stage combination, computed from shared memory.
//
//   * thread block = TX x TY threads owning an x-y tile of TX x (TY*NY) nodes.  In 3-D it marches along
//     z over a chunk of planes on a ring of 2*3+2 planes; in 2-D the ring is a single plane.  Every plane
//     (tile + 3-cell halo, corners included, so curvature's mixed differences are covered too) is
//     brought into the ring ONCE with cp.async (LDGSTS, no register staging) one iteration ahead of its
//     first use.  Stored coefficient fields (velocity, speed, b, S0) and phi^n are staged the same way
//     in double-buffered "aux" tiles, so the compute phase reads shared memory only.
//   * ghost cells: periodic / Neumann / symmetry / stored-halo boundaries are index maps with weight 1
//     (boundaryconditions.jl:107-153), so boundary tiles fill their ghosts by copying from the REMAPPED
//     address — no arithmetic, no divergence in the compute phase.  ExtrapolationBC{P>=1} (a weighted
//     stencil) takes the REMAP=false instantiation, whose boundary tiles call lsm_bc.cuh.
//   * the B200 FP64 pipe (measured 63 lane-ops/clk/SM, tools/fp64_peak.cu) is a co-bound of these
//     stencils, so every Hamiltonian is restructured to minimise issue slots while staying within
//     1e-10 of the reference (DESIGN.md §5):
//       - WENO5: samples are read in UPWIND ORDER q_k = phi[i - s*(3-k)], s = sign(u), which turns
//         u * (u > 0 ? weno5- : weno5+) into (|u|/h) * W(q) with no selects; W works on undivided
//         differences (WENO5 is homogeneous of degree 1), smoothness indicators and candidates are
//         written on second differences, the three weight divisions + three normalisations become
//         ONE reciprocal (MUFU.RCP64H + 2 Newton steps), and max(v^2) is a compare-select chain:
//         ~47 DP instructions per evaluation instead of ~65 + 6 divisions (13.6 slots each);
//       - Godunov/ENO2 terms use undivided differences and the positive homogeneity of minmod;
//       - curvature uses kappa*|grad phi| = (tr(H) q - g'Hg)/q, i.e. no pow() and no sqrt().
//
// Compiled with FMA contraction ON.  Parity with the CPU oracle is checked in tests/ (<= 1e-10 after
// 100 RK3 steps in Float64, <= 1e-4 in Float32).
#include "lsm_tile_util.cuh"

namespace lsm {

namespace {

#ifndef LSM_MINB_2D
#define LSM_MINB_2D 4      // 2-D blocks process a single tile (load, wait, compute): latency bound, so favour resident blocks
#endif
#ifndef LSM_MINB_EIK
#define LSM_MINB_EIK 3    // Eikonal kernel: latency-bound at 16 warps/SM (ncu: 'wait' + short-scoreboard stalls lead); 3 blocks of 74 KB fit.
                          // Also the single-term Float32 WENO advection kernels: 45 KB each, so 3 blocks fit and the bound keeps their
                          // registers from ruling that out
#endif

template <class T, int NDIM, int TX, int TY, int NY>
struct TileGeom {
    // A TMA box must start at a 16-byte-aligned element (measured: tools/tma_probe.cu — a Float64 box at an odd x
    // faults with "illegal instruction"), so the tile starts XL = 4 columns left of x0 (one unused column on each
    // side of the 3-cell halo) and rows are W = TX + 8 wide for both dtypes.
    static constexpr int XL = 4;
    static constexpr int W = TX + 2 * XL;
    static constexpr int HH = TY * NY + 2 * HAL;
    static constexpr int PLANE = ((W * HH + 31) / 32) * 32;              // slot stride: tile + halo, padded to 128 B
    static constexpr int TILE = TX * TY * NY;     // owned nodes of one plane of the tile
    static constexpr int NT = TX * TY;
    static constexpr int NW = NT / 32;
    static constexpr int PD = 1;                                    // planes prefetched ahead of the one being computed (2 measured no faster, costs smem)
    static constexpr int RING = NDIM == 3 ? 2 * HAL + 1 + PD : 1;   // phi planes resident in shared memory
    static constexpr int NBUF = NDIM == 3 ? PD + 1 : 1;             // aux tiles (coefficients, phi^n) in flight
    static size_t smem_bytes(int naux) { return ((size_t)RING * PLANE + (size_t)NBUF * naux * TILE) * sizeof(T) + 128 + 16; }   // + alignment slack + mbarrier
};


// Fused stage kernel.  MASK = which term kinds the instantiation carries code for; the terms themselves
// (order, coefficients) are runtime data, applied one after the other like the reference
// (x = base; x -= c*H_1; x -= c*H_2; ..., timestepping.jl:128-202).
template <class T, int NDIM, int MASK, int NTS, int COEFK, bool REMAP, int TX, int TY, int NY, int MINB, int TK, int SB>
__global__ void __launch_bounds__(TX * TY, (NDIM == 2 ? LSM_MINB_2D
                                                   : ((MASK == M_EIK && TK >= 0) || (sizeof(T) == 4 && MASK == M_ADV_WENO && NTS == 1) ? LSM_MINB_EIK : MINB)))
stage_tiled_kernel(const __grid_constant__ StageParams<T> P, const __grid_constant__ AuxList A, const __grid_constant__ TmaMaps M, const int cz) {
    using G = TileGeom<T, NDIM, TX, TY, NY>;
    constexpr int RING = G::RING;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned char* const sm128 = smem_raw + ((128u - ((unsigned)__cvta_generic_to_shared(smem_raw) & 127u)) & 127u);   // TMA wants 128 B
    T* const ring = reinterpret_cast<T*>(sm128);
    T* const aux = ring + (size_t)RING * G::PLANE;                   // [NBUF][naux][TILE]
    unsigned long long* const bar = reinterpret_cast<unsigned long long*>(aux + (size_t)G::NBUF * A.n * G::TILE);

    const int n0 = P.in.n[0], n1 = P.in.n[1], n2 = NDIM == 3 ? P.in.n[2] : 1;
    const long vs1 = P.in.s1, vs2 = NDIM == 3 ? P.in.s2 : 0;
    const T* __restrict__ const vp = P.in.p;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int lane = tx & 31, warp = (ty * TX + tx) >> 5;
    // block -> tile: the grid's own coordinates, or (narrow band) brick blockIdx.x of the list, a tile of cz = BRICK_Z planes
    unsigned bx = blockIdx.x, by = blockIdx.y, bz = blockIdx.z;
    if (P.bricks) {
        if ((int)blockIdx.x >= P.bricks[0]) return;
        const unsigned b = (unsigned)P.bricks[1 + blockIdx.x];
        const unsigned nbx = (n0 + TX - 1) / TX, nby = (n1 + TY * NY - 1) / (TY * NY);
        bx = b % nbx; by = (b / nbx) % nby; bz = b / (nbx * nby);
    }
    const int x0 = bx * TX, y0 = by * (TY * NY);
    // range of the LAST dimension to update: z planes in 3-D, rows in 2-D (slab decomposition splits it)
    const int zbeg = NDIM == 3 ? P.r0 + bz * cz : 0;
    const int zend = NDIM == 3 ? min(P.r1, zbeg + cz) : 1;
    if (zbeg >= zend) return;
    const int ylo = NDIM == 2 ? P.r0 : 0, yhi = NDIM == 2 ? P.r1 : n1;
    if (NDIM == 2 && (y0 >= yhi || y0 + TY * NY <= ylo)) return;

    // whole tile + halo inside the stored x-y extent -> plain copies; otherwise resolve ghosts
    const bool y_lo_ok = (y0 - HAL >= 0) || (NDIM == 2 && P.in.bc[1][0].kind == BC_HALO);
    const bool y_hi_ok = (y0 + TY * NY + HAL <= n1) || (NDIM == 2 && P.in.bc[1][1].kind == BC_HALO);
    const bool xy_in = (x0 - G::XL >= 0) && (x0 - G::XL + G::W <= n0) && y_lo_ok && y_hi_ok;
    const int kzl = P.in.bc[2][0].kind, kzh = P.in.bc[2][1].kind;
    // TMA fill (one cp.async.bulk.tensor per plane, issued by thread 0, completed on an mbarrier) for tiles that need
    // no ghost resolution; everything else goes through the LDGSTS paths below.
    const bool tma_phi = NDIM == 3 && M.enabled && xy_in;
    const bool tma_aux = NDIM == 3 && M.enabled && (x0 + TX <= n0) && (y0 + TY * NY <= n1);
    const bool leader = (tx | ty) == 0;
    unsigned phase = 0;
    if (NDIM == 3 && M.enabled) {
        if (leader) mbar_init(bar, 1);
        __syncthreads();
    }

    // ---- ring fill.  One warp per row of the (tile + halo) plane: lanes 0..31 copy columns 0..31, lanes 0..W-33
    // also columns 32..W-1.  The source address of a thread's element is  rowptr + zz * vs2, where rowptr depends
    // only on the thread (x / y ghost remap included) and zz only on the plane, so everything per-thread is hoisted
    // out of the z loop and a copy costs one 64-bit add.
    constexpr int RPW = (G::HH + G::NW - 1) / G::NW;          // rows per warp
    const T* rowp[RPW];
    int dxb;                                                  // column offset of the second element (32 unless clamped)
    {
        int gxa = x0 - G::XL + lane, gxb = x0 - G::XL + 32 + lane;
        if (!xy_in && REMAP) {
            // columns / rows beyond the grid + halo of a partial tile are never read: clamp them into range
            gxa = min(max(remap_index(gxa, n0, P.in.bc[0][0].kind, P.in.bc[0][1].kind), 0), n0 - 1);
            gxb = min(max(remap_index(gxb, n0, P.in.bc[0][0].kind, P.in.bc[0][1].kind), 0), n0 - 1);
        }
        dxb = gxb - gxa;
#pragma unroll
        for (int m = 0; m < RPW; ++m) {
            int gy = y0 - HAL + warp + m * G::NW;
            if (!xy_in && REMAP) {
                gy = remap_index(gy, n1, P.in.bc[1][0].kind, P.in.bc[1][1].kind);
                if (NDIM == 2) gy = min(max(gy, P.in.bc[1][0].kind == BC_HALO ? -HAL : 0), P.in.bc[1][1].kind == BC_HALO ? n1 - 1 + HAL : n1 - 1);
                else gy = min(max(gy, 0), n1 - 1);
            }
            rowp[m] = vp + (long)gy * vs1 + gxa;
        }
    }
    const int dst0 = warp * G::W + lane;                      // element offset of row `warp`, column `lane` in a slot
    auto load_phi = [&](int z, int slot, unsigned& txb) {
        T* dst = ring + slot * G::PLANE + dst0;
        const bool z_plain = NDIM == 2 || ((z >= 0 || kzl == BC_HALO) && (z < n2 || kzh == BC_HALO));
        if (tma_phi && z_plain) {
            if (leader) tma_load_3d(ring + slot * G::PLANE, &M.phi, x0 - G::XL, y0 - HAL, z + P.in.halo, bar);
            txb += (unsigned)(G::W * G::HH * sizeof(T));
        } else if (REMAP || (xy_in && z_plain)) {
            const int zz = (NDIM == 3 && REMAP) ? remap_index(z, n2, kzl, kzh) : z;
            const long zoff = NDIM == 3 ? (long)zz * vs2 : 0;
#pragma unroll
            for (int m = 0; m < RPW; ++m) {
                if (RPW * G::NW == G::HH || warp + m * G::NW < G::HH) {
                    const T* sp = rowp[m] + zoff;
                    cp_async(dst + m * G::NW * G::W, sp, sizeof(T) == 8);
                    if (lane < G::W - 32) cp_async(dst + m * G::NW * G::W + 32, sp + dxb, sizeof(T) == 8);
                }
            }
        } else {
            for (int r = warp; r < G::HH; r += G::NW) {
                T* d = ring + slot * G::PLANE + r * G::W;
                d[lane] = getindex_slow<NDIM, T>(P.in, x0 - G::XL + lane, y0 - HAL + r, z);
                if (lane < G::W - 32) d[32 + lane] = getindex_slow<NDIM, T>(P.in, x0 - G::XL + 32 + lane, y0 - HAL + r, z);
            }
        }
    };
    // stored coefficients and phi^n of the owned nodes of plane z: per-thread node offsets are loop invariants
    long aoff[NY];
#pragma unroll
    for (int k = 0; k < NY; ++k) {
        const int ii = x0 + tx, jj = y0 + ty + k * TY;
        aoff[k] = (ii < n0 && jj < n1) ? (long)ii + (long)jj * vs1 : -1;
    }
    auto load_aux = [&](int z, int buf, unsigned& txb) {
        T* dst = aux + (size_t)buf * A.n * G::TILE + ty * TX + tx;
        const long zoff = (long)z * vs2;
        if (tma_aux) {
            if (leader)
                for (int a = 0; a < A.n; ++a) tma_load_3d(aux + ((size_t)buf * A.n + a) * G::TILE, &M.aux[a], x0, y0, z, bar);
            txb += (unsigned)(A.n * G::TILE * sizeof(T));
        } else for (int a = 0; a < A.n; ++a) {
            const T* sp = static_cast<const T*>(A.src[a]) + zoff;
#pragma unroll
            for (int k = 0; k < NY; ++k)
                if (aoff[k] >= 0) cp_async(dst + a * G::TILE + k * TY * TX, sp + aoff[k], sizeof(T) == 8);
        }
    };

    // Software pipeline (3-D): plane p lives in ring slot (p - (zbeg - HAL)) mod RING.  Iteration z issues the copies
    // of plane z + HAL + PD and of the aux tiles of plane z + PD as ONE cp.async group, computes plane z, then waits
    // until at most PD - 1 groups are pending — so a plane has PD iterations to arrive and DRAM latency is paid once
    // per chunk, not once per plane.  The slot written in iteration z held plane z - HAL - 1, last read in z - 1.
    constexpr int PD = G::PD;
    static_assert(PD == 1, "the TMA mbarrier protocol below assumes one plane of prefetch");
    {
        unsigned txb = 0;
        if (NDIM == 3) for (int p = 0; p <= 2 * HAL; ++p) load_phi(zbeg - HAL + p, p, txb);
        else load_phi(0, 0, txb);
        load_aux(zbeg, 0, txb);
        if (txb && leader) mbar_expect_tx(bar, txb);
        cp_async_commit();
        cp_async_wait_all();
        if (txb) { mbar_wait(bar, phase); phase ^= 1u; }
    }
    __syncthreads();

    const double ih[3] = {1.0 / P.h[0], 1.0 / P.h[1], NDIM == 3 ? 1.0 / P.h[2] : 0.0};
    const int i = x0 + tx;
    // separable velocity u_d = ((s_d X_d[i]) Y_d[j]) Z_d[z] (single-term advection kernels): the x-y factor is a per-thread
    // loop invariant, the z factor is block-uniform — same product order as the reference-side tables, so bit-identical
    double pxy[NY][3];
    if (TK < 0 && COEFK == COEF_SEPARABLE) {
#pragma unroll
        for (int k = 0; k < NY; ++k) {
            const int jj = min(y0 + ty + k * TY, n1 - 1), ii = min(i, n0 - 1);
#pragma unroll
            for (int d = 0; d < NDIM; ++d) pxy[k][d] = (P.terms[0].cval[d] * __ldg(P.terms[0].tab[d][0] + ii)) * __ldg(P.terms[0].tab[d][1] + jj);
        }
    }
    int s0 = 0;        // ring slot of plane z - HAL
    int ab = 0;        // aux buffer of plane z
    // element offsets of the ring slots of planes z-3 .. z+3 (block-uniform); shifted by one entry per plane
    int zo[2 * HAL + 1];
#pragma unroll
    for (int k = 0; k <= 2 * HAL; ++k) zo[k] = NDIM == 3 ? k * G::PLANE : 0;
    // output / phi^n addressing: element offset of this thread's nodes in plane z, advanced by vs2 per plane
    long lin_k[NY];
#pragma unroll
    for (int k = 0; k < NY; ++k) lin_k[k] = (long)i + (long)(y0 + ty + k * TY) * vs1 + (long)zbeg * vs2;

    // which of this thread's NY nodes exist (partial tiles / 2-D row range): a loop invariant kept as a bit mask
    unsigned act = 0;
#pragma unroll
    for (int k = 0; k < NY; ++k) {
        const int j = y0 + ty + k * TY;
        if (i < n0 && j < n1 && (NDIM == 3 || (j >= ylo && j < yhi))) act |= 1u << k;
    }

    for (int z = zbeg; z < zend; ++z) {
        unsigned txb = 0;
        if (NDIM == 3) {
            int sl = s0 + 2 * HAL + PD; sl = sl >= RING ? sl - RING : sl;
            int bf = ab + PD;           bf = bf >= G::NBUF ? bf - G::NBUF : bf;
            if (z + HAL + PD <= zend - 1 + HAL) load_phi(z + HAL + PD, sl, txb);
            if (z + PD < zend) load_aux(z + PD, bf, txb);
            if (txb && leader) mbar_expect_tx(bar, txb);
            cp_async_commit();
        }
        const T* cur = ring + zo[HAL];
        const T* auxz = aux + (size_t)ab * A.n * G::TILE;
#pragma unroll
        for (int k = 0; k < NY; ++k) {
            const int r = ty + k * TY;
            const int j = y0 + r;
            if ((act >> k) & 1u) {
                const int sc = (r + HAL) * G::W + tx + G::XL;
                const int st = r * TX + tx;
                const T* c0 = cur + sc;
                const T qc = c0[0];
                // sample at offset m along dimension d (all inside the tile + halo)
                auto at = [&](int d, int m) -> T {          // m is a compile-time constant at every call site
                    if (d == 0) return c0[m];
                    if (d == 1) return c0[m * G::W];
                    return ring[zo[HAL + m] + sc];
                };
                // upwind-ordered sample: offset mult * s along d, s = +-1 (mult compile-time)
                auto up = [&](int d, int mult, int s) -> T {
                    if (d == 0) return c0[mult * s];
                    if (d == 1) return c0[mult * s * G::W];
                    return ring[(s > 0 ? zo[HAL + mult] : zo[HAL - mult]) + sc];
                };
                auto at2 = [&](int d1, int m1, int d2, int m2) -> T {      // d1 < d2
                    const int off = (d1 == 0 ? m1 : m1 * G::W) + (d2 == 1 ? m2 * G::W : 0);
                    if (d2 == 2) return ring[zo[HAL + m2] + sc + off];
                    return c0[off];
                };
                // coefficient component d of term k (times g(t))
                auto coef_gen = [&](const TermDev& tm, int kk, int d, const bool SCALE, auto kc) -> double {
                    double v;
                    constexpr int KK = decltype(kc)::value;                 // term index when it is a compile-time constant, else -1
                    constexpr int SCK = sig_coef(COEFK, KK);                // compile-time coefficient kind (static signature)
                    constexpr int SFIRST = TK >= 0 ? sig_first(TK, COEFK, KK, NDIM) : 0;
                    const int ck = SCK >= 0 ? SCK : tm.coef_kind;
                    if (ck == COEF_FIELD) {
                        if (SCK >= 0 || A.first[kk] >= 0) v = double(auxz[((SCK >= 0 ? SFIRST : A.first[kk]) + d) * G::TILE + st]);
                        else {   // Float64 coefficient with a Float32 state (S0): read directly
                            const long node = (long)i + (long)j * vs1 + (long)z * vs2;
                            v = static_cast<const double*>(tm.coef)[(long)d * tm.cstride + node];
                        }
                    } else if (TK < 0 && COEFK == COEF_SEPARABLE) {
                        v = pxy[k][d];
                        if (NDIM == 3) v = v * __ldg(tm.tab[d][2] + z);
                    } else if (ck == COEF_SEPARABLE) {
                        v = (tm.cval[d] * __ldg(tm.tab[d][0] + i)) * __ldg(tm.tab[d][1] + j);
                        if (NDIM == 3) v = v * __ldg(tm.tab[d][2] + z);
                    } else v = tm.cval[d];
                    if (SCALE && tm.scaled) v = v * tm.g;
                    return v;
                };
                auto coef = [&](const TermDev& tm, int kk, int d, auto kc) -> double { return coef_gen(tm, kk, d, true, kc); };
                auto coef_raw = [&](const TermDev& tm, int kk, int d, auto kc) -> double { return coef_gen(tm, kk, d, false, kc); };
                // second-order ENO pair along d, undivided: returns h*neg, h*pos (levelsetterms.jl:156-170, 252-265)
                auto eno2 = [&](int d, double& ng, double& ps) {
                    const T pm2 = at(d, -2), pm1 = at(d, -1), pp1 = at(d, 1), pp2 = at(d, 2);
                    const double dm = double(T(qc - pm1)), dp = double(T(pp1 - qc));
                    const double cc = double(T(pp1 - T(2) * qc + pm1));
                    const double cm = double(T(pm2 - T(2) * pm1 + qc)), cp = double(T(qc - T(2) * pp1 + pp2));
                    ng = fma(0.5, minmod(cm, cc), dm);
                    ps = fma(-0.5, minmod(cp, cc), dp);
                };

                // static base mode SB (see SB_* below): which RK combination this launch forms, whether phi^n / corr is staged (and in
                // which aux slot) and whether a second accumulator is written are compile-time facts; SB < 0 reads them at run time
                constexpr int SP0 = TK >= 0 ? sig_first(TK, COEFK, NTS, NDIM) : (COEFK == COEF_FIELD ? NDIM : 0);   // aux slot of phi^n (static kernels)
                const int base = SB < 0 ? P.base : (SB == SB_IN || SB == SB_IN_OUT2 ? BASE_IN : SB == SB_S2 ? BASE_RK3_S2 : SB == SB_S3 ? BASE_RK3_S3 : BASE_P0);
                const bool has_p0 = SB < 0 ? A.p0 >= 0 : (SB == SB_S2 || SB == SB_S3 || SB == SB_P0);
                const bool has_out2 = SB < 0 ? P.out2 != nullptr : SB == SB_IN_OUT2;
                T x = qc;
                if (has_p0) {
                    const T pn = auxz[(SB < 0 ? A.p0 : SP0) * G::TILE + st];
                    if (base == BASE_RK3_S2) x = T(fma(0.75, double(pn), 0.25 * double(qc)));       // timestepping.jl:183
                    else if (base == BASE_RK3_S3) x = div3(T(pn + T(2) * qc));                       // timestepping.jl:194
                    else x = pn;                                                                       // RK2 S2 (corr)
                }
                T x2 = qc;

                constexpr bool ONE = (MASK & (MASK - 1)) == 0;      // single kind: no runtime kind tests
                auto one_term = [&](const TermDev& tm, const int kk, auto kc) {
                    constexpr int SKIND = sig_kind(TK, decltype(kc)::value);     // compile-time kind of this term (static signature) or -1
                    constexpr int SCK = sig_coef(COEFK, decltype(kc)::value);
                    const bool k_weno = SKIND >= 0 ? SKIND == SK_ADV_WENO : (ONE || (tm.kind == TERM_ADVECTION && tm.scheme == SCHEME_WENO5));
                    const bool k_upw = SKIND >= 0 ? SKIND == SK_ADV_UPWIND : (ONE || tm.kind == TERM_ADVECTION);
                    const bool k_god = SKIND >= 0 ? (SKIND == SK_NORMAL || SKIND == SK_EIK) : (ONE || tm.kind == TERM_NORMAL || tm.kind == TERM_EIKONAL);
                    const bool k_curv = SKIND >= 0 ? SKIND == SK_CURV : (ONE || tm.kind == TERM_CURVATURE);
                    const bool k_normal = SKIND >= 0 ? SKIND == SK_NORMAL : (MASK & M_NORMAL) && (!(MASK & M_EIK) || tm.kind == TERM_NORMAL);
                    const bool c_none = SCK >= 0 ? SCK == COEF_NONE : tm.coef_kind == COEF_NONE;
                    double H = 0.0;
                    if ((MASK & M_ADV_WENO) && k_weno) {
                        // levelsetterms.jl:73-82 : H = sum_d u_d * weno(d) = sum_d (|u_d| / h_d) * W_d, left to right
                        const double g = tm.scaled ? tm.g : 1.0;
                        const int ghi = __double2hiint(g);
#pragma unroll
                        for (int d = 0; d < NDIM; ++d) {
                            const double u = coef_raw(tm, kk, d, kc);             // velocity before the time factor g(t)
                            // v = u*g; v > 0 selects the minus-biased stencil.  sign(v) = sign(u)*sign(g); |v|/h = |u| * (|g|/h)
                            // s from the sign bits (integer ops instead of 8 DSETP): when u*g == 0 the reference takes the plus-biased
                            // stencil but multiplies it by zero, so either ordering yields the same 0 contribution (a == 0).
                            const int s = ((__double2hiint(u) ^ ghi) >> 31) | 1;                 // = sign(u*g); upwind-ordered sampling: q_k = phi[i - s*(3-k)]
                            // 2-D Float32 kernels are not faster with the FP32 evaluation (they are latency / fill bound) and C2's curvature term
                            // amplifies its 1e-7 deviations past the 1e-4 bar at 512^2 (notch corners): they take Julia's promoted form
                            const double w = (NDIM == 2 || !ONE) ? weno5_up_f64<T>(A.wk, up(d, -3, s), up(d, -2, s), up(d, -1, s), qc, up(d, 1, s), up(d, 2, s))
                                                                 : weno5_up<T>(A.wk, up(d, -3, s), up(d, -2, s), up(d, -1, s), qc, up(d, 1, s), up(d, 2, s));
                            const double a = fabs(u) * (fabs(g) * ih[d]);
                            H = d == 0 ? a * w : fma(a, w, H);
                        }
                    } else if ((MASK & M_ADV_UPWIND) && k_upw) {
#pragma unroll
                        for (int d = 0; d < NDIM; ++d) {
                            const double u = coef(tm, kk, d, kc);
                            double der = u > 0 ? double(T(qc - at(d, -1))) : double(T(at(d, 1) - qc));
                            if (P.skip_zero_u && u == 0.0) der = 0.0;
                            const double a = u * ih[d];
                            H = d == 0 ? a * der : fma(a, der, H);
                        }
                    } else if ((MASK & (M_NORMAL | M_EIK)) && k_god) {
                        // Godunov |grad phi| from the ENO2 pair (levelsetterms.jl:156-170, 252-265).  Only ONE of the two
                        // upwind selections is ever used at a node — grad+ when the sign source (speed v, frozen S0, or phi
                        // itself) is > 0, grad- otherwise — so only that one is accumulated.
                        double cf = 0.0;                      // v or S0
                        bool sp;
                        if (k_normal) { cf = coef(tm, kk, 0, kc); sp = cf > 0; }
                        else if (c_none) sp = qc > T(0);
                        else { cf = coef(tm, kk, 0, kc); sp = cf > 0; }
                        double gsel = 0.0;
#pragma unroll
                        for (int d = 0; d < NDIM; ++d) {
                            double ng, ps;
                            eno2(d, ng, ps);
                            // grad+: positive(neg)^2 + negative(pos)^2 ; grad-: negative(neg)^2 + positive(pos)^2
                            const double a = ((ng > 0) == sp) ? ng : 0.0;
                            const double b = ((ps < 0) == sp) ? ps : 0.0;
                            gsel = fma(fma(a, a, b * b), ih[d] * ih[d], gsel);
                        }
                        const double nrm = sqrt(gsel);
                        if (k_normal) {
                            // positive(v)*sqrt(grad+) + negative(v)*sqrt(grad-): one of the two products is exactly 0
                            // (a NaN speed gives 0 like positive()/negative() do)
                            H = (cf > 0 ? cf : (cf < 0 ? cf : 0.0)) * nrm;
                        } else if (c_none) {                             // live sign, O&F 7.6 (levelsetterms.jl:237-242)
                            const double den = sqrt(double(T(qc * qc)) + (nrm * nrm) * (P.dxmin * P.dxmin));
                            const double S = den == 0.0 ? 0.0 : double(qc) / den;
                            H = S * (nrm - 1.0);
                        } else {                                         // frozen sign, O&F 7.5 (levelsetterms.jl:243-247)
                            H = cf * (nrm - 1.0);
                        }
                    } else if ((MASK & M_CURV) && k_curv) {
                        // levelsetterms.jl:111-121 + levelsetops.jl:197-244:  b * kappa * |grad phi| = b * (tr(H) q - g'Hg) / q
                        double g[3] = {0, 0, 0}, Hd[3] = {0, 0, 0};
#pragma unroll
                        for (int d = 0; d < NDIM; ++d) {
                            const T pp = at(d, 1), pm = at(d, -1);
                            g[d] = double(T(pp - pm)) * (0.5 * ih[d]);
                            Hd[d] = double(T(pp - T(2) * qc + pm)) * (ih[d] * ih[d]);
                        }
                        auto mixed = [&](int d1, int d2) -> double {
                            const double a = double(T(at2(d1, 1, d2, 1) - at2(d1, 1, d2, -1)));
                            const double b = double(T(at2(d1, -1, d2, 1) - at2(d1, -1, d2, -1)));
                            return (a - b) * (0.25 * ih[d1] * ih[d2]);
                        };
                        const double h01 = mixed(0, 1);
                        double q = fma(g[1], g[1], g[0] * g[0]);
                        double tr = Hd[0] + Hd[1];
                        double quad = fma(Hd[1] * g[1], g[1], fma(Hd[0] * g[0], g[0], 2.0 * (h01 * g[0] * g[1])));
                        if (NDIM == 3) {
                            const double h02 = mixed(0, 2), h12 = mixed(1, 2);
                            q = fma(g[2], g[2], q);
                            tr += Hd[2];
                            quad = fma(Hd[2] * g[2], g[2], quad) + 2.0 * (h02 * g[0] * g[2] + h12 * g[1] * g[2]);
                        }
                        const double eps = sizeof(T) == 8 ? 2.220446049250313e-16 : 1.1920928955078125e-07;
                        const double b = coef(tm, kk, 0, kc);
                        H = q < eps ? b * 0.0 : b * (fma(tr, q, -quad) * fast_rcp<2>(q));
                    }
                    x = T(fma(-P.c, H, double(x)));
                    if (has_out2) x2 = T(fma(-P.c2, H, double(x2)));
                };
                if (NTS > 0) {
                    one_term(P.terms[0], 0, std::integral_constant<int, 0>{});
                    if (NTS > 1) one_term(P.terms[1], 1, std::integral_constant<int, 1>{});
                    static_assert(NTS <= 2, "static term lists hold at most two terms");
                } else {
                    for (int kk = 0; kk < P.nterms; ++kk) one_term(P.terms[kk], kk, std::integral_constant<int, -1>{});
                }
                const long lin = lin_k[k];
                P.out[lin] = x;
                if (has_out2) P.out2[lin] = x2;
            }
        }
        if (NDIM == 3) {
            cp_async_wait_pending<PD - 1>();
            if (txb) { mbar_wait(bar, phase); phase ^= 1u; }
            __syncthreads();
            s0 = s0 + 1 == RING ? 0 : s0 + 1;
            ab = ab + 1 == G::NBUF ? 0 : ab + 1;
#pragma unroll
            for (int k = 0; k < 2 * HAL; ++k) zo[k] = zo[k + 1];
            { int sl = s0 + 2 * HAL; sl = sl >= RING ? sl - RING : sl; zo[2 * HAL] = sl * G::PLANE; }
#pragma unroll
            for (int k = 0; k < NY; ++k) lin_k[k] += vs2;
        }
    }
}

#ifndef LSM_MINB_2D
#define LSM_MINB_2D 4      // 2-D blocks process a single tile (load, wait, compute): latency bound, so favour resident blocks
#endif
#ifndef LSM_TX
#define LSM_TX 32
#define LSM_TY 8
#define LSM_NY 2
#define LSM_MINB 2
#endif


template <class T, int NDIM, int MASK, int NTS, int COEFK, bool REMAP, int TK = -1, int SB = -1>
cudaError_t launch_tiled(const StageParams<T>& P, const AuxList& A, cudaStream_t s) {
    constexpr int TX = LSM_TX, TY = LSM_TY, NY = LSM_NY;
    using G = TileGeom<T, NDIM, TX, TY, NY>;
    auto kern = stage_tiled_kernel<T, NDIM, MASK, NTS, COEFK, REMAP, TX, TY, NY, LSM_MINB, TK, SB>;
    const size_t smem = G::smem_bytes(A.n);
    static size_t attr_smem[16] = {};
    { cudaError_t e = ensure_dyn_smem(kern, smem, attr_smem); if (e != cudaSuccess) return e; }
    const View<T>& v = P.in;
    // TMA tensor maps: 3-D, rows a multiple of 16 bytes, 16-byte aligned bases, and a grid big enough to care
    TmaMaps M;
    M.enabled = 0;
    if (NDIM == 3 && (v.n[0] * sizeof(T)) % 16 == 0 && (long)v.n[0] * v.n[1] * v.n[2] >= 32L * 32 * 32 && !tma_disabled()) {
        const T* base = v.p - (long)v.halo * v.s2;
        bool ok = ((uintptr_t)base % 16 == 0) && cached_map3<T>(&M.phi, base, v.n[0], v.n[1], (long)v.n[2] + 2L * v.halo, G::W, G::HH);
        for (int a = 0; ok && a < A.n; ++a)
            ok = ((uintptr_t)A.src[a] % 16 == 0) && cached_map3<T>(&M.aux[a], A.src[a], v.n[0], v.n[1], v.n[2], TX, TY * NY);
        M.enabled = ok ? 1 : 0;
    }
    dim3 block(TX, TY), grid;
    int cz = 1;
    if (P.bricks) {
        // one block per brick of the whole box: blocks past the list's device-side count exit at once, so the host never reads it
        static_assert(TX == BRICK_X && TY * NY == BRICK_Y, "a narrow-band brick is one x-y tile");
        cz = BRICK_Z;
        const long nb = (long)((v.n[0] + TX - 1) / TX) * ((v.n[1] + TY * NY - 1) / (TY * NY)) * (NDIM == 3 ? (v.n[2] + cz - 1) / cz : 1);
        grid = dim3((unsigned)nb, 1, 1);
    } else if (NDIM == 3) {
        const int nr = P.r1 - P.r0;
        cz = nr >= 128 ? 64 : (nr >= 32 ? 32 : nr);
        grid = dim3((v.n[0] + TX - 1) / TX, (v.n[1] + TY * NY - 1) / (TY * NY), (nr + cz - 1) / cz);
    } else {
        grid = dim3((v.n[0] + TX - 1) / TX, (v.n[1] + TY * NY - 1) / (TY * NY), 1);
    }
    kern<<<grid, block, smem, s>>>(P, A, M, cz);
    return cudaGetLastError();
}

// Static-signature kernels also fix the RK base mode at compile time (5 legal combinations of BASE_* and out2); anything
// unexpected (phi^n staged in another aux slot) takes the runtime-base instantiation.
template <class T, int NDIM, int MASK, int NTS, int COEFK, bool REMAP, int TK>
cudaError_t launch_static(const StageParams<T>& P, const AuxList& A, cudaStream_t s) {
    constexpr int SP0 = TK >= 0 ? sig_first(TK, COEFK, NTS, NDIM) : (COEFK == COEF_FIELD ? NDIM : 0);
    const int sb = static_base(P, A, SP0);
    // (cannot happen with the aux list launch_stage_tiled builds; the all-terms kernel handles anything)
    if (sb < 0) return launch_tiled<T, NDIM, M_ALL, 0, -1, REMAP>(P, A, s);
    return with_static_base(sb, [&](auto SB) { return launch_tiled<T, NDIM, MASK, NTS, COEFK, REMAP, TK, decltype(SB)::value>(P, A, s); });
}

template <class T, int NDIM, bool REMAP>
cudaError_t launch_by_mask(int mask, const StageParams<T>& P, const AuxList& A, cudaStream_t s) {
    if constexpr (REMAP) {
        switch (mask) {
            case M_ADV_WENO:
                if (P.nterms == 1) {
                    const TermDev& t0 = P.terms[0];
                    if (t0.coef_kind == COEF_FIELD && A.first[0] == 0) return launch_static<T, NDIM, M_ADV_WENO, 1, COEF_FIELD, REMAP, -1>(P, A, s);
                    if (t0.coef_kind == COEF_SEPARABLE) return launch_static<T, NDIM, M_ADV_WENO, 1, COEF_SEPARABLE, REMAP, -1>(P, A, s);
                    if (t0.coef_kind == COEF_CONST) return launch_static<T, NDIM, M_ADV_WENO, 1, COEF_CONST, REMAP, -1>(P, A, s);
                }
                break;
            // static signatures (term kinds, coefficient kinds and aux-tile slots known at compile time) for the BASELINE
            // configurations; any other ordering / coefficient kind takes the runtime-dispatch instantiation of the same mask
            case M_EIK:
                if (P.nterms == 1) {
                    const TermDev& t0 = P.terms[0];
                    if (t0.coef_kind == COEF_FIELD && A.first[0] == 0) return launch_static<T, NDIM, M_EIK, 1, COEF_FIELD, REMAP, SK_EIK>(P, A, s);
                    if (t0.coef_kind == COEF_NONE) return launch_static<T, NDIM, M_EIK, 1, COEF_NONE, REMAP, SK_EIK>(P, A, s);
                    return launch_tiled<T, NDIM, M_EIK, 1, -1, REMAP>(P, A, s);
                }
                break;
            case M_NORMAL | M_ADV_WENO:
                if (P.nterms == 2) {
                    const TermDev &t0 = P.terms[0], &t1 = P.terms[1];
                    if (t0.kind == TERM_NORMAL && t0.coef_kind == COEF_FIELD && A.first[0] == 0 && t1.coef_kind == COEF_FIELD && A.first[1] == 1)
                        return launch_static<T, NDIM, M_NORMAL | M_ADV_WENO, 2, COEF_FIELD | (COEF_FIELD << 2), REMAP, SK_NORMAL | (SK_ADV_WENO << 3)>(P, A, s);
                    return launch_tiled<T, NDIM, M_NORMAL | M_ADV_WENO, 2, -1, REMAP>(P, A, s);
                }
                break;
            case M_ADV_WENO | M_CURV:
                if (P.nterms == 2) {
                    const TermDev &t0 = P.terms[0], &t1 = P.terms[1];
                    if (t0.kind == TERM_ADVECTION && t0.coef_kind == COEF_FIELD && A.first[0] == 0 && t1.coef_kind == COEF_CONST)
                        return launch_static<T, NDIM, M_ADV_WENO | M_CURV, 2, COEF_FIELD | (COEF_CONST << 2), REMAP, SK_ADV_WENO | (SK_CURV << 3)>(P, A, s);
                    return launch_tiled<T, NDIM, M_ADV_WENO | M_CURV, 2, -1, REMAP>(P, A, s);
                }
                break;
            default: break;
        }
    }
    return launch_tiled<T, NDIM, M_ALL, 0, -1, REMAP>(P, A, s);
}

int term_mask(const TermDev& t) {
    switch (t.kind) {
        case TERM_ADVECTION: return t.scheme == SCHEME_WENO5 ? M_ADV_WENO : M_ADV_UPWIND;
        case TERM_NORMAL:    return M_NORMAL;
        case TERM_CURVATURE: return M_CURV;
        default:             return M_EIK;
    }
}

template <class T>
bool stage_tiled_supported(int ndim, const StageParams<T>& P) {
    if (ndim != 2 && ndim != 3) return false;
    if (P.nterms < 1 || P.nterms > 4) return false;
    for (int d = 0; d < ndim; ++d) if (P.in.n[d] < 8) return false;      // tiny grids: strict kernel
    int naux = P.p0 ? 1 : 0;
    for (int k = 0; k < P.nterms; ++k) {
        const TermDev& t = P.terms[k];
        if (t.coef_kind == COEF_FIELD && !(t.coef_f64 && sizeof(T) == 4)) naux += t.kind == TERM_ADVECTION ? ndim : 1;
        if (t.coef_kind == COEF_SEPARABLE && t.kind != TERM_ADVECTION) return false;
    }
    return naux <= 8;
}

}  // namespace

template <class T>
cudaError_t launch_stage_tiled(int ndim, const StageParams<T>& P, int kernel, int sm_count, cudaStream_t s, int* used_pair) {
    if (!stage_tiled_supported<T>(ndim, P)) return cudaErrorNotSupported;
    if (P.r1 <= P.r0) return cudaSuccess;
    AuxList A{};
    A.n = 0; A.p0 = -1; A.wk = weno_constants();
    int mask = 0;
    for (int k = 0; k < 4; ++k) A.first[k] = -1;
    for (int k = 0; k < P.nterms; ++k) {
        const TermDev& t = P.terms[k];
        mask |= term_mask(t);
        if (t.coef_kind == COEF_FIELD && !(t.coef_f64 && sizeof(T) == 4)) {
            A.first[k] = A.n;
            const int nc = t.kind == TERM_ADVECTION ? ndim : 1;
            for (int d = 0; d < nc; ++d) A.src[A.n++] = static_cast<const T*>(t.coef) + (long)d * t.cstride;
        }
    }
    if (P.p0) { A.p0 = A.n; A.src[A.n++] = P.p0; }
    // the x-pair kernels (lsm_pair3d.cu, lsm_pair2d.cu) report cudaErrorNotSupported for what they do not cover; they have no
    // brick-list mode
    if (kernel != 3 && !P.bricks) {
        const cudaError_t e = ndim == 3 ? launch_stage_pair3d<T>(P, A, s, kernel == 4) : launch_stage_pair2d<T>(P, A, s, kernel == 2, sm_count);
        if (e != cudaErrorNotSupported) { *used_pair = 1; return e; }
    }
    bool remap = true;     // every BC an index map?
    for (int d = 0; d < ndim; ++d)
        for (int sd = 0; sd < 2; ++sd) remap = remap && bc_index_map(P.in.bc[d][sd].kind, P.in.bc[d][sd].P);
    if (ndim == 3) return remap ? launch_by_mask<T, 3, true>(mask, P, A, s) : launch_by_mask<T, 3, false>(mask, P, A, s);
    return remap ? launch_by_mask<T, 2, true>(mask, P, A, s) : launch_by_mask<T, 2, false>(mask, P, A, s);
}

// The Makefile compiles this file twice (-DLSM_TILED_F32 / -DLSM_TILED_F64) so that the two halves of the ~160 kernel
// instantiations build in parallel; without either macro both are instantiated here.
#if !defined(LSM_TILED_F64)
template cudaError_t launch_stage_tiled<float>(int, const StageParams<float>&, int, int, cudaStream_t, int*);
#endif
#if !defined(LSM_TILED_F32)
template cudaError_t launch_stage_tiled<double>(int, const StageParams<double>&, int, int, cudaStream_t, int*);
#endif

}  // namespace lsm
