// lsm_pair3d.cu — the headline kernel: one fused RK stage of 3-D WENO5 advection (BASELINE config 3 and, in its variants,
// configs 4 and 5), re-designed around the measured issue model of round 1
// (DESIGN.md §4.1: a Float64 instruction costs two issue slots, everything else one, and the kernel is issue bound):
//
//   * every thread owns TWO ADJACENT x nodes (i, i+1) of one row (RY = 1) or of two adjacent rows (RY = 2) and
//     marches along z.  All shared-memory traffic is 128-bit (LDS.128 / STG.128 for Float64 pairs): one load
//     serves both nodes, so a node costs ~10 shared loads per stage instead of 20, and the x differences (and,
//     for RY = 2, the y differences) that neighbouring nodes have in common are computed once
//     (derivatives.jl:89-121 evaluates ϕ[I-3..I+3] per node; adjacent nodes share 6 of their 7 samples);
//   * the upwind side is resolved by BRANCHING on the sign bits of u·g(t) for the pair — the velocity is smooth,
//     so warps are almost always uniform — instead of address arithmetic per sample: each side's code reads its
//     samples at immediate offsets, and the mixed case (a sign change inside the pair or the warp) simply diverges;
//   * EVERY tile is filled by TMA (cp.async.bulk.tensor.3d + mbarrier), one elected thread per plane; tiles that
//     touch the x / y boundary get zero-filled out-of-range cells from the TMA unit and a LAZY ghost fix-up: the
//     ghost cells of plane z+1 (an index map with weight 1 for periodic / Neumann / symmetry,
//     boundaryconditions.jl:107-153) are fetched from their remapped global address while plane z is being
//     computed and stored before the barrier.  Ghost planes in z are whole-plane index remaps of the TMA coordinate.
//
// Variants (template parameters): CK = stored / separable velocity, or PAIR_EIK = the frozen-sign EikonalReinitializationTerm of
// BASELINE config 4; HASN = NormalMotionTerm + AdvectionTerm (config 5: the ENO2 pair of the Godunov norm and WENO5 share the
// first / second differences of a node); ISO = equal mesh size (per-dimension scaling folded into the stage coefficient);
// XMAX = exact max|d| for the WENO epsilon instead of the 20-bit one (lsm_tile_util.cuh: absmax5_hi); Float32 fields evaluate
// the two nodes with packed FFMA2 / FADD2 / FMUL2 (lsm_pair_common.cuh: weno_core2).
//
// With XMAX the arithmetic is the SAME sequence of operations as lsm_tiled.cu's weno5_up / eno2 / stage combination, so the two
// kernels agree bit for bit (tests/test_gpu_parity.py::test_pair_kernel_bitwise_vs_tiled, ::test_pair_kernel_eikonal_bitwise_vs_tiled);
// the default (20-bit epsilon maximum) stays within 1e-13 of that and within 1e-10 of the oracle after 100 RK3 steps.
#include <algorithm>
#include "lsm_pair_common.cuh"

namespace lsm {

namespace {

template <class T, int RY, int NT>
struct PairGeom {
    static constexpr int BX = 64;                 // nodes per tile row: 32 lanes x 2 adjacent nodes
    static constexpr int TYT = NT / 32;           // thread rows
    static constexpr int BY = TYT * RY;           // tile rows
    static constexpr int XL = 4;                  // a TMA box starts at a 16-byte aligned element: 4 columns left of x0
    static constexpr int W = BX + 2 * XL;
    static constexpr int HH = BY + 2 * HAL;
    static constexpr int PLANE = ((W * HH * (int)sizeof(T) + 127) / 128) * 128 / (int)sizeof(T);     // slot stride (elements), 128 B granules
    static constexpr int TILE = BX * BY;
    static constexpr int RING = 2 * HAL + 2;      // planes z-3 .. z+3 and the one in flight
    static constexpr int NBUF = 2;                // coefficient / phi^n tiles: the plane in use and the one in flight
    static constexpr int NGC = (6 * HH + 6 * W + NT - 1) / NT;     // ghost candidates per thread (boundary tiles)
    static size_t smem_bytes(int naux) { return ((size_t)RING * PLANE + (size_t)NBUF * naux * TILE) * sizeof(T) + 128 + 16; }
};

// One dimension of "NormalMotionTerm + AdvectionTerm(WENO5)" (BASELINE config 5) for two nodes.  The six first differences
// D[k] = phi[k-2] - phi[k-3] and five second differences E[k] = D[k+1] - D[k] of a node feed BOTH terms:
//   * the second-order ENO pair of the Godunov norm (levelsetterms.jl:156-170): D-  = D[2], D+ = D[3], D2-- = E[1], D20 = E[2],
//     D2++ = E[3] (undivided; the reference forms D20 = (phi+ - 2 phi0 + phi-)/h^2 directly, this is the same value up to rounding);
//   * WENO5 on D[0..4] (minus-biased) or D[5..1] with negated E (plus-biased).
// sp = (speed > 0) selects grad+ / grad-; g accumulates the selected squares (times w = 1/h_d^2 unless the mesh is isotropic).
template <bool XMAX, bool ISO>
__device__ __forceinline__ void pair_eval_n(const WenoK& K, const double (&a)[7], const double (&b)[7], int xa, int xb, bool spa, bool spb,
                                            double w, double& WA, double& WB, double& ga, double& gb) {
    double DA[6], DB[6], EA[5], EB[5];
#pragma unroll
    for (int k = 0; k < 6; ++k) { DA[k] = a[k + 1] - a[k]; DB[k] = b[k + 1] - b[k]; }
#pragma unroll
    for (int k = 0; k < 5; ++k) { EA[k] = DA[k + 1] - DA[k]; EB[k] = DB[k + 1] - DB[k]; }
    {
        const double nga = fma(0.5, minmod(EA[1], EA[2]), DA[2]), psa = fma(-0.5, minmod(EA[3], EA[2]), DA[3]);
        const double ngb = fma(0.5, minmod(EB[1], EB[2]), DB[2]), psb = fma(-0.5, minmod(EB[3], EB[2]), DB[3]);
        const double a1 = ((nga > 0) == spa) ? nga : 0.0, a2 = ((psa < 0) == spa) ? psa : 0.0;
        const double b1 = ((ngb > 0) == spb) ? ngb : 0.0, b2 = ((psb < 0) == spb) ? psb : 0.0;
        if (ISO) { ga = fma(a1, a1, fma(a2, a2, ga)); gb = fma(b1, b1, fma(b2, b2, gb)); }
        else { ga = fma(fma(a1, a1, a2 * a2), w, ga); gb = fma(fma(b1, b1, b2 * b2), w, gb); }
    }
    if ((xa | xb) >= 0) {
        WA = weno_core_de<XMAX>(K, DA[0], DA[1], DA[2], DA[3], DA[4], EA[0], EA[1], EA[2], EA[3]);
        WB = weno_core_de<XMAX>(K, DB[0], DB[1], DB[2], DB[3], DB[4], EB[0], EB[1], EB[2], EB[3]);
    } else if ((xa & xb) < 0) {
        WA = weno_core_de<XMAX>(K, DA[5], DA[4], DA[3], DA[2], DA[1], -EA[4], -EA[3], -EA[2], -EA[1]);
        WB = weno_core_de<XMAX>(K, DB[5], DB[4], DB[3], DB[2], DB[1], -EB[4], -EB[3], -EB[2], -EB[1]);
    } else {
        WA = xa >= 0 ? weno_core_de<XMAX>(K, DA[0], DA[1], DA[2], DA[3], DA[4], EA[0], EA[1], EA[2], EA[3])
                     : weno_core_de<XMAX>(K, DA[5], DA[4], DA[3], DA[2], DA[1], -EA[4], -EA[3], -EA[2], -EA[1]);
        WB = xb >= 0 ? weno_core_de<XMAX>(K, DB[0], DB[1], DB[2], DB[3], DB[4], EB[0], EB[1], EB[2], EB[3])
                     : weno_core_de<XMAX>(K, DB[5], DB[4], DB[3], DB[2], DB[1], -EB[4], -EB[3], -EB[2], -EB[1]);
    }
}

constexpr int PAIR_EIK = 100;    // value of the CK template parameter that selects the Eikonal variant

// CK: COEF_FIELD (stored velocity, staged by TMA next to the phi ring) or COEF_SEPARABLE (u_d = s_d X_d[i] Y_d[j] Z_d[k] from tables).
// SB: static RK base mode (SB_* of lsm_tile_util.cuh).
template <class T, int RY, int NT, int CK, int SB, bool ISO, bool XMAX, bool HASN>
__global__ void __launch_bounds__(NT, 2)
pair3d_kernel(const __grid_constant__ StageParams<T> P, const __grid_constant__ AuxList A, const __grid_constant__ TmaMaps M, const int cz) {
    using G = PairGeom<T, RY, NT>;
    using V2 = typename Vec2<T>::type;
    constexpr int RING = G::RING, W = G::W, PLANE = G::PLANE, TILE = G::TILE;
    constexpr bool HAS_P0 = SB == SB_S2 || SB == SB_S3 || SB == SB_P0;
    constexpr bool HAS_OUT2 = SB == SB_IN_OUT2;
    // HASN: the term list is (NormalMotionTerm(stored speed), AdvectionTerm(stored velocity, WENO5)) — BASELINE config 5; else the
    // single advection term.  Aux tiles: [speed,] u1, u2, u3 [, phi^n]
    // CK == PAIR_EIK: the single term is EikonalReinitializationTerm with a frozen, stored S0 (BASELINE config 4): aux tiles S0 [, phi^n]
    constexpr bool EIK = CK == PAIR_EIK;
    constexpr int TA = HASN ? 1 : 0;                       // index of the advection term
    constexpr int AU = HASN ? 1 : 0;                       // first velocity tile
    constexpr int NVEL = EIK ? 1 : (CK == COEF_FIELD ? 3 : 0) + AU;  // tiles before phi^n
    constexpr int NAUX = NVEL + (HAS_P0 ? 1 : 0);
    static_assert(!HASN || (CK == COEF_FIELD && sizeof(T) == 8 && RY == 1), "the two-term variant is Float64, stored coefficients");
    static_assert(!EIK || (!HASN && RY == 1), "the Eikonal variant is a single term");
    constexpr unsigned PHI_BYTES = (unsigned)(W * G::HH * sizeof(T));
    constexpr unsigned AUX_BYTES = (unsigned)(NAUX * TILE * sizeof(T));

    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned char* const sm128 = smem_raw + ((128u - ((unsigned)__cvta_generic_to_shared(smem_raw) & 127u)) & 127u);
    T* const ring = reinterpret_cast<T*>(sm128);
    T* const aux = ring + (size_t)RING * PLANE;                      // [NBUF][NAUX][TILE]
    unsigned long long* const bar = reinterpret_cast<unsigned long long*>(aux + (size_t)G::NBUF * NAUX * TILE);

    const int n0 = P.in.n[0], n1 = P.in.n[1], n2 = P.in.n[2];
    const long vs1 = P.in.s1, vs2 = P.in.s2;
    const T* __restrict__ const vp = P.in.p;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * 32 + tx;
    const int x0 = blockIdx.x * G::BX, y0 = blockIdx.y * G::BY;
    const int zbeg = P.r0 + blockIdx.z * cz;
    const int zend = min(P.r1, zbeg + cz);
    if (zbeg >= zend) return;
    const int kzl = P.in.bc[2][0].kind, kzh = P.in.bc[2][1].kind;
    const bool leader = tid == 0;

    auto issue_phi = [&](int z, int off) {                        // off: BYTE offset of the destination slot
        tma_load_3d(reinterpret_cast<unsigned char*>(ring) + off, &M.phi, x0 - G::XL, y0 - HAL, remap_index(z, n2, kzl, kzh) + P.in.halo, bar);
    };
    auto issue_aux = [&](int z, int boff) {                       // boff: BYTE offset of the destination buffer
#pragma unroll
        for (int a = 0; a < NAUX; ++a) tma_load_3d(reinterpret_cast<unsigned char*>(aux) + boff + a * TILE * (int)sizeof(T), &M.aux[a], x0, y0, z, bar);
    };

    if (leader) mbar_init(bar, 1);
    __syncthreads();
    if (leader) {
        mbar_expect_tx(bar, (2 * HAL + 1) * PHI_BYTES + AUX_BYTES);
        for (int p = 0; p <= 2 * HAL; ++p) issue_phi(zbeg - HAL + p, p * PLANE * (int)sizeof(T));
        issue_aux(zbeg, 0);
    }

    // ---- loop invariants (computed while the first planes are in flight) ------------------------------------------------
    // ghost cells of a boundary tile: candidate c of this thread -> (source offset inside a plane, destination offset inside a slot)
    const bool need_fix = (x0 == 0) || (x0 + G::BX + HAL > n0) || (y0 < HAL) || (y0 + G::BY + HAL > n1);
    int gsrc[G::NGC], gdst[G::NGC];
#pragma unroll
    for (int g = 0; g < G::NGC; ++g) { gsrc[g] = -1; gdst[g] = 0; }
    if (need_fix) {
#pragma unroll
        for (int g = 0; g < G::NGC; ++g) {
            const int c = tid + g * NT;
            int col = -1, row = -1;
            if (c < 6 * G::HH) {                                   // x ghost columns: 3 left of the grid, 3 right of it, every row of the box
                const int side = c / (3 * G::HH), k = (c % (3 * G::HH)) / G::HH;
                row = c % G::HH;
                const int gx = side == 0 ? -1 - k : n0 + k;
                col = gx - (x0 - G::XL);
            } else if (c < 6 * G::HH + 6 * W) {                    // y ghost rows: 3 below the grid, 3 above it, every column of the box
                const int c2 = c - 6 * G::HH;
                const int side = c2 / (3 * W), k = (c2 % (3 * W)) / W;
                col = c2 % W;
                const int gy = side == 0 ? -1 - k : n1 + k;
                row = gy - (y0 - HAL);
            }
            if (col >= 0 && col < W && row >= 0 && row < G::HH) {
                const int gx = x0 - G::XL + col, gy = y0 - HAL + row;
                if (gx >= -HAL && gx < n0 + HAL && gy >= -HAL && gy < n1 + HAL) {
                    const int sx = min(max(remap_index(gx, n0, P.in.bc[0][0].kind, P.in.bc[0][1].kind), 0), n0 - 1);
                    const int sy = min(max(remap_index(gy, n1, P.in.bc[1][0].kind, P.in.bc[1][1].kind), 0), n1 - 1);
                    gsrc[g] = sx + sy * (int)vs1;
                    gdst[g] = row * W + col;
                }
            }
        }
    }
    // this thread's nodes: columns i, i+1 of rows j0 .. j0+RY-1
    const int i = x0 + 2 * tx;
    const int j0 = y0 + ty * RY;
    const int sc = (ty * RY + HAL) * W + G::XL + 2 * tx;          // element offset of node (i, j0) inside a ring slot (even: 16-byte aligned pairs)
    const int st = (ty * RY) * G::BX + 2 * tx;                    // same inside an aux tile
    bool act[RY];
#pragma unroll
    for (int r = 0; r < RY; ++r) act[r] = i < n0 && (j0 + r) < n1;
    const double g = P.terms[TA].scaled ? P.terms[TA].g : 1.0;
    const double gN = HASN && P.terms[0].scaled ? P.terms[0].g : 1.0;
    const double ihsq[3] = {(1.0 / P.h[0]) * (1.0 / P.h[0]), (1.0 / P.h[1]) * (1.0 / P.h[1]), (1.0 / P.h[2]) * (1.0 / P.h[2])};
    const int ghi = __double2hiint(g);
    const double gih[3] = {g * (1.0 / P.h[0]), g * (1.0 / P.h[1]), g * (1.0 / P.h[2])};
    // ISO (equal mesh size in the three dimensions, the usual case): sum_d (u_d g / h) W_d = (g / h) sum_d u_d W_d, so the per-
    // dimension scaling (3 DMUL per node) folds into the stage coefficient: x -= (c g / h) * sum_d u_d W_d.
    const double cH = ISO ? P.c * gih[0] : P.c, cH2 = ISO ? P.c2 * gih[0] : P.c2;
    const double cN = ISO ? P.c * (1.0 / P.h[0]) : P.c, cN2 = ISO ? P.c2 * (1.0 / P.h[0]) : P.c2;     // normal term: sqrt(sum / h^2) = sqrt(sum) / h
    auto scl = [&](double u, int d) -> double { return ISO ? u : u * gih[d]; };
    // separable velocity: the x-y factor of every node is a loop invariant (same product order as the stored tables)
    double pxy[RY][2][3];
    if (CK == COEF_SEPARABLE) {
#pragma unroll
        for (int r = 0; r < RY; ++r)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int ii = min(i + c, n0 - 1), jj = min(j0 + r, n1 - 1);
#pragma unroll
                for (int d = 0; d < 3; ++d) pxy[r][c][d] = (P.terms[TA].cval[d] * __ldg(P.terms[TA].tab[d][0] + ii)) * __ldg(P.terms[TA].tab[d][1] + jj);
            }
    }
    const WenoK KR = weno_regs<XMAX>(A.wk);
    long lin = (long)i + (long)j0 * vs1 + (long)zbeg * vs2;       // output / phi^n element offset of node (i, j0, z)

    mbar_wait(bar, 0);
    unsigned phase = 1;
    if (need_fix) {                                                // ghosts of the first plane (slot HAL): fetched and stored on the spot
#pragma unroll
        for (int gk = 0; gk < G::NGC; ++gk)
            if (gsrc[gk] >= 0) ring[HAL * PLANE + gdst[gk]] = vp[(long)zbeg * vs2 + gsrc[gk]];
    }
    __syncthreads();

    constexpr int ES = (int)sizeof(T);
    constexpr int ABUF = NAUX * TILE * ES;                         // bytes of one aux buffer
    int zo[2 * HAL + 1];                                           // BYTE offsets of the slots of planes z-3 .. z+3 (block-uniform)
#pragma unroll
    for (int k = 0; k <= 2 * HAL; ++k) zo[k] = k * PLANE * ES;
    int onew = (2 * HAL + 1) * PLANE * ES;                         // slot receiving plane z + 4
    int ab = 0;                                                    // byte offset of the aux buffer of plane z (0 or ABUF)
    const unsigned sc_a = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)(sc * ES);      // node (i, j0) in slot 0
    const unsigned st_a = (unsigned)__cvta_generic_to_shared(aux) + (unsigned)(st * ES);       // node (i, j0) in aux tile 0 of buffer 0

    for (int z = zbeg; z < zend; ++z) {
        const bool lp = z + HAL + 1 <= zend - 1 + HAL;             // plane z+4 will be read by a later iteration
        const bool la = z + 1 < zend;
        if (leader && (lp || la)) {
            mbar_expect_tx(bar, (lp ? PHI_BYTES : 0u) + (la ? AUX_BYTES : 0u));
            if (lp) issue_phi(z + HAL + 1, onew);
            if (la) issue_aux(z + 1, ABUF - ab);
        }
        // ghost cells of plane z+1 (arrived three iterations ago, current in the next one): fetch now, store before the barrier
        T gval[G::NGC];
        const bool fix = need_fix && la;
        if (fix) {
            const T* src = vp + (long)(z + 1) * vs2;
#pragma unroll
            for (int gk = 0; gk < G::NGC; ++gk) gval[gk] = gsrc[gk] >= 0 ? __ldg(src + gsrc[gk]) : T(0);
        }

        const unsigned cur = sc_a + (unsigned)zo[HAL];
        const unsigned auxz = st_a + (unsigned)ab;
        if constexpr (EIK) {
            if (act[0]) {
                // EikonalReinitializationTerm, frozen sign (levelsetterms.jl:234-265, O&F 7.5): H = S0 (|grad phi|_Godunov - 1) with the
                // second-order ENO pair of every dimension; the operations are those of lsm_tiled.cu (direct second differences:
                // C4 is the rounding-sensitive configuration), evaluated for the two nodes of the thread from 128-bit loads.
                const V2 xm = lds_pair(cur - 2 * ES, T()), c0 = lds_pair(cur, T()), xp = lds_pair(cur + 2 * ES, T());
                const V2 s0 = lds_pair(auxz, T());
                const double cf[2] = {double(s0.x), double(s0.y)};
                const bool sp[2] = {cf[0] > 0, cf[1] > 0};
                double gsel[2] = {0.0, 0.0};
                auto eno2 = [&](T pm2, T pm1, T qc, T pp1, T pp2, double w, bool spc, double& acc) {
                    const double dm = double(T(qc - pm1)), dp = double(T(pp1 - qc));
                    const double c2 = double(T(pp1 - T(2) * qc + pm1));
                    const double cm = double(T(pm2 - T(2) * pm1 + qc)), cp = double(T(qc - T(2) * pp1 + pp2));
                    const double ng = fma(0.5, minmod(cm, c2), dm);
                    const double ps = fma(-0.5, minmod(cp, c2), dp);
                    const double a = ((ng > 0) == spc) ? ng : 0.0;
                    const double b = ((ps < 0) == spc) ? ps : 0.0;
                    acc = fma(fma(a, a, b * b), w, acc);
                };
                // x: nodes i (c0.x) and i+1 (c0.y)
                eno2(xm.x, xm.y, c0.x, c0.y, xp.x, ihsq[0], sp[0], gsel[0]);
                eno2(xm.y, c0.x, c0.y, xp.x, xp.y, ihsq[0], sp[1], gsel[1]);
                {   // y
                    const V2 a2 = lds_pair(cur - 2 * W * ES, T()), a1 = lds_pair(cur - W * ES, T()), b1 = lds_pair(cur + W * ES, T()), b2 = lds_pair(cur + 2 * W * ES, T());
                    eno2(a2.x, a1.x, c0.x, b1.x, b2.x, ihsq[1], sp[0], gsel[0]);
                    eno2(a2.y, a1.y, c0.y, b1.y, b2.y, ihsq[1], sp[1], gsel[1]);
                }
                {   // z
                    const V2 a2 = lds_pair(sc_a + (unsigned)zo[HAL - 2], T()), a1 = lds_pair(sc_a + (unsigned)zo[HAL - 1], T()),
                             b1 = lds_pair(sc_a + (unsigned)zo[HAL + 1], T()), b2 = lds_pair(sc_a + (unsigned)zo[HAL + 2], T());
                    eno2(a2.x, a1.x, c0.x, b1.x, b2.x, ihsq[2], sp[0], gsel[0]);
                    eno2(a2.y, a1.y, c0.y, b1.y, b2.y, ihsq[2], sp[1], gsel[1]);
                }
                T xb[2] = {c0.x, c0.y};
                if (HAS_P0) {
                    const V2 pn = lds_pair(auxz + TILE * ES, T());
                    const T pv[2] = {pn.x, pn.y};
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        if (SB == SB_S2) xb[c] = T(fma(0.75, double(pv[c]), 0.25 * double(xb[c])));
                        else if (SB == SB_S3) xb[c] = div3(T(pv[c] + T(2) * xb[c]));
                        else xb[c] = pv[c];
                    }
                }
                V2 o, o2;
                const double h0 = cf[0] * (sqrt(gsel[0]) - 1.0), h1 = cf[1] * (sqrt(gsel[1]) - 1.0);
                o.x = T(fma(-P.c, h0, double(xb[0]))); o.y = T(fma(-P.c, h1, double(xb[1])));
                *reinterpret_cast<V2*>(P.out + lin) = o;
                if (HAS_OUT2) {
                    o2.x = T(fma(-P.c2, h0, double(c0.x))); o2.y = T(fma(-P.c2, h1, double(c0.y)));
                    *reinterpret_cast<V2*>(P.out2 + lin) = o2;
                }
            }
        } else if (act[0]) {
            double H[RY][2];
            V2 cc[RY];
            // normal-motion term (HASN): speed of the two nodes, which Godunov norm it selects, and the accumulated squares
            double vn[RY][2], gn[RY][2];
            bool sp[RY][2];
#pragma unroll
            for (int r = 0; r < RY; ++r) {
                if (HASN) {
                    const V2 vv = lds_pair(auxz + r * G::BX * ES, T());
                    vn[r][0] = double(vv.x) * gN; vn[r][1] = double(vv.y) * gN;
                    if (!P.terms[0].scaled) { vn[r][0] = double(vv.x); vn[r][1] = double(vv.y); }
                } else { vn[r][0] = vn[r][1] = 0.0; }
                sp[r][0] = vn[r][0] > 0; sp[r][1] = vn[r][1] > 0;
                gn[r][0] = gn[r][1] = 0.0;
            }
            // one dimension for the pair (a, b): the single-term evaluation, or the shared-difference two-term one
            auto evalp = [&](const T (&a)[7], const T (&b)[7], double ua, double ub, int d, int r, double& wa, double& wb) {
                if constexpr (HASN) {
                    const double ad[7] = {double(a[0]), double(a[1]), double(a[2]), double(a[3]), double(a[4]), double(a[5]), double(a[6])};
                    const double bd[7] = {double(b[0]), double(b[1]), double(b[2]), double(b[3]), double(b[4]), double(b[5]), double(b[6])};
                    pair_eval_n<XMAX, ISO>(KR, ad, bd, __double2hiint(ua) ^ ghi, __double2hiint(ub) ^ ghi, sp[r][0], sp[r][1], ihsq[d], wa, wb, gn[r][0], gn[r][1]);
                } else {
                    pair_eval<T, XMAX>(KR, a, b, __double2hiint(ua) ^ ghi, __double2hiint(ub) ^ ghi, wa, wb);
                }
            };
            // ---- x: the two nodes of a row share 6 of their 7 samples
#pragma unroll
            for (int r = 0; r < RY; ++r) {
                const unsigned row = cur + r * W * ES;
                const V2 m2 = lds_pair(row - 4 * ES, T()), m1 = lds_pair(row - 2 * ES, T()), c0 = lds_pair(row, T()),
                         p1 = lds_pair(row + 2 * ES, T()), p2 = lds_pair(row + 4 * ES, T());
                cc[r] = c0;
                const T a[7] = {m2.y, m1.x, m1.y, c0.x, c0.y, p1.x, p1.y};
                const T b[7] = {m1.x, m1.y, c0.x, c0.y, p1.x, p1.y, p2.x};
                double ua, ub;
                if (CK == COEF_FIELD) {
                    const V2 u = lds_pair(auxz + (AU * TILE + r * G::BX) * ES, T());
                    ua = double(u.x); ub = double(u.y);
                } else { ua = pxy[r][0][0] * __ldg(P.terms[TA].tab[0][2] + z); ub = pxy[r][1][0] * __ldg(P.terms[TA].tab[0][2] + z); }
                double wa, wb;
                evalp(a, b, ua, ub, 0, r, wa, wb);
                H[r][0] = scl(ua, 0) * wa;
                H[r][1] = scl(ub, 0) * wb;
            }
            // ---- y
            {
                V2 yv[7 + RY - 1];
#pragma unroll
                for (int k = 0; k < 7 + RY - 1; ++k) yv[k] = (k >= HAL && k < HAL + RY) ? cc[k - HAL] : lds_pair(cur + (k - HAL) * W * ES, T());
                double u[RY][2];
#pragma unroll
                for (int r = 0; r < RY; ++r) {
                    if (CK == COEF_FIELD) {
                        const V2 uu = lds_pair(auxz + ((AU + 1) * TILE + r * G::BX) * ES, T());
                        u[r][0] = double(uu.x); u[r][1] = double(uu.y);
                    } else { u[r][0] = pxy[r][0][1] * __ldg(P.terms[TA].tab[1][2] + z); u[r][1] = pxy[r][1][1] * __ldg(P.terms[TA].tab[1][2] + z); }
                }
                if (RY == 1) {
                    const T a[7] = {yv[0].x, yv[1].x, yv[2].x, yv[3].x, yv[4].x, yv[5].x, yv[6].x};
                    const T b[7] = {yv[0].y, yv[1].y, yv[2].y, yv[3].y, yv[4].y, yv[5].y, yv[6].y};
                    double wa, wb;
                    evalp(a, b, u[0][0], u[0][1], 1, 0, wa, wb);
                    H[0][0] = fma(scl(u[0][0], 1), wa, H[0][0]);
                    H[0][1] = fma(scl(u[0][1], 1), wb, H[0][1]);
                } else {
                    // rows j0, j0+1 of the same column share their samples
                    const T a0[7] = {yv[0].x, yv[1].x, yv[2].x, yv[3].x, yv[4].x, yv[5].x, yv[6].x};
                    const T a1[7] = {yv[1].x, yv[2].x, yv[3].x, yv[4].x, yv[5].x, yv[6].x, yv[6 + RY - 1].x};
                    const T b0[7] = {yv[0].y, yv[1].y, yv[2].y, yv[3].y, yv[4].y, yv[5].y, yv[6].y};
                    const T b1[7] = {yv[1].y, yv[2].y, yv[3].y, yv[4].y, yv[5].y, yv[6].y, yv[6 + RY - 1].y};
                    double w00, w10, w01, w11;
                    pair_eval<T, XMAX>(KR, a0, a1, __double2hiint(u[0][0]) ^ ghi, __double2hiint(u[RY - 1][0]) ^ ghi, w00, w10);
                    pair_eval<T, XMAX>(KR, b0, b1, __double2hiint(u[0][1]) ^ ghi, __double2hiint(u[RY - 1][1]) ^ ghi, w01, w11);
                    H[0][0] = fma(scl(u[0][0], 1), w00, H[0][0]);
                    H[0][1] = fma(scl(u[0][1], 1), w01, H[0][1]);
                    H[RY - 1][0] = fma(scl(u[RY - 1][0], 1), w10, H[RY - 1][0]);
                    H[RY - 1][1] = fma(scl(u[RY - 1][1], 1), w11, H[RY - 1][1]);
                }
            }
            // ---- z: the column of every node through the ring
#pragma unroll
            for (int r = 0; r < RY; ++r) {
                V2 zv[7];
#pragma unroll
                for (int k = 0; k < 7; ++k) zv[k] = k == HAL ? cc[r] : lds_pair(sc_a + (unsigned)zo[k] + r * W * ES, T());
                const T a[7] = {zv[0].x, zv[1].x, zv[2].x, zv[3].x, zv[4].x, zv[5].x, zv[6].x};
                const T b[7] = {zv[0].y, zv[1].y, zv[2].y, zv[3].y, zv[4].y, zv[5].y, zv[6].y};
                double ua, ub;
                if (CK == COEF_FIELD) {
                    const V2 u = lds_pair(auxz + ((AU + 2) * TILE + r * G::BX) * ES, T());
                    ua = double(u.x); ub = double(u.y);
                } else { ua = pxy[r][0][2] * __ldg(P.terms[TA].tab[2][2] + z); ub = pxy[r][1][2] * __ldg(P.terms[TA].tab[2][2] + z); }
                double wa, wb;
                evalp(a, b, ua, ub, 2, r, wa, wb);
                H[r][0] = fma(scl(ua, 2), wa, H[r][0]);
                H[r][1] = fma(scl(ub, 2), wb, H[r][1]);
            }
            // ---- RK stage combination (timestepping.jl:128-202) and the pair store
#pragma unroll
            for (int r = 0; r < RY; ++r) {
                if (r > 0 && !act[r]) break;
                T xb[2] = {cc[r].x, cc[r].y};
                if (HAS_P0) {
                    const V2 pn = lds_pair(auxz + (NVEL * TILE + r * G::BX) * ES, T());
                    const T pv[2] = {pn.x, pn.y};
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        if (SB == SB_S2) xb[c] = T(fma(0.75, double(pv[c]), 0.25 * double(xb[c])));       // timestepping.jl:183
                        else if (SB == SB_S3) xb[c] = div3(T(pv[c] + T(2) * xb[c]));                       // timestepping.jl:194
                        else xb[c] = pv[c];                                                                // RK2 S2 (corr)
                    }
                }
                // terms are subtracted one after the other with a rounding to the storage type in between, like the reference
                // (x = base; x -= c H_normal; x -= c H_advection, timestepping.jl:128-202)
                T x2[2] = {cc[r].x, cc[r].y};
                if (HASN) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        // positive(v) sqrt(grad+) + negative(v) sqrt(grad-): one of the two products is exactly 0; a NaN speed gives 0
                        const double v = vn[r][c];
                        const double hn = (v > 0 ? v : (v < 0 ? v : 0.0)) * sqrt(gn[r][c]);
                        xb[c] = T(fma(-cN, hn, double(xb[c])));
                        if (HAS_OUT2) x2[c] = T(fma(-cN2, hn, double(x2[c])));
                    }
                }
                V2 o;
                o.x = T(fma(-cH, H[r][0], double(xb[0])));
                o.y = T(fma(-cH, H[r][1], double(xb[1])));
                *reinterpret_cast<V2*>(P.out + lin + r * vs1) = o;
                if (HAS_OUT2) {
                    V2 o2;
                    o2.x = T(fma(-cH2, H[r][0], double(x2[0])));
                    o2.y = T(fma(-cH2, H[r][1], double(x2[1])));
                    *reinterpret_cast<V2*>(P.out2 + lin + r * vs1) = o2;
                }
            }
        }
        if (fix) {
            T* dst = reinterpret_cast<T*>(reinterpret_cast<unsigned char*>(ring) + zo[HAL + 1]);
#pragma unroll
            for (int gk = 0; gk < G::NGC; ++gk)
                if (gsrc[gk] >= 0) dst[gdst[gk]] = gval[gk];
        }
        if (lp || la) { mbar_wait(bar, phase); phase ^= 1u; }
        __syncthreads();
        {
            const int freed = zo[0];                               // plane z-3 is dead: its slot receives plane z+5 in the next iteration
#pragma unroll
            for (int k = 0; k < 2 * HAL; ++k) zo[k] = zo[k + 1];
            zo[2 * HAL] = onew;
            onew = freed;
        }
        ab = ABUF - ab;
        lin += vs2;
    }
}

#ifndef LSM_PAIR_RY
#define LSM_PAIR_RY 1
#define LSM_PAIR_NT 256
#endif

template <class T, int CK, int SB, bool ISO, bool XMAX, bool HASN = false>
cudaError_t launch_pair_x(const StageParams<T>& P, const AuxList& A, cudaStream_t s) {
    constexpr int RY = LSM_PAIR_RY, NT = LSM_PAIR_NT;
    using G = PairGeom<T, RY, NT>;
    auto kern = pair3d_kernel<T, RY, NT, CK, SB, ISO, XMAX, HASN>;
    constexpr bool HAS_P0 = SB == SB_S2 || SB == SB_S3 || SB == SB_P0;
    constexpr int NAUX = (CK == PAIR_EIK ? 1 : (CK == COEF_FIELD ? 3 : 0) + (HASN ? 1 : 0)) + (HAS_P0 ? 1 : 0);
    const size_t smem = G::smem_bytes(NAUX);
    static size_t attr_smem[16] = {};
    { cudaError_t e = ensure_dyn_smem(kern, smem, attr_smem); if (e != cudaSuccess) return e; }
    const View<T>& v = P.in;
    TmaMaps M;
    M.enabled = 1;
    const T* base = v.p - (long)v.halo * v.s2;
    if ((uintptr_t)base % 16 != 0 || !cached_map3<T>(&M.phi, base, v.n[0], v.n[1], (long)v.n[2] + 2L * v.halo, G::W, G::HH)) return cudaErrorNotSupported;
    for (int a = 0; a < NAUX; ++a)
        if ((uintptr_t)A.src[a] % 16 != 0 || !cached_map3<T>(&M.aux[a], A.src[a], v.n[0], v.n[1], v.n[2], G::BX, G::BY)) return cudaErrorNotSupported;
    // z chunk per block: ~64 planes (the 7-plane prologue of a chunk is then < 3 % of its time and hides behind the SM's other block),
    // split evenly (120 planes of a 1024^3 / 8-GPU slab -> 2 x 60, not 32 + 32 + 32 + 24), but short enough that the grid still fills
    // the 148 x 2 block slots about twice
    const int nr = P.r1 - P.r0;
    const long tiles = (long)((v.n[0] + G::BX - 1) / G::BX) * ((v.n[1] + G::BY - 1) / G::BY);
    int nchunks = std::max(1, (nr + 32) / 64);
    const long want = (2L * 296 + tiles - 1) / tiles;                  // chunks needed for ~2 waves
    if (nchunks < want) nchunks = (int)std::min<long>(want, std::max(1, nr / 8));
    static const int cz_env = [] { const char* e = getenv("LSM_B200_CZ"); return e ? atoi(e) : 0; }();     // experiments only
    const int cz = cz_env > 0 ? std::min(cz_env, nr) : (nr + nchunks - 1) / nchunks;
    dim3 block(32, NT / 32), grid((v.n[0] + G::BX - 1) / G::BX, (v.n[1] + G::BY - 1) / G::BY, (nr + cz - 1) / cz);
    kern<<<grid, block, smem, s>>>(P, A, M, cz);
    return cudaGetLastError();
}

template <class T, int CK, int SB, bool HASN>
cudaError_t launch_pair(const StageParams<T>& P, const AuxList& A, cudaStream_t s, bool exact_eps) {
    if constexpr (CK == PAIR_EIK) return launch_pair_x<T, CK, SB, false, false, false>(P, A, s);
    const bool iso = P.h[0] == P.h[1] && P.h[1] == P.h[2];
    if (sizeof(T) == 4 || !exact_eps)      // (the Float32 evaluation normalises by the exact FP32 maximum either way)
        return iso ? launch_pair_x<T, CK, SB, true, false, HASN>(P, A, s) : launch_pair_x<T, CK, SB, false, false, HASN>(P, A, s);
    if constexpr (sizeof(T) == 8)
        return iso ? launch_pair_x<T, CK, SB, true, true, HASN>(P, A, s) : launch_pair_x<T, CK, SB, false, true, HASN>(P, A, s);
    return cudaErrorNotSupported;
}

template <class T, int CK, bool HASN = false>
cudaError_t launch_pair_sb(const StageParams<T>& P, const AuxList& A, cudaStream_t s, bool exact_eps) {
    constexpr int SP0 = CK == PAIR_EIK ? 1 : (CK == COEF_FIELD ? 3 : 0) + (HASN ? 1 : 0);
    if (A.p0 >= 0 && A.p0 != SP0) return cudaErrorNotSupported;
    if (P.base == BASE_IN && !P.p0) {
        if (!P.out2) return launch_pair<T, CK, SB_IN, HASN>(P, A, s, exact_eps);
        return launch_pair<T, CK, SB_IN_OUT2, HASN>(P, A, s, exact_eps);
    }
    if (P.base == BASE_RK3_S2 && P.p0 && !P.out2) return launch_pair<T, CK, SB_S2, HASN>(P, A, s, exact_eps);
    if (P.base == BASE_RK3_S3 && P.p0 && !P.out2) return launch_pair<T, CK, SB_S3, HASN>(P, A, s, exact_eps);
    if (P.base == BASE_P0 && P.p0 && !P.out2) return launch_pair<T, CK, SB_P0, HASN>(P, A, s, exact_eps);
    return cudaErrorNotSupported;
}

}  // namespace

// Single-term 3-D WENO5 advection with index-map boundary conditions on a TMA-compatible box; anything else reports
// cudaErrorNotSupported and the caller takes the general tiled kernel.
template <class T>
cudaError_t launch_stage_pair3d(const StageParams<T>& P, const AuxList& A, cudaStream_t s, bool exact_eps) {
    if (pair_kernel_disabled() || tma_disabled() || !encode_tiled_fn()) return cudaErrorNotSupported;
    if (P.nterms != 1 && P.nterms != 2) return cudaErrorNotSupported;
    const TermDev& ta = P.terms[P.nterms - 1];          // the advection term (last)
    const bool eik = P.nterms == 1 && ta.kind == TERM_EIKONAL && ta.coef_kind == COEF_FIELD && !ta.coef_f64 && A.first[0] == 0;
    if (!eik && (ta.kind != TERM_ADVECTION || ta.scheme != SCHEME_WENO5)) return cudaErrorNotSupported;
    const View<T>& v = P.in;
    if ((v.n[0] * sizeof(T)) % 16 != 0 || v.n[0] < 8 || v.n[1] < 8 || v.n[2] < 4) return cudaErrorNotSupported;
    if ((long)v.n[0] * v.n[1] >= (1L << 31)) return cudaErrorNotSupported;
    for (int d = 0; d < 3; ++d)
        for (int sd = 0; sd < 2; ++sd) {
            const BCDev& b = v.bc[d][sd];
            const bool index_map = b.kind == BC_PERIODIC || b.kind == BC_SYMMETRY || (b.kind == BC_EXTRAP && b.P == 0) || (b.kind == BC_HALO && d == 2);
            if (!index_map) return cudaErrorNotSupported;
        }
    if (eik) return launch_pair_sb<T, PAIR_EIK>(P, A, s, exact_eps);
    if (P.nterms == 2) {
        // (NormalMotionTerm(stored speed), AdvectionTerm(stored velocity)) in this order, Float64
        if constexpr (sizeof(T) == 8) {
            const TermDev& tn = P.terms[0];
            if (tn.kind != TERM_NORMAL || tn.coef_kind != COEF_FIELD || tn.coef_f64 != 0 || A.first[0] != 0) return cudaErrorNotSupported;
            if (ta.coef_kind != COEF_FIELD || ta.coef_f64 != 0 || A.first[1] != 1) return cudaErrorNotSupported;
            return launch_pair_sb<T, COEF_FIELD, true>(P, A, s, exact_eps);
        }
        return cudaErrorNotSupported;
    }
    if (ta.coef_kind == COEF_FIELD && A.first[0] == 0 && !ta.coef_f64) return launch_pair_sb<T, COEF_FIELD>(P, A, s, exact_eps);
    if (ta.coef_kind == COEF_SEPARABLE) return launch_pair_sb<T, COEF_SEPARABLE>(P, A, s, exact_eps);
    return cudaErrorNotSupported;
}

// The Makefile compiles this file twice (-DLSM_PAIR_F32 / -DLSM_PAIR_F64) so that the two halves build in parallel.
#if !defined(LSM_PAIR_F64)
template cudaError_t launch_stage_pair3d<float>(const StageParams<float>&, const AuxList&, cudaStream_t, bool);
#endif
#if !defined(LSM_PAIR_F32)
template cudaError_t launch_stage_pair3d<double>(const StageParams<double>&, const AuxList&, cudaStream_t, bool);
#endif

}  // namespace lsm
