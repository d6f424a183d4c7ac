// lsm_simplex.cuh — the Freudenthal–Kuhn triangulation of the node lattice, shared by the zero-level-set extraction
// (lsm_interface.cu), the closest-point redistancing (lsm_redistance.cu) and the level-set integrals (lsm_integrals.cu): corner
// classification of a node's cell, the simplices of a cell, the primitives (points / segments / triangles) each simplex contributes,
// in the order include/lsm_b200.h states, and their vertex coordinates.
#pragma once
#include <cstddef>
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>
#include "lsm_kernels.h"

namespace lsm {
namespace {

// corner k of a cell is c + sum_d bit_d(k) e_d.  Chain of simplex p (lexicographic permutation order) and the sign of p.
__constant__ unsigned char c_chain3[6][4] = {{0, 1, 3, 7}, {0, 1, 5, 7}, {0, 2, 3, 7}, {0, 2, 6, 7}, {0, 4, 5, 7}, {0, 4, 6, 7}};
__constant__ signed char c_sign3[6] = {1, -1, -1, 1, 1, -1};
__constant__ unsigned char c_chain2[2][3] = {{0, 1, 3}, {0, 2, 3}};
__constant__ signed char c_sign2[2] = {1, -1};

template <int N> __device__ __forceinline__ int nsimplices() { return N == 3 ? 6 : N == 2 ? 2 : 1; }
template <int N> __device__ __forceinline__ int chain(int p, int k) {
    if (N == 3) return c_chain3[p][k];
    if (N == 2) return c_chain2[p][k];
    return k;
}
template <int N> __device__ __forceinline__ int psign(int p) { return N == 3 ? c_sign3[p] : N == 2 ? c_sign2[p] : 1; }
template <int N> __device__ __forceinline__ unsigned chain_mask(int p) {
    unsigned m = 0;
    for (int k = 0; k <= N; ++k) m |= 1u << chain<N>(p, k);
    return m;
}

__device__ __forceinline__ long long corner_off(const IfaceArgs& A, int k) {
    return (long long)(k & 1) + ((k >> 1) & 1) * A.s1 + ((k >> 2) & 1) * A.s2;
}

template <class T> __device__ __forceinline__ double sval(const IfaceArgs& A, long long j) {
    return double(static_cast<const T*>(A.phi)[j]) - A.level;
}

// corner classification of the cell of node idx: in-box, inside (s <= 0) and NaN bit masks over the 2^N corners
struct Masks { unsigned box, in, nan; };

template <class T, int N>
__device__ __forceinline__ Masks classify(const IfaceArgs& A, long long idx, const int* i) {
    unsigned up = 0;                      // axes along which the node has an upper neighbour in the box
    for (int d = 0; d < N; ++d) if (i[d] + 1 < A.m[d]) up |= 1u << d;
    Masks M{0, 0, 0};
    for (int k = 0; k < (1 << N); ++k) {
        if ((k & up) != k) continue;
        const double s = sval<T>(A, idx + corner_off(A, k));
        M.box |= 1u << k;
        if (s <= 0.0) M.in |= 1u << k;
        if (s != s) M.nan |= 1u << k;
    }
    return M;
}

// cut edges owned by the node: (a, a + e) for the in-box corners e != 0, both ends valid, one inside and one outside
template <int N> __device__ __forceinline__ unsigned cut_edges(const Masks& M) {
    if (M.nan & 1u) return 0;
    const unsigned valid = M.box & ~M.nan;
    return valid & ((M.in & 1u) ? ~M.in : M.in) & ~1u;
}

template <int N> __device__ __forceinline__ int prims_of_simplex(const Masks& M, int p) {
    const unsigned cm = chain_mask<N>(p);
    if (cm & M.nan) return 0;
    const int k = __popc(cm & M.in);
    if (k == 0 || k == N + 1) return 0;
    return (N == 3 && k == 2) ? 2 : 1;
}

template <int N> __device__ __forceinline__ int cell_prims(const Masks& M) {
    constexpr unsigned full = (1u << (1 << N)) - 1u;
    const unsigned valid = M.box & ~M.nan;
    if (M.box != full || !(valid & M.in) || !(valid & ~M.in)) return 0;
    int np = 0;
    for (int p = 0; p < nsimplices<N>(); ++p) np += prims_of_simplex<N>(M, p);
    return np;
}

// The primitives of simplex p of a cell (prims_of_simplex(M, p) > 0), in the contract's order.  emit(w, e) is called once per
// primitive: w[0..N] are the simplex's chain corners, e[j] = (x, y), x < y chain positions, is the simplex edge (w_x, w_y) whose
// crossing is vertex j of the primitive; the edge's lattice form is (c + w_x, c + w_x + (w_x ^ w_y)).
template <int N, class Emit>
__device__ __forceinline__ void simplex_prims(const Masks& M, int p, int hsign, Emit&& emit) {
    int w[N + 1], inside = 0;
    for (int k = 0; k <= N; ++k) { w[k] = chain<N>(p, k); inside |= ((M.in >> w[k]) & 1) << k; }
    auto E = [](int x, int y) { return x < y ? make_int2(x, y) : make_int2(y, x); };
    if constexpr (N == 1) {
        const int2 e[1] = {E(0, 1)};
        emit(w, e);
        return;
    }
    const int sgn = psign<N>(p) * hsign;
    const int k = __popc(inside);
    if (N == 2 || k != 2) {
        // lone vertex q (the only inside or the only outside one); r < s (< u) the others in chain order.  The
        // simplex (q, r, s[, u]) has orientation sgn (-1)^q: with a positive one, (qr, qs[, qu]) has q on its left
        // (2-D) / its normal pointing away from q (3-D); the normal must point outside and the inside must lie left.
        const int q = __ffs(k == 1 ? inside : (~inside & ((1 << (N + 1)) - 1))) - 1;
        int o[3], no = 0;
        for (int x = 0; x <= N; ++x) if (x != q) o[no++] = x;
        const int sigma = (q & 1) ? -sgn : sgn;
        const bool q_outside = k == N;
        const bool flip = (sigma < 0) != q_outside;
        if constexpr (N == 2) {
            const int2 e[2] = {flip ? E(q, o[1]) : E(q, o[0]), flip ? E(q, o[0]) : E(q, o[1])};
            emit(w, e);
        } else {
            const int2 e[3] = {E(q, o[0]), flip ? E(q, o[2]) : E(q, o[1]), flip ? E(q, o[1]) : E(q, o[2])};
            emit(w, e);
        }
    } else if constexpr (N == 3) {
        // 3-D, inside {a < b}, outside {c < d}: quad (ac, ad, bd, bc) split into (ac, ad, bd), (ac, bd, bc); with
        // (a, b, c, d) positively oriented that ordering has its normal pointing to c, d (outside)
        int ins[2], outs[2], ni = 0, nu = 0;
        for (int x = 0; x <= 3; ++x) { if ((inside >> x) & 1) ins[ni++] = x; else outs[nu++] = x; }
        const int seq[4] = {ins[0], ins[1], outs[0], outs[1]};
        int inv = 0;
        for (int x = 0; x < 4; ++x) for (int y = x + 1; y < 4; ++y) inv += seq[x] > seq[y];
        const int sigma = (inv & 1) ? -sgn : sgn;
        const int2 ac = E(ins[0], outs[0]), ad = E(ins[0], outs[1]), bd = E(ins[1], outs[1]), bc = E(ins[1], outs[0]);
        if (sigma > 0) { const int2 t0[3] = {ac, ad, bd}, t1[3] = {ac, bd, bc}; emit(w, t0); emit(w, t1); }
        else           { const int2 t0[3] = {ac, bd, ad}, t1[3] = {ac, bc, bd}; emit(w, t0); emit(w, t1); }
    }
}

// corner values of cell c (all corners in the box) and their classification
template <class T, int N>
__device__ __forceinline__ Masks cell_corners(const IfaceArgs& A, long long cidx, double* s) {
    Masks M{(1u << (1 << N)) - 1u, 0, 0};
    for (int k = 0; k < (1 << N); ++k) {
        s[k] = sval<T>(A, cidx + corner_off(A, k));
        if (s[k] <= 0.0) M.in |= 1u << k;
        if (s[k] != s[k]) M.nan |= 1u << k;
    }
    return M;
}

// vertices V[j][d] of the primitives of simplex p of cell c, as lsm_interface.cu computes them on the lattice edge (c + w_x, c + w_y),
// passed to f(V).  With a field F, given as F_at(k) = double(F) at corner k of the cell, f(V, Fv) also gets the vertex values
// Fv[j] = Fa + t (Fb - Fa), Fa = F_at(w_x), Fb = F_at(w_y), with the t of the coordinates.
template <int N, class Fn, class FAt = std::nullptr_t>
__device__ __forceinline__ void simplex_vertices(const IfaceArgs& A, const int* c, const double* s, const Masks& M, int p, Fn&& f,
                                                 FAt&& F_at = nullptr) {
    constexpr bool WITH_F = !std::is_same_v<std::decay_t<FAt>, std::nullptr_t>;
    simplex_prims<N>(M, p, A.hsign, [&](const int* w, const int2* e) {
        double V[N][3];
        [[maybe_unused]] double Fv[N];
        for (int j = 0; j < N; ++j) {
            const int a = w[e[j].x], b = w[e[j].y];
            const double t = s[a] / (s[a] - s[b]);
            for (int d = 0; d < N; ++d) {
                const double g = double(c[d] + ((a >> d) & 1));
                V[j][d] = (((a ^ b) >> d) & 1) ? A.lc[d] + (g + t) * A.h[d] : A.lc[d] + g * A.h[d];
            }
            if constexpr (WITH_F) {
                const double fa = F_at(a), fb = F_at(b);
                Fv[j] = fa + t * (fb - fa);
            }
        }
        if constexpr (WITH_F) f(V, Fv);
        else f(V);
    });
}

__device__ __forceinline__ void node_index(const IfaceArgs& A, long long idx, int* i) {
    i[0] = (int)(idx % A.m[0]);
    const long long q = idx / A.m[0];
    i[1] = (int)(q % A.m[1]);
    i[2] = (int)(q / A.m[1]);
}
__device__ __forceinline__ void next_index(const IfaceArgs& A, int* i) {
    if (++i[0] == A.m[0]) { i[0] = 0; if (++i[1] == A.m[1]) { i[1] = 0; ++i[2]; } }
}

}  // namespace
}  // namespace lsm
