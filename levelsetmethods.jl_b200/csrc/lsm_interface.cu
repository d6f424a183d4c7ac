// lsm_interface.cu — extraction of the zero level set {phi = level} as a piecewise-linear mesh (lsm_interface_extract).
//
// Marching simplices on the Freudenthal–Kuhn triangulation of the node lattice: cell c (its lower corner) is split into N!
// simplices, one per permutation pi of the axes in lexicographic order, with vertices w_0 = c, w_k = w_{k-1} + e_pi(k).  Every
// lattice edge (a, a + e), e in {0,1}^N \ {0}, that joins an inside node (s = phi - level <= 0) to an outside node (s > 0) is a
// mesh vertex; NaN nodes are neither, and a simplex with a NaN vertex emits nothing.  There are no case tables and no ambiguous
// cases, and the mesh is watertight by construction.  Vertex keys, orientation rules and output order are stated in
// include/lsm_b200.h; tests/interface_ref.py restates them in NumPy and the two agree bit for bit (this file is compiled with
// -fmad=false).
//
// Three passes over the node box, in tiles of 1024 nodes (4 consecutive nodes per thread):
//   count : classify the 2^N corners of every node's cell, count its cut edges and its primitives, one pair of totals per tile;
//   scan  : exclusive scan of the tile totals (one block), and the two grand totals for the host;
//   emit  : vertices in key order (emit_vertices), then primitives in cell order (emit_prims), each tile at its scanned offset.
// A primitive refers to edges owned by neighbouring nodes, possibly in later tiles: emit_prims finds their vertex indices by
// bisection on the keys emit_vertices wrote, within the key range of the tile that owns the edge's lower node.  The only scratch
// is 24 bytes per tile; output order depends on the data alone.
#include <cstdint>
#include <cuda_runtime.h>
#include "lsm_kernels.h"

namespace lsm {
namespace {

constexpr int TPB = 256, NPT = 4, TILE = TPB * NPT;

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

__device__ __forceinline__ void node_index(const IfaceArgs& A, long long idx, int* i) {
    i[0] = (int)(idx % A.m[0]);
    const long long q = idx / A.m[0];
    i[1] = (int)(q % A.m[1]);
    i[2] = (int)(q / A.m[1]);
}
__device__ __forceinline__ void next_index(const IfaceArgs& A, int* i) {
    if (++i[0] == A.m[0]) { i[0] = 0; if (++i[1] == A.m[1]) { i[1] = 0; ++i[2]; } }
}

// block-wide exclusive scan of (a, b) pairs over TPB threads; also returns the block totals
template <int BS, class V>
__device__ __forceinline__ void block_scan2(V a, V b, V* ea, V* eb, V* ta, V* tb) {
    __shared__ V sa[BS / 32], sb[BS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    V ia = a, ib = b;
    for (int o = 1; o < 32; o <<= 1) {
        const V xa = __shfl_up_sync(0xffffffffu, ia, o), xb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += xa; ib += xb; }
    }
    if (lane == 31) { sa[w] = ia; sb[w] = ib; }
    __syncthreads();
    V pa = 0, pb = 0, qa = 0, qb = 0;
    for (int k = 0; k < BS / 32; ++k) {
        if (k < w) { pa += sa[k]; pb += sb[k]; }
        qa += sa[k]; qb += sb[k];
    }
    *ea = pa + ia - a; *eb = pb + ib - b; *ta = qa; *tb = qb;
    __syncthreads();
}

template <class T, int N>
__global__ void __launch_bounds__(TPB) iface_count_kernel(const __grid_constant__ IfaceArgs A, int2* __restrict__ tile_cnt) {
    const long long first = (long long)blockIdx.x * TILE + (long long)threadIdx.x * NPT;
    int nv = 0, np = 0;
    if (first < A.nodes) {
        int i[3];
        node_index(A, first, i);
        for (int j = 0; j < NPT && first + j < A.nodes; ++j, next_index(A, i)) {
            const Masks M = classify<T, N>(A, first + j, i);
            nv += __popc(cut_edges<N>(M));
            np += cell_prims<N>(M);
        }
    }
    int ev, ep, tv, tp;
    block_scan2<TPB, int>(nv, np, &ev, &ep, &tv, &tp);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = make_int2(tv, tp);
}

// one block: off_v / off_p[t] = totals of the tiles before t, [ntiles] = grand totals, also written to tot[0..1]
constexpr int SCAN_TPB = 1024;
__global__ void __launch_bounds__(SCAN_TPB) iface_scan_kernel(const int2* __restrict__ tile_cnt, long long ntiles, long long* __restrict__ off_v,
                                                         long long* __restrict__ off_p, long long* __restrict__ tot) {
    const long long chunk = (ntiles + SCAN_TPB - 1) / SCAN_TPB;
    const long long b = threadIdx.x * chunk, e = b + chunk < ntiles ? b + chunk : ntiles;
    long long sv = 0, sp = 0;
    for (long long t = b; t < e; ++t) { const int2 c = tile_cnt[t]; sv += c.x; sp += c.y; }
    long long ev, ep, tv, tp;
    block_scan2<SCAN_TPB, long long>(sv, sp, &ev, &ep, &tv, &tp);
    for (long long t = b; t < e; ++t) { const int2 c = tile_cnt[t]; off_v[t] = ev; off_p[t] = ep; ev += c.x; ep += c.y; }
    if (threadIdx.x == 0) { off_v[ntiles] = tv; off_p[ntiles] = tp; tot[0] = tv; tot[1] = tp; }
}

template <class T, int N>
__global__ void __launch_bounds__(TPB) iface_vertices_kernel(const __grid_constant__ IfaceArgs A, const long long* __restrict__ off_v,
                                                             double* __restrict__ verts, long long* __restrict__ keys) {
    const long long first = (long long)blockIdx.x * TILE + (long long)threadIdx.x * NPT;
    unsigned cut[NPT] = {};
    int nv = 0;
    int i0[3] = {0, 0, 0};
    if (first < A.nodes) {
        node_index(A, first, i0);
        int i[3] = {i0[0], i0[1], i0[2]};
        for (int j = 0; j < NPT && first + j < A.nodes; ++j, next_index(A, i)) {
            cut[j] = cut_edges<N>(classify<T, N>(A, first + j, i));
            nv += __popc(cut[j]);
        }
    }
    int ev, ep, tv, tp;
    block_scan2<TPB, int>(nv, 0, &ev, &ep, &tv, &tp);
    if (!nv) return;
    long long out = off_v[blockIdx.x] + ev;
    constexpr long long ncode = (1 << N) - 1;
    int i[3] = {i0[0], i0[1], i0[2]};
    for (int j = 0; j < NPT; ++j, next_index(A, i)) {
        if (!cut[j]) continue;
        const long long idx = first + j;
        const double sa = sval<T>(A, idx);
        int g[3] = {i[0], i[1], i[2]};
        g[N - 1] += A.first_last;
        for (int e = 1; e <= (int)ncode; ++e) {
            if (!((cut[j] >> e) & 1u)) continue;
            const double sb = sval<T>(A, idx + corner_off(A, e));
            const double t = sa / (sa - sb);
            for (int d = 0; d < N; ++d)
                verts[out * N + d] = ((e >> d) & 1) ? A.lc[d] + (double(g[d]) + t) * A.h[d] : A.lc[d] + double(g[d]) * A.h[d];
            keys[out] = (A.lin0 + idx) * ncode + (e - 1);
            ++out;
        }
    }
}

// index of `key` in keys[lo, hi) (it is there: every cut edge of every cell is a vertex)
__device__ __forceinline__ int find_key(const long long* __restrict__ keys, long long lo, long long hi, long long key) {
    while (lo < hi) {
        const long long mid = lo + ((hi - lo) >> 1);
        if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    return (int)lo;
}

template <class T, int N>
__global__ void __launch_bounds__(TPB) iface_prims_kernel(const __grid_constant__ IfaceArgs A, const long long* __restrict__ off_v,
                                                          const long long* __restrict__ off_p, const long long* __restrict__ keys,
                                                          int* __restrict__ prims) {
    const long long first = (long long)blockIdx.x * TILE + (long long)threadIdx.x * NPT;
    Masks Ms[NPT];
    int cnt[NPT] = {};
    int np = 0;
    if (first < A.nodes) {
        int i[3];
        node_index(A, first, i);
        for (int j = 0; j < NPT; ++j, next_index(A, i)) {
            if (first + j >= A.nodes) { Ms[j] = Masks{0, 0, 0}; continue; }
            Ms[j] = classify<T, N>(A, first + j, i);
            cnt[j] = cell_prims<N>(Ms[j]);
            np += cnt[j];
        }
    }
    int ev, ep, tv, tp;
    block_scan2<TPB, int>(0, np, &ev, &ep, &tv, &tp);
    if (!np) return;
    long long out = off_p[blockIdx.x] + ep;
    constexpr long long ncode = (1 << N) - 1;
    for (int j = 0; j < NPT; ++j) {
        if (!cnt[j]) continue;
        const long long idx = first + j;
        const Masks& M = Ms[j];
        for (int p = 0; p < nsimplices<N>(); ++p) {
            if (!prims_of_simplex<N>(M, p)) continue;
            int w[N + 1], inside = 0;
            for (int k = 0; k <= N; ++k) { w[k] = chain<N>(p, k); inside |= ((M.in >> w[k]) & 1) << k; }
            // vertex index of simplex edge (w_x, w_y): bisection over the keys of the tile that owns the edge's lower node
            auto vid = [&](int x, int y) {
                const int a = x < y ? w[x] : w[y], b = x < y ? w[y] : w[x];
                const long long na = idx + corner_off(A, a), ta = na / TILE;
                return find_key(keys, off_v[ta], off_v[ta + 1], (A.lin0 + na) * ncode + ((a ^ b) - 1));
            };
            const int sgn = psign<N>(p) * A.hsign;
            if constexpr (N == 1) {
                prims[out++] = vid(0, 1);
                continue;
            }
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
                    const int v0 = vid(q, o[0]), v1 = vid(q, o[1]);
                    prims[out * 2] = flip ? v1 : v0; prims[out * 2 + 1] = flip ? v0 : v1;
                } else {
                    const int v0 = vid(q, o[0]), v1 = vid(q, o[1]), v2 = vid(q, o[2]);
                    prims[out * 3] = v0; prims[out * 3 + 1] = flip ? v2 : v1; prims[out * 3 + 2] = flip ? v1 : v2;
                }
                ++out;
            } else if constexpr (N == 3) {
                // 3-D, inside {a < b}, outside {c < d}: quad (ac, ad, bd, bc) split into (ac, ad, bd), (ac, bd, bc); with
                // (a, b, c, d) positively oriented that ordering has its normal pointing to c, d (outside)
                int ins[2], outs[2], ni = 0, nu = 0;
                for (int x = 0; x <= 3; ++x) { if ((inside >> x) & 1) ins[ni++] = x; else outs[nu++] = x; }
                const int seq[4] = {ins[0], ins[1], outs[0], outs[1]};
                int inv = 0;
                for (int x = 0; x < 4; ++x) for (int y = x + 1; y < 4; ++y) inv += seq[x] > seq[y];
                const int sigma = (inv & 1) ? -sgn : sgn;
                const int ac = vid(ins[0], outs[0]), ad = vid(ins[0], outs[1]), bd = vid(ins[1], outs[1]), bc = vid(ins[1], outs[0]);
                int* P = prims + out * 3;
                if (sigma > 0) { P[0] = ac; P[1] = ad; P[2] = bd; P[3] = ac; P[4] = bd; P[5] = bc; }
                else           { P[0] = ac; P[1] = bd; P[2] = ad; P[3] = ac; P[4] = bc; P[5] = bd; }
                out += 2;
            }
        }
    }
}

template <class T, int N>
cudaError_t launch_n(const IfaceArgs& A, int pass, void* scratch, double* verts, long long* keys, int* prims, cudaStream_t s) {
    const unsigned grid = (unsigned)A.ntiles;
    int2* cnt = static_cast<int2*>(scratch);
    long long* off_v = reinterpret_cast<long long*>(cnt + A.ntiles + (A.ntiles & 1));   // 16-byte aligned
    long long* off_p = off_v + A.ntiles + 1;
    long long* tot = off_p + A.ntiles + 1;
    if (pass == 0) {
        iface_count_kernel<T, N><<<grid, TPB, 0, s>>>(A, cnt);
        iface_scan_kernel<<<1, SCAN_TPB, 0, s>>>(cnt, A.ntiles, off_v, off_p, tot);
    } else if (pass == 1) {
        iface_vertices_kernel<T, N><<<grid, TPB, 0, s>>>(A, off_v, verts, keys);
    } else {
        iface_prims_kernel<T, N><<<grid, TPB, 0, s>>>(A, off_v, off_p, keys, prims);
    }
    return cudaGetLastError();
}

template <class T>
cudaError_t launch_t(const IfaceArgs& A, int pass, void* scratch, double* verts, long long* keys, int* prims, cudaStream_t s) {
    switch (A.ndim) {
        case 1: return launch_n<T, 1>(A, pass, scratch, verts, keys, prims, s);
        case 2: return launch_n<T, 2>(A, pass, scratch, verts, keys, prims, s);
        default: return launch_n<T, 3>(A, pass, scratch, verts, keys, prims, s);
    }
}

}  // namespace

long long iface_tiles(long long nodes) { return (nodes + TILE - 1) / TILE; }

size_t iface_scratch_bytes(long long ntiles) {
    return sizeof(int2) * (size_t)(ntiles + (ntiles & 1)) + sizeof(long long) * (size_t)(2 * (ntiles + 1) + 2);
}

long long* iface_totals(const IfaceArgs& A, void* scratch) {
    int2* cnt = static_cast<int2*>(scratch);
    return reinterpret_cast<long long*>(cnt + A.ntiles + (A.ntiles & 1)) + 2 * (A.ntiles + 1);
}

cudaError_t launch_iface(const IfaceArgs& A, int pass, void* scratch, double* verts, long long* keys, int* prims, cudaStream_t s) {
    return A.f64 ? launch_t<double>(A, pass, scratch, verts, keys, prims, s) : launch_t<float>(A, pass, scratch, verts, keys, prims, s);
}

}  // namespace lsm
