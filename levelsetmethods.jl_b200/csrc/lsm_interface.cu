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
#include "lsm_simplex.cuh"

namespace lsm {
namespace {

constexpr int TPB = 256, NPT = 4, TILE = TPB * NPT;

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
            simplex_prims<N>(M, p, A.hsign, [&](const int* w, const int2* e) {
                // vertex index of simplex edge (w_x, w_y): bisection over the keys of the tile that owns the edge's lower node
                for (int j = 0; j < N; ++j) {
                    const int a = w[e[j].x], b = w[e[j].y];
                    const long long na = idx + corner_off(A, a), ta = na / TILE;
                    prims[out * N + j] = find_key(keys, off_v[ta], off_v[ta + 1], (A.lin0 + na) * ncode + ((a ^ b) - 1));
                }
                ++out;
            });
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
