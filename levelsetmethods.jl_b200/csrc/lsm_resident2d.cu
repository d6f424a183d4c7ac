// lsm_resident2d.cu — small 2-D grids (the reference's own CPU-sized cases, e.g. 128 x 128): the WHOLE time loop in ONE kernel.
//
// A 128^2 RK3 step is three stage launches of a few microseconds each — launch latency and the fill / drain of every kernel
// dominate (10.9 us per step even when a CUDA graph replays the launches).  Here one thread-block CLUSTER of 16 CTAs keeps the
// state, the RK stage buffers and the velocity in its DISTRIBUTED SHARED MEMORY for the whole `integrate!` call:
//
//   * CTA q owns a strip of rows (split evenly, at least 3 per CTA); its shared memory holds three (rows + 6) x (n0 + 8) buffers
//     (state and two stage buffers, each with 3 halo rows and 3 ghost columns per side) and |u_d| / h_d of its nodes;
//   * every thread owns the same (at most NPT) nodes for the whole run, so everything that does not change — shared-memory
//     offset, upwind direction per axis (the velocity is static), which ghost columns and which halo rows of which CTA mirror the
//     node under the boundary conditions' index maps — is worked out once;
//   * a stage = evaluate the owned nodes with the arithmetic of the tiled 2-D kernel (lsm_tiled.cu: promoted Float64 WENO5, same
//     operation order -> bit-identical results), store the result into the own buffer AND PUSH it into the ghost columns / the
//     neighbouring CTAs' halo rows that mirror it with st.async (a DSMEM store that counts its bytes on the destination CTA's
//     mbarrier): a stage ends with __syncthreads + a wait for the 6 * n0 halo values of the own strip — point-to-point, no
//     cluster-wide barrier and no memory fence (a cluster barrier with release semantics costs MEMBAR.ALL.GPU + ~500 cycles:
//     20 % of the first version's time);
//   * the host knows every dt in advance (static velocity: dt = min(dt_max, cfl * dt_cfl, tf - tc), timestepping.jl:104-118), so
//     the kernel receives the run-length encoded dt sequence and touches global memory twice: at the start and at the end.
//
// Covered: one AdvectionTerm(u stored, WENO5) without a time factor, index-map boundary conditions, ForwardEuler / RK2 / RK3,
// Float64 and Float32, 8 <= n0, 48 <= n1, at most 2^15 nodes, a single rank.  Everything else takes the per-stage kernels.
#include "lsm_tile_util.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace lsm {

namespace {

constexpr int RES_CS = 16;        // CTAs of the cluster (non-portable size: one GPC)
constexpr int RES_NT = 512;       // threads per CTA
constexpr int RES_MAXD = 4;       // destinations of one row among the halo rows of the cluster (<= 4 when every strip has >= 3 rows)
constexpr long RES_MAX_NODES = 1L << 15;
constexpr size_t RES_MAX_SMEM = 200u << 10;

// even split of n1 rows over the cluster: the first n1 % CS strips hold one row more
__host__ __device__ inline int strip_begin(int q, int n1) { const int b = n1 / RES_CS, r = n1 % RES_CS; return q * b + (q < r ? q : r); }
__host__ __device__ inline int strip_rows(int q, int n1) { return n1 / RES_CS + (q < n1 % RES_CS ? 1 : 0); }
__device__ inline int strip_owner(int row, int n1) {
    const int b = n1 / RES_CS, r = n1 % RES_CS;
    return row < r * (b + 1) ? row / (b + 1) : r + (row - r * (b + 1)) / b;
}

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ unsigned mapa_u32(unsigned addr, int rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// remote store that signals the destination CTA's mbarrier (complete_tx) when the datum has landed
__device__ __forceinline__ void st_async(unsigned raddr, double v, unsigned rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                 ::"r"(raddr), "l"(__double_as_longlong(v)), "r"(rbar) : "memory");
}
__device__ __forceinline__ void st_async(unsigned raddr, float v, unsigned rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                 ::"r"(raddr), "r"(__float_as_uint(v)), "r"(rbar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Wait for a phase of the CTA's halo mbarrier.  The protocol cannot dead-lock (see the kernel), but a resident kernel that spins
// for ever would take the whole device with it, so the wait is bounded: after ~2 s (or as soon as another thread has given up)
// the status word is set, every later wait returns at once and the host reports the failure.
__device__ __noinline__ void mbar_wait_slow(unsigned bar, unsigned parity, unsigned long long* status, bool& dead) {
    const long long t0 = clock64();
    long long next = 1LL << 20;
    for (;;) {
        if (mbar_try_wait(bar, parity)) return;
        const long long el = clock64() - t0;
        if (el > next) {
            next = el + (1LL << 20);
            if (*reinterpret_cast<volatile unsigned long long*>(status) != 0ULL) { dead = true; return; }
            if (el > (1LL << 32)) { atomicMax(status, 2ULL); dead = true; return; }
        }
    }
}
__device__ __forceinline__ void mbar_wait_guarded(unsigned bar, unsigned parity, unsigned long long* status, bool& dead) {
    if (dead) return;
#pragma unroll 1
    for (int i = 0; i < 16; ++i) if (mbar_try_wait(bar, parity)) return;
    mbar_wait_slow(bar, parity, status, dead);
}

template <class T, int NPT, int NST>
__global__ void __launch_bounds__(RES_NT, 1) resident2d_kernel(const __grid_constant__ ResidentArgs<T> R) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int tid = threadIdx.x;
    const int n0 = R.n[0], n1 = R.n[1];
    const int W = n0 + 8;                                   // 4 columns left of x = 0 (3 ghosts + 1 pad keeps rows 16-byte aligned)
    const int RMAX = (n1 + RES_CS - 1) / RES_CS;            // rows of the largest strip: every CTA uses the same buffer layout
    const int r_beg = strip_begin(rank, n1), rows = strip_rows(rank, n1), nodes = rows * n0;
    const int BUF = (RMAX + 2 * HAL) * W;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long* const bar = reinterpret_cast<unsigned long long*>(smem_raw);      // [2] halo mbarriers (even / odd stages)
    double* const A0 = reinterpret_cast<double*>(smem_raw + 16);   // |u_x| / h_x of the owned nodes, [RMAX * n0]
    double* const A1 = A0 + RMAX * n0;                       // |u_y| / h_y
    T* const U = reinterpret_cast<T*>(A1 + RMAX * n0);       // [3][RMAX + 6][W]
    int* const hcnt = reinterpret_cast<int*>(U + 3 * BUF);   // [RMAX] halo-row destinations of each owned row
    int* const hdst = hcnt + RMAX;                           // [RMAX][RES_MAXD]: (CTA << 16) | buffer row
    const int bx0 = R.bc[0][0], bx1 = R.bc[0][1], by0 = R.bc[1][0], by1 = R.bc[1][1];

    // ---- which halo rows of the cluster mirror my rows (boundaryconditions.jl:107-153 as index maps, meshfield.jl:248-260)
    for (int r = tid; r < RMAX; r += RES_NT) hcnt[r] = 0;
    if (tid == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); }
    __syncthreads();
    if (tid < RES_CS * 2 * HAL) {
        const int q = tid / (2 * HAL), j = tid - q * (2 * HAL);
        const int rq = strip_rows(q, n1);
        const int rel = j < HAL ? j - HAL : rq + (j - HAL);
        int gr = remap_index(strip_begin(q, n1) + rel, n1, by0, by1);
        gr = min(max(gr, 0), n1 - 1);
        if (strip_owner(gr, n1) == rank) {
            const int lr = gr - r_beg;
            const int slot = atomicAdd(&hcnt[lr], 1);
            if (slot < RES_MAXD) hdst[lr * RES_MAXD + slot] = (q << 16) | (rel + HAL);
            else atomicMax(R.status, 1ULL);                  // cannot happen when every strip has >= 3 rows
        }
    }
    __syncthreads();

    // ---- per-thread node descriptors (the thread owns nodes tid, tid + NT, ... of the strip for the whole run)
    int nsc[NPT];            // shared-memory offset of the node inside a buffer
    unsigned ninf[NPT];      // bit 0 / 1: u_x / u_y negative; bits 2-7: ghost columns -3,-2,-1,n0,n0+1,n0+2 mirror this node; bits 8-10: halo destinations
    int nxr[NPT];            // x | row << 16
    const double ihx = 1.0 / R.h[0], ihy = 1.0 / R.h[1];
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
        const int e = tid + k * RES_NT;
        nsc[k] = 0; ninf[k] = 0; nxr[k] = 0;
        if (e < nodes) {
            const int row = e / n0, x = e - row * n0;
            const long g = (long)(r_beg + row) * R.s1 + x;
            const double u0 = double(R.u[0][g]), u1 = double(R.u[1][g]);
            A0[e] = fabs(u0) * ihx;                          // = |u| * (|g| / h) of lsm_tiled.cu with g = 1
            A1[e] = fabs(u1) * ihy;
            unsigned inf = ((unsigned)__double2hiint(u0) >> 31) | (((unsigned)__double2hiint(u1) >> 31) << 1);
#pragma unroll
            for (int j = 0; j < 2 * HAL; ++j) {
                const int gx = j < HAL ? j - HAL : n0 + (j - HAL);
                const int sx = min(max(remap_index(gx, n0, bx0, bx1), 0), n0 - 1);
                if (sx == x) inf |= 4u << j;
            }
            inf |= (unsigned)min(hcnt[row], RES_MAXD) << 8;
            nsc[k] = (row + HAL) * W + 4 + x; ninf[k] = inf; nxr[k] = x | (row << 16);
        }
    }

    // store a node value: own buffer, the ghost columns, and the halo rows (of any CTA) that mirror it — those with st.async,
    // which counts the bytes on the destination CTA's mbarrier `rb`
    const unsigned bar_u32 = smem_u32(bar);
    auto put = [&](T* buf, const int sc, const unsigned inf, const int xr, const T val, const unsigned rb) {
        buf[sc] = val;
        if (inf & 0x7FCu) {
            const int x = xr & 0xFFFF, row = xr >> 16;
            if (inf & 0xFCu) {
                T* const r0 = buf + sc - x;
#pragma unroll
                for (int j = 0; j < 2 * HAL; ++j)
                    if (inf & (4u << j)) r0[j < HAL ? j - HAL : n0 + (j - HAL)] = val;
            }
            const int nd = (inf >> 8) & 7;
            for (int j = 0; j < nd; ++j) {
                const int d = hdst[row * RES_MAXD + j];
                const unsigned la = smem_u32(buf) + (unsigned)(((d & 0xFFFF) * W + 4 + x) * (int)sizeof(T));
                st_async(mapa_u32(la, d >> 16), val, mapa_u32(rb, d >> 16));
            }
        }
    };
    // End of a stage: own stores visible to the CTA (__syncthreads), all 6 * n0 halo values of the buffer just written have
    // arrived from their owners (mbarrier of the stage's parity).  No cluster-wide barrier: a CTA can be at most one stage ahead
    // of the CTAs it exchanges rows with (it needs their rows of the previous stage), it pushes into a buffer they read two
    // stages ago at the latest — or, for RK2's corrector, into halo rows whose readers are exactly the threads whose pushes it
    // has waited for — and the even / odd mbarriers keep the byte counts of consecutive stages apart.
    const unsigned halo_bytes = (unsigned)(2 * HAL * n0 * (int)sizeof(T));
    unsigned gstage = 0;
    bool dead = false;
    auto stage_end = [&]() {
        const unsigned b = bar_u32 + 8u * (gstage & 1u);
        __syncthreads();
        if (tid == 0) mbar_expect_tx(bar + (gstage & 1u), halo_bytes);
        mbar_wait_guarded(b, (gstage >> 1) & 1u, R.status, dead);
        ++gstage;
    };

    cluster.sync();                                          // every CTA of the cluster is running and has initialised its mbarriers
#pragma unroll
    for (int k = 0; k < NPT; ++k)
        if (tid + k * RES_NT < nodes) {
            const int x = nxr[k] & 0xFFFF, row = nxr[k] >> 16;
            put(U, nsc[k], ninf[k], nxr[k], R.phi[(long)(r_beg + row) * R.s1 + x], bar_u32);
        }
    stage_end();

    const WenoK& K = R.wk;
    // stages per step: compile-time in the 2-nodes-per-thread kernels, so the buffer roles of a stage are too (NST = 0: runtime —
    // with 4 nodes per thread the unrolled stages would spill)
    const int nst = NST > 0 ? NST : R.nstages;
    int cur = 0;                                             // buffer holding the state
    for (int r = 0; r < R.nruns; ++r) {
        const double dt = R.dt[r];
        for (long step = 0; step < R.count[r]; ++step) {
            T* const a = U + cur * BUF;
            T* const b = U + (cur == 2 ? 0 : cur + 1) * BUF;
            T* const c = U + (cur == 0 ? 2 : cur - 1) * BUF;
#pragma unroll(NST > 0 ? NST : 1)
            for (int s = 0; s < nst; ++s) {
                // one RK stage: out = base(in, p0) - cc * H(in)   [out2 = in - c2 * H(in)]     (timestepping.jl:128-202)
                T *in, *out, *out2 = nullptr;
                const T* p0 = a;
                int base = BASE_IN;
                double cc = dt, c2 = 0.0;
                if (nst == 3) {
                    if (s == 0) { in = a; out = b; }
                    else if (s == 1) { in = b; out = c; base = BASE_RK3_S2; cc = 0.25 * dt; }
                    else { in = c; out = a; base = BASE_RK3_S3; cc = (2.0 / 3.0) * dt; }
                } else if (nst == 2) {
                    if (s == 0) { in = a; out = b; out2 = c; c2 = 0.5 * dt; }
                    else { in = b; out = a; p0 = c; base = BASE_P0; cc = 0.5 * dt; }
                } else { in = a; out = b; }
                const unsigned rbar = bar_u32 + 8u * (gstage & 1u);
#pragma unroll
                for (int k = 0; k < NPT; ++k) {
                    if (tid + k * RES_NT < nodes) {
                        const int sc = nsc[k];
                        const unsigned inf = ninf[k];
                        const T* const c0 = in + sc;
                        const T qc = c0[0];
                        // levelsetterms.jl:73-82 in the form of lsm_tiled.cu: H = sum_d (|u_d| / h_d) * W_d on upwind-ordered samples
                        const int s0 = (inf & 1u) ? -1 : 1, t1 = (inf & 2u) ? -W : W;
                        const double w0 = weno5_up_f64<T>(K, c0[-3 * s0], c0[-2 * s0], c0[-s0], qc, c0[s0], c0[2 * s0]);
                        const double w1 = weno5_up_f64<T>(K, c0[-3 * t1], c0[-2 * t1], c0[-t1], qc, c0[t1], c0[2 * t1]);
                        double H = A0[tid + k * RES_NT] * w0;
                        H = fma(A1[tid + k * RES_NT], w1, H);
                        T xb = qc;
                        if (base == BASE_RK3_S2) xb = T(fma(0.75, double(p0[sc]), 0.25 * double(qc)));     // timestepping.jl:183
                        else if (base == BASE_RK3_S3) xb = div3(T(p0[sc] + T(2) * qc));                      // timestepping.jl:194
                        else if (base == BASE_P0) xb = p0[sc];                                               // RK2 corrector
                        put(out, sc, inf, nxr[k], T(fma(-cc, H, double(xb))), rbar);
                        if (out2) out2[sc] = T(fma(-c2, H, double(qc)));
                    }
                }
                stage_end();
            }
            if (nst == 1) cur = cur == 2 ? 0 : cur + 1;      // ForwardEuler: the output buffer becomes the state
        }
    }

    cluster.sync();                                          // nobody exits while a neighbour may still address its shared memory
    const T* const fin = U + cur * BUF;
#pragma unroll
    for (int k = 0; k < NPT; ++k)
        if (tid + k * RES_NT < nodes) {
            const int x = nxr[k] & 0xFFFF, row = nxr[k] >> 16;
            R.out[(long)(r_beg + row) * R.s1 + x] = fin[nsc[k]];
        }
}

template <class T>
size_t resident_smem(int n0, int n1) {
    const size_t rmax = (size_t)(n1 + RES_CS - 1) / RES_CS;
    return 2 * rmax * n0 * sizeof(double) + 3 * (rmax + 2 * HAL) * (n0 + 8) * sizeof(T) + 16 + rmax * (1 + RES_MAXD) * sizeof(int);
}

}  // namespace

template <class T>
bool resident2d_supported(int n0, int n1) {
    // n1 >= 3 * CS: every strip holds at least the 3 rows its neighbours' halos need (and a row has at most RES_MAXD mirrors)
    // n0 >= 8 like the tiled kernels (tinier grids take the strict kernel, whose rounding differs)
    if (n0 < 8 || n0 > 0xFFFF || n1 < HAL * RES_CS || (long)n0 * n1 > RES_MAX_NODES) return false;
    const long per_cta = (long)((n1 + RES_CS - 1) / RES_CS) * n0;
    return per_cta <= 4L * RES_NT && resident_smem<T>(n0, n1) <= RES_MAX_SMEM;
}

namespace {
template <class T, int NPT, int NST>
cudaError_t launch_npt(const ResidentArgs<T>& R, cudaStream_t s) {
    const size_t smem = resident_smem<T>(R.n[0], R.n[1]);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    // per-device function attributes, set once (contexts of one process may launch from several threads: the calls are idempotent)
    static bool ready[64] = {};
    if (dev < 0 || dev >= 64) return cudaErrorNotSupported;
    if (!ready[dev]) {
        e = cudaFuncSetAttribute(resident2d_kernel<T, NPT, NST>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(resident2d_kernel<T, NPT, NST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RES_MAX_SMEM);
        if (e != cudaSuccess) { cudaGetLastError(); return cudaErrorNotSupported; }
        ready[dev] = true;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(RES_CS, 1, 1);
    cfg.blockDim = dim3(RES_NT, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = RES_CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int ncl = 0;
    e = cudaOccupancyMaxActiveClusters(&ncl, resident2d_kernel<T, NPT, NST>, &cfg);          // a 16-CTA cluster needs one GPC with 16 free SMs
    if (e != cudaSuccess || ncl < 1) { cudaGetLastError(); return cudaErrorNotSupported; }
    return cudaLaunchKernelEx(&cfg, resident2d_kernel<T, NPT, NST>, R);
}
}  // namespace

template <class T>
cudaError_t launch_resident2d(const ResidentArgs<T>& R, cudaStream_t s) {
    if (!resident2d_supported<T>(R.n[0], R.n[1])) return cudaErrorNotSupported;
    const long per_cta = (long)((R.n[1] + RES_CS - 1) / RES_CS) * R.n[0];
    const bool two = per_cta <= 2L * RES_NT;
    switch (R.nstages) {
        case 1: return two ? launch_npt<T, 2, 1>(R, s) : launch_npt<T, 4, 0>(R, s);
        case 2: return two ? launch_npt<T, 2, 2>(R, s) : launch_npt<T, 4, 0>(R, s);
        case 3: return two ? launch_npt<T, 2, 3>(R, s) : launch_npt<T, 4, 0>(R, s);
        default: return cudaErrorNotSupported;
    }
}

template bool resident2d_supported<double>(int, int);
template bool resident2d_supported<float>(int, int);
template cudaError_t launch_resident2d<double>(const ResidentArgs<double>&, cudaStream_t);
template cudaError_t launch_resident2d<float>(const ResidentArgs<float>&, cudaStream_t);

}  // namespace lsm
