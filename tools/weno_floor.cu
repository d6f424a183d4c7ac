// weno_floor.cu — the FP64 floor of the headline stage kernel, measured (VERDICT r01 item 1: "prove it with a register-only
// microkernel that executes just the minimal DP arithmetic and report its time as the kernel's floor").
//
// Every thread owns a pair of adjacent x nodes like pair3d_kernel and executes, per node-pair-stage, exactly the arithmetic of the
// production kernel's C3 instantiation — three pair_eval<double, XMAX> calls from csrc/lsm_pair_common.cuh (x with the shared
// differences of the pair, y, z), the isotropic-mesh fold sum_d u_d W_d and the RK update — on operands that LIVE IN REGISTERS:
// no shared or global loads, no TMA, no barriers, no upwind-direction logic (the minus-biased branch is selected at compile time),
// no address arithmetic.  The 7-point windows are 8-entry register rings rotated by unrolling the loop 8 times (no MOVs); the value
// entering a window is the previous result of the pair, so nothing can be hoisted out of the loop.
// The five windows of a pair are 40 doubles, so a thread needs ~170 registers: ONE CTA of 256 threads per SM (production: two, with the
// windows in shared memory); the 6 independent WENO evaluations of a pair give each of the 2 warps per scheduler ample ILP.
// 148 SMs; 1776 pair-stages per thread = one 512^3 stage launch.
// Per node-stage in SASS (sm_100a, CUDA 12.9): 125.8 FP64 + 43.2 other instructions with the 20-bit eps maximum and the completed-square
// smoothness indicators (139.4 + 43.1 with the 13/3 form before it), 118.8 + 35.2 with z reuse, 151.4 + 61.6 with the exact maximum.
//
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I levelsetmethods.jl_b200/csrc -I include tools/weno_floor.cu -o tools/weno_floor
#include <cstdio>
#include <cuda_runtime.h>
#include "lsm_pair_common.cuh"

using namespace lsm;

__device__ __forceinline__ double flip(double x, int bits) { return __hiloint2double(__double2hiint(x), __double2loint(x) ^ bits); }

template <bool XMAX, bool ZREUSE>
__global__ void __launch_bounds__(256, 1) floor_kernel(double* out, const WenoK K0, const double c, const int blocks8) {
    const WenoK K = weno_regs<XMAX>(K0);     // the constants held in registers like the production kernel does
    const double t = 1e-3 * (threadIdx.x % 13) + 1e-4 * (blockIdx.x % 7);
    double X[8], YA[8], YB[8], ZA[8], ZB[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        X[j] = 0.01 * j + t * (j & 1);
        YA[j] = 0.011 * j + t; YB[j] = 0.012 * j - t;
        ZA[j] = 0.009 * j + 2 * t; ZB[j] = 0.008 * j - 2 * t;
    }
    const double ua0 = 0.31 + t, ub0 = 0.32 + t, ua1 = 0.21 + t, ub1 = 0.22 + t, ua2 = 0.11 + t, ub2 = 0.12 + t;
    for (int blk = 0; blk < blocks8; ++blk) {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            // logical window element j lives in ring slot (it + j) & 7
            const double ax[7] = {X[(it + 0) & 7], X[(it + 1) & 7], X[(it + 2) & 7], X[(it + 3) & 7], X[(it + 4) & 7], X[(it + 5) & 7], X[(it + 6) & 7]};
            const double bx[7] = {X[(it + 1) & 7], X[(it + 2) & 7], X[(it + 3) & 7], X[(it + 4) & 7], X[(it + 5) & 7], X[(it + 6) & 7], X[(it + 7) & 7]};
            const double ay[7] = {YA[(it + 0) & 7], YA[(it + 1) & 7], YA[(it + 2) & 7], YA[(it + 3) & 7], YA[(it + 4) & 7], YA[(it + 5) & 7], YA[(it + 6) & 7]};
            const double by[7] = {YB[(it + 0) & 7], YB[(it + 1) & 7], YB[(it + 2) & 7], YB[(it + 3) & 7], YB[(it + 4) & 7], YB[(it + 5) & 7], YB[(it + 6) & 7]};
            const double az[7] = {ZA[(it + 0) & 7], ZA[(it + 1) & 7], ZA[(it + 2) & 7], ZA[(it + 3) & 7], ZA[(it + 4) & 7], ZA[(it + 5) & 7], ZA[(it + 6) & 7]};
            const double bz[7] = {ZB[(it + 0) & 7], ZB[(it + 1) & 7], ZB[(it + 2) & 7], ZB[(it + 3) & 7], ZB[(it + 4) & 7], ZB[(it + 5) & 7], ZB[(it + 6) & 7]};
            double wa, wb;
            pair_eval<double, XMAX>(K, ax, bx, 0, 0, wa, wb);
            double Ha = ua0 * wa, Hb = ub0 * wb;
            pair_eval<double, XMAX>(K, ay, by, 0, 0, wa, wb);
            Ha = fma(ua1, wa, Ha); Hb = fma(ub1, wb, Hb);
            pair_eval<double, XMAX>(K, az, bz, 0, 0, wa, wb);
            Ha = fma(ua2, wa, Ha); Hb = fma(ub2, wb, Hb);
            const double oa = fma(-c, Ha, ax[3]), ob = fma(-c, Hb, bx[3]);      // BASE_IN: x = phi - c * H
            // Next plane.  x and y windows hold entirely NEW samples in every plane of the real march: all their entries are refreshed
            // (low mantissa bits flipped by bits of the new results — one LOP3 each, standing in for the kernel's LDS; data-dependent,
            // so that nothing folds across iterations).  The z window of a node SHIFTS by one plane: with ZREUSE the compiler keeps
            // the differences of the previous plane (what a perfect z-register-blocked kernel could do), without it the z window is
            // refreshed like the others (what pair3d_kernel does: every plane recomputes its z differences).
            const int ka = __double2loint(oa), kb = __double2loint(ob);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                X[j] = flip(X[j], ka & 1);
                YA[j] = flip(YA[j], kb & 2); YB[j] = flip(YB[j], ka & 4);
                if (!ZREUSE) { ZA[j] = flip(ZA[j], kb & 8); ZB[j] = flip(ZB[j], ka & 16); }
            }
            X[it & 7] = oa;
            YA[(it + 7) & 7] = ob; YB[(it + 7) & 7] = flip(oa, 1);
            ZA[(it + 7) & 7] = flip(ob, 2); ZB[(it + 7) & 7] = flip(oa, 4);
        }
    }
    double s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += X[j] + YA[j] + YB[j] + ZA[j] + ZB[j];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <bool XMAX, bool ZREUSE>
void run(const char* name, double* d) {
    const int grid = 148, block = 256;
    const long pairs = 512L * 512 * 512 / 2;
    const int blocks8 = (int)((pairs + (long)grid * block * 8 - 1) / ((long)grid * block * 8));     // 222 -> 1776 pair-stages per thread
    const double done = (double)grid * block * 8.0 * blocks8 * 2.0;                                   // node-stages executed
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    floor_kernel<XMAX, ZREUSE><<<grid, block>>>(d, weno_constants(), 1e-3, 4);
    float best = 1e30f, sum = 0;
    const int reps = 20;
    for (int r = 0; r < reps; ++r) {
        cudaEventRecord(e0); floor_kernel<XMAX, ZREUSE><<<grid, block>>>(d, weno_constants(), 1e-3, blocks8); cudaEventRecord(e1); cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1); if (ms < best) best = ms; sum += ms;
    }
    const double scale = 134217728.0 / done;       // to exactly 512^3 node-stages
    printf("%-34s best %.4f ms  mean %.4f ms per 512^3 node-stages (one stage launch); %.1f G node-stages/s\n", name, best * scale, sum / reps * scale,
           done / (sum / reps) * 1e-6);
}

int main() {
    double* d; cudaMalloc(&d, 148 * 256 * sizeof(double));
    run<false, false>("20-bit eps max (pair3d default)", d);
    run<false, true>("20-bit eps max, z differences reused", d);
    run<true, false>("exact eps max (LSM_OPT_KERNEL=4)", d);
    cudaError_t e = cudaDeviceSynchronize();
    printf("status: %s\n", cudaGetErrorString(e));
    return e != cudaSuccess;
}
