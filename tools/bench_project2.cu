// Phase E inner-loop variants, stand-alone (points in shared memory): does a register tile of TWO views per thread
// (each point loaded once for both) beat one view per thread, with scalar FFMA and with packed FFMA2?
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -I odam_b200/csrc -o build/bp2 tools/bench_project2.cu
// Prints SM cycles per point-view per scheduler-warp-lane (lower is better; 18.5 = the FP32 roofline of the 37-flop count).
#include <cstdio>
#include <cuda_runtime.h>
#include "sq_device.cuh"
using namespace odam;

// scalar FFMA form of project_uv2<false>, one point per call
__device__ __forceinline__ void project_scalar(const float (&M)[12], float X, float Y, float Z, float &u, float &w)
{
    float qx = __fmaf_rn(X, M[0], __fmaf_rn(Y, M[1], __fmaf_rn(Z, M[2], M[3])));
    float qy = __fmaf_rn(X, M[4], __fmaf_rn(Y, M[5], __fmaf_rn(Z, M[6], M[7])));
    float qz = __fmaf_rn(X, M[8], __fmaf_rn(Y, M[9], __fmaf_rn(Z, M[10], M[11])));
    float r = rcp_approx(qz);
    u = __fmul_rn(qx, r);
    w = __fmul_rn(qy, r);
}

template <bool PACKED>
__device__ __forceinline__ void proj4(const float (&M)[12], const float4 x, const float4 y, const float4 z, float (&u)[4], float (&w)[4])
{
    if (PACKED) {
        project_uv2<false>(M, x.x, x.y, y.x, y.y, z.x, z.y, u[0], u[1], w[0], w[1]);
        project_uv2<false>(M, x.z, x.w, y.z, y.w, z.z, z.w, u[2], u[3], w[2], w[3]);
    } else {
        project_scalar(M, x.x, y.x, z.x, u[0], w[0]);
        project_scalar(M, x.y, y.y, z.y, u[1], w[1]);
        project_scalar(M, x.z, y.z, z.z, u[2], w[2]);
        project_scalar(M, x.w, y.w, z.w, u[3], w[3]);
    }
}

__device__ __forceinline__ void upd(float (&n)[4], const float (&u)[4], const float (&w)[4])
{
    n[0] = fmin3(n[0], u[0], u[1]); n[1] = fmax3(n[1], u[0], u[1]); n[2] = fmin3(n[2], w[0], w[1]); n[3] = fmax3(n[3], w[0], w[1]);
    n[0] = fmin3(n[0], u[2], u[3]); n[1] = fmax3(n[1], u[2], u[3]); n[2] = fmin3(n[2], w[2], w[3]); n[3] = fmax3(n[3], w[2], w[3]);
}

// the same with 2-input min/max (FMNMX: one issue cycle on the ALU pipe, partly overlapping the FMA pipe)
__device__ __forceinline__ void upd_2in(float (&n)[4], const float (&u)[4], const float (&w)[4])
{
#pragma unroll
    for (int h = 0; h < 4; h++) { n[0] = fminf(n[0], u[h]); n[1] = fmaxf(n[1], u[h]); n[2] = fminf(n[2], w[h]); n[3] = fmaxf(n[3], w[h]); }
}
// ... and with a pairwise pre-combine (min/max of two points first, then one 2-input update per pair and side)
__device__ __forceinline__ void upd_tree(float (&n)[4], const float (&u)[4], const float (&w)[4])
{
    n[0] = fminf(n[0], fminf(fminf(u[0], u[1]), fminf(u[2], u[3]))); n[1] = fmaxf(n[1], fmaxf(fmaxf(u[0], u[1]), fmaxf(u[2], u[3])));
    n[2] = fminf(n[2], fminf(fminf(w[0], w[1]), fminf(w[2], w[3]))); n[3] = fmaxf(n[3], fmaxf(fmaxf(w[0], w[1]), fmaxf(w[2], w[3])));
}

// VIEWS views per thread, GROUP points per straight-line block, 16-point chunks with chunk-id tracking as in the kernel
// MINMAX: 0 = 3-input FMNMX3, 1 = 2-input chain, 2 = 2-input tree
template <int VIEWS, bool PACKED, int GROUP, int MINB, int MINMAX = 0>
__global__ void __launch_bounds__(512, MINB) k(const float *Ms, float *out, int reps)
{
    __shared__ __align__(16) float px[1024], py[1024], pz[1024];
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) { px[i] = 0.3f * __sinf(i * 0.37f); py[i] = 0.3f * __cosf(i * 0.11f); pz[i] = 0.2f * __sinf(i * 0.73f); }
    __syncthreads();
    float M[VIEWS][12];
    for (int v = 0; v < VIEWS; v++)
        for (int k2 = 0; k2 < 12; k2++) M[v][k2] = Ms[((threadIdx.x * VIEWS + v) % 50) * 12 + k2];
    float best[VIEWS][4];
    int cid[VIEWS][4];
    for (int v = 0; v < VIEWS; v++) { best[v][0] = 1e6f; best[v][1] = -1e6f; best[v][2] = 1e6f; best[v][3] = -1e6f; cid[v][0] = cid[v][1] = cid[v][2] = cid[v][3] = -1; }
    for (int rep = 0; rep < reps; rep++) {
#pragma unroll 1
        for (int c = 0; c < 62; c++) {
            float n[VIEWS][4];
#pragma unroll
            for (int v = 0; v < VIEWS; v++) { n[v][0] = best[v][0]; n[v][1] = best[v][1]; n[v][2] = best[v][2]; n[v][3] = best[v][3]; }
#pragma unroll 1
            for (int g = 0; g < 16; g += GROUP) {
#pragma unroll
                for (int h = 0; h < GROUP / 4; h++) {
                    const float4 x = reinterpret_cast<const float4 *>(px + c * 16 + g)[h], y = reinterpret_cast<const float4 *>(py + c * 16 + g)[h],
                                 z = reinterpret_cast<const float4 *>(pz + c * 16 + g)[h];
#pragma unroll
                    for (int v = 0; v < VIEWS; v++) {
                        float u[4], w[4];
                        proj4<PACKED>(M[v], x, y, z, u, w);
                        if (MINMAX == 0) upd(n[v], u, w); else if (MINMAX == 1) upd_2in(n[v], u, w); else upd_tree(n[v], u, w);
                    }
                }
            }
#pragma unroll
            for (int v = 0; v < VIEWS; v++) {
                if (n[v][0] < best[v][0]) { best[v][0] = n[v][0]; cid[v][0] = c; }
                if (n[v][1] > best[v][1]) { best[v][1] = n[v][1]; cid[v][1] = c; }
                if (n[v][2] < best[v][2]) { best[v][2] = n[v][2]; cid[v][2] = c; }
                if (n[v][3] > best[v][3]) { best[v][3] = n[v][3]; cid[v][3] = c; }
            }
        }
        M[0][3] += 1e-3f;
    }
    float r = 0.f;
    for (int v = 0; v < VIEWS; v++) r += best[v][0] + best[v][1] + best[v][2] + best[v][3] + cid[v][0] + cid[v][1] + cid[v][2] + cid[v][3];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

template <int VIEWS, bool PACKED, int GROUP, int MINB, int MINMAX = 0>
static void run(const char *name, const float *dM, float *out, int threads, int blocks_per_sm)
{
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int reps = 20, blocks = 148 * blocks_per_sm;
    float ms = 0, best = 1e30f;
    for (int r = 0; r < 4; r++) {
        cudaEventRecord(e0);
        k<VIEWS, PACKED, GROUP, MINB, MINMAX><<<blocks, threads>>>(dM, out, reps);
        cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
        if (r && ms < best) best = ms;
    }
    const double pv = (double)blocks * threads * reps * 62 * 16 * VIEWS;
    cudaFuncAttributes fa; cudaFuncGetAttributes(&fa, k<VIEWS, PACKED, GROUP, MINB, MINMAX>);
    printf("%-44s T=%d x %d/SM regs=%3d  %.3f ms  %6.1f TFLOP/s(37)  %.2f cycles/point-view\n", name, threads, blocks_per_sm, fa.numRegs, best,
           pv * 37 / best / 1e9, best * 1e-3 * 1.965e9 * 148 * 4 / (pv / 32));
}

int main()
{
    float hM[50 * 12];
    for (int v = 0; v < 50; v++) { float m[12] = {1170, 0, 648, 100.f + v, 0, 1170, 484, 50, 0, 0, 1, 3.0f + 0.01f * v}; for (int k2 = 0; k2 < 12; k2++) hM[v * 12 + k2] = m[k2]; }
    float *dM, *out; cudaMalloc(&dM, sizeof hM); cudaMalloc(&out, 4 * 148 * 4 * 512); cudaMemcpy(dM, hM, sizeof hM, cudaMemcpyHostToDevice);
    for (int occ = 0; occ < 2; occ++) {
        const int threads = occ ? 512 : 256, bps = occ ? 1 : 4;   // dense: 4 x 256; latency regime: one 512-thread CTA per SM
        printf("--- %s\n", occ ? "one 512-thread CTA per SM (latency regime)" : "4 x 256 threads per SM (dense regime)");
        run<1, false, 16, 2>("1 view, scalar FFMA, 16-point blocks", dM, out, threads, bps);
        run<1, false, 4, 2>("1 view, scalar FFMA, 4-point blocks", dM, out, threads, bps);
        run<1, true, 16, 2>("1 view, FFMA2, 16-point blocks", dM, out, threads, bps);
        run<1, true, 16, 2, 1>("1 view, FFMA2, 16-pt, 2-input min/max chain", dM, out, threads, bps);
        run<1, true, 16, 2, 2>("1 view, FFMA2, 16-pt, 2-input min/max tree", dM, out, threads, bps);
        run<1, false, 16, 2, 1>("1 view, scalar, 16-pt, 2-input min/max chain", dM, out, threads, bps);
        run<1, false, 16, 2, 2>("1 view, scalar, 16-pt, 2-input min/max tree", dM, out, threads, bps);
        run<1, true, 8, 2>("1 view, FFMA2, 8-point blocks", dM, out, threads, bps);
        run<1, true, 4, 2>("1 view, FFMA2, 4-point blocks", dM, out, threads, bps);
        run<2, false, 4, 2>("2 views, scalar FFMA, 4-point blocks (64 regs)", dM, out, threads, bps);
        run<2, true, 4, 2>("2 views, FFMA2, 4-point blocks (64 regs)", dM, out, threads, bps);
        run<2, true, 8, 2>("2 views, FFMA2, 8-point blocks (64 regs)", dM, out, threads, bps);
        if (occ) {
            run<2, true, 8, 1>("2 views, FFMA2, 8-point blocks (128 regs)", dM, out, threads, bps);
            run<2, false, 8, 1>("2 views, scalar, 8-point blocks (128 regs)", dM, out, threads, bps);
            run<4, true, 4, 1>("4 views, FFMA2, 4-point blocks (128 regs)", dM, out, threads, bps);
        }
    }
    return 0;
}
