// Stand-alone throughput test of phase E's inner loop variants (points in shared memory, one view per thread).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -I odam_b200/csrc -o /tmp/bp tools/bench_project.cu
#include <cstdio>
#include <cuda_runtime.h>
#include "sq_device.cuh"
using namespace odam;

__device__ __forceinline__ void proj_valid(const float (&M)[12], float X, float Y, float Z, float &u, float &w)
{
    float qx = __fmaf_rn(X, M[0], __fmaf_rn(Y, M[1], __fmaf_rn(Z, M[2], M[3])));
    float qy = __fmaf_rn(X, M[4], __fmaf_rn(Y, M[5], __fmaf_rn(Z, M[6], M[7])));
    float qz = __fmaf_rn(X, M[8], __fmaf_rn(Y, M[9], __fmaf_rn(Z, M[10], M[11])));
    float r = rcp_approx(__fadd_rn(fabsf(qz), 1e-6f));
    r = qz > 0.5f ? r : __int_as_float(0x7fc00000);
    u = __fmul_rn(qx, r); w = __fmul_rn(qy, r);
}
__device__ __forceinline__ void proj_novalid(const float (&M)[12], float X, float Y, float Z, float &u, float &w)
{
    float qx = __fmaf_rn(X, M[0], __fmaf_rn(Y, M[1], __fmaf_rn(Z, M[2], M[3])));
    float qy = __fmaf_rn(X, M[4], __fmaf_rn(Y, M[5], __fmaf_rn(Z, M[6], M[7])));
    float qz = __fmaf_rn(X, M[8], __fmaf_rn(Y, M[9], __fmaf_rn(Z, M[10], M[11])));
    float r = rcp_approx(__fadd_rn(fabsf(qz), 1e-6f));
    u = __fmul_rn(qx, r); w = __fmul_rn(qy, r);
}
__device__ __forceinline__ void proj_folded(const float (&M)[12], float X, float Y, float Z, float &u, float &w)
{   // M[11] already holds m11 + 1e-6
    float qx = __fmaf_rn(X, M[0], __fmaf_rn(Y, M[1], __fmaf_rn(Z, M[2], M[3])));
    float qy = __fmaf_rn(X, M[4], __fmaf_rn(Y, M[5], __fmaf_rn(Z, M[6], M[7])));
    float qz = __fmaf_rn(X, M[8], __fmaf_rn(Y, M[9], __fmaf_rn(Z, M[10], M[11])));
    float r = rcp_approx(qz);
    u = __fmul_rn(qx, r); w = __fmul_rn(qy, r);
}
__device__ __forceinline__ void proj_folded_valid(const float (&M)[12], float X, float Y, float Z, float &u, float &w)
{
    float qx = __fmaf_rn(X, M[0], __fmaf_rn(Y, M[1], __fmaf_rn(Z, M[2], M[3])));
    float qy = __fmaf_rn(X, M[4], __fmaf_rn(Y, M[5], __fmaf_rn(Z, M[6], M[7])));
    float qz = __fmaf_rn(X, M[8], __fmaf_rn(Y, M[9], __fmaf_rn(Z, M[10], M[11])));
    float r = rcp_approx(qz);
    r = qz > 0.500001f ? r : __int_as_float(0x7fc00000);
    u = __fmul_rn(qx, r); w = __fmul_rn(qy, r);
}

template <int VAR>
__global__ void __launch_bounds__(512, 2) k(const float *Ms, float *out, int reps)
{
    __shared__ __align__(16) float px[1024], py[1024], pz[1024];
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) { px[i] = 0.3f * __sinf(i * 0.37f); py[i] = 0.3f * __cosf(i * 0.11f); pz[i] = 0.2f * __sinf(i * 0.73f); }
    __syncthreads();
    float M[12];
    for (int k2 = 0; k2 < 12; k2++) M[k2] = Ms[(threadIdx.x % 50) * 12 + k2];
    float best[4] = {1e6f, -1e6f, 1e6f, -1e6f};
    int cid[4] = {-1, -1, -1, -1};
    for (int rep = 0; rep < reps; rep++) {
        constexpr int CH = VAR == 4 ? 16 : 8;
        for (int c = 0; c < 1000 / CH; c++) {
            float u[CH], w[CH];
#pragma unroll
            for (int h = 0; h < CH / 4; h++) {
                float4 x = reinterpret_cast<const float4 *>(px + c * CH)[h], y = reinterpret_cast<const float4 *>(py + c * CH)[h],
                       z = reinterpret_cast<const float4 *>(pz + c * CH)[h];
#define P(a, i)                                                                     \
    if (VAR == 0) proj_valid(M, x.a, y.a, z.a, u[4 * h + i], w[4 * h + i]);          \
    else if (VAR == 1) proj_novalid(M, x.a, y.a, z.a, u[4 * h + i], w[4 * h + i]);   \
    else if (VAR == 5) proj_folded_valid(M, x.a, y.a, z.a, u[4 * h + i], w[4 * h + i]); \
    else proj_folded(M, x.a, y.a, z.a, u[4 * h + i], w[4 * h + i]);
                P(x, 0) P(y, 1) P(z, 2) P(w, 3)
            }
            float n0 = best[0], n1 = best[1], n2 = best[2], n3 = best[3];
            if (VAR == 3) {
#pragma unroll
                for (int h = 0; h < CH; h++) { n0 = fminf(n0, u[h]); n1 = fmaxf(n1, u[h]); n2 = fminf(n2, w[h]); n3 = fmaxf(n3, w[h]); }
            } else {
#pragma unroll
                for (int h = 0; h < CH; h += 2) { n0 = fmin3(n0, u[h], u[h + 1]); n1 = fmax3(n1, u[h], u[h + 1]); n2 = fmin3(n2, w[h], w[h + 1]); n3 = fmax3(n3, w[h], w[h + 1]); }
            }
            if (n0 < best[0]) { best[0] = n0; cid[0] = c; }
            if (n1 > best[1]) { best[1] = n1; cid[1] = c; }
            if (n2 < best[2]) { best[2] = n2; cid[2] = c; }
            if (n3 > best[3]) { best[3] = n3; cid[3] = c; }
        }
        M[3] += 1e-3f;
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = best[0] + best[1] + best[2] + best[3] + cid[0] + cid[1] + cid[2] + cid[3];
}

int main()
{
    float hM[50 * 12];
    for (int v = 0; v < 50; v++) { float m[12] = {1170, 0, 648, 100 + v, 0, 1170, 484, 50, 0, 0, 1, 3.0f + 0.01f * v}; for (int k2 = 0; k2 < 12; k2++) hM[v * 12 + k2] = m[k2]; }
    float *dM, *out; cudaMalloc(&dM, sizeof hM); cudaMalloc(&out, 4 * 148 * 4 * 512); cudaMemcpy(dM, hM, sizeof hM, cudaMemcpyHostToDevice);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    const char *names[] = {"V0 validity", "V1 no validity", "V2 no validity + folded eps", "V3 = V2 with 2-input min/max", "V4 = V2 with 16-point chunks", "V5 folded eps + validity"};
    for (int threads = 256; threads <= 512; threads *= 2)
    for (int var = 0; var < 6; var++) {
        int reps = 20, blocks = 148 * (1024 / threads);
        float ms = 0;
        for (int r = 0; r < 3; r++) {
            cudaEventRecord(e0);
            switch (var) { case 0: k<0><<<blocks, threads>>>(dM, out, reps); break; case 1: k<1><<<blocks, threads>>>(dM, out, reps); break;
                case 2: k<2><<<blocks, threads>>>(dM, out, reps); break; case 3: k<3><<<blocks, threads>>>(dM, out, reps); break;
                case 4: k<4><<<blocks, threads>>>(dM, out, reps); break; case 5: k<5><<<blocks, threads>>>(dM, out, reps); break; }
            cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
        }
        double pv = (double)blocks * threads * reps * 1000.0;
        printf("T=%d %-32s %.3f ms  %.2f Gpoint-view/s  = %.1f TFLOP/s (37 flop)  %.2f cycles/point-view/SMSP-warp\n", threads, names[var], ms, pv / ms / 1e6, pv * 37 / ms / 1e9,
               ms * 1e-3 * 1.965e9 * 148 * 4 / (pv / 32));
    }
    return 0;
}
