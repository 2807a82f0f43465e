// sq_kernels.cu -- fused multi-view superquadric optimiser for B200 (sm_100a) + its C ABI (include/odam_sq.h).
//
// One CTA per object, one persistent launch for all iterations.  Per iteration, entirely on chip:
//   A  derived quantities (a = s^2, e = 0.2 + 1.4 sigmoid(h), rotation)                  [sq_libs.py:577-584]
//   B  two 201-entry equal-arc-length grids, one warp each, level-synchronous            [sampling.cpp:76-125]
//   C  sequential fp32 CDF + normalisation (warp 0, overlapping the omega grid of warp 1) [sampling.cpp:137-148]
//   D  per sample: CDF bisection -> (eta, omega) grid indices -> surface point -> world   [sampling.cpp:151-154,210-212;
//      point, kept in shared memory (SoA, 12 KB)                                           sampling.py:591-615]
//   E  per (view, point slice): project all points, track the 4 extrema with 3-input      [sq_libs.py:395-413]
//      min/max, resolve the arg-extreme index by rescanning one 8-point chunk
//   F  per (view, side): L1 term and analytic gradient through the arg-extreme point      [sq_libs.py:420-430 + autograd]
//   G  deterministic CTA reduction of 9 gradients + 4 side sums, prior, Adam              [sq_libs.py:463-472]
//
// No tensor cores: the path is FP32 FMA + min/max + one MUFU.RCP per point-view.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "../../include/odam_sq.h"

#ifndef SQ_FFMA2
#define SQ_FFMA2 1   // phase E on packed fp32 pairs (FFMA2/FMUL2); 0 = scalar FFMA build for A/B timing
#endif
#include "sq_device.cuh"
#include "sq_postproc.cuh"
#include "sq_stage.h"

namespace cg = cooperative_groups;

namespace odam {

constexpr int kMaxCluster = 4;   // CTAs per object (view-tiled thread-block cluster)
constexpr int kRed = 13;  // 9 gradients + 4 side sums

struct alignas(16) Smem {
    float px[kNPad], py[kNPad], pz[kNPad];  // world points, SoA
    GridTab ge, go;
    alignas(16) float cdf[kGPad];
    uint8_t pj[kNPad];                      // eta-grid index of each sample
    float xred[2][kMaxCluster][kRed + 3];   // per-CTA partial sums exchanged through DSMEM, double-buffered by iteration parity
    alignas(8) uint64_t xbar[2];            // one mbarrier per buffer: completes when all C*13 floats have landed
    alignas(8) uint64_t tma_bar;            // completion of the one-off TMA staging of this CTA's views
    float par[12], m[12], v[12], s0[4], grad[12], prior[12];
    Pose pose;
    int status;
    int bad[2];
    float adam_now[4];                       // this iteration's row of the Adam table (fetched early)
    long long tmark, cyc[16];                // per-phase clock64() accumulation by thread 0 (diagnostics)
};

// only when the caller asked for the per-phase cycle counts (`prof` in scope): the clock read and the shared-memory
// round trip sit on thread 0's critical path otherwise
#define SQ_MARK(S, tid, k)                                                \
    do {                                                                   \
        if (prof && (tid) == 0) {                                          \
            long long now_ = clock64();                                    \
            (S).cyc[k] += now_ - (S).tmark;                                \
            (S).tmark = now_;                                              \
        }                                                                  \
    } while (0)

constexpr size_t kSpecBytes = 2 * sizeof(GridSpec);
constexpr size_t kFwdSmem = kSpecBytes;  // forward-only kernels: dynamic part = B0 scratch (Smem itself is static)

struct OptArgs {
    const float *init; const int32_t *cls; const int32_t *view_off;
    const float *Ms; const float *box; const uint8_t *mask; const float *prior;
    int n, n_iters, optimize_shapes, max_slices, cluster, red_offset;
    int stage_offset, stage_views;   // >0: this many views per CTA fit the staging area at scratch + stage_offset
    const float *adam_tab;  // [n_iters][4]: -lr/bc1, -lr_shape/bc1, sqrt(bc2), unused
    float beta1w, beta2, beta2w, eps;
    const float *m0, *v0, *s0;
    float *out_params, *out_loss; int32_t *out_status;
    float *out_m, *out_v, *out_grad, *out_pred; int32_t *out_arg; uint8_t *out_eta_idx; float *out_grids;
    float *out_param_hist;
    long long *out_cycles;
};

// phase A: what the sampler and the surface need of parameter `k` (one lane per parameter), plus the per-iteration
// resets of the sampler state (lane 9).  Runs once before the first iteration and then fused with the Adam update.
__device__ __forceinline__ void derive_param(Smem &S, int k)
{
    Pose &P = S.pose;
    const float p = S.par[k];
    if (k < 3) P.t[k] = p;
    else if (k == 3) {
        double sd, cd;
        sq_sincos_pi(p, sd, cd);  // yaw: correctly rounded cos/sin for |angle| < ~1e5 rad
        P.cz = (float)cd; P.sz = (float)sd;
    } else if (k < 7) P.a[k - 4] = __fmul_rn(p, p);
    else if (k < 9) {
        // torch.sigmoid, correctly rounded: t = exp(-|p|) in (0, 1], sigma = 1/(1+t) or t/(1+t)
        const double t = p > -700.f && p < 700.f ? sq_exp_neg(-fabs((double)p)) : 0.0;
        float sg = (float)((p >= 0.f ? 1.0 : t) / (1.0 + t));
        P.sig[k - 7] = sg;
        P.e[k - 7] = __fadd_rn(__fmul_rn(sg, 1.4f), 0.2f);
    } else if (k == 9) {
        S.bad[0] = 0; S.bad[1] = 0;
        S.ge.fix_lo = S.ge.count; S.go.fix_lo = S.go.count;
        S.ge.changed = 0; S.go.changed = 0;
    }
}

// phases B-D: derived quantities in S.pose -> 1000 world points in S.px/py/pz (+ S.pj, grids)
// kCompact: both grids through one copy of the B0/walk code (see the loop below); otherwise one specialised copy each.
template <bool kCompact>
__device__ __forceinline__ void sample_surface(Smem &S, GridSpec *spec, int tid, int nthreads, bool have_prev,
                                               bool prof = false)
{
    const int warp = tid >> 5, lane = tid & 31;
    // ---- B0: node pool of the previous tree -> powers, split ratios, slots; B: fix-up walk; C: CDF ----
    // (every kernel here runs at least two warps)
    const float pi = 3.14159274101257324f;       // (float)acos(-1), sampling.cpp:14
    const float pi_2 = __fmul_rn(pi, 0.5f);      // pi/2, :15
    const Pose &P = S.pose;
    if constexpr (kCompact) {
        // Both grids run through ONE copy of the code (instruction-cache footprint): pass 0 is the eta grid with every
        // thread, pass 1 the omega grid with warps >= 1 behind named barrier 1 -- meanwhile warp 0 finishes the eta
        // grid (fix-up walk over new nodes -- everything on the first iteration -- then the strictly serial CDF).
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {
            GridTab &g = pass ? S.go : S.ge;
            GridSpec &sp = spec[pass];
            const float a2 = pass ? P.a[1] : P.a[2];
            int bad = 0;
            if (warp >= pass) {
                const int t = tid - 32 * pass, n = nthreads - 32 * pass;
                pool_powers(g, sp, P.e[pass], g_logtab[pass], pi_2, t, n);
                asm volatile("bar.sync %0, %1;" ::"r"(pass), "r"(n) : "memory");
                pool_ratios(g, sp, P.a[0], a2, t, n);
                asm volatile("bar.sync %0, %1;" ::"r"(pass), "r"(n) : "memory");
                if (g.changed) {   // uniform: some split count differs from the cached tree -> replay the placement
                    pool_place(g, sp, t, n, bad);
                    asm volatile("bar.sync %0, %1;" ::"r"(pass), "r"(n) : "memory");
                }
                if (pass == 0) SQ_MARK(S, tid, 8);
            }
            if (warp == pass) {  // the grid's serial tail belongs to one warp: sampling.cpp:183-190 / :202-209
                const float tb = pass ? pi : pi_2;
                pool_walk(g, sp, P.a[0], a2, P.e[pass], tb, -tb, g_logtab[pass], pi_2, lane, bad);
                if (pass == 0) {
                    SQ_MARK(S, tid, 1);
                    build_cdf_warp(S.ge, S.cdf, __fadd_rn(P.a[0], P.a[1]), lane);  // :191-199
                    SQ_MARK(S, tid, 7);
                }
            }
            if (bad) S.bad[pass] = 1;
        }
    } else {
        // The same schedule with a specialised copy of the code per grid (compile-time shared-memory addresses).
        int bad = 0;
        pool_powers(S.ge, spec[0], P.e[0], g_logtab[0], pi_2, tid, nthreads);
        __syncthreads();
        pool_ratios(S.ge, spec[0], P.a[0], P.a[2], tid, nthreads);
        __syncthreads();
        if (S.ge.changed) {   // uniform: some split count differs from the cached tree -> replay the placement
            pool_place(S.ge, spec[0], tid, nthreads, bad);
            if (bad) S.bad[0] = 1;
            __syncthreads();
        }
        SQ_MARK(S, tid, 8);
        bad = 0;
        if (warp == 0) {
            pool_walk(S.ge, spec[0], P.a[0], P.a[2], P.e[0], pi_2, -pi_2, g_logtab[0], pi_2, lane, bad);  // :183-190
            SQ_MARK(S, tid, 1);
            build_cdf_warp(S.ge, S.cdf, __fadd_rn(P.a[0], P.a[1]), lane);                                // :191-199
            if (bad) S.bad[0] = 1;
            SQ_MARK(S, tid, 7);
        } else {
            const int t1 = tid - 32, n1 = nthreads - 32;
            pool_powers(S.go, spec[1], P.e[1], g_logtab[1], pi_2, t1, n1);
            asm volatile("bar.sync 1, %0;" ::"r"(n1) : "memory");
            pool_ratios(S.go, spec[1], P.a[0], P.a[1], t1, n1);
            asm volatile("bar.sync 1, %0;" ::"r"(n1) : "memory");
            if (S.go.changed) {
                pool_place(S.go, spec[1], t1, n1, bad);
                asm volatile("bar.sync 1, %0;" ::"r"(n1) : "memory");
            }
            if (warp == 1) pool_walk(S.go, spec[1], P.a[0], P.a[1], P.e[1], pi, -pi, g_logtab[1], pi_2, lane, bad);  // :202-209
            if (bad) S.bad[1] = 1;
        }
    }
    __syncthreads();
    SQ_MARK(S, tid, 10);
    // ---- D ----
    {
        const Pose P = S.pose;
        for (int i = tid; i < kNPad; i += nthreads) {
            if (i < kN) {
                // CDF bucket of this sample.  The bucket of the previous iteration is almost always still right;
                // on the (monotone) CDF, "cdf[j-1] < u <= cdf[j]" is exactly what the bisection returns.
                const float uu = g_u_eta[i];
                int j = 0;
                bool ok = false;
                if (have_prev) {
                    j = S.pj[i];
                    float hi = S.cdf[j], lo = j > 0 ? S.cdf[j - 1] : -1.f;
                    bool up = hi < uu, down = !(lo < uu);
                    ok = !up && !down;
                    if (__any_sync(__activemask(), !ok)) {  // most moves are to a neighbouring bucket
                        int j1 = min(max(j + (up ? 1 : (down ? -1 : 0)), 0), kG - 1);
                        float hi1 = S.cdf[j1], lo1 = j1 > 0 ? S.cdf[j1 - 1] : -1.f;
                        if (!ok && !(hi1 < uu) && lo1 < uu) { j = j1; ok = true; }
                    }
                }
                if (!ok) j = lower_bound_201(S.cdf, uu);
                int k = g_k_omega[i];
                float x0, y0, z0, X, Y, Z;
                local_point(P, lds_f4(&S.ge.slot[j]), lds_f4(&S.go.slot[k]), x0, y0, z0);
                to_world(P, clamp_eps(x0), clamp_eps(y0), clamp_eps(z0), X, Y, Z);
                S.px[i] = X; S.py[i] = Y; S.pz[i] = Z; S.pj[i] = (uint8_t)j;
            } else {  // padding: never valid (NaN is ignored by min/max)
                float nanv = __int_as_float(0x7fc00000);
                S.px[i] = nanv; S.py[i] = nanv; S.pz[i] = nanv; S.pj[i] = 0;
            }
        }
    }
    __syncthreads();
    SQ_MARK(S, tid, 2);
}

template <bool kStaged>
__device__ __forceinline__ void load_M(const float *Ms, int gv, float (&M)[12])
{
    const float4 *p = reinterpret_cast<const float4 *>(Ms + (size_t)gv * 12);
    float4 r0, r1, r2;
    if (kStaged) { r0 = p[0]; r1 = p[1]; r2 = p[2]; }             // shared memory (staged by TMA)
    else { r0 = __ldg(p); r1 = __ldg(p + 1); r2 = __ldg(p + 2); }  // global, read-only path
    M[0] = r0.x; M[1] = r0.y; M[2] = r0.z; M[3] = r0.w;
    M[4] = r1.x; M[5] = r1.y; M[6] = r1.z; M[7] = r1.w;
    M[8] = r2.x; M[9] = r2.y; M[10] = r2.z; M[11] = r2.w;
}

// phase E for one (view, slice) item: extrema over chunks [c0, c1) and, per side, the chunk that produced it
// (-1 = no valid point improved on the +-1e6 sentinel).  The arg index is resolved later, only for the slice that
// wins the cross-slice combine.
// kGroup = points per straight-line block (a divisor of kChunk, multiple of 4): the whole chunk when one CTA owns the SM
// (latency regime, most ILP), 4 when several CTAs in different phases share the instruction caches.
template <bool kCheck, int kGroup>
__device__ __forceinline__ void scan_item(const Smem &S, const float (&M)[12], int c0, int c1,
                                          float (&best)[4], int (&cid)[4])
{
    best[0] = 1000000.f; best[1] = -1000000.f; best[2] = 1000000.f; best[3] = -1000000.f;
    cid[0] = cid[1] = cid[2] = cid[3] = -1;
#pragma unroll 1
    for (int c = c0; c < c1; c++) {
        float n0 = best[0], n1 = best[1], n2 = best[2], n3 = best[3];
#pragma unroll 1
        for (int g = 0; g < kChunk; g += kGroup) {
            const float4 *xs = reinterpret_cast<const float4 *>(S.px + c * kChunk + g);
            const float4 *ys = reinterpret_cast<const float4 *>(S.py + c * kChunk + g);
            const float4 *zs = reinterpret_cast<const float4 *>(S.pz + c * kChunk + g);
            float u[kGroup], w[kGroup];
#pragma unroll
            for (int h = 0; h < kGroup / 4; h++) {
                float4 x = xs[h], y = ys[h], z = zs[h];
#if SQ_FFMA2
                project_uv2<kCheck>(M, x.x, x.y, y.x, y.y, z.x, z.y, u[4 * h + 0], u[4 * h + 1], w[4 * h + 0], w[4 * h + 1]);
                project_uv2<kCheck>(M, x.z, x.w, y.z, y.w, z.z, z.w, u[4 * h + 2], u[4 * h + 3], w[4 * h + 2], w[4 * h + 3]);
#else
                project_uv<kCheck>(M, x.x, y.x, z.x, u[4 * h + 0], w[4 * h + 0]);
                project_uv<kCheck>(M, x.y, y.y, z.y, u[4 * h + 1], w[4 * h + 1]);
                project_uv<kCheck>(M, x.z, y.z, z.z, u[4 * h + 2], w[4 * h + 2]);
                project_uv<kCheck>(M, x.w, y.w, z.w, u[4 * h + 3], w[4 * h + 3]);
#endif
            }
#pragma unroll
            for (int h = 0; h < kGroup; h += 2) {
                n0 = fmin3(n0, u[h], u[h + 1]);
                n1 = fmax3(n1, u[h], u[h + 1]);
                n2 = fmin3(n2, w[h], w[h + 1]);
                n3 = fmax3(n3, w[h], w[h + 1]);
            }
        }
        // strict improvement only: the first chunk (lowest indices) keeps ties
        if (n0 < best[0]) { best[0] = n0; cid[0] = c; }
        if (n1 > best[1]) { best[1] = n1; cid[1] = c; }
        if (n2 < best[2]) { best[2] = n2; cid[2] = c; }
        if (n3 > best[3]) { best[3] = n3; cid[3] = c; }
    }
}

// two rows of a camera matrix: `row` (0 = x, 1 = y) and the z row
template <bool kStaged>
__device__ __forceinline__ void load_M2(const float *Ms, int gv, int row, float (&Mr)[4], float (&Mz)[4])
{
    const float4 *p = reinterpret_cast<const float4 *>(Ms + (size_t)gv * 12);
    float4 r, z;
    if (kStaged) { r = p[row]; z = p[2]; }
    else { r = __ldg(p + row); z = __ldg(p + 2); }
    Mr[0] = r.x; Mr[1] = r.y; Mr[2] = r.z; Mr[3] = r.w;
    Mz[0] = z.x; Mz[1] = z.y; Mz[2] = z.z; Mz[3] = z.w;
}

// first point of chunk `c` whose projected coordinate (the same operations as project_uv<true>, for the one image
// axis this side lives on) equals the extremum `best`
__device__ __forceinline__ int resolve_arg(const Smem &S, const float (&Mr)[4], const float (&Mz)[4], int c, float best)
{
    // Every thread searches its own chunk, so at the same step neighbouring lanes would read addresses 16 words apart
    // -- two shared-memory banks for the whole warp, a 16-way conflict (measured: 5 wavefronts per load).  Each lane
    // therefore walks its chunk from a different starting offset; the lowest matching index wins, as before.
    int found = kNPad;
    const int base = c * kChunk;
    const float mz3 = __fadd_rn(Mz[3], 1e-6f);  // as in the scan
    const int rot = threadIdx.x & (kChunk - 1);
#pragma unroll 4
    for (int t = 0; t < kChunk; t++) {
        const int h = base + ((t + rot) & (kChunk - 1));
        const float X = S.px[h], Y = S.py[h], Z = S.pz[h];
        const float q = __fmaf_rn(X, Mr[0], __fmaf_rn(Y, Mr[1], __fmaf_rn(Z, Mr[2], Mr[3])));
        const float qz = __fmaf_rn(X, Mz[0], __fmaf_rn(Y, Mz[1], __fmaf_rn(Z, Mz[2], mz3)));
        float r = rcp_approx(qz);
        r = qz > 0.500001f ? r : __int_as_float(0x7fc00000);
        if (__fmul_rn(q, r) == best) found = min(found, h);
    }
    return found < kNPad ? found : -1;
}

#ifndef SQ_COMPACT_BLOCKS
#define SQ_COMPACT_BLOCKS 4
#endif
// Resident CTAs per SM the register allocation aims at: the compact build 4 x 256 threads, the straight-line build 1024
// threads' worth (64 registers each) -- except kSolo, the build for launches where every CTA has an SM to itself (the
// latency regime): one 512-thread CTA may then use 128 registers per thread, which removes every spill and most of
// the rematerialised address arithmetic from the serial phases (+3..6 % there, bit-identical results).
#define SQ_MIN_BLOCKS(threads, compact, solo) ((compact) ? SQ_COMPACT_BLOCKS : ((solo) ? 1 : 1024 / (threads)))
// phase-E work item -> view << 16 | first chunk << 8 | end chunk: item = slice * V + view, the 63 chunks split evenly
__device__ __forceinline__ unsigned item_code(int item, int V, int slices)
{
    const int sl = item / V, v = item - sl * V;
    return ((unsigned)v << 16) | (unsigned)(((sl * kNChunks) / slices) << 8) | (unsigned)(((sl + 1) * kNChunks) / slices);
}

// kCompact selects the small-instruction-footprint build (odam_sq_options::code_layout): same arithmetic either way.
// kProf: the instantiation that accumulates the per-phase cycle counts (odam_sq_options::out_cycles).  The marks are
// compiled out of the production kernels: a predicate test, a branch and a volatile clock read at 15 places cost
// 2.6 % (config 2) to 4.8 % (config 5) of the throughput even when no count is taken.
template <int kMaxThreads, bool kCompact, bool kSolo = false, bool kProf = false>
__global__ void __launch_bounds__(kMaxThreads, SQ_MIN_BLOCKS(kMaxThreads, kCompact, kSolo)) sq_optimize_kernel(OptArgs A)
{
    // fixed state in static shared memory (compile-time addresses), per-launch scratch in dynamic shared memory
    __shared__ Smem S;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
#ifdef SQ_E_GROUP
    constexpr int kGroup = SQ_E_GROUP;
#else
    constexpr int kGroup = kCompact ? 4 : kChunk;
#endif
    const int tid = threadIdx.x, T = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarps = T >> 5;
    constexpr bool prof = kProf;
    // A cluster of C CTAs shares one object: every CTA runs the (cheap, deterministic) sampler redundantly and
    // projects its own tile of the views; the 13 partial sums meet through distributed shared memory once per iteration.
    const int C = A.cluster;
    const int obj = blockIdx.x / C, crank = blockIdx.x - obj * C;
    const int v_obj = A.view_off[obj];
    const int Vall = A.view_off[obj + 1] - v_obj;
    const int v_begin = v_obj + (Vall * crank) / C;
    const int V = v_obj + (Vall * (crank + 1)) / C - v_begin;   // this CTA's views
    // per-(item, side) results of phase E live after the fixed part of shared memory: {key, chunk id} where key is the
    // extremum for the min sides and MINUS the extremum for the max sides, so that phase F combines slices with "<" only
    float2 *ext = reinterpret_cast<float2 *>(scratch_raw);
    // cross-warp reduction scratch sits behind the per-item area (its size depends on the CTA size, not on 32 warps)
    float(*red)[kRed + 3] = reinterpret_cast<float(*)[kRed + 3]>(scratch_raw + A.red_offset);

    int slices = V > 0 ? T / V : 1;
    slices = max(1, min(slices, A.max_slices));
    const int n_items = V * slices;

    if (tid < 9) {
        S.par[tid] = A.init[(size_t)obj * 9 + tid];
        S.m[tid] = A.m0 ? A.m0[(size_t)obj * 9 + tid] : 0.f;
        S.v[tid] = A.v0 ? A.v0[(size_t)obj * 9 + tid] : 0.f;
        if (A.prior) S.prior[tid] = A.prior[(size_t)min(max(A.cls[obj], 0), 7) * 9 + tid];  // host entry validates; device entry clamps
    }
    if (tid < 3) S.s0[tid] = A.s0 ? A.s0[(size_t)obj * 3 + tid] : A.init[(size_t)obj * 9 + 4 + tid];
    if (tid == 0) {
        S.status = 0;
        for (int k = 0; k < 16; k++) S.cyc[k] = 0;
        S.tmark = clock64();
        const float pi = 3.14159274101257324f, pi_2 = __fmul_rn(pi, 0.5f);
        pool_init(S.ge, pi_2, -pi_2);
        pool_init(S.go, pi, -pi);
        if (C > 1) {
            mbar_init(&S.xbar[0], 1);
            mbar_init(&S.xbar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    __syncthreads();
    if (C > 1) cg::this_cluster().sync();  // every CTA of the cluster is resident and its barriers are initialised

    // One-off staging of this CTA's camera matrices and boxes into shared memory by TMA bulk copies (when the launch
    // reserved room: few, wide CTAs); masks are bytes at 4-byte granularity, copied by plain loads.
    const bool staged = A.stage_views > 0 && V <= A.stage_views;
    float *sMs = reinterpret_cast<float *>(scratch_raw + A.stage_offset);
    float *sBox = sMs + (size_t)A.stage_views * 12;
    uint8_t *sMask = reinterpret_cast<uint8_t *>(sBox + (size_t)A.stage_views * 4);
    if (staged && V > 0) {
        if (tid == 0) {
            mbar_init(&S.tma_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_arrive_expect_tx(&S.tma_bar, (uint32_t)V * 64u);
            tma_bulk_g2s(sMs, A.Ms + (size_t)v_begin * 12, (uint32_t)V * 48u, &S.tma_bar);
            tma_bulk_g2s(sBox, A.box + (size_t)v_begin * 4, (uint32_t)V * 16u, &S.tma_bar);
        }
        for (int i = tid; i < V; i += T) reinterpret_cast<uint32_t *>(sMask)[i] = reinterpret_cast<const uint32_t *>(A.mask)[v_begin + i];
        __syncthreads();
        mbar_wait(&S.tma_bar, 0);
    }
    const float *Msrc = staged ? sMs : A.Ms + (size_t)v_begin * 12;
    const float *Bsrc = staged ? sBox : A.box + (size_t)v_begin * 4;
    const uint8_t *Ksrc = staged ? sMask : A.mask + (size_t)v_begin * 4;

    const unsigned my_item = tid < n_items ? item_code(tid, V, slices) : 0u;
    const float invV = Vall > 0 ? __fdiv_rn(1.f, (float)Vall) : 0.f;
    if (tid < 10) derive_param(S, tid);
    __syncthreads();

    for (int it = 0; it < A.n_iters; it++) {
        // this iteration's Adam step sizes, fetched now: the load is off the critical path by the time phase G wants them
        if (tid < 3) S.adam_now[tid] = A.adam_tab[it * 4 + tid];
        sample_surface<kCompact>(S, reinterpret_cast<GridSpec *>(scratch_raw), tid, T, it > 0, prof);
        const bool last = it == A.n_iters - 1;

        // ---- E ----
        for (int item = tid; item < n_items; item += T) {
            unsigned code = my_item;   // this thread's first item was decoded once, before the first iteration
            if (item != tid) code = item_code(item, V, slices);
            const int v = code >> 16, c0 = (code >> 8) & 0xff, c1 = code & 0xff;
            float M[12];
            if (staged) load_M<true>(Msrc, v, M); else load_M<false>(Msrc, v, M);
            M[11] = __fadd_rn(M[11], 1e-6f);  // the reference's |z| + 1e-6, folded (see project_uv)
            float best[4];
            int cid[4];
            if (view_all_valid(M, S.pose)) scan_item<false, kGroup>(S, M, c0, c1, best, cid);
            else scan_item<true, kGroup>(S, M, c0, c1, best, cid);
            reinterpret_cast<float4 *>(ext)[2 * item] = make_float4(best[0], __int_as_float(cid[0]), -best[1], __int_as_float(cid[1]));
            reinterpret_cast<float4 *>(ext)[2 * item + 1] = make_float4(best[2], __int_as_float(cid[2]), -best[3], __int_as_float(cid[3]));
        }
        __syncthreads();
        SQ_MARK(S, tid, 3);

        // ---- F ----
        float acc[kRed];
#pragma unroll
        for (int k = 0; k < kRed; k++) acc[k] = 0.f;
        const Pose P = S.pose;
        float lside = 0.f;               // this thread's side is fixed: sd = tid & 3 (T is a multiple of 4)
        const int sd = tid & 3;
        for (int pr = tid; pr < 4 * V; pr += T) {
            int v = pr >> 2;
            // combine slices in index order; strict comparison keeps the first index on ties
            float2 rec = ext[pr];
#pragma unroll 4
            for (int sl = 1; sl < slices; sl++) {   // branch-free so that the loads of several slices are in flight
                const float2 b = ext[sl * 4 * V + pr];
                const bool better = b.x < rec.x;
                rec.x = better ? b.x : rec.x;
                rec.y = better ? b.y : rec.y;
            }
            float best = (sd & 1) ? -rec.x : rec.x;
            const int cid = __float_as_int(rec.y);
            SQ_MARK(S, tid, 0);
            int gv = v_begin + v;
            float target = Bsrc[v * 4 + sd];
            float mk = Ksrc[v * 4 + sd] ? 1.f : 0.f;
            // Only two rows of the camera matrix matter to this side: Mr = the x row (sides 0,1) or the y row (2,3), Mz.
            // The scan ranks points with a 1-ulp reciprocal; the winner's coordinate is now re-evaluated with the
            // reference's own rounding sequence (k-ordered FMA chain of the CPU GEMM, IEEE division) so that the
            // loss carries the same fp32 noise as the reference's instead of an independent sample of it.
            float Mr[4], Mz[4];
            float num = 0.f, qz = 1.f, d = 1.f;
            int arg = -1;
            if (cid >= 0) {
                if (staged) load_M2<true>(Msrc, v, sd >> 1, Mr, Mz); else load_M2<false>(Msrc, v, sd >> 1, Mr, Mz);
                arg = resolve_arg(S, Mr, Mz, cid, best);
            }
            if (arg >= 0) {
                float X = S.px[arg], Y = S.py[arg], Z = S.pz[arg];
                num = __fadd_rn(__fmaf_rn(Z, Mr[2], __fmaf_rn(Y, Mr[1], __fmul_rn(X, Mr[0]))), Mr[3]);
                qz = __fadd_rn(__fmaf_rn(Z, Mz[2], __fmaf_rn(Y, Mz[1], __fmul_rn(X, Mz[0]))), Mz[3]);
                d = __fadd_rn(fabsf(qz), 1e-6f);
                best = __fdiv_rn(num, d);
            }
            SQ_MARK(S, tid, 5);
            float diff = __fsub_rn(best, target);
            float l = fabsf(diff);
            if (!(l == l)) l = 0.f;  // sq_libs.py:426-427
            lside = __fadd_rn(lside, __fmul_rn(l, mk));
            if (last) {
                if (A.out_pred) A.out_pred[(size_t)gv * 4 + sd] = best;
                if (A.out_arg) A.out_arg[(size_t)gv * 4 + sd] = arg;
            }
            if (arg < 0 && mk != 0.f) atomicOr(&S.status, ODAM_SQ_ST_NO_VALID_PT);
            if (arg < 0 || mk == 0.f || !(diff == diff)) continue;
            // gradient through the arg-extreme point.  point_vjp (sq_autograd.cuh) holds the same chain rule for the
            // differentiable ops; this copy stays inline on purpose: phase F is register-capped tuned code, and moving
            // it onto the shared helper would need its own A/B timing.
            float c = __fmul_rn(__fmul_rn(sgnf(diff), mk), invV);
            float g_lin = __fdiv_rn(c, d);                                        // d(u)/d(q_x or q_y)
            float g_z = -__fmul_rn(__fdiv_rn(__fmul_rn(c, num), __fmul_rn(d, d)), sgnf(qz));  // d(u)/d(q_z)
            float gp0 = __fmaf_rn(Mz[0], g_z, __fmul_rn(Mr[0], g_lin));
            float gp1 = __fmaf_rn(Mz[1], g_z, __fmul_rn(Mr[1], g_lin));
            float gp2 = __fmaf_rn(Mz[2], g_z, __fmul_rn(Mr[2], g_lin));
            int j = S.pj[arg], k = g_k_omega[arg];
            const float4 se = S.ge.slot[j], so = S.go.slot[k];
            float x0, y0, z0;
            local_point(P, se, so, x0, y0, z0);
            float x = clamp_eps(x0), y = clamp_eps(y0);
            acc[0] += gp0; acc[1] += gp1; acc[2] += gp2;
            acc[3] += gp0 * (-x * P.sz - y * P.cz) + gp1 * (x * P.cz - y * P.sz);
            float gl0 = (P.cz * gp0 + P.sz * gp1) * clamp_grad(x0);
            float gl1 = (-P.sz * gp0 + P.cz * gp1) * clamp_grad(y0);
            float gl2 = gp2 * clamp_grad(z0);
            float fce = se.y, fse = se.z, fco = so.y, fso = so.z;
            acc[4] += 2.f * S.par[4] * (gl0 * fce * fco);
            acc[5] += 2.f * S.par[5] * (gl1 * fce * fso);
            acc[6] += 2.f * S.par[6] * (gl2 * fse);
            if (A.optimize_shapes) {
                float lce, lse, lco, lso;
                slot_logs(S.ge, j, g_logtab[0], lce, lse);
                slot_logs(S.go, k, g_logtab[1], lco, lso);
                float ge1 = (gl0 * x0 + gl1 * y0) * lce + gl2 * z0 * lse;
                float ge2 = gl0 * x0 * lco + gl1 * y0 * lso;
                acc[7] += ge1 * 1.4f * P.sig[0] * (1.f - P.sig[0]);
                acc[8] += ge2 * 1.4f * P.sig[1] * (1.f - P.sig[1]);
            }
        }
        SQ_MARK(S, tid, 9);
        // ---- G: deterministic reduction (butterfly inside the warp, warp order across) ----
#pragma unroll
        for (int k = 0; k < 4; k++) acc[9 + k] = sd == k ? lside : 0.f;
        const int nred = min(nwarps, (4 * V + 31) >> 5);  // warps that had (view, side) pairs
        if (warp < nred) {
#pragma unroll
            for (int k = 0; k < kRed; k++) {
                float x = acc[k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(kFull, x, o);
                acc[k] = x;
            }
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < kRed; k++) red[warp][k] = acc[k];
            }
        }
        __syncthreads();
        SQ_MARK(S, tid, 4);
        if (tid < kRed) {
            float x = 0.f;
            for (int wi = 0; wi < nred; wi++) x += red[wi][tid];
            red[0][tid] = x;
            if (C > 1) {
                // hand this CTA's partial to every CTA of the cluster (including itself): asynchronous remote stores
                // that complete on the receiver's mbarrier; buffers and barriers alternate with the iteration parity
                const int pb = it & 1;
                if (tid == 0) mbar_arrive_expect_tx(&S.xbar[pb], (uint32_t)(C * kRed * sizeof(float)));
                const uint32_t dst = smem_u32(&S.xred[pb][crank][tid]), bar = smem_u32(&S.xbar[pb]);
                for (int r = 0; r < C; r++) st_async_f32(mapa_u32(dst, r), x, mapa_u32(bar, r));
                mbar_wait(&S.xbar[pb], (uint32_t)((it >> 1) & 1));
                x = 0.f;  // same rank order in every CTA -> identical sums -> identical Adam steps
                for (int r = 0; r < C; r++) x += S.xred[pb][r][tid];
                red[0][tid] = x;
            }
        }
        SQ_MARK(S, tid, 12);
        __syncthreads();
        SQ_MARK(S, tid, 13);
        // ---- G: gradient (+ prior), Adam (torch/optim/adam.py _single_tensor_adam; roundings as probed against torch's
        // CPU kernels) and the derived quantities for the next iteration, one lane per parameter; the loss on one more
        // lane.  The divergent code paths (prior, loss, sin/cos of the yaw, sigmoid of the shapes) sit on different
        // warps so that they run side by side instead of one after the other: lane index = parameter index in every
        // warp, so that warps may double up when the CTA has fewer than four.
        {
            int k = -1;
            if (warp == 0 && lane < 7 && lane != 3) k = lane;       // translation, scales (+ prior)
            if (warp == min(3, nwarps - 1) && lane == 3) k = 3;     // yaw -> sin, cos
            if (warp == min(2, nwarps - 1) && (lane == 7 || lane == 8)) k = lane;  // shapes -> sigmoid
            const bool loss_lane = warp == 1 && lane == 9;
            if (k >= 0) {
                float g = red[0][k];
                if (A.prior && k >= 4 && k < 7) {  // d/ds of 20 (s0-s)^T A (s0-s)  (sq_libs.py:463-466)
                    const int r = k - 4;
                    float sym = 0.f;
                    for (int cc = 0; cc < 3; cc++)
                        sym = __fmaf_rn(S.prior[3 * r + cc] + S.prior[3 * cc + r], S.s0[cc] - S.par[4 + cc], sym);
                    g += -20.f * sym;
                }
                if (k >= 7 && !A.optimize_shapes) g = 0.f;
                S.grad[k] = g;
                if (!isfinite(g)) atomicOr(&S.status, ODAM_SQ_ST_NONFINITE);
            }
            float dd[3] = {0.f, 0.f, 0.f};
            if (loss_lane) { dd[0] = S.s0[0] - S.par[4]; dd[1] = S.s0[1] - S.par[5]; dd[2] = S.s0[2] - S.par[6]; }
            // warps 0 and 1: every read of the scales of this iteration comes before their update
            if (warp < 2) asm volatile("bar.sync 2, 64;" ::: "memory");
            if (loss_lane) {
                // loss = sum over sides of mean over ALL views (sq_libs.py:428-429) + prior (:463-466)
                float loss = 0.f;
                for (int sd2 = 0; sd2 < 4; sd2++) loss = __fadd_rn(loss, __fdiv_rn(red[0][9 + sd2], (float)Vall));
                if (A.prior) {
                    float q3 = 0.f;
                    for (int r = 0; r < 3; r++) {
                        float row = 0.f;
                        for (int cc = 0; cc < 3; cc++) row = __fmaf_rn(S.prior[3 * r + cc], dd[cc], row);
                        q3 = __fmaf_rn(dd[r], row, q3);
                    }
                    loss = __fadd_rn(loss, __fmul_rn(q3, 20.f));
                }
                if (crank == 0) A.out_loss[(size_t)obj * A.n_iters + it] = loss;
                if (!isfinite(loss)) atomicOr(&S.status, ODAM_SQ_ST_NONFINITE);
                if (S.bad[0] | S.bad[1]) atomicOr(&S.status, ODAM_SQ_ST_SAMPLER);
                derive_param(S, 9);  // per-iteration resets of the sampler state
            }
            if (k >= 0) {
                if (k < 7 || A.optimize_shapes) {
                    float g = S.grad[k], m = S.m[k], v = S.v[k], p = S.par[k];
                    const float alpha = S.adam_now[k < 7 ? 0 : 1], bc2s = S.adam_now[2];
                    m = __fmaf_rn(A.beta1w, __fsub_rn(g, m), m);
                    v = __fmul_rn(v, A.beta2);
                    v = __fmaf_rn(__fmul_rn(A.beta2w, g), g, v);
                    float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2s), A.eps);
                    p = __fadd_rn(p, __fdiv_rn(__fmul_rn(alpha, m), denom));
                    S.m[k] = m; S.v[k] = v; S.par[k] = p;
                }
                if (A.out_param_hist && crank == 0) A.out_param_hist[((size_t)obj * A.n_iters + it) * 9 + k] = S.par[k];
                derive_param(S, k);
            }
        }
        SQ_MARK(S, tid, 14);
        if (last && crank == 0) {
            if (A.out_eta_idx) for (int i = tid; i < kN; i += T) A.out_eta_idx[(size_t)obj * kN + i] = S.pj[i];
            if (A.out_grids) for (int i = tid; i < kG; i += T) {
                A.out_grids[((size_t)obj * 2 + 0) * kG + i] = S.ge.slot[i].x;
                A.out_grids[((size_t)obj * 2 + 1) * kG + i] = S.go.slot[i].x;
            }
        }
        __syncthreads();
        SQ_MARK(S, tid, 6);
    }
    if (tid == 0) S.cyc[11] = S.ge.rebuilds + S.go.rebuilds;  // slot 11: tree rebuilds (both grids)
    __syncthreads();
    if (A.out_cycles && crank == 0 && tid < 16) A.out_cycles[(size_t)obj * 16 + tid] = S.cyc[tid];
    if (tid < 9 && crank == 0) {
        float p = S.par[tid];
        A.out_params[(size_t)obj * 9 + tid] = p;
        if (!isfinite(p)) atomicOr(&S.status, ODAM_SQ_ST_NONFINITE);
        if (A.out_m) A.out_m[(size_t)obj * 9 + tid] = S.m[tid];
        if (A.out_v) A.out_v[(size_t)obj * 9 + tid] = S.v[tid];
        if (A.out_grad) A.out_grad[(size_t)obj * 9 + tid] = S.grad[tid];
    }
    __syncthreads();
    if (tid == 0 && A.out_status && S.status) atomicOr(&A.out_status[obj], S.status);  // zeroed by the host before the launch
    if (C > 1) cg::this_cluster().sync();  // no CTA exits while a peer may still store into its shared memory
}

// forward only: compute_ellipsoid_points for n objects, one CTA each
__global__ void __launch_bounds__(256) sq_points_kernel(const float *params, int n, float *out_xyz)
{
    __shared__ Smem S;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int tid = threadIdx.x, obj = blockIdx.x;
    if (tid < 9) S.par[tid] = params[(size_t)obj * 9 + tid];
    if (tid == 0) {
        const float pi = 3.14159274101257324f, pi_2 = __fmul_rn(pi, 0.5f);
        pool_init(S.ge, pi_2, -pi_2);
        pool_init(S.go, pi, -pi);
    }
    __syncthreads();
    if (tid < 10) derive_param(S, tid);
    __syncthreads();
    sample_surface<true>(S, reinterpret_cast<GridSpec *>(scratch_raw), tid, blockDim.x, false);
    for (int i = tid; i < kN; i += blockDim.x) {
        float *o = out_xyz + ((size_t)obj * kN + i) * 3;
        o[0] = S.px[i]; o[1] = S.py[i]; o[2] = S.pz[i];
    }
}

#include "sq_autograd.cuh"

// The reference's own native entry point (sampling.hpp:5-15 sample_on_batch, B*M primitives, N=1000,
// buffer_size=201, seed=0): a[n][3], e[n][2] -> etas[n][1000], omegas[n][1000].  One CTA (2 warps) per primitive.
// u_eta / k_omega: per-primitive draws [n][1000] of ONE generator that keeps drawing across the primitives of a call
// (sampling.cpp:169-214: primitive p consumes uniforms 2000p .. 2000p+1999), or NULL = the tables of primitive 0.
__global__ void __launch_bounds__(64) sq_angles_kernel(const float *a, const float *e, int n, float *etas, float *omegas,
                                                       const float *u_eta, const uint8_t *k_omega)
{
    __shared__ Smem S;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, obj = blockIdx.x;
    const float pi = 3.14159274101257324f, pi_2 = __fmul_rn(pi, 0.5f);
    const float a1 = a[obj * 3 + 0], a2 = a[obj * 3 + 1], a3 = a[obj * 3 + 2];
    const float e1 = e[obj * 2 + 0], e2 = e[obj * 2 + 1];
    int bad = 0;
    GridSpec *spec = reinterpret_cast<GridSpec *>(scratch_raw);
    if (tid == 0) { pool_init(S.ge, pi_2, -pi_2); pool_init(S.go, pi, -pi); }
    __syncthreads();
    pool_powers(S.ge, spec[0], e1, g_logtab[0], pi_2, tid, blockDim.x);      // end points only (empty pool)
    pool_powers(S.go, spec[1], e2, g_logtab[1], pi_2, blockDim.x - 1 - tid, blockDim.x);
    __syncthreads();
    if (warp == 0) {
        pool_walk(S.ge, spec[0], a1, a3, e1, pi_2, -pi_2, g_logtab[0], pi_2, lane, bad);
        build_cdf_warp(S.ge, S.cdf, __fadd_rn(a1, a2), lane);
    } else {
        pool_walk(S.go, spec[1], a1, a2, e2, pi, -pi, g_logtab[1], pi_2, lane, bad);
    }
    __syncthreads();
    for (int i = tid; i < kN; i += blockDim.x) {
        const float uu = u_eta ? u_eta[(size_t)obj * kN + i] : g_u_eta[i];
        const int ko = k_omega ? k_omega[(size_t)obj * kN + i] : g_k_omega[i];
        etas[(size_t)obj * kN + i] = S.ge.slot[lower_bound_201(S.cdf, uu)].x;
        omegas[(size_t)obj * kN + i] = S.go.slot[ko].x;
    }
}

// compute_ellipsoid_points + compute_oriented_bbox (run_multi_view.py:66-67): params -> the 8 corners of the oriented
// box of the 1000 surface points (float64, upper four first), one CTA per object; optionally the points themselves.
__global__ void __launch_bounds__(256) sq_obb_kernel(const float *params, int n, double *out_corners, int32_t *out_flag,
                                                      float *out_xyz)
{
    __shared__ Smem S;
    __shared__ HullScratch H;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int tid = threadIdx.x, obj = blockIdx.x;
    if (tid < 9) S.par[tid] = params[(size_t)obj * 9 + tid];
    if (tid == 0) {
        const float pi = 3.14159274101257324f, pi_2 = __fmul_rn(pi, 0.5f);
        pool_init(S.ge, pi_2, -pi_2);
        pool_init(S.go, pi, -pi);
    }
    __syncthreads();
    if (tid < 10) derive_param(S, tid);
    __syncthreads();
    sample_surface<true>(S, reinterpret_cast<GridSpec *>(scratch_raw), tid, blockDim.x, false);
    if (out_xyz)
        for (int i = tid; i < kN; i += blockDim.x) {
            float *o = out_xyz + ((size_t)obj * kN + i) * 3;
            o[0] = S.px[i]; o[1] = S.py[i]; o[2] = S.pz[i];
        }
    obb_of_points(H, S.px, S.py, S.pz, kN, out_corners + (size_t)obj * 24, out_flag ? out_flag + obj : nullptr);
}

// compute_oriented_bbox of arbitrary point sets: pts[n][n_pts][3] float32, n_pts <= 1024
__global__ void __launch_bounds__(256) sq_obb_points_kernel(const float *pts, int n, int n_pts, double *out_corners,
                                                             int32_t *out_flag)
{
    __shared__ float px[kHullMax], py[kHullMax], pz[kHullMax];
    __shared__ HullScratch H;
    const int obj = blockIdx.x;
    for (int i = threadIdx.x; i < n_pts; i += blockDim.x) {
        const float *p = pts + ((size_t)obj * n_pts + i) * 3;
        px[i] = p[0]; py[i] = p[1]; pz[i] = p[2];
    }
    __syncthreads();
    obb_of_points(H, px, py, pz, n_pts, out_corners + (size_t)obj * 24, out_flag ? out_flag + obj : nullptr);
}

// merge_process's pair costs (run_merge.py:90-121): cost[i][j] = 1 - box3d_iou(box_i, box_j)[0] when the classes allow
// a merge (equal, or both in {4, 5}), else 1; symmetric, zero diagonal.  One thread per pair i < j.
// cls == NULL: every pair is evaluated.  iou3d / iou2d (optional, [n][n]): the raw values for i < j, zero elsewhere.
__global__ void sq_merge_cost_kernel(const double *boxes, const int32_t *cls, int n, double *cost, double *iou3d, double *iou2d)
{
    const long long total = (long long)n * n;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / n), j = (int)(t - (long long)i * n);
        if (i > j) continue;
        if (i == j) {
            if (cost) cost[t] = 0.0;
            if (iou3d) iou3d[t] = 0.0;
            if (iou2d) iou2d[t] = 0.0;
            continue;
        }
        bool mergable = true;
        if (cls) {
            const int a = cls[i], b = cls[j];
            mergable = a == b || ((a == 4 || a == 5) && (b == 4 || b == 5));
        }
        double v3 = 0.0, v2 = 0.0;
        if (mergable) box3d_iou_pair(boxes + (size_t)i * 24, boxes + (size_t)j * 24, &v3, &v2);
        const double c = mergable ? 1.0 - v3 : 1.0;
        if (cost) { cost[t] = c; cost[(size_t)j * n + i] = c; }
        if (iou3d) { iou3d[t] = v3; iou3d[(size_t)j * n + i] = 0.0; }
        if (iou2d) { iou2d[t] = v2; iou2d[(size_t)j * n + i] = 0.0; }
    }
}

// get_bbox (sq_libs.py:547-554): plain projective division, no validity test; one CTA per object,
// one thread per view (looping when V > blockDim).
__global__ void __launch_bounds__(256) sq_boxes_kernel(const float *params, const int32_t *view_off,
                                                        const float *Ms, int n, float *out_box)
{
    __shared__ Smem S;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int tid = threadIdx.x, obj = blockIdx.x;
    if (tid < 9) S.par[tid] = params[(size_t)obj * 9 + tid];
    if (tid == 0) {
        const float pi = 3.14159274101257324f, pi_2 = __fmul_rn(pi, 0.5f);
        pool_init(S.ge, pi_2, -pi_2);
        pool_init(S.go, pi, -pi);
    }
    __syncthreads();
    if (tid < 10) derive_param(S, tid);
    __syncthreads();
    sample_surface<true>(S, reinterpret_cast<GridSpec *>(scratch_raw), tid, blockDim.x, false);
    const int v_begin = view_off[obj], V = view_off[obj + 1] - v_begin;
    for (int v = tid; v < V; v += blockDim.x) {
        float M[12];
        load_M<false>(Ms, v_begin + v, M);
        float b0 = INFINITY, b1 = -INFINITY, b2 = INFINITY, b3 = -INFINITY;
        for (int i = 0; i < kN; i++) {
            float X = S.px[i], Y = S.py[i], Z = S.pz[i];
            float qx = __fmaf_rn(X, M[0], __fmaf_rn(Y, M[1], __fmaf_rn(Z, M[2], M[3])));
            float qy = __fmaf_rn(X, M[4], __fmaf_rn(Y, M[5], __fmaf_rn(Z, M[6], M[7])));
            float qz = __fmaf_rn(X, M[8], __fmaf_rn(Y, M[9], __fmaf_rn(Z, M[10], M[11])));
            float u = __fdiv_rn(qx, qz), w = __fdiv_rn(qy, qz);
            b0 = fminf(b0, u); b1 = fmaxf(b1, u); b2 = fminf(b2, w); b3 = fmaxf(b3, w);
        }
        float *o = out_box + (size_t)(v_begin + v) * 4;
        o[0] = b0; o[1] = b1; o[2] = b2; o[3] = b3;
    }
}

// FP32 FMA-pipe roofline probe: 8 independent FFMA chains per thread, no memory traffic.
// self-test of the split IEEE division (sq_device.cuh: div_rn_recip / div_rn_by) against __fdiv_rn on random operands
// covering the whole range div_rn_safe() admits; every 4th pair shares its divisor's neighbourhood in the last place
__global__ void div_selftest_kernel(uint32_t seed, long long n, unsigned long long *mismatches)
{
    unsigned long long bad = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint64_t x = (uint64_t)i * 0x9E3779B97F4A7C15ull + seed;   // splitmix64
        x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
        uint32_t ma = (uint32_t)x & 0x7fffffu, mb = (uint32_t)(x >> 23) & 0x7fffffu;
        uint32_t ea = 67u + (uint32_t)((x >> 46) % 121u), eb = 67u + (uint32_t)((x >> 54) % 121u);   // 2^-60 .. 2^60
        if ((i & 3) == 3) { mb = ma ^ ((uint32_t)(x >> 60) & 7u); eb = ea; }        // quotients next to 1
        const float a = __uint_as_float((ea << 23) | ma), b = __uint_as_float((eb << 23) | mb);
        const float sa = (x >> 63) ? -a : a;
        if (!(div_rn_safe(sa) && div_rn_safe(b))) { bad++; continue; }
        if (__float_as_uint(div_rn_by(sa, b, div_rn_recip(b))) != __float_as_uint(__fdiv_rn(sa, b))) bad++;
    }
    if (bad) atomicAdd(mismatches, bad);
}

__global__ void __launch_bounds__(1024) fma_peak_kernel(float *sink, int iters, float a, float b)
{
    float x0 = threadIdx.x, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f,
          x7 = x0 + 7.f;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            x0 = __fmaf_rn(x0, a, b); x1 = __fmaf_rn(x1, a, b); x2 = __fmaf_rn(x2, a, b); x3 = __fmaf_rn(x3, a, b);
            x4 = __fmaf_rn(x4, a, b); x5 = __fmaf_rn(x5, a, b); x6 = __fmaf_rn(x6, a, b); x7 = __fmaf_rn(x7, a, b);
        }
    }
    float r = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (r == 123.456f) sink[0] = r;  // never true; keeps the chains alive
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static thread_local char g_cuda_err[256] = "";
static int cuda_fail(cudaError_t e, const char *what)
{
    snprintf(g_cuda_err, sizeof g_cuda_err, "%s: %s", what, cudaGetErrorString(e));
    return ODAM_SQ_ERR_CUDA;
}
#define CU(x)                                         \
    do {                                              \
        cudaError_t e_ = (x);                         \
        if (e_ != cudaSuccess) return cuda_fail(e_, #x); \
    } while (0)

// libstdc++'s mt19937 + uniform_real_distribution<float> (sampling.cpp:18-28), seed 0 (_sampler.pyx:438)
static void host_uniforms(uint32_t seed, int n, float *out)
{
    std::vector<uint32_t> mt(624);
    mt[0] = seed;
    for (int i = 1; i < 624; i++) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    int idx = 624;
    for (int k = 0; k < n; k++) {
        if (idx == 624) {
            for (int i = 0; i < 624; i++) {
                uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
                mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            idx = 0;
        }
        uint32_t y = mt[idx++];
        y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
        float r = (float)y / 4294967296.0f;
        if (r >= 1.0f) r = nextafterf(1.0f, 0.0f);
        out[k] = r;
    }
}

// libm's log2_inline of |cosf(theta)| and |sinf(theta)| (the first half of the reference's powf calls) at the dyadic
// angles of a D&C tree rooted at (ta, tb); heap-indexed.  Evaluated with the same host+device code the kernels use.
static double2 logs_at(float th)
{
    const float c = fabsf(sq_glibc_cosf(th)), s = fabsf(sq_glibc_sinf(th));
    return make_double2(sq_glibc_log2(c), s == 0.f ? -1e300 : sq_glibc_log2(s));
}
static void gen_logtab(float ta, float tb, int pos, std::vector<double2> &tab)
{
    if (pos >= kTabSize) return;
    const float th = (ta + tb) * 0.5f;
    tab[pos] = logs_at(th);
    gen_logtab(ta, th, 2 * pos, tab);
    gen_logtab(th, tb, 2 * pos + 1, tab);
}

// restores the caller's current device on every return path of the *_host entry points
struct DeviceGuard {
    int prev = -1;
    cudaError_t enter(int device)
    {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) { prev = -1; return e; }
        return cudaSetDevice(device);
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

struct AdamTab {   // bias-correction table of one (stream, schedule): kept until evicted, never shared across streams
    cudaStream_t stream; int iters, step0; double lr, lrs; float *dev; int cap;
};

struct DeviceState {
    bool ready = false;
    std::mutex host_mu;   // one *_host call at a time per device: they share the staging workspace and the stream
    std::vector<AdamTab> tabs;
    int sm_count = 0;
    int max_smem_optin = 0;
    int excl_clusters[kMaxCluster + 1] = {0, 0, 0, 0, 0};   // [c]: clusters of c CTAs that can be resident at once with one
                                                          // CTA per SM (cudaOccupancyMaxActiveClusters), 0 = unknown
    // workspace of the *_host entry points
    cudaStream_t stream = nullptr;
    void *dbuf = nullptr; size_t dbytes = 0;
    void *hbuf = nullptr; size_t hbytes = 0;   // pinned staging
};
static DeviceState g_dev[64];
static std::mutex g_mu;

using OptKernel = void (*)(OptArgs);

// every instantiation is capped at 64 registers/thread (1024 resident threads per SM worth of registers); the compact
// layout only exists for CTAs of up to 256 threads (it is for many small CTAs per SM)
static OptKernel pick_kernel(int threads, int compact, int solo = 0, int prof = 0)
{
    if (prof) {   // the same builds with the cycle marks compiled in
        if (solo && !compact && threads <= 512) return sq_optimize_kernel<512, false, true, true>;
        if (compact) return threads <= 256 ? sq_optimize_kernel<256, true, false, true> : nullptr;
        return threads <= 256 ? sq_optimize_kernel<256, false, false, true>
                              : (threads <= 512 ? sq_optimize_kernel<512, false, false, true> : sq_optimize_kernel<1024, false, false, true>);
    }
    if (solo && !compact && threads <= 512) return sq_optimize_kernel<512, false, true>;   // one CTA per SM: 128 registers
    if (compact) return threads <= 256 ? sq_optimize_kernel<256, true> : nullptr;
    return threads <= 256 ? sq_optimize_kernel<256, false>
                          : (threads <= 512 ? sq_optimize_kernel<512, false> : sq_optimize_kernel<1024, false>);
}

static int ensure_init(int device)
{
    if (device < 0 || device >= 64) return ODAM_SQ_ERR_ARG;
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceState &D = g_dev[device];
    if (D.ready) return ODAM_SQ_OK;
    DeviceGuard guard;
    CU(guard.enter(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return ODAM_SQ_ERR_DEVICE;
    D.sm_count = prop.multiProcessorCount;
    D.max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    std::vector<float> u(2 * kN);
    host_uniforms(0u, 2 * kN, u.data());
    std::vector<uint8_t> kom(kN);
    for (int i = 0; i < kN; i++) kom[i] = (uint8_t)(int)(u[kN + i] * (float)kG);  // sampling.cpp:211
    CU(cudaMemcpyToSymbol(g_u_eta, u.data(), sizeof(float) * kN));
    CU(cudaMemcpyToSymbol(g_k_omega, kom.data(), kN));
    {
        const float pi = 3.14159274101257324f, pi_2 = pi * 0.5f;
        std::vector<double2> tab(2 * kTabSize, make_double2(0.0, 0.0));
        std::vector<double2> one(kTabSize, make_double2(0.0, 0.0));
        gen_logtab(pi_2, -pi_2, 1, one);
        one[0] = logs_at(pi_2);
        std::copy(one.begin(), one.end(), tab.begin());
        gen_logtab(pi, -pi, 1, one);
        one[0] = logs_at(pi);
        std::copy(one.begin(), one.end(), tab.begin() + kTabSize);
        CU(cudaMemcpyToSymbol(g_logtab, tab.data(), sizeof(double2) * 2 * kTabSize));
    }
    for (int compact = 0; compact < 2; compact++)
        for (int threads : {256, 512, 1024})
            for (int prof = 0; prof < 2; prof++)
                if (auto kern = pick_kernel(threads, compact, 0, prof))
                    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, D.max_smem_optin - (int)sizeof(Smem)));
    for (int prof = 0; prof < 2; prof++)
        CU(cudaFuncSetAttribute(pick_kernel(512, 0, 1, prof), cudaFuncAttributeMaxDynamicSharedMemorySize, D.max_smem_optin - (int)sizeof(Smem)));
    // How many view-tiled clusters can have every CTA on an SM of its own?  A cluster must fit one GPC, and the GPCs
    // of a 148-SM B200 do not hold a whole number of 3- or 4-CTA clusters: measured, 45 x 3 and 32 x 4 CTAs run one
    // per SM while 46 x 3 or 34 x 4 put two CTAs on some SMs and are 10..19 % slower than the next smaller cluster.
    // Asking for (almost) all of an SM's shared memory makes the occupancy query count one CTA per SM.
    for (int c = 2; c <= kMaxCluster; c++) {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3(c * D.sm_count); cfg.blockDim = dim3(512);
        cfg.dynamicSmemBytes = D.max_smem_optin - (int)sizeof(Smem);
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = c; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        int num = 0;
        if (cudaOccupancyMaxActiveClusters(&num, sq_optimize_kernel<512, false>, &cfg) == cudaSuccess) D.excl_clusters[c] = num;
        else cudaGetLastError();
    }
    CU(cudaFuncSetAttribute(sq_points_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    CU(cudaFuncSetAttribute(sq_boxes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    CU(cudaFuncSetAttribute(sq_angles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    CU(cudaFuncSetAttribute(sq_obb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    CU(cudaFuncSetAttribute(sq_points_vjp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    CU(cudaFuncSetAttribute(sq_sides_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSidesSmem));
    CU(cudaFuncSetAttribute(sq_sides_vjp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    CU(cudaStreamCreateWithFlags(&D.stream, cudaStreamNonBlocking));
    D.ready = true;
    return ODAM_SQ_OK;
}

constexpr double kCompactMaxViews = 40;  // mean views per CTA up to which the compact layout wins (measured)
struct LaunchCfg { int threads, max_slices, smem, cluster, red_offset, stage_offset, stage_views, compact, solo; };

// view statistics -> CTA size.  Small tracks get several point slices per view so that a CTA has >=4 warps.
static int choose_launch(int max_views, double mean_views, int n, const odam_sq_options *opt, int sm_count,
                         int smem_optin, const int *excl_clusters, LaunchCfg &L)
{
    // objects that can have a cluster of c CTAs each with every CTA alone on its SM (see ensure_init); the fallback
    // margins are the measured B200 numbers (45 clusters of 3, 32 of 4)
    auto fits = [&](int c) {
        const int cap = excl_clusters && excl_clusters[c] > 0 ? excl_clusters[c]
                        : (c == 2 ? sm_count / 2 : c == 3 ? (sm_count - sm_count / 12) / 3 : (sm_count - sm_count / 8) / 4);
        return n <= cap;
    };
    // view-tiled clusters: while every CTA can still have an SM to itself, 2, 3 or 4 CTAs (on different SMs) share an
    // object; long tracks (>= 128 views) are split in two in any case (finer load balance across SMs)
    int cluster = opt ? opt->cluster : 0;
    // (3 CTAs: measured +3 % over 2 at 40..45 objects x 30..50 views; with 147 of 148 SMs asked for -- 49 objects --
    // the clusters no longer all fit their GPCs at once and the launch is 19 % SLOWER, hence the margin)
    if (cluster == 0)
        cluster = (fits(4) && mean_views >= 32) ? 4
                  : (fits(3) && mean_views >= 24) ? 3
                  : (((fits(2) && mean_views >= 16) || mean_views >= 128) ? 2 : 1);
    if (cluster < 1 || cluster > kMaxCluster) return ODAM_SQ_ERR_ARG;
    // two regimes (measured, tools/regime_sweep.sh): "latency" = no more CTAs than SMs, one wide CTA per SM;
    // "dense" = CTAs share SMs, 256-thread CTAs
    const bool dense = n * cluster > sm_count;
    // point slices per view: many for a lone CTA, 8 when CTAs share SMs (16 for very short tracks)
    // at most two CTAs per SM and short tracks: two wide CTAs (512 threads x 64 registers each = the whole register file)
    // beat four narrow ones at half occupancy -- measured with 160..296 objects: +7..9 % at 20 and 30 views, -5 % at 50
    const bool two_wide = dense && (long)n * cluster <= 2L * sm_count && mean_views <= 40.0 * cluster;
    int max_slices = opt && opt->max_slices ? opt->max_slices
                     : (dense ? (two_wide ? (mean_views < 24 * cluster ? 12 : 8) : (mean_views < 12 * cluster ? 16 : 8)) : 25);
    if (max_slices < 1 || max_slices > 25) return ODAM_SQ_ERR_ARG;
    mean_views = std::max(1.0, mean_views / cluster);
    max_views = (max_views + cluster - 1) / cluster;
    int threads = opt ? opt->threads : 0;
    // code layout: compact when several CTAs in different phases share an SM and the sampler/backward phases are a
    // sizeable part of the iteration (few views); long tracks spend their time in the projection loop either way
    int layout = opt ? opt->code_layout : 0;
    if (layout < 0 || layout > 2) return ODAM_SQ_ERR_ARG;
    if (layout == 0)
        layout = (dense && mean_views <= kCompactMaxViews && (threads == 0 ? !two_wide : threads <= 256)) ? 2 : 1;
    if (layout == 2 && threads > 256) return ODAM_SQ_ERR_ARG;
    if (threads == 0) {
        // measured on B200 (DESIGN.md section 5): in the throughput regime (several CTAs per SM) 256 threads, 320 for
        // long tracks; in the latency regime (fewer CTAs than SMs) a wide CTA with many point slices per view
        int v = std::max(1, (int)(mean_views + 0.5));
        if (dense) {
            threads = two_wide ? 512 : (v <= 110 ? 256 : 320);
        } else {
            int s = std::max(1, std::min(max_slices, 512 / v));
            // at least 512: short tracks leave threads idle in the projection, but the sampler's node-parallel
            // phases and the 1000-point surface want them (50 objects x 20 views: +5 % over 256 threads)
            threads = std::max(512, std::min(1024, ((v * s + 31) / 32) * 32));
        }
    }
    if (threads % 32 || threads < 64 || threads > 1024) return ODAM_SQ_ERR_ARG;  // two warps share the sampler's tail
    long items = std::max(threads, max_views);  // V * min(max_slices, threads / V) <= threads when V <= threads
    long red_offset = std::max<long>(items * 4 * 8, (long)kSpecBytes);  // phase-E results alias the B0 scratch
    long smem = red_offset + (threads / 32) * (kRed + 3) * 4;            // + cross-warp reduction rows
    // Each CTA's camera matrices, boxes and masks are staged into shared memory once, by TMA bulk copies (68 bytes
    // per view): always in the latency regime (few, wide CTAs: shared memory is plentiful), and in the dense regime
    // whenever the staging area does not cost a resident CTA (4 x 256 threads, 3 x 320 or 2 x 512 per SM)
    long stage_offset = (smem + 15) & ~15L;
    int stage_views = max_views <= 256 ? ((max_views + 3) & ~3) : 0;
    if (stage_views && dense) {
        const long ctas = two_wide ? 2 : 1024 / threads;
        const long per_cta = (long)sizeof(Smem) + stage_offset + (long)stage_views * 68 + 1024;   // + the driver's 1 KB
        if (ctas * per_cta > 228L * 1024) stage_views = 0;
    }
    if (stage_views) smem = stage_offset + (long)stage_views * 68;
    if (smem + (long)sizeof(Smem) > smem_optin) return ODAM_SQ_ERR_CONFIG;
    L.threads = threads; L.max_slices = max_slices; L.smem = (int)smem; L.cluster = cluster; L.red_offset = (int)red_offset;
    L.stage_offset = (int)stage_offset; L.stage_views = stage_views; L.compact = layout == 2;
    L.solo = !dense;   // every CTA alone on its SM
    return ODAM_SQ_OK;
}

static void fill_adam_tab(std::vector<float> &tab, int n_iters, int step0, double lr, double lr_shape)
{
    tab.resize((size_t)n_iters * 4);
    for (int it = 0; it < n_iters; it++) {
        double step = (double)(step0 + it + 1);
        double bc1 = 1.0 - pow(0.9, step), bc2 = 1.0 - pow(0.999, step);
        tab[it * 4 + 0] = (float)(-(lr / bc1));
        tab[it * 4 + 1] = (float)(-(lr_shape / bc1));
        tab[it * 4 + 2] = (float)pow(bc2, 0.5);
        tab[it * 4 + 3] = 0.f;
    }
}

static int launch_optimize(DeviceState &D, const OptArgs &A0, const LaunchCfg &L, cudaStream_t st)
{
    OptArgs A = A0;
    A.max_slices = L.max_slices;
    A.beta1w = (float)(1.0 - 0.9); A.beta2 = (float)0.999; A.beta2w = (float)(1.0 - 0.999); A.eps = (float)1e-8;
    A.cluster = L.cluster;
    A.red_offset = L.red_offset;
    A.stage_offset = L.stage_offset; A.stage_views = L.stage_views;
    if (A.out_status) CU(cudaMemsetAsync(A.out_status, 0, sizeof(int32_t) * A.n, st));  // CTAs OR their flags in
    OptKernel kern = pick_kernel(L.threads, L.compact, L.solo, A.out_cycles != nullptr);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
#ifndef SQ_EXTRA_SMEM
#define SQ_EXTRA_SMEM 0   // diagnostics: unused dynamic shared memory per CTA, to lower the number of resident CTAs
#endif
    cfg.gridDim = dim3(A.n * L.cluster); cfg.blockDim = dim3(L.threads); cfg.dynamicSmemBytes = L.smem + SQ_EXTRA_SMEM; cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = L.cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
    CU(cudaLaunchKernelEx(&cfg, kern, A));
    return ODAM_SQ_OK;
}

struct Carver {  // hands out 256-byte aligned offsets into one packed staging buffer
    size_t off = 0;
    template <class T> size_t take(size_t count) {
        off = (off + 255) & ~(size_t)255;
        size_t at = off;
        off += sizeof(T) * count;
        return at;
    }
};
int ensure_ws(DeviceState &D, size_t bytes)
{
    if (D.dbytes < bytes) {
        if (D.dbuf) cudaFree(D.dbuf);
        if (D.hbuf) cudaFreeHost(D.hbuf);
        D.dbuf = D.hbuf = nullptr; D.dbytes = D.hbytes = 0;
        size_t cap = bytes + bytes / 4 + (1 << 20);
        CU(cudaMalloc(&D.dbuf, cap));
        CU(cudaMallocHost(&D.hbuf, cap));
        D.dbytes = D.hbytes = cap;
    }
    return ODAM_SQ_OK;
}

}  // namespace odam

using namespace odam;

extern "C" {

int odam_sq_abi_version(void) { return ODAM_SQ_ABI_VERSION; }

const char *odam_sq_error_string(int code)
{
    switch (code) {
        case ODAM_SQ_OK: return "ok";
        case ODAM_SQ_ERR_ARG: return "invalid argument";
        case ODAM_SQ_ERR_CUDA: return "CUDA runtime error";
        case ODAM_SQ_ERR_DEVICE: return "device is not compute capability 10.x (B200 required)";
        case ODAM_SQ_ERR_CONFIG: return "launch configuration not realisable (too many views for shared memory)";
        default: return "unknown error";
    }
}

const char *odam_sq_last_cuda_error(void) { return g_cuda_err; }

int odam_sq_init(int device) { return ensure_init(device); }

int odam_sq_cluster_capacity(int device, int cluster, int *objects)
{
    if (!objects || cluster < 2 || cluster > kMaxCluster) return ODAM_SQ_ERR_ARG;
    int rc = ensure_init(device);
    if (rc) return rc;
    *objects = g_dev[device].excl_clusters[cluster];
    return ODAM_SQ_OK;
}

int odam_sq_query_launch(const int32_t *view_off, int n, const odam_sq_options *opt, int *threads, int *smem_bytes,
                         int *ctas_per_sm, int *cluster, int *code_layout, int *max_slices)
{
    if (!view_off || n <= 0) return ODAM_SQ_ERR_ARG;
    int maxv = 0;
    for (int i = 0; i < n; i++) maxv = std::max(maxv, view_off[i + 1] - view_off[i]);
    LaunchCfg L;
    int sm_count = 148, smem_optin = 232448;   // B200; the current device's own numbers once it is initialised
    const int *excl = nullptr;
    {
        int dev = -1;
        if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64 && g_dev[dev].ready) {
            sm_count = g_dev[dev].sm_count;
            smem_optin = g_dev[dev].max_smem_optin;
            excl = g_dev[dev].excl_clusters;
        } else {
            cudaGetLastError();
        }
    }
    int rc = choose_launch(maxv, (double)(view_off[n] - view_off[0]) / n, n, opt, sm_count, smem_optin, excl, L);
    if (rc) return rc;
    if (threads) *threads = L.threads;
    if (cluster) *cluster = L.cluster;
    if (code_layout) *code_layout = L.compact ? 2 : 1;
    if (max_slices) *max_slices = L.max_slices;
    if (smem_bytes) *smem_bytes = L.smem;
    if (smem_bytes) *smem_bytes += (int)sizeof(Smem);
    const int regs = (L.solo && !L.compact && L.threads <= 512) ? 128 : 64;   // the build pick_kernel() selects
    if (ctas_per_sm) *ctas_per_sm = std::min({32, 2048 / L.threads, 65536 / (regs * L.threads), (233472 - 1024) / (L.smem + (int)sizeof(Smem) + 1024)});
    return ODAM_SQ_OK;
}

// device-pointer entry: view statistics are needed on the host to pick the CTA size, so the caller's
// options may carry them (threads != 0); otherwise view_off is read back (one small D2H copy).
int odam_sq_optimize(const float *init, const int32_t *cls, const int32_t *view_off, const float *Ms,
                     const float *box, const uint8_t *mask, const float *prior, int n, int n_iters,
                     int representation, float lr, float lr_shape, float *out_params, float *out_loss,
                     int32_t *out_status, const odam_sq_options *opt, void *stream)
{
    if (!init || !view_off || !Ms || !box || !mask || !out_params || !out_loss || n < 0 || n_iters < 0)
        return ODAM_SQ_ERR_ARG;
    if (prior && !cls) return ODAM_SQ_ERR_ARG;
    if (representation < 0 || representation > 2) return ODAM_SQ_ERR_ARG;
    if (n == 0 || n_iters == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    cudaStream_t st = (cudaStream_t)stream;
    int maxv = opt ? opt->max_views : 0;
    double meanv = maxv;
    if (!(opt && opt->threads && maxv > 0)) {
        std::vector<int32_t> voff(n + 1);
        CU(cudaMemcpyAsync(voff.data(), view_off, sizeof(int32_t) * (n + 1), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        maxv = 0;
        for (int i = 0; i < n; i++) {
            if (voff[i + 1] < voff[i]) return ODAM_SQ_ERR_ARG;
            maxv = std::max(maxv, voff[i + 1] - voff[i]);
        }
        meanv = (double)(voff[n] - voff[0]) / n;
    }
    LaunchCfg L;
    rc = choose_launch(maxv, meanv, n, opt, D.sm_count, D.max_smem_optin, D.excl_clusters, L);
    if (rc) return rc;
    // Adam bias-correction table (host doubles, as torch computes them in Python floats); one cached table per
    // (stream, schedule), so launches on different streams never share -- or overwrite -- each other's table
    const float *adam_dev = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        const int step0 = opt ? opt->step0 : 0;
        for (const AdamTab &t : D.tabs)
            if (t.stream == st && t.iters == n_iters && t.step0 == step0 && t.lr == (double)lr && t.lrs == (double)lr_shape)
                adam_dev = t.dev;
        if (!adam_dev) {
            AdamTab *slot = nullptr;
            for (AdamTab &t : D.tabs)
                if (t.stream == st) slot = &t;                    // this stream's previous schedule: reuse its buffer
            if (!slot && D.tabs.size() >= 16) slot = &D.tabs[0];  // bounded cache: recycle the oldest entry
            if (slot) {
                CU(cudaStreamSynchronize(slot->stream));          // its last launch may still read the table
                if (slot->cap < n_iters) { cudaFree(slot->dev); slot->dev = nullptr; slot->cap = 0; }
            } else {
                D.tabs.push_back(AdamTab{st, 0, 0, 0, 0, nullptr, 0});
                slot = &D.tabs.back();
            }
            if (!slot->dev) {
                CU(cudaMalloc(&slot->dev, sizeof(float) * 4 * n_iters));
                slot->cap = n_iters;
            }
            std::vector<float> tab;
            fill_adam_tab(tab, n_iters, step0, (double)lr, (double)lr_shape);
            // pageable source: the copy has left the host vector when the call returns
            CU(cudaMemcpyAsync(slot->dev, tab.data(), sizeof(float) * tab.size(), cudaMemcpyHostToDevice, st));
            slot->stream = st; slot->iters = n_iters; slot->step0 = step0; slot->lr = (double)lr; slot->lrs = (double)lr_shape;
            adam_dev = slot->dev;
        }
    }
    OptArgs A;
    memset(&A, 0, sizeof A);
    A.init = init; A.cls = cls; A.view_off = view_off; A.Ms = Ms; A.box = box; A.mask = mask; A.prior = prior;
    A.n = n; A.n_iters = n_iters; A.optimize_shapes = representation == ODAM_SQ_REPR_SUPER_QUADRIC;
    A.adam_tab = adam_dev;
    A.out_params = out_params; A.out_loss = out_loss; A.out_status = out_status;
    if (opt) {
        A.m0 = opt->m0; A.v0 = opt->v0; A.s0 = opt->s0;
        A.out_m = opt->out_m; A.out_v = opt->out_v; A.out_grad = opt->out_grad; A.out_pred = opt->out_pred;
        A.out_arg = opt->out_arg; A.out_eta_idx = opt->out_eta_idx; A.out_grids = opt->out_grids;
        A.out_param_hist = opt->out_param_hist;
        A.out_cycles = (long long *)opt->out_cycles;
    }
    rc = launch_optimize(D, A, L, st);
    if (rc) return rc;
    if (opt && opt->out_corners) {   // run_multi_view.py:66-67 right behind the optimiser, same stream
        sq_obb_kernel<<<n, 256, kFwdSmem, st>>>(out_params, n, opt->out_corners, opt->out_box_flag, nullptr);
        CU(cudaGetLastError());
    }
    return ODAM_SQ_OK;
}

int odam_sq_sample_points(const float *params, int n, float *out_xyz, void *stream)
{
    if (!params || !out_xyz || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    sq_points_kernel<<<n, 256, kFwdSmem, (cudaStream_t)stream>>>(params, n, out_xyz);
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

int odam_sq_project_boxes(const float *params, const int32_t *view_off, const float *Ms, int n, float *out_box,
                          void *stream)
{
    if (!params || !view_off || !Ms || !out_box || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    sq_boxes_kernel<<<n, 256, kFwdSmem, (cudaStream_t)stream>>>(params, view_off, Ms, n, out_box);
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

// ---- differentiable ops (sq_autograd.cuh): device pointers, enqueued on `stream` ----

int odam_sq_sample_points_vjp(const float *params, const float *grad_xyz, int n, float *out_grad_params, void *stream)
{
    if (!params || !grad_xyz || !out_grad_params || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    sq_points_vjp_kernel<<<n, kAgThreads, kFwdSmem, (cudaStream_t)stream>>>(params, grad_xyz, n, out_grad_params);
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

int odam_sq_box_sides(const float *params, const int32_t *view_off, const float *Ms, int n, int total_views,
                      float *out_pred, int32_t *out_arg, void *stream)
{
    if (!params || !view_off || !Ms || !out_pred || !out_arg || n < 0 || total_views < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    sq_sides_kernel<<<n, kAgThreads, kSidesSmem, (cudaStream_t)stream>>>(params, view_off, Ms, n, total_views, out_pred,
                                                                          out_arg);
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

int odam_sq_box_sides_vjp(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                          const float *grad_pred, int n, int total_views, float *out_grad_params, void *stream)
{
    if (!params || !view_off || !Ms || !arg || !grad_pred || !out_grad_params || n < 0 || total_views < 0)
        return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    sq_sides_vjp_kernel<<<n, kAgThreads, kFwdSmem, (cudaStream_t)stream>>>(params, view_off, Ms, arg, grad_pred, n,
                                                                            total_views, out_grad_params);
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

// ---- host-pointer entry points: H2D, kernel, D2H on the library's own stream ----

int odam_sq_optimize_host(const float *init, const int32_t *cls, const int32_t *view_off, const float *Ms,
                          const float *box, const uint8_t *mask, const float *prior, int n, int n_iters,
                          int representation, float lr, float lr_shape, float *out_params, float *out_loss,
                          int32_t *out_status, const odam_sq_options *opt, int device)
{
    if (!init || !view_off || !Ms || !box || !mask || !out_params || !out_loss || n < 0 || n_iters < 0)
        return ODAM_SQ_ERR_ARG;
    if (prior && !cls) return ODAM_SQ_ERR_ARG;
    if (representation < 0 || representation > 2) return ODAM_SQ_ERR_ARG;
    if (n == 0 || n_iters == 0) return ODAM_SQ_OK;
    int maxv = 0;
    for (int i = 0; i < n; i++) {
        if (view_off[i + 1] < view_off[i]) return ODAM_SQ_ERR_ARG;
        maxv = std::max(maxv, view_off[i + 1] - view_off[i]);
    }
    if (view_off[0] != 0) return ODAM_SQ_ERR_ARG;
    if (prior)
        for (int i = 0; i < n; i++)
            if (cls[i] < 0 || cls[i] > 7) return ODAM_SQ_ERR_ARG;   // 8 classes (sq_libs.py:13-22)
    const size_t SV = (size_t)view_off[n];
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    LaunchCfg L;
    rc = choose_launch(maxv, (double)SV / n, n, opt, D.sm_count, D.max_smem_optin, D.excl_clusters, L);
    if (rc) return rc;

    // one packed staging buffer: inputs first, outputs after; same layout on host (pinned) and device
    size_t in_bytes = 0, total = 0;
    size_t o_init, o_cls, o_voff, o_Ms, o_box, o_mask, o_prior, o_tab, o_m0, o_v0, o_s0;
    size_t o_par, o_loss, o_st, o_m, o_v, o_g, o_pred, o_arg, o_eta, o_grids, o_hist, o_cor, o_flag;
    auto lay = [&](Carver &C) {
        o_init = C.take<float>((size_t)n * 9); o_cls = C.take<int32_t>(n);
        o_voff = C.take<int32_t>(n + 1); o_Ms = C.take<float>(SV * 12);
        o_box = C.take<float>(SV * 4); o_mask = C.take<uint8_t>(SV * 4);
        o_prior = C.take<float>(72); o_tab = C.take<float>((size_t)n_iters * 4);
        o_m0 = C.take<float>(opt && opt->m0 ? (size_t)n * 9 : 0); o_v0 = C.take<float>(opt && opt->v0 ? (size_t)n * 9 : 0);
        o_s0 = C.take<float>(opt && opt->s0 ? (size_t)n * 3 : 0);
        in_bytes = (C.off + 255) & ~(size_t)255;
        o_par = C.take<float>((size_t)n * 9); o_loss = C.take<float>((size_t)n * n_iters);
        o_st = C.take<int32_t>(n);
        o_m = C.take<float>(opt && opt->out_m ? (size_t)n * 9 : 0); o_v = C.take<float>(opt && opt->out_v ? (size_t)n * 9 : 0);
        o_g = C.take<float>(opt && opt->out_grad ? (size_t)n * 9 : 0); o_pred = C.take<float>(opt && opt->out_pred ? SV * 4 : 0);
        o_arg = C.take<int32_t>(opt && opt->out_arg ? SV * 4 : 0);
        o_eta = C.take<uint8_t>(opt && opt->out_eta_idx ? (size_t)n * kN : 0);
        o_grids = C.take<float>(opt && opt->out_grids ? (size_t)n * 2 * kG : 0);
        o_hist = C.take<float>(opt && opt->out_param_hist ? (size_t)n * n_iters * 9 : 0);
        o_cor = C.take<double>(opt && opt->out_corners ? (size_t)n * 24 : 0);
        o_flag = C.take<int32_t>(opt && opt->out_corners ? n : 0);
        total = C.off;
    };
    { Carver C; lay(C); }
    {
        std::lock_guard<std::mutex> lk(g_mu);
        rc = ensure_ws(D, total);
    }
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h + o_init, init, sizeof(float) * 9 * n);
    if (cls) memcpy(h + o_cls, cls, sizeof(int32_t) * n);
    memcpy(h + o_voff, view_off, sizeof(int32_t) * (n + 1));
    memcpy(h + o_Ms, Ms, sizeof(float) * 12 * SV);
    memcpy(h + o_box, box, sizeof(float) * 4 * SV);
    memcpy(h + o_mask, mask, SV * 4);
    if (prior) memcpy(h + o_prior, prior, sizeof(float) * 72);
    std::vector<float> tab;
    fill_adam_tab(tab, n_iters, opt ? opt->step0 : 0, (double)lr, (double)lr_shape);
    memcpy(h + o_tab, tab.data(), sizeof(float) * tab.size());
    if (opt && opt->m0) memcpy(h + o_m0, opt->m0, sizeof(float) * 9 * n);
    if (opt && opt->v0) memcpy(h + o_v0, opt->v0, sizeof(float) * 9 * n);
    if (opt && opt->s0) memcpy(h + o_s0, opt->s0, sizeof(float) * 3 * n);
    cudaStream_t st = D.stream;
    CU(cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, st));

    OptArgs A;
    memset(&A, 0, sizeof A);
    A.init = (float *)(d + o_init); A.cls = cls ? (int32_t *)(d + o_cls) : nullptr;
    A.view_off = (int32_t *)(d + o_voff); A.Ms = (float *)(d + o_Ms); A.box = (float *)(d + o_box);
    A.mask = d + o_mask; A.prior = prior ? (float *)(d + o_prior) : nullptr;
    A.n = n; A.n_iters = n_iters; A.optimize_shapes = representation == ODAM_SQ_REPR_SUPER_QUADRIC;
    A.adam_tab = (float *)(d + o_tab);
    A.out_params = (float *)(d + o_par); A.out_loss = (float *)(d + o_loss); A.out_status = (int32_t *)(d + o_st);
    if (opt) {
        A.m0 = opt->m0 ? (float *)(d + o_m0) : nullptr; A.v0 = opt->v0 ? (float *)(d + o_v0) : nullptr;
        A.s0 = opt->s0 ? (float *)(d + o_s0) : nullptr;
        A.out_m = opt->out_m ? (float *)(d + o_m) : nullptr; A.out_v = opt->out_v ? (float *)(d + o_v) : nullptr;
        A.out_grad = opt->out_grad ? (float *)(d + o_g) : nullptr;
        A.out_pred = opt->out_pred ? (float *)(d + o_pred) : nullptr;
        A.out_arg = opt->out_arg ? (int32_t *)(d + o_arg) : nullptr;
        A.out_eta_idx = opt->out_eta_idx ? d + o_eta : nullptr;
        A.out_grids = opt->out_grids ? (float *)(d + o_grids) : nullptr;
        A.out_param_hist = opt->out_param_hist ? (float *)(d + o_hist) : nullptr;
    }
    rc = launch_optimize(D, A, L, st);
    if (rc) return rc;
    if (opt && opt->out_corners) {   // run_multi_view.py:66-67 right behind the optimiser: no second call, copy or sync
        sq_obb_kernel<<<n, 256, kFwdSmem, st>>>((float *)(d + o_par), n, (double *)(d + o_cor), (int32_t *)(d + o_flag), nullptr);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(h + in_bytes, d + in_bytes, total - in_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    memcpy(out_params, h + o_par, sizeof(float) * 9 * n);
    memcpy(out_loss, h + o_loss, sizeof(float) * (size_t)n * n_iters);
    if (out_status) memcpy(out_status, h + o_st, sizeof(int32_t) * n);
    if (opt) {
        if (opt->out_m) memcpy(opt->out_m, h + o_m, sizeof(float) * 9 * n);
        if (opt->out_v) memcpy(opt->out_v, h + o_v, sizeof(float) * 9 * n);
        if (opt->out_grad) memcpy(opt->out_grad, h + o_g, sizeof(float) * 9 * n);
        if (opt->out_pred) memcpy(opt->out_pred, h + o_pred, sizeof(float) * 4 * SV);
        if (opt->out_arg) memcpy(opt->out_arg, h + o_arg, sizeof(int32_t) * 4 * SV);
        if (opt->out_eta_idx) memcpy(opt->out_eta_idx, h + o_eta, (size_t)n * kN);
        if (opt->out_grids) memcpy(opt->out_grids, h + o_grids, sizeof(float) * 2 * kG * n);
        if (opt->out_param_hist) memcpy(opt->out_param_hist, h + o_hist, sizeof(float) * 9 * (size_t)n * n_iters);
        if (opt->out_corners) memcpy(opt->out_corners, h + o_cor, sizeof(double) * 24 * n);
        if (opt->out_corners && opt->out_box_flag) memcpy(opt->out_box_flag, h + o_flag, sizeof(int32_t) * n);
    }
    return ODAM_SQ_OK;
}

int odam_sq_sample_points_host(const float *params, int n, float *out_xyz, int device)
{
    if (!params || !out_xyz || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    size_t in_b = ((sizeof(float) * 9 * n + 255) / 256) * 256, out_b = sizeof(float) * 3 * kN * (size_t)n;
    { std::lock_guard<std::mutex> lk(g_mu); rc = ensure_ws(D, in_b + out_b); }
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h, params, sizeof(float) * 9 * n);
    CU(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, D.stream));
    sq_points_kernel<<<n, 256, kFwdSmem, D.stream>>>((float *)d, n, (float *)(d + in_b));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + in_b, d + in_b, out_b, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    memcpy(out_xyz, h + in_b, out_b);
    return ODAM_SQ_OK;
}

int odam_sq_project_boxes_host(const float *params, const int32_t *view_off, const float *Ms, int n, float *out_box,
                               int device)
{
    if (!params || !view_off || !Ms || !out_box || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    const size_t SV = (size_t)view_off[n];
    Carver C;
    size_t o_p = C.take<float>((size_t)n * 9), o_v = C.take<int32_t>(n + 1), o_M = C.take<float>(SV * 12);
    size_t in_b = (C.off + 255) & ~(size_t)255;
    size_t out_b = sizeof(float) * 4 * SV;
    { std::lock_guard<std::mutex> lk(g_mu); rc = ensure_ws(D, in_b + out_b); }
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h + o_p, params, sizeof(float) * 9 * n);
    memcpy(h + o_v, view_off, sizeof(int32_t) * (n + 1));
    memcpy(h + o_M, Ms, sizeof(float) * 12 * SV);
    CU(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, D.stream));
    sq_boxes_kernel<<<n, 256, kFwdSmem, D.stream>>>((float *)(d + o_p), (int32_t *)(d + o_v), (float *)(d + o_M), n,
                                                         (float *)(d + in_b));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + in_b, d + in_b, out_b, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    memcpy(out_box, h + in_b, out_b);
    return ODAM_SQ_OK;
}

int odam_sq_oriented_boxes_host(const float *params, int n, double *out_corners, int32_t *out_flag, float *out_xyz,
                                int device)
{
    if (!params || !out_corners || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    Carver C;
    size_t o_p = C.take<float>((size_t)n * 9);
    size_t in_b = (C.off + 255) & ~(size_t)255;
    C.off = in_b;
    size_t o_c = C.take<double>((size_t)n * 24), o_f = C.take<int32_t>(n);
    size_t o_x = C.take<float>(out_xyz ? (size_t)n * kN * 3 : 0);
    rc = ensure_ws(D, C.off);
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h + o_p, params, sizeof(float) * 9 * n);
    CU(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, D.stream));
    sq_obb_kernel<<<n, 256, kFwdSmem, D.stream>>>((float *)(d + o_p), n, (double *)(d + o_c), (int32_t *)(d + o_f),
                                                      out_xyz ? (float *)(d + o_x) : nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + in_b, d + in_b, C.off - in_b, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    memcpy(out_corners, h + o_c, sizeof(double) * 24 * n);
    if (out_flag) memcpy(out_flag, h + o_f, sizeof(int32_t) * n);
    if (out_xyz) memcpy(out_xyz, h + o_x, sizeof(float) * 3 * kN * (size_t)n);
    return ODAM_SQ_OK;
}

int odam_sq_oriented_boxes(const float *params, int n, double *out_corners, int32_t *out_flag, float *out_xyz,
                           void *stream)
{
    if (!params || !out_corners || n < 0) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int device = 0;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    sq_obb_kernel<<<n, 256, kFwdSmem, (cudaStream_t)stream>>>(params, n, out_corners, out_flag, out_xyz);
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

int odam_sq_oriented_boxes_of_points_host(const float *points, int n, int n_pts, double *out_corners, int32_t *out_flag,
                                          int device)
{
    if (!points || !out_corners || n < 0 || n_pts < 1 || n_pts > kHullMax) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    Carver C;
    size_t o_p = C.take<float>((size_t)n * n_pts * 3);
    size_t in_b = (C.off + 255) & ~(size_t)255;
    C.off = in_b;
    size_t o_c = C.take<double>((size_t)n * 24), o_f = C.take<int32_t>(n);
    rc = ensure_ws(D, C.off);
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h + o_p, points, sizeof(float) * 3 * (size_t)n * n_pts);
    CU(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, D.stream));
    sq_obb_points_kernel<<<n, 256, 0, D.stream>>>((float *)(d + o_p), n, n_pts, (double *)(d + o_c), (int32_t *)(d + o_f));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + in_b, d + in_b, C.off - in_b, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    memcpy(out_corners, h + o_c, sizeof(double) * 24 * n);
    if (out_flag) memcpy(out_flag, h + o_f, sizeof(int32_t) * n);
    return ODAM_SQ_OK;
}

int odam_sq_merge_cost_host(const double *boxes, const int32_t *cls, int n, double *out_cost, double *out_iou3d,
                            double *out_iou2d, int device)
{
    if (!boxes || n < 0 || !(out_cost || out_iou3d || out_iou2d)) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    const size_t nn = (size_t)n * n;
    Carver C;
    size_t o_b = C.take<double>((size_t)n * 24), o_cls = C.take<int32_t>(cls ? n : 0);
    size_t in_b = (C.off + 255) & ~(size_t)255;
    C.off = in_b;
    size_t o_c = C.take<double>(out_cost ? nn : 0), o_3 = C.take<double>(out_iou3d ? nn : 0), o_2 = C.take<double>(out_iou2d ? nn : 0);
    rc = ensure_ws(D, C.off);
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h + o_b, boxes, sizeof(double) * 24 * n);
    if (cls) memcpy(h + o_cls, cls, sizeof(int32_t) * n);
    CU(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, D.stream));
    const int threads = 128;
    const int blocks = (int)std::min<size_t>((nn + threads - 1) / threads, (size_t)D.sm_count * 16);
    sq_merge_cost_kernel<<<blocks, threads, 0, D.stream>>>((double *)(d + o_b), cls ? (int32_t *)(d + o_cls) : nullptr, n,
                                                           out_cost ? (double *)(d + o_c) : nullptr,
                                                           out_iou3d ? (double *)(d + o_3) : nullptr,
                                                           out_iou2d ? (double *)(d + o_2) : nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + in_b, d + in_b, C.off - in_b, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    if (out_cost) memcpy(out_cost, h + o_c, sizeof(double) * nn);
    if (out_iou3d) memcpy(out_iou3d, h + o_3, sizeof(double) * nn);
    if (out_iou2d) memcpy(out_iou2d, h + o_2, sizeof(double) * nn);
    return ODAM_SQ_OK;
}

int odam_sq_sample_on_batch_host(const float *shapes, const float *epsilons, float *etas, float *omegas, int B, int M,
                                 int N, int buffer_size, int seed, int device)
{
    if (!shapes || !epsilons || !etas || !omegas || B < 0 || M < 0) return ODAM_SQ_ERR_ARG;
    if (N != kN || buffer_size != kG || seed != 0) return ODAM_SQ_ERR_ARG;  // the only configuration the path uses
    const int n = B * M;
    if (n == 0) return ODAM_SQ_OK;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    Carver C;
    size_t o_a = C.take<float>((size_t)n * 3), o_e = C.take<float>((size_t)n * 2);
    // one generator per CALL, drawing on across the primitives (sampling.cpp:169): primitive p uses uniforms
    // [2000p, 2000p+1000) for its etas and [2000p+1000, 2000p+2000) for its omega indices
    const bool many = n > 1;
    size_t o_u = C.take<float>(many ? (size_t)n * kN : 0), o_k = C.take<uint8_t>(many ? (size_t)n * kN : 0);
    size_t in_b = (C.off + 255) & ~(size_t)255;
    C.off = in_b;
    size_t o_eta = C.take<float>((size_t)n * kN), o_om = C.take<float>((size_t)n * kN);
    { std::lock_guard<std::mutex> lk(g_mu); rc = ensure_ws(D, C.off); }
    if (rc) return rc;
    unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
    memcpy(h + o_a, shapes, sizeof(float) * 3 * n);
    memcpy(h + o_e, epsilons, sizeof(float) * 2 * n);
    if (many) {
        std::vector<float> u((size_t)2 * kN * n);
        host_uniforms(0u, 2 * kN * n, u.data());
        float *hu = (float *)(h + o_u);
        uint8_t *hk = h + o_k;
        for (int p = 0; p < n; p++)
            for (int i = 0; i < kN; i++) {
                hu[(size_t)p * kN + i] = u[(size_t)2 * kN * p + i];
                hk[(size_t)p * kN + i] = (uint8_t)(int)(u[(size_t)2 * kN * p + kN + i] * (float)kG);  // sampling.cpp:211
            }
    }
    CU(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, D.stream));
    sq_angles_kernel<<<n, 64, kFwdSmem, D.stream>>>((float *)(d + o_a), (float *)(d + o_e), n, (float *)(d + o_eta),
                                                         (float *)(d + o_om), many ? (float *)(d + o_u) : nullptr,
                                                         many ? d + o_k : nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + in_b, d + in_b, C.off - in_b, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    memcpy(etas, h + o_eta, sizeof(float) * kN * (size_t)n);
    memcpy(omegas, h + o_om, sizeof(float) * kN * (size_t)n);
    return ODAM_SQ_OK;
}

int odam_sq_fma_peak(int device, double *tflops)
{
    if (!tflops) return ODAM_SQ_ERR_ARG;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    { std::lock_guard<std::mutex> lk(g_mu); rc = ensure_ws(D, 4096); }
    if (rc) return rc;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    const int iters = 4096, blocks = D.sm_count * 2, threads = 1024;
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(e0, D.stream));
        fma_peak_kernel<<<blocks, threads, 0, D.stream>>>((float *)D.dbuf, iters, 0.999f, 0.001f);
        CU(cudaEventRecord(e1, D.stream));
        CU(cudaEventSynchronize(e1));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        double fl = 2.0 * 8 * 16 * (double)iters * blocks * threads;
        if (rep) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops = best;
    return ODAM_SQ_OK;
}

int odam_sq_selftest(int device, uint32_t seed, long long n, long long *mismatches)
{
    if (!mismatches || n < 0) return ODAM_SQ_ERR_ARG;
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    { std::lock_guard<std::mutex> lk(g_mu); rc = ensure_ws(D, 4096); }
    if (rc) return rc;
    CU(cudaMemsetAsync(D.dbuf, 0, 8, D.stream));
    div_selftest_kernel<<<D.sm_count * 4, 256, 0, D.stream>>>(seed, n, (unsigned long long *)D.dbuf);
    unsigned long long h = 0;
    CU(cudaMemcpyAsync(&h, D.dbuf, 8, cudaMemcpyDeviceToHost, D.stream));
    CU(cudaStreamSynchronize(D.stream));
    *mismatches = (long long)h;
    return ODAM_SQ_OK;
}

}  // extern "C"
