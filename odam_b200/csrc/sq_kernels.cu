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

#include "sq_device.cuh"
#include "sq_postproc.cuh"
#include "sq_stage.h"

namespace cg = cooperative_groups;

namespace odam {

constexpr int kMaxCluster = 4;   // CTAs per object (view-tiled thread-block cluster)
constexpr int kRed = 13;  // 9 gradients + 4 side sums
constexpr float kPi = 3.14159274101257324f;   // (float)acos(-1), sampling.cpp:14

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

// pi/2 (sampling.cpp:15).  Same value as a constexpr kPi * 0.5f, but that form changes the code ptxas generates for the
// sampler kernels.
__device__ __forceinline__ float half_pi() { return __fmul_rn(kPi, 0.5f); }

// the roots of both grids' trees: eta over [-pi/2, pi/2], omega over [-pi, pi] (one thread)
__device__ __forceinline__ void init_grid_roots(Smem &S)
{
    const float pi_2 = half_pi();
    pool_init(S.ge, pi_2, -pi_2);
    pool_init(S.go, kPi, -kPi);
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
    const float pi_2 = half_pi();
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
                const float tb = pass ? kPi : pi_2;
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
            if (warp == 1) pool_walk(S.go, spec[1], P.a[0], P.a[1], P.e[1], kPi, -kPi, g_logtab[1], pi_2, lane, bad);  // :202-209
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

// the common start of the one-CTA-per-object kernels: params[obj] -> the sampler state in shared memory (parameters,
// pose, both grids, the eta bucket of every sample in S.pj) and the 1000 world points
__device__ __forceinline__ void sample_object(Smem &S, const float *params, int obj, unsigned char *scratch)
{
    const int tid = threadIdx.x;
    if (tid < 9) S.par[tid] = params[(size_t)obj * 9 + tid];
    if (tid == 0) init_grid_roots(S);
    __syncthreads();
    if (tid < 10) derive_param(S, tid);
    __syncthreads();
    sample_surface<true>(S, reinterpret_cast<GridSpec *>(scratch), tid, blockDim.x, false);
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
                project_uv2<kCheck>(M, x.x, x.y, y.x, y.y, z.x, z.y, u[4 * h + 0], u[4 * h + 1], w[4 * h + 0], w[4 * h + 1]);
                project_uv2<kCheck>(M, x.z, x.w, y.z, y.w, z.z, z.w, u[4 * h + 2], u[4 * h + 3], w[4 * h + 2], w[4 * h + 3]);
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

// first point of chunk `c` whose projected coordinate equals the extremum `best`: one half of project_uv2<true>'s
// sequence, for the one image axis this side lives on: FMA chains for q and q_z with the 1e-6 folded into M[11]
// (Mz[3] here), MUFU.RCP of q_z, NaN unless q_z > 0.500001, one rounded product
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

// Resident CTAs per SM the register allocation aims at: the compact build 4 x 256 threads, the straight-line build 1024
// threads' worth (64 registers each) -- except kSolo, the build for launches where every CTA has an SM to itself (the
// latency regime): one 512-thread CTA may then use 128 registers per thread, which removes every spill and most of
// the rematerialised address arithmetic from the serial phases (+3..6 % there, bit-identical results).
constexpr int min_blocks(int threads, bool compact, bool solo) { return compact ? 4 : (solo ? 1 : 1024 / threads); }
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
__global__ void __launch_bounds__(kMaxThreads, min_blocks(kMaxThreads, kCompact, kSolo)) sq_optimize_kernel(OptArgs A)
{
    // fixed state in static shared memory (compile-time addresses), per-launch scratch in dynamic shared memory
    __shared__ Smem S;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    constexpr int kGroup = kCompact ? 4 : kChunk;
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
        init_grid_roots(S);
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
            M[11] = __fadd_rn(M[11], 1e-6f);  // the reference's |z| + 1e-6, folded (see project_uv2)
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
            // differentiable ops; this copy stays inline on purpose: phase F is register-capped tuned code, and on the
            // shared helper it measured 0.2 % slower (config 2, B200 at 1000 W).
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
    sample_object(S, params, blockIdx.x, scratch_raw);
    const int tid = threadIdx.x, obj = blockIdx.x;
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
    const float pi_2 = half_pi();
    const float a1 = a[obj * 3 + 0], a2 = a[obj * 3 + 1], a3 = a[obj * 3 + 2];
    const float e1 = e[obj * 2 + 0], e2 = e[obj * 2 + 1];
    int bad = 0;
    GridSpec *spec = reinterpret_cast<GridSpec *>(scratch_raw);
    if (tid == 0) init_grid_roots(S);
    __syncthreads();
    pool_powers(S.ge, spec[0], e1, g_logtab[0], pi_2, tid, blockDim.x);      // end points only (empty pool)
    pool_powers(S.go, spec[1], e2, g_logtab[1], pi_2, blockDim.x - 1 - tid, blockDim.x);
    __syncthreads();
    if (warp == 0) {
        pool_walk(S.ge, spec[0], a1, a3, e1, pi_2, -pi_2, g_logtab[0], pi_2, lane, bad);
        build_cdf_warp(S.ge, S.cdf, __fadd_rn(a1, a2), lane);
    } else {
        pool_walk(S.go, spec[1], a1, a2, e2, kPi, -kPi, g_logtab[1], pi_2, lane, bad);
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
    sample_object(S, params, obj, scratch_raw);
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
    sample_object(S, params, obj, scratch_raw);
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

// Device copy of the Adam bias-correction table for a launch on `st` (host doubles, as torch computes them in Python
// floats); one cached table per (stream, schedule), so launches on different streams never share -- or overwrite --
// each other's table
static int adam_table(DeviceState &D, cudaStream_t st, int n_iters, int step0, float lr, float lr_shape,
                      const float *&dev)
{
    std::lock_guard<std::mutex> lk(g_mu);
    dev = nullptr;
    for (const AdamTab &t : D.tabs)
        if (t.stream == st && t.iters == n_iters && t.step0 == step0 && t.lr == (double)lr && t.lrs == (double)lr_shape)
            dev = t.dev;
    if (dev) return ODAM_SQ_OK;
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
    dev = slot->dev;
    return ODAM_SQ_OK;
}

using OptKernel = void (*)(OptArgs);

// The builds of sq_optimize_kernel, each with its cycle-mark twin (prof), in ascending CTA size within each layout.
// Their register budget follows from __launch_bounds__: min_blocks() CTAs of `threads` share the 64K registers.
// The compact layout only exists for CTAs of up to 256 threads (it is for many small CTAs per SM).
struct OptBuild { int threads; bool compact, solo, prof; OptKernel kern; };
static const OptBuild kOptBuilds[] = {
    {256, false, false, false, sq_optimize_kernel<256, false, false, false>},
    {512, false, false, false, sq_optimize_kernel<512, false, false, false>},
    {1024, false, false, false, sq_optimize_kernel<1024, false, false, false>},
    {256, true, false, false, sq_optimize_kernel<256, true, false, false>},
    {512, false, true, false, sq_optimize_kernel<512, false, true, false>},
    {256, false, false, true, sq_optimize_kernel<256, false, false, true>},
    {512, false, false, true, sq_optimize_kernel<512, false, false, true>},
    {1024, false, false, true, sq_optimize_kernel<1024, false, false, true>},
    {256, true, false, true, sq_optimize_kernel<256, true, false, true>},
    {512, false, true, true, sq_optimize_kernel<512, false, true, true>},
};

// the smallest build of the layout that fits `threads` CTA threads; the solo build when every CTA has an SM to itself
// and it fits, else the shared one; NULL: no such build
static const OptBuild *pick_build(int threads, bool compact, bool solo, bool prof)
{
    for (int want_solo = solo && !compact; want_solo >= 0; want_solo--)
        for (const OptBuild &B : kOptBuilds)
            if (B.compact == compact && B.solo == (bool)want_solo && B.prof == prof && threads <= B.threads) return &B;
    return nullptr;
}

static int opt_regs(const OptBuild &B) { return 65536 / (B.threads * min_blocks(B.threads, B.compact, B.solo)); }

// Dynamic shared memory of each per-object kernel: its launcher asks for this much and ensure_init() sets the kernel's
// attribute to it (sq_sides_kernel's kSidesSmem is in sq_autograd.cuh)
constexpr size_t kPointsSmem = kFwdSmem, kObbSmem = kFwdSmem, kBoxesSmem = kFwdSmem, kAnglesSmem = kFwdSmem;
constexpr size_t kPointsVjpSmem = kFwdSmem, kSidesVjpSmem = kFwdSmem;

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
        std::vector<double2> tab(2 * kTabSize, make_double2(0.0, 0.0));
        std::vector<double2> one(kTabSize, make_double2(0.0, 0.0));
        const float pi_2 = kPi * 0.5f;
        gen_logtab(pi_2, -pi_2, 1, one);
        one[0] = logs_at(pi_2);
        std::copy(one.begin(), one.end(), tab.begin());
        gen_logtab(kPi, -kPi, 1, one);
        one[0] = logs_at(kPi);
        std::copy(one.begin(), one.end(), tab.begin() + kTabSize);
        CU(cudaMemcpyToSymbol(g_logtab, tab.data(), sizeof(double2) * 2 * kTabSize));
    }
    for (const OptBuild &B : kOptBuilds)
        CU(cudaFuncSetAttribute(B.kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                D.max_smem_optin - (int)sizeof(Smem)));
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
        if (cudaOccupancyMaxActiveClusters(&num, pick_build(512, false, false, false)->kern, &cfg) == cudaSuccess)
            D.excl_clusters[c] = num;
        else cudaGetLastError();
    }
    const struct { const void *kern; size_t smem; } per_object[] = {
        {(const void *)sq_points_kernel, kPointsSmem},
        {(const void *)sq_boxes_kernel, kBoxesSmem},
        {(const void *)sq_angles_kernel, kAnglesSmem},
        {(const void *)sq_obb_kernel, kObbSmem},
        {(const void *)sq_points_vjp_kernel, kPointsVjpSmem},
        {(const void *)sq_sides_kernel, kSidesSmem},
        {(const void *)sq_sides_vjp_kernel<false>, kSidesVjpSmem},
        {(const void *)sq_sides_vjp_kernel<true>, kSidesVjpSmem},
    };
    for (const auto &k : per_object)
        CU(cudaFuncSetAttribute(k.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
    CU(cudaStreamCreateWithFlags(&D.stream, cudaStreamNonBlocking));
    D.ready = true;
    return ODAM_SQ_OK;
}

static int check_launch()
{
    CU(cudaGetLastError());
    return ODAM_SQ_OK;
}

// body(D) of a device-pointer entry with validated arguments: nothing for n == 0, else on the caller's current device
template <class F>
static int on_current_device(int n, F &&body)
{
    if (n == 0) return ODAM_SQ_OK;
    int device;
    CU(cudaGetDevice(&device));
    int rc = ensure_init(device);
    if (rc) return rc;
    return body(g_dev[device]);
}

// One launcher per kernel: the only place that names its grid and CTA size, with the dynamic shared memory declared
// above ensure_init().  One CTA per object unless stated.
static int launch_points(const float *params, int n, float *xyz, cudaStream_t st)
{
    sq_points_kernel<<<n, 256, kPointsSmem, st>>>(params, n, xyz);
    return check_launch();
}

static int launch_obb(const float *params, int n, double *corners, int32_t *flag, float *xyz, cudaStream_t st)
{
    sq_obb_kernel<<<n, 256, kObbSmem, st>>>(params, n, corners, flag, xyz);
    return check_launch();
}

static int launch_boxes(const float *params, const int32_t *view_off, const float *Ms, int n, float *box,
                        cudaStream_t st)
{
    sq_boxes_kernel<<<n, 256, kBoxesSmem, st>>>(params, view_off, Ms, n, box);
    return check_launch();
}

static int launch_points_vjp(const float *params, const float *grad_xyz, int n, float *grad_params, cudaStream_t st)
{
    sq_points_vjp_kernel<<<n, kAgThreads, kPointsVjpSmem, st>>>(params, grad_xyz, n, grad_params);
    return check_launch();
}

static int launch_sides(const float *params, const int32_t *view_off, const float *Ms, int n, int total_views,
                        float *pred, int32_t *arg, cudaStream_t st)
{
    sq_sides_kernel<<<n, kAgThreads, kSidesSmem, st>>>(params, view_off, Ms, n, total_views, pred, arg);
    return check_launch();
}

template <bool kCams>
static int launch_sides_vjp(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                            const float *grad_pred, int n, int total_views, float *grad_params, float *grad_Ms,
                            cudaStream_t st)
{
    sq_sides_vjp_kernel<kCams><<<n, kAgThreads, kSidesVjpSmem, st>>>(params, view_off, Ms, arg, grad_pred, n,
                                                                      total_views, grad_params, grad_Ms);
    return check_launch();
}

static int launch_obb_points(const float *points, int n, int n_pts, double *corners, int32_t *flag, cudaStream_t st)
{
    sq_obb_points_kernel<<<n, 256, 0, st>>>(points, n, n_pts, corners, flag);
    return check_launch();
}

// grid-stride over the n x n pairs, at most 16 CTAs per SM
static int launch_merge_cost(const double *boxes, const int32_t *cls, int n, double *cost, double *iou3d, double *iou2d,
                             int sm_count, cudaStream_t st)
{
    const int threads = 128;
    const int blocks = (int)std::min<size_t>(((size_t)n * n + threads - 1) / threads, (size_t)sm_count * 16);
    sq_merge_cost_kernel<<<blocks, threads, 0, st>>>(boxes, cls, n, cost, iou3d, iou2d);
    return check_launch();
}

static int launch_angles(const float *shapes, const float *epsilons, int n, float *etas, float *omegas,
                         const float *u_eta, const uint8_t *k_omega, cudaStream_t st)
{
    sq_angles_kernel<<<n, 64, kAnglesSmem, st>>>(shapes, epsilons, n, etas, omegas, u_eta, k_omega);
    return check_launch();
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
    // a layout with no build of this CTA size (the compact one above 256 threads, also when it was asked for with
    // threads chosen here): every configuration this returns has a build, and pick_build() relies on it
    if (!pick_build(threads, layout == 2, !dense, false)) return ODAM_SQ_ERR_ARG;
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

static int launch_optimize(const OptArgs &A0, const LaunchCfg &L, cudaStream_t st)
{
    OptArgs A = A0;
    A.max_slices = L.max_slices;
    A.beta1w = (float)(1.0 - 0.9); A.beta2 = (float)0.999; A.beta2w = (float)(1.0 - 0.999); A.eps = (float)1e-8;
    A.cluster = L.cluster;
    A.red_offset = L.red_offset;
    A.stage_offset = L.stage_offset; A.stage_views = L.stage_views;
    if (A.out_status) CU(cudaMemsetAsync(A.out_status, 0, sizeof(int32_t) * A.n, st));  // CTAs OR their flags in
    OptKernel kern = pick_build(L.threads, L.compact, L.solo, A.out_cycles != nullptr)->kern;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(A.n * L.cluster); cfg.blockDim = dim3(L.threads); cfg.dynamicSmemBytes = L.smem; cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = L.cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
    CU(cudaLaunchKernelEx(&cfg, kern, A));
    return ODAM_SQ_OK;
}

// The workspace of the host-pointer entries (D.stream, D.dbuf, D.hbuf) belongs to whoever holds D.host_mu.
static int ensure_ws(DeviceState &D, size_t bytes)
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

// body(D) of a host-pointer entry: `device` current (the caller's is restored), D.host_mu held, a workspace of at
// least `bytes`
template <class F>
static int with_workspace(int device, size_t bytes, F &&body)
{
    int rc = ensure_init(device);
    if (rc) return rc;
    DeviceState &D = g_dev[device];
    DeviceGuard guard;
    CU(guard.enter(device));
    std::lock_guard<std::mutex> host_lock(D.host_mu);
    rc = ensure_ws(D, bytes);
    if (rc) return rc;
    return body(D);
}

// The round trip of a host-pointer entry on the library's stream.  in() and out() declare a host array through the
// caller's pointer variable.  run() packs the inputs into the pinned workspace (256-byte aligned, inputs first, the
// same layout on the device) and sends them with one H2D copy, points every declared variable at its device copy
// (NULL stays NULL), calls launch(stream), fetches the outputs with one D2H copy and unpacks them after the
// synchronise.
class Staging {
    struct Buf { const void *src; void *dst; size_t bytes, off; void *var; void (*point)(void *var, void *at); };
    std::vector<Buf> bufs;
    template <class T> static void point_at(void *var, void *at) { *static_cast<T **>(var) = static_cast<T *>(at); }

  public:
    template <class T> void in(T *&p, size_t count) { bufs.push_back({p, nullptr, p ? sizeof(T) * count : 0, 0, &p, point_at<T>}); }
    template <class T> void out(T *&p, size_t count) { bufs.push_back({nullptr, p, p ? sizeof(T) * count : 0, 0, &p, point_at<T>}); }

    template <class F> int run(int device, F &&launch)
    {
        size_t in_bytes = 0, end = 0;
        for (int pass = 0; pass < 2; pass++) {   // inputs, then outputs
            for (Buf &b : bufs)
                if ((b.dst != nullptr) == (pass == 1)) { b.off = end; end += (b.bytes + 255) & ~(size_t)255; }
            if (pass == 0) in_bytes = end;
        }
        return with_workspace(device, end, [&](DeviceState &D) {
            unsigned char *h = (unsigned char *)D.hbuf, *d = (unsigned char *)D.dbuf;
            for (const Buf &b : bufs) {
                if (b.src) memcpy(h + b.off, b.src, b.bytes);
                b.point(b.var, b.src || b.dst ? d + b.off : nullptr);
            }
            CU(cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, D.stream));
            int rc = launch(D.stream);
            if (rc) {   // the H2D copy may still read the workspace: let it finish before host_mu is released
                cudaStreamSynchronize(D.stream);
                return rc;
            }
            CU(cudaMemcpyAsync(h + in_bytes, d + in_bytes, end - in_bytes, cudaMemcpyDeviceToHost, D.stream));
            CU(cudaStreamSynchronize(D.stream));
            for (const Buf &b : bufs)
                if (b.dst) memcpy(b.dst, h + b.off, b.bytes);
            return ODAM_SQ_OK;
        });
    }
};

// most views of an object, from view offsets in host memory; *ordered: whether the offsets never decrease
static int most_views(const int32_t *view_off, int n, bool *ordered = nullptr)
{
    int maxv = 0;
    bool ok = true;
    for (int i = 0; i < n; i++) {
        ok = ok && view_off[i + 1] >= view_off[i];
        maxv = std::max(maxv, view_off[i + 1] - view_off[i]);
    }
    if (ordered) *ordered = ok;
    return maxv;
}

// host view offsets: start at 0 and never decrease (so they index the staged arrays); maxv = most views of an object
static int check_view_off(const int32_t *view_off, int n, int &maxv)
{
    bool ordered;
    maxv = most_views(view_off, n, &ordered);
    return view_off[0] == 0 && ordered ? ODAM_SQ_OK : ODAM_SQ_ERR_ARG;
}

// the checks shared by the device- and host-pointer entry of each operation
static int check_sample_points(const float *params, int n, const float *xyz)
{
    return !params || !xyz || n < 0 ? ODAM_SQ_ERR_ARG : ODAM_SQ_OK;
}

static int check_project_boxes(const float *params, const int32_t *view_off, const float *Ms, int n, const float *box)
{
    return !params || !view_off || !Ms || !box || n < 0 ? ODAM_SQ_ERR_ARG : ODAM_SQ_OK;
}

static int check_oriented_boxes(const float *params, int n, const double *corners)
{
    return !params || !corners || n < 0 ? ODAM_SQ_ERR_ARG : ODAM_SQ_OK;
}

// odam_sq_box_sides_vjp(_cameras): `out` is the gradient the entry must write
static int check_sides_vjp(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                           const float *grad_pred, int n, int total_views, const float *out)
{
    return !params || !view_off || !Ms || !arg || !grad_pred || !out || n < 0 || total_views < 0 ? ODAM_SQ_ERR_ARG
                                                                                                  : ODAM_SQ_OK;
}

// the arguments of odam_sq_optimize(_host); the launch fields and adam_tab are set later
static OptArgs opt_args(const float *init, const int32_t *cls, const int32_t *view_off, const float *Ms, const float *box,
                        const uint8_t *mask, const float *prior, int n, int n_iters, int representation,
                        float *out_params, float *out_loss, int32_t *out_status, const odam_sq_options *opt)
{
    OptArgs A;
    memset(&A, 0, sizeof A);
    A.init = init; A.cls = cls; A.view_off = view_off; A.Ms = Ms; A.box = box; A.mask = mask; A.prior = prior;
    A.n = n; A.n_iters = n_iters; A.optimize_shapes = representation == ODAM_SQ_REPR_SUPER_QUADRIC;
    A.out_params = out_params; A.out_loss = out_loss; A.out_status = out_status;
    if (opt) {
        A.m0 = opt->m0; A.v0 = opt->v0; A.s0 = opt->s0;
        A.out_m = opt->out_m; A.out_v = opt->out_v; A.out_grad = opt->out_grad; A.out_pred = opt->out_pred;
        A.out_arg = opt->out_arg; A.out_eta_idx = opt->out_eta_idx; A.out_grids = opt->out_grids;
        A.out_param_hist = opt->out_param_hist;
        A.out_cycles = (long long *)opt->out_cycles;
    }
    return A;
}

static int check_opt_args(const OptArgs &A, int representation)
{
    if (!A.init || !A.view_off || !A.Ms || !A.box || !A.mask || !A.out_params || !A.out_loss || A.n < 0 || A.n_iters < 0)
        return ODAM_SQ_ERR_ARG;
    if (A.prior && !A.cls) return ODAM_SQ_ERR_ARG;
    if (representation < 0 || representation > 2) return ODAM_SQ_ERR_ARG;
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
    const int maxv = most_views(view_off, n);
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
    const int regs = opt_regs(*pick_build(L.threads, L.compact, L.solo, false));
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
    OptArgs A = opt_args(init, cls, view_off, Ms, box, mask, prior, n, n_iters, representation, out_params, out_loss,
                         out_status, opt);
    int rc = check_opt_args(A, representation);
    if (rc || n_iters == 0) return rc;
    return on_current_device(n, [&](DeviceState &D) {
        cudaStream_t st = (cudaStream_t)stream;
        int maxv = opt ? opt->max_views : 0;
        double meanv = maxv;
        if (!(opt && opt->threads && maxv > 0)) {
            std::vector<int32_t> voff(n + 1);
            CU(cudaMemcpyAsync(voff.data(), view_off, sizeof(int32_t) * (n + 1), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            bool ordered;
            maxv = most_views(voff.data(), n, &ordered);
            if (!ordered) return ODAM_SQ_ERR_ARG;
            meanv = (double)(voff[n] - voff[0]) / n;
        }
        LaunchCfg L;
        rc = choose_launch(maxv, meanv, n, opt, D.sm_count, D.max_smem_optin, D.excl_clusters, L);
        if (rc) return rc;
        rc = adam_table(D, st, n_iters, opt ? opt->step0 : 0, lr, lr_shape, A.adam_tab);
        if (rc) return rc;
        rc = launch_optimize(A, L, st);
        if (rc || !(opt && opt->out_corners)) return rc;
        // run_multi_view.py:66-67 right behind the optimiser, same stream
        return launch_obb(out_params, n, opt->out_corners, opt->out_box_flag, nullptr, st);
    });
}

int odam_sq_sample_points(const float *params, int n, float *out_xyz, void *stream)
{
    if (int rc = check_sample_points(params, n, out_xyz)) return rc;
    return on_current_device(n, [&](DeviceState &) { return launch_points(params, n, out_xyz, (cudaStream_t)stream); });
}

int odam_sq_project_boxes(const float *params, const int32_t *view_off, const float *Ms, int n, float *out_box,
                          void *stream)
{
    if (int rc = check_project_boxes(params, view_off, Ms, n, out_box)) return rc;
    return on_current_device(n, [&](DeviceState &) {
        return launch_boxes(params, view_off, Ms, n, out_box, (cudaStream_t)stream);
    });
}

// ---- differentiable ops (sq_autograd.cuh): device pointers, enqueued on `stream` ----

int odam_sq_sample_points_vjp(const float *params, const float *grad_xyz, int n, float *out_grad_params, void *stream)
{
    if (!params || !grad_xyz || !out_grad_params || n < 0) return ODAM_SQ_ERR_ARG;
    return on_current_device(n, [&](DeviceState &) {
        return launch_points_vjp(params, grad_xyz, n, out_grad_params, (cudaStream_t)stream);
    });
}

int odam_sq_box_sides(const float *params, const int32_t *view_off, const float *Ms, int n, int total_views,
                      float *out_pred, int32_t *out_arg, void *stream)
{
    if (!params || !view_off || !Ms || !out_pred || !out_arg || n < 0 || total_views < 0) return ODAM_SQ_ERR_ARG;
    return on_current_device(n, [&](DeviceState &) {
        return launch_sides(params, view_off, Ms, n, total_views, out_pred, out_arg, (cudaStream_t)stream);
    });
}

int odam_sq_box_sides_vjp(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                          const float *grad_pred, int n, int total_views, float *out_grad_params, void *stream)
{
    if (int rc = check_sides_vjp(params, view_off, Ms, arg, grad_pred, n, total_views, out_grad_params)) return rc;
    return on_current_device(n, [&](DeviceState &) {
        return launch_sides_vjp<false>(params, view_off, Ms, arg, grad_pred, n, total_views, out_grad_params, nullptr,
                                       (cudaStream_t)stream);
    });
}

int odam_sq_box_sides_vjp_cameras(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                                  const float *grad_pred, int n, int total_views, float *out_grad_params,
                                  float *out_grad_Ms, void *stream)
{
    if (int rc = check_sides_vjp(params, view_off, Ms, arg, grad_pred, n, total_views, out_grad_Ms)) return rc;
    return on_current_device(n, [&](DeviceState &) {
        return launch_sides_vjp<true>(params, view_off, Ms, arg, grad_pred, n, total_views, out_grad_params,
                                      out_grad_Ms, (cudaStream_t)stream);
    });
}

// ---- host-pointer entry points: one Staging round trip on the library's own stream ----

int odam_sq_optimize_host(const float *init, const int32_t *cls, const int32_t *view_off, const float *Ms,
                          const float *box, const uint8_t *mask, const float *prior, int n, int n_iters,
                          int representation, float lr, float lr_shape, float *out_params, float *out_loss,
                          int32_t *out_status, const odam_sq_options *opt, int device)
{
    OptArgs A = opt_args(init, cls, view_off, Ms, box, mask, prior, n, n_iters, representation, out_params, out_loss,
                         out_status, opt);
    int maxv, rc = check_opt_args(A, representation);
    if (rc || n == 0 || n_iters == 0) return rc;
    rc = check_view_off(view_off, n, maxv);
    if (rc) return rc;
    if (prior)
        for (int i = 0; i < n; i++)
            if (cls[i] < 0 || cls[i] > 7) return ODAM_SQ_ERR_ARG;   // 8 classes (sq_libs.py:13-22)
    const size_t SV = (size_t)view_off[n];
    rc = ensure_init(device);
    if (rc) return rc;
    const DeviceState &D = g_dev[device];
    LaunchCfg L;
    rc = choose_launch(maxv, (double)SV / n, n, opt, D.sm_count, D.max_smem_optin, D.excl_clusters, L);
    if (rc) return rc;
    std::vector<float> tab;
    fill_adam_tab(tab, n_iters, opt ? opt->step0 : 0, (double)lr, (double)lr_shape);
    A.adam_tab = tab.data();
    A.out_cycles = nullptr;   // a device-pointer option
    double *corners = opt ? opt->out_corners : nullptr;
    int32_t *box_flag = corners ? opt->out_box_flag : nullptr;
    const size_t n9 = (size_t)n * 9;
    Staging S;
    S.in(A.init, n9); S.in(A.cls, n); S.in(A.view_off, n + 1); S.in(A.Ms, SV * 12); S.in(A.box, SV * 4);
    S.in(A.mask, SV * 4); S.in(A.prior, 72); S.in(A.adam_tab, tab.size());
    S.in(A.m0, n9); S.in(A.v0, n9); S.in(A.s0, (size_t)n * 3);
    S.out(A.out_params, n9); S.out(A.out_loss, (size_t)n * n_iters); S.out(A.out_status, n);
    S.out(A.out_m, n9); S.out(A.out_v, n9); S.out(A.out_grad, n9); S.out(A.out_pred, SV * 4); S.out(A.out_arg, SV * 4);
    S.out(A.out_eta_idx, (size_t)n * kN); S.out(A.out_grids, (size_t)n * 2 * kG);
    S.out(A.out_param_hist, n9 * n_iters); S.out(corners, (size_t)n * 24); S.out(box_flag, n);
    return S.run(device, [&](cudaStream_t st) {
        rc = launch_optimize(A, L, st);
        if (rc || !corners) return rc;
        // run_multi_view.py:66-67 right behind the optimiser: no second call, copy or sync
        return launch_obb(A.out_params, n, corners, box_flag, nullptr, st);
    });
}

int odam_sq_sample_points_host(const float *params, int n, float *out_xyz, int device)
{
    if (int rc = check_sample_points(params, n, out_xyz)) return rc;
    if (n == 0) return ODAM_SQ_OK;
    Staging S;
    S.in(params, (size_t)n * 9);
    S.out(out_xyz, (size_t)n * kN * 3);
    return S.run(device, [&](cudaStream_t st) { return launch_points(params, n, out_xyz, st); });
}

int odam_sq_project_boxes_host(const float *params, const int32_t *view_off, const float *Ms, int n, float *out_box,
                               int device)
{
    if (int rc = check_project_boxes(params, view_off, Ms, n, out_box)) return rc;
    if (n == 0) return ODAM_SQ_OK;
    int maxv, rc = check_view_off(view_off, n, maxv);
    if (rc) return rc;
    const size_t SV = (size_t)view_off[n];
    Staging S;
    S.in(params, (size_t)n * 9); S.in(view_off, n + 1); S.in(Ms, SV * 12);
    S.out(out_box, SV * 4);
    return S.run(device, [&](cudaStream_t st) { return launch_boxes(params, view_off, Ms, n, out_box, st); });
}

int odam_sq_oriented_boxes_host(const float *params, int n, double *out_corners, int32_t *out_flag, float *out_xyz,
                                int device)
{
    if (int rc = check_oriented_boxes(params, n, out_corners)) return rc;
    if (n == 0) return ODAM_SQ_OK;
    Staging S;
    S.in(params, (size_t)n * 9);
    S.out(out_corners, (size_t)n * 24); S.out(out_flag, n); S.out(out_xyz, (size_t)n * kN * 3);
    return S.run(device, [&](cudaStream_t st) { return launch_obb(params, n, out_corners, out_flag, out_xyz, st); });
}

int odam_sq_oriented_boxes(const float *params, int n, double *out_corners, int32_t *out_flag, float *out_xyz,
                           void *stream)
{
    if (int rc = check_oriented_boxes(params, n, out_corners)) return rc;
    return on_current_device(n, [&](DeviceState &) {
        return launch_obb(params, n, out_corners, out_flag, out_xyz, (cudaStream_t)stream);
    });
}

int odam_sq_oriented_boxes_of_points_host(const float *points, int n, int n_pts, double *out_corners, int32_t *out_flag,
                                          int device)
{
    if (!points || !out_corners || n < 0 || n_pts < 1 || n_pts > kHullMax) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    Staging S;
    S.in(points, (size_t)n * n_pts * 3);
    S.out(out_corners, (size_t)n * 24); S.out(out_flag, n);
    return S.run(device, [&](cudaStream_t st) {
        return launch_obb_points(points, n, n_pts, out_corners, out_flag, st);
    });
}

int odam_sq_merge_cost_host(const double *boxes, const int32_t *cls, int n, double *out_cost, double *out_iou3d,
                            double *out_iou2d, int device)
{
    if (!boxes || n < 0 || !(out_cost || out_iou3d || out_iou2d)) return ODAM_SQ_ERR_ARG;
    if (n == 0) return ODAM_SQ_OK;
    const size_t nn = (size_t)n * n;
    Staging S;
    S.in(boxes, (size_t)n * 24); S.in(cls, n);
    S.out(out_cost, nn); S.out(out_iou3d, nn); S.out(out_iou2d, nn);
    return S.run(device, [&](cudaStream_t st) {
        return launch_merge_cost(boxes, cls, n, out_cost, out_iou3d, out_iou2d, g_dev[device].sm_count, st);
    });
}

int odam_sq_sample_on_batch_host(const float *shapes, const float *epsilons, float *etas, float *omegas, int B, int M,
                                 int N, int buffer_size, int seed, int device)
{
    if (!shapes || !epsilons || !etas || !omegas || B < 0 || M < 0) return ODAM_SQ_ERR_ARG;
    if (N != kN || buffer_size != kG || seed != 0) return ODAM_SQ_ERR_ARG;  // the only configuration the path uses
    const int n = B * M;
    if (n == 0) return ODAM_SQ_OK;
    // one generator per CALL, drawing on across the primitives (sampling.cpp:169): primitive p uses uniforms
    // [2000p, 2000p+1000) for its etas and [2000p+1000, 2000p+2000) for its omega indices; one primitive uses the
    // kernel's own tables
    std::vector<float> u_eta;
    std::vector<uint8_t> k_omega;
    if (n > 1) {
        std::vector<float> u((size_t)2 * kN * n);
        host_uniforms(0u, 2 * kN * n, u.data());
        u_eta.resize((size_t)n * kN);
        k_omega.resize((size_t)n * kN);
        for (int p = 0; p < n; p++)
            for (int i = 0; i < kN; i++) {
                u_eta[(size_t)p * kN + i] = u[(size_t)2 * kN * p + i];
                k_omega[(size_t)p * kN + i] = (uint8_t)(int)(u[(size_t)2 * kN * p + kN + i] * (float)kG);  // sampling.cpp:211
            }
    }
    const float *u_ptr = n > 1 ? u_eta.data() : nullptr;
    const uint8_t *k_ptr = n > 1 ? k_omega.data() : nullptr;
    Staging S;
    S.in(shapes, (size_t)n * 3); S.in(epsilons, (size_t)n * 2); S.in(u_ptr, u_eta.size()); S.in(k_ptr, k_omega.size());
    S.out(etas, (size_t)n * kN); S.out(omegas, (size_t)n * kN);
    return S.run(device, [&](cudaStream_t st) {
        return launch_angles(shapes, epsilons, n, etas, omegas, u_ptr, k_ptr, st);
    });
}

int odam_sq_fma_peak(int device, double *tflops)
{
    if (!tflops) return ODAM_SQ_ERR_ARG;
    return with_workspace(device, 4096, [&](DeviceState &D) {
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
    });
}

int odam_sq_selftest(int device, uint32_t seed, long long n, long long *mismatches)
{
    if (!mismatches || n < 0) return ODAM_SQ_ERR_ARG;
    return with_workspace(device, 4096, [&](DeviceState &D) {
        CU(cudaMemsetAsync(D.dbuf, 0, 8, D.stream));
        div_selftest_kernel<<<D.sm_count * 4, 256, 0, D.stream>>>(seed, n, (unsigned long long *)D.dbuf);
        unsigned long long h = 0;
        CU(cudaMemcpyAsync(&h, D.dbuf, 8, cudaMemcpyDeviceToHost, D.stream));
        CU(cudaStreamSynchronize(D.stream));
        *mismatches = (long long)h;
        return ODAM_SQ_OK;
    });
}

}  // extern "C"
