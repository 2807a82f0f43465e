// sq_autograd.cuh -- forward and backward kernels of the differentiable ops (odam_b200/autograd.py; C ABI
// odam_sq_sample_points_vjp, odam_sq_box_sides, odam_sq_box_sides_vjp, odam_sq_box_sides_vjp_cameras).  Included by
// sq_kernels.cu inside namespace odam, after Smem and sample_object.
//
// Every kernel runs one CTA of kAgThreads threads per object and starts with sample_object, like sq_points_kernel.
// Backward kernels recompute the sampler instead of saving anything from the forward pass: it is deterministic, so
// both passes see the same samples.
//
// Reductions are deterministic: each thread's items follow a fixed stride, then a warp butterfly, then a fixed warp
// order.  An object's gradient is therefore the same bits from run to run and whether it is launched alone or in a
// batch.  Each CTA clamps its views [view_off[i], view_off[i+1]) to [0, total_views], so inconsistent offsets never
// read or write out of bounds.
#pragma once

constexpr int kAgThreads = 256;
constexpr int kAgMaxSlices = 64;                       // point slices per view in sq_sides_kernel
constexpr size_t kSidesSmem = kAgThreads * 4 * 8;      // per-(item, side) {value, code}; aliases the sampler's scratch
static_assert(kSidesSmem >= kSpecBytes, "the sampler's scratch must fit the dynamic shared memory");

// Chain rule of one surface sample: d(point)/d(params) applied to the upstream gradient gp = dL/d(world point), added
// into acc[9] (sq_libs.py:577-595 + sampling.py:598-615).  The same arithmetic as phase F of sq_optimize_kernel, which
// keeps its own copy: phase F is register-capped tuned code, and on this helper it measured 0.2 % slower (config 2,
// B200 at 1000 W).  Unlike phase F the shape gradient is always formed (at h = -10000 the sigmoid factor makes it 0 by itself),
// and NaN or Inf in gp propagates.
__device__ __forceinline__ void point_vjp(const Smem &S, const Pose &P, int j, int k, float gp0, float gp1, float gp2,
                                          float (&acc)[9])
{
    const float4 se = S.ge.slot[j], so = S.go.slot[k];
    float x0, y0, z0;
    local_point(P, se, so, x0, y0, z0);
    const float x = clamp_eps(x0), y = clamp_eps(y0);
    acc[0] += gp0; acc[1] += gp1; acc[2] += gp2;
    acc[3] += gp0 * (-x * P.sz - y * P.cz) + gp1 * (x * P.cz - y * P.sz);
    const float gl0 = (P.cz * gp0 + P.sz * gp1) * clamp_grad(x0);
    const float gl1 = (-P.sz * gp0 + P.cz * gp1) * clamp_grad(y0);
    const float gl2 = gp2 * clamp_grad(z0);
    const float fce = se.y, fse = se.z, fco = so.y, fso = so.z;
    acc[4] += 2.f * S.par[4] * (gl0 * fce * fco);
    acc[5] += 2.f * S.par[5] * (gl1 * fce * fso);
    acc[6] += 2.f * S.par[6] * (gl2 * fse);
    float lce, lse, lco, lso;
    slot_logs(S.ge, j, g_logtab[0], lce, lse);
    slot_logs(S.go, k, g_logtab[1], lco, lso);
    const float ge1 = (gl0 * x0 + gl1 * y0) * lce + gl2 * z0 * lse;
    const float ge2 = gl0 * x0 * lco + gl1 * y0 * lso;
    acc[7] += ge1 * 1.4f * P.sig[0] * (1.f - P.sig[0]);
    acc[8] += ge2 * 1.4f * P.sig[1] * (1.f - P.sig[1]);
}

// acc[9] of every thread -> out[9]: warp butterfly, then the warps in order.  red: 9 floats per warp.
__device__ __forceinline__ void ag_reduce9(float (&acc)[9], float (*red)[9], float *out)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < 9; k++) {
        float x = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(kFull, x, o);
        if (lane == 0) red[warp][k] = x;
    }
    __syncthreads();
    if (tid < 9) {
        float x = 0.f;
        for (int w = 0; w < nwarps; w++) x += red[w][tid];
        out[tid] = x;
    }
}

__device__ __forceinline__ void ag_views(const int32_t *view_off, int obj, int total_views, int &v_begin, int &V)
{
    const int lo = min(max(view_off[obj], 0), total_views);
    const int hi = min(max(view_off[obj + 1], lo), total_views);
    v_begin = lo; V = hi - lo;
}

// grad_params[n][9] = sum over the 1000 samples of grad_xyz . d(point)/d(params)
__global__ void __launch_bounds__(kAgThreads) sq_points_vjp_kernel(const float *params, const float *grad_xyz, int n,
                                                                   float *out_grad)
{
    __shared__ Smem S;
    __shared__ float red[kAgThreads / 32][9];
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int obj = blockIdx.x, tid = threadIdx.x;
    sample_object(S, params, obj, scratch_raw);
    float acc[9];
#pragma unroll
    for (int k = 0; k < 9; k++) acc[k] = 0.f;
    const Pose P = S.pose;
    for (int i = tid; i < kN; i += blockDim.x) {
        const float *g = grad_xyz + ((size_t)obj * kN + i) * 3;
        point_vjp(S, P, S.pj[i], g_k_omega[i], g[0], g[1], g[2], acc);
    }
    ag_reduce9(acc, red, out_grad + (size_t)obj * 9);
}

// one camera matrix, scalar loads (the caller's Ms need not be 16-byte aligned)
__device__ __forceinline__ void ag_load_M(const float *Ms, int gv, float (&M)[12])
{
#pragma unroll
    for (int k = 0; k < 12; k++) M[k] = __ldg(Ms + (size_t)gv * 12 + k);
}

// projection of one point with the reference's rounding sequence (the k-ordered FMA chain of the CPU GEMM, as in
// phase F): numerator of one image row and q_z
__device__ __forceinline__ float ag_row(const float *Mr, float X, float Y, float Z)
{
    return __fadd_rn(__fmaf_rn(Z, Mr[2], __fmaf_rn(Y, Mr[1], __fmul_rn(X, Mr[0]))), Mr[3]);
}

// torch.min / torch.max over a row: NaN wins over numbers, and an earlier entry keeps a tie
__device__ __forceinline__ bool ag_better(float c, float b, bool is_max)
{
    return (is_max ? c > b : c < b) || (c != c && b == b);
}

// constraint_2d (sq_libs.py:397-413): per (view, side) the extremum over the 1000 samples of
// valid ? coord : +-1e6 (valid = q_z > 0.5, coord = q / (|q_z| + 1e-6) by IEEE division), first index on ties;
// arg = the winning sample, or -1 when the winning entry is a sentinel.  Items are (view, point slice) so that short
// tracks still use the CTA; the slices of a view are combined lower slice first, which keeps first-index ties.
// No +-1e6 clipping and no 1-ulp reciprocal ranking: unlike phase E of the fused kernel this is the reference's rule
// exactly.
__global__ void __launch_bounds__(kAgThreads) sq_sides_kernel(const float *params, const int32_t *view_off, const float *Ms,
                                                              int n, int total_views, float *out_pred, int32_t *out_arg)
{
    __shared__ Smem S;
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int obj = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    sample_object(S, params, obj, scratch_raw);
    int v_begin, V;
    ag_views(view_off, obj, total_views, v_begin, V);
    float(*val)[4] = reinterpret_cast<float(*)[4]>(scratch_raw);                  // [T][4]
    int(*code)[4] = reinterpret_cast<int(*)[4]>(scratch_raw + (size_t)T * 16);     // [T][4]: i, or -1 - i for a sentinel
    for (int vr = 0; vr < V; vr += T) {   // rounds of at most T views
        const int Vr = min(T, V - vr);
        const int slices = max(1, min(T / Vr, kAgMaxSlices));
        if (tid < Vr * slices) {
            const int sl = tid / Vr, v = tid - sl * Vr;
            const int i0 = (sl * kN) / slices, i1 = ((sl + 1) * kN) / slices;
            float M[12];
            ag_load_M(Ms, v_begin + vr + v, M);
            float best[4];
            int bc[4];
            for (int i = i0; i < i1; i++) {
                const float X = S.px[i], Y = S.py[i], Z = S.pz[i];
                const float qz = ag_row(M + 8, X, Y, Z);
                const bool valid = qz > 0.5f;
                float c[4];
                if (valid) {
                    const float d = __fadd_rn(fabsf(qz), 1e-6f);
                    c[0] = c[1] = __fdiv_rn(ag_row(M, X, Y, Z), d);
                    c[2] = c[3] = __fdiv_rn(ag_row(M + 4, X, Y, Z), d);
                } else {
                    c[0] = c[2] = 1000000.f;
                    c[1] = c[3] = -1000000.f;
                }
                const int ci = valid ? i : -1 - i;
#pragma unroll
                for (int s = 0; s < 4; s++)
                    if (i == i0 || ag_better(c[s], best[s], s & 1)) { best[s] = c[s]; bc[s] = ci; }
            }
#pragma unroll
            for (int s = 0; s < 4; s++) { val[tid][s] = best[s]; code[tid][s] = bc[s]; }
        }
        __syncthreads();
        for (int pr = tid; pr < 4 * Vr; pr += T) {
            const int v = pr >> 2, s = pr & 3;
            float b = val[v][s];
            int c = code[v][s];
            for (int sl = 1; sl < slices; sl++) {
                const float x = val[sl * Vr + v][s];
                if (ag_better(x, b, s & 1)) { b = x; c = code[sl * Vr + v][s]; }
            }
            const size_t o = (size_t)(v_begin + vr + v) * 4 + s;
            out_pred[o] = b;
            out_arg[o] = c >= 0 ? c : -1;
        }
        __syncthreads();
    }
}

// d pred / d q and d pred / d q_z of one side, scaled by its upstream gradient c = grad_pred[o]: pred = q / d with
// d = |q_z| + 1e-6, g_lin = c / d, g_z = -c q sign(q_z) / d^2.  Both passes of sq_sides_vjp_kernel form them here, so
// the camera gradient uses the same scalars as the parameter gradient.
__device__ __forceinline__ void side_scalars(float num, float qz, const float *grad_pred, size_t o, float &g_lin,
                                             float &g_z)
{
    const float d = __fadd_rn(fabsf(qz), 1e-6f);
    const float c = grad_pred[o];
    g_lin = __fdiv_rn(c, d);
    g_z = -__fmul_rn(__fdiv_rn(__fmul_rn(c, num), __fmul_rn(d, d)), sgnf(qz));
}

// vector-Jacobian product of sq_sides_kernel: one item per (view, side) with arg >= 0, through the arg sample.
// side_scalars, then the camera rows M[:, :3]^T and the per-sample chain of point_vjp.
// kCams = false: Ms is a constant and out_grad is required (odam_sq_box_sides_vjp).
// kCams = true (odam_sq_box_sides_vjp_cameras): out_grad may be NULL (the params pass is skipped); then one thread per
// view writes out_grad_Ms[gv][12] = sum over the live sides s, in the order x_min, x_max, y_min, y_max, of
// g_lin ph into row s >> 1 and g_z ph into row 2, ph = [X, Y, Z, 1] the arg sample.  No atomics: every row has one
// writer and a fixed order.  Rows outside every object's clamped view range are not written.
template <bool kCams>
__global__ void __launch_bounds__(kAgThreads) sq_sides_vjp_kernel(const float *params, const int32_t *view_off,
                                                                  const float *Ms, const int32_t *arg, const float *grad_pred,
                                                                  int n, int total_views, float *out_grad, float *out_grad_Ms)
{
    __shared__ Smem S;
    __shared__ float red[kAgThreads / 32][9];
    extern __shared__ __align__(16) unsigned char scratch_raw[];
    const int obj = blockIdx.x, tid = threadIdx.x;
    sample_object(S, params, obj, scratch_raw);
    int v_begin, V;
    ag_views(view_off, obj, total_views, v_begin, V);
    if (!kCams || out_grad) {
        float acc[9];
#pragma unroll
        for (int k = 0; k < 9; k++) acc[k] = 0.f;
        const Pose P = S.pose;
        for (int pr = tid; pr < 4 * V; pr += blockDim.x) {
            const size_t o = (size_t)v_begin * 4 + pr;
            const int a = arg[o];
            if (a < 0 || a >= kN) continue;   // a sentinel won: the side does not depend on the parameters
            const int gv = v_begin + (pr >> 2), s = pr & 3;
            float Mr[4], Mz[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                Mr[k] = __ldg(Ms + (size_t)gv * 12 + 4 * (s >> 1) + k);
                Mz[k] = __ldg(Ms + (size_t)gv * 12 + 8 + k);
            }
            const float X = S.px[a], Y = S.py[a], Z = S.pz[a];
            float g_lin, g_z;
            side_scalars(ag_row(Mr, X, Y, Z), ag_row(Mz, X, Y, Z), grad_pred, o, g_lin, g_z);
            const float gp0 = __fmaf_rn(Mz[0], g_z, __fmul_rn(Mr[0], g_lin));
            const float gp1 = __fmaf_rn(Mz[1], g_z, __fmul_rn(Mr[1], g_lin));
            const float gp2 = __fmaf_rn(Mz[2], g_z, __fmul_rn(Mr[2], g_lin));
            point_vjp(S, P, S.pj[a], g_k_omega[a], gp0, gp1, gp2, acc);
        }
        ag_reduce9(acc, red, out_grad + (size_t)obj * 9);
    }
    if (kCams) {
        for (int v = tid; v < V; v += blockDim.x) {
            const int gv = v_begin + v;
            float M[12], g[12];
            ag_load_M(Ms, gv, M);
#pragma unroll
            for (int k = 0; k < 12; k++) g[k] = 0.f;
#pragma unroll
            for (int s = 0; s < 4; s++) {
                const size_t o = (size_t)gv * 4 + s;
                const int a = arg[o];
                if (a < 0 || a >= kN) continue;
                const float ph[4] = {S.px[a], S.py[a], S.pz[a], 1.f};
                const int r = s >> 1;
                float g_lin, g_z;
                side_scalars(ag_row(M + 4 * r, ph[0], ph[1], ph[2]), ag_row(M + 8, ph[0], ph[1], ph[2]), grad_pred, o,
                             g_lin, g_z);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    g[4 * r + k] = __fadd_rn(g[4 * r + k], __fmul_rn(g_lin, ph[k]));
                    g[8 + k] = __fadd_rn(g[8 + k], __fmul_rn(g_z, ph[k]));
                }
            }
#pragma unroll
            for (int k = 0; k < 12; k++) out_grad_Ms[(size_t)gv * 12 + k] = g[k];
        }
    }
}
