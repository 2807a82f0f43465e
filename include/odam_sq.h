/*
 * odam_sq.h -- C ABI of the B200-native multi-view superquadric optimiser.
 *
 * This is the drop-in boundary for ONE path of likojack/ODAM: the per-track optimisation that
 *   src/scripts/run_multi_view.py:56-67   (SuperQuadricOptimizer(...); .run(bbox_lines, None, P_cws, n_iters);
 *                                          Q_est.compute_ellipsoid_points(use_numpy=True))
 * performs object by object on the CPU, i.e.
 *   src/super_quadric/sq_libs.py:432-475  SuperQuadricOptimizer.run            -> odam_sq_optimize[_host]
 *   src/super_quadric/sq_libs.py:577-595  SuperQuadric.compute_ellipsoid_points -> odam_sq_sample_points[_host]
 *   src/super_quadric/sq_libs.py:547-554  SuperQuadric.get_bbox                -> odam_sq_project_boxes[_host]
 *   src/super_quadric/learnable_primitives/fast_sampler/sampling.hpp:5-15 sample_on_batch (the reference's
 *   own native entry point, bound by _sampler.pyx:413-454) is subsumed: the sampler runs inside the kernels.
 *
 * Everything is plain pointers and sizes; no C++/torch types.  All objects of a call are optimised
 * in ONE persistent kernel launch (one CTA per object, all iterations on chip).
 *
 * Layouts (all little-endian, densely packed, row-major)
 *   params  [n][9]  float   translate x,y,z | yaw angle | scales s1,s2,s3 (= sqrt(dim/2), sq_libs.py:361)
 *                           | shape logits h1,h2 (e = 0.2 + 1.4*sigmoid(h), sq_libs.py:26-27)
 *   cls     [n]     int32   class id 0..7 (sq_libs.py:13-22), only read when a prior is given
 *   view_off[n+1]   int32   CSR offsets into the per-view arrays; object i owns views view_off[i]..view_off[i+1]-1
 *   Ms      [SV][12] float  P_cw = K @ inv(T_wc)[:3,:] (processor.py:311), row-major 3x4
 *   box     [SV][4] float   detected box sides in pixels, order x_min,x_max,y_min,y_max
 *                           (= -line[-1] of the reference's line dicts, sq_libs.py:449)
 *   mask    [SV][4] uint8   1 = side present (sides within 20 px of the image border are dropped by the
 *                           caller, quadric_helper.py:87-107), 0 = absent
 *   prior   [8][9]  float   per-class 3x3 matrices of src/super_quadric/scale_prior, or NULL = no prior
 *   loss    [n][n_iters] float  total loss (2-D term + prior) BEFORE each step = the reference's loss_log
 *   status  [n]     int32   bit flags ODAM_SQ_ST_*
 *
 * Pointers of the *_host entry points are HOST memory (copies happen inside, on an internal stream,
 * and the call returns when the results are in the output buffers).  Pointers of the other entry
 * points are DEVICE memory on the current CUDA device; the work is enqueued on `stream`
 * (a cudaStream_t passed as void*, NULL = default stream) and the call returns without synchronising.
 *
 * Error convention: 0 = success, negative = ODAM_SQ_ERR_*; never throws, never aborts.
 * Thread safety: one host thread per device at a time (the *_host calls share a per-device workspace).
 */
#ifndef ODAM_SQ_H_
#define ODAM_SQ_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ODAM_SQ_ABI_VERSION 4
#define ODAM_SQ_N_SAMPLES 1000 /* sq_libs.py:545  EqualDistanceSamplerSQ(1000) */
#define ODAM_SQ_GRID 201       /* _sampler.pyx:423 buffer_size */
#define ODAM_SQ_N_PARAMS 9

/* representation (sq_libs.py:363-387) */
#define ODAM_SQ_REPR_SUPER_QUADRIC 0 /* shapes optimised, lr_shape                    */
#define ODAM_SQ_REPR_CUBE 1          /* shapes frozen (caller passes h = -10000)      */
#define ODAM_SQ_REPR_QUADRIC 2       /* shapes frozen (caller passes h = -0)          */

/* status bits */
#define ODAM_SQ_ST_NONFINITE 1   /* a parameter, gradient or loss became NaN/Inf (the reference would raise
                                    from torch anomaly mode, sq_libs.py:456)                                */
#define ODAM_SQ_ST_SAMPLER 2     /* degenerate geometry inside the equal-arc-length sampler (NaN split)     */
#define ODAM_SQ_ST_NO_VALID_PT 4 /* some masked-in side of some view had no point with z > 0.5 (+-1e6 used) */

/* error codes */
#define ODAM_SQ_OK 0
#define ODAM_SQ_ERR_ARG (-1)     /* NULL/negative/inconsistent argument          */
#define ODAM_SQ_ERR_CUDA (-2)    /* a CUDA runtime call failed; see odam_sq_last_cuda_error() */
#define ODAM_SQ_ERR_DEVICE (-3)  /* device is not compute capability 10.x        */
#define ODAM_SQ_ERR_CONFIG (-4)  /* launch configuration not realisable          */

/* Optional knobs and test-only inputs/outputs; zero-initialise, then set what you need. */
typedef struct odam_sq_options {
    int threads;            /* CTA size (multiple of 32, 64..1024); 0 = choose from the view counts   */
    int max_slices;         /* max point-slices per view (1..25); 0 = default                          */
    int cluster;            /* CTAs per object (thread-block cluster, views tiled across them): 1..4; 0 = auto
                               (2, 3 or 4 when there are fewer objects than SMs)                              */
    int max_views;          /* device-pointer entry only: max views of any object, if the caller knows it
                               (with threads != 0 this avoids reading view_off back to the host)         */
    int code_layout;        /* 0 = auto.  1 = straight-line build of the kernel (16-point blocks, one copy of the sampler
                               per grid: most ILP, for a CTA that has its SM to itself);  2 = compact build (4-point
                               blocks, both grids through one copy: small instruction-cache footprint, for many CTAs
                               per SM in different phases).  Same arithmetic, bit-identical results.        */
    /* teacher forcing (tests): start from a recorded optimiser state instead of a fresh one          */
    const float *m0;        /* [n][9] Adam exp_avg     (NULL = zeros)                                  */
    const float *v0;        /* [n][9] Adam exp_avg_sq  (NULL = zeros)                                  */
    int step0;              /* Adam steps already taken                                                */
    const float *s0;        /* [n][3] prior anchor scales (NULL = the scales in `init`, sq_libs.py:454) */
    /* extra outputs (any may be NULL)                                                                 */
    float *out_m;           /* [n][9]                                                                  */
    float *out_v;           /* [n][9]                                                                  */
    float *out_grad;        /* [n][9]  gradient of the LAST iteration                                  */
    float *out_pred;        /* [SV][4] predicted box sides of the LAST iteration                       */
    int32_t *out_arg;       /* [SV][4] arg-extreme sample index of the LAST iteration (-1 = sentinel)  */
    uint8_t *out_eta_idx;   /* [n][1000] eta-grid index of every sample, LAST iteration                */
    float *out_grids;       /* [n][2][201] eta grid then omega grid, LAST iteration                    */
    float *out_param_hist;  /* [n][n_iters][9] parameters after every step                             */
    int64_t *out_cycles;    /* device-pointer entry only: [n][16] SM cycles per phase as seen by thread 0, summed over iterations
                               (see tools/prof_run.py for the slot names) */
    /* the step that follows the optimiser at the reference's call site (run_multi_view.py:66-67), fused behind it:
       a second launch on the same stream samples the final surfaces and computes their oriented boxes (see
       odam_sq_oriented_boxes) -- one call, one synchronisation, one copy back instead of two                    */
    double *out_corners;    /* [n][8][3] oriented boxes of the optimised objects (NULL = not wanted)             */
    int32_t *out_box_flag;  /* [n] flags of odam_sq_oriented_boxes (may be NULL)                                 */
} odam_sq_options;

int odam_sq_abi_version(void);
const char *odam_sq_error_string(int code);
const char *odam_sq_last_cuda_error(void);

/* Loads the sampler's constant tables (the 2000 uniforms of mt19937(seed=0), sampling.cpp:18-28,169)
 * onto `device` and sizes the kernels' shared memory.  Idempotent; called lazily by every entry point. */
int odam_sq_init(int device);

/* Opt-in objective of odam_sq_optimize_objective[_host], for detections noisier than the reference assumes.  Object i
 * with V views (all of them, as the reference divides) minimises
 *     sum over sides s and views v of  w[v][s] * mask[v][s] * rho(pred[v][s] - box[v][s]) / V   (+ the prior, unchanged)
 * with rho one of
 *     ODAM_SQ_LOSS_L1         |r|  (the reference)
 *     ODAM_SQ_LOSS_SMOOTH_L1  0.5 r^2 / beta if |r| < beta, else |r| - 0.5 beta  (torch's smooth_l1_loss), beta = loss_scale
 *     ODAM_SQ_LOSS_CAUCHY     0.5 c^2 log1p((r / c)^2), rho' = r / (1 + (r / c)^2), c = loss_scale
 * A NaN residual contributes nothing.  Weights are finite and >= 0 and multiply the mask: a side whose w * mask is 0
 * contributes nothing to the loss or the gradient and never raises ODAM_SQ_ST_NO_VALID_PT, exactly as a masked-out side.
 * lr_scale[it] (it = 0 .. n_iters-1 of the call) multiplies both learning rates of iteration it, as a torch scheduler
 * that sets group["lr"] = lr * lr_scale[it]; the bias corrections continue from step0 as before.
 * The kernel build with weights and robust kinds runs only when side_weight != NULL or loss != L1; a schedule alone runs
 * the builds of odam_sq_optimize.  The new build has no cycle-mark twin: out_cycles with it is ODAM_SQ_ERR_ARG. */
#define ODAM_SQ_LOSS_L1 0
#define ODAM_SQ_LOSS_SMOOTH_L1 1
#define ODAM_SQ_LOSS_CAUCHY 2
typedef struct odam_sq_objective {
    const float *side_weight;  /* [SV][4] per-side weights; NULL = 1.  DEVICE memory for odam_sq_optimize_objective,
                                  which does not validate them (as for cls); HOST memory for the _host entry, which
                                  rejects negative or non-finite weights                                          */
    int loss;                  /* ODAM_SQ_LOSS_*                                                                    */
    float loss_scale;          /* beta / c in pixels, finite and > 0 for the robust kinds; ignored for L1           */
    const float *lr_scale;     /* HOST [n_iters] finite, >= 0 multipliers of both learning rates; NULL = constant   */
} odam_sq_objective;

/* SuperQuadricOptimizer.run for n objects at once (sq_libs.py:432-475).  Device pointers. */
int odam_sq_optimize(const float *init, const int32_t *cls, const int32_t *view_off,
                     const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                     int n, int n_iters, int representation, float lr, float lr_shape,
                     float *out_params, float *out_loss, int32_t *out_status,
                     const odam_sq_options *opt, void *stream);

/* Same, HOST pointers; total_views = view_off[n].  This is what the Python drop-in calls. */
int odam_sq_optimize_host(const float *init, const int32_t *cls, const int32_t *view_off,
                          const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                          int n, int n_iters, int representation, float lr, float lr_shape,
                          float *out_params, float *out_loss, int32_t *out_status,
                          const odam_sq_options *opt, int device);

/* odam_sq_optimize[_host] with the objective above; obj == NULL is exactly the entry without it.  Besides the checks of
 * odam_sq_optimize[_host], ODAM_SQ_ERR_ARG (before any CUDA call) for an unknown loss, a robust kind without a finite
 * loss_scale > 0, a negative or non-finite lr_scale entry, opt->out_cycles with the weighted/robust build, and at the
 * _host entry a negative or non-finite weight. */
int odam_sq_optimize_objective(const float *init, const int32_t *cls, const int32_t *view_off,
                               const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                               int n, int n_iters, int representation, float lr, float lr_shape,
                               float *out_params, float *out_loss, int32_t *out_status,
                               const odam_sq_objective *obj, const odam_sq_options *opt, void *stream);
int odam_sq_optimize_objective_host(const float *init, const int32_t *cls, const int32_t *view_off,
                                    const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                                    int n, int n_iters, int representation, float lr, float lr_shape,
                                    float *out_params, float *out_loss, int32_t *out_status,
                                    const odam_sq_objective *obj, const odam_sq_options *opt, int device);

/* Opt-in early stopping of odam_sq_optimize_converge[_host]: each object stops once its loss stops improving, and may
 * return its lowest-loss iterate instead of the last one.
 *
 * The rule is per object.  L[k] is the loss before step k, the value written to out_loss.  keep is
 * (float)(1.0 - (double)rel_tol), computed on the host.  All comparisons are in fp32.
 *
 *     best = +inf; b = -1; last = 0
 *     for k in 0 .. n_iters-1:
 *         (iteration k: loss L[k] at the current params, then the Adam step)
 *         if isfinite(L[k]):
 *             if b < 0 or L[k] < best * keep:  last = k       # a significant improvement (fp32 product, round to nearest)
 *             if b < 0 or L[k] < best:         best = L[k]; b = k   # strict: first index on ties
 *         if patience > 0 and k - last >= patience:  stop; iters = k + 1
 *
 * Outputs of an object that stopped: out_loss[iters:] and the rows out_param_hist[iters:] are NaN.  out_params holds
 * the parameters after step iters - 1; with keep_best, those at which L[b] was evaluated instead (init when b = 0, else
 * the parameters after step b - 1; the last ones when no loss was finite).  out_m, out_v and out_grad describe the
 * last step run, and out_corners the boxes of whatever out_params holds.  The status flags keep their meaning;
 * out_iters < n_iters is the signal that an object stopped.
 * Until an object stops, it runs the arithmetic of odam_sq_optimize_objective: with patience = 0 and keep_best = 0
 * every output equals that entry's.  The kernel build with the rule has no cycle-mark twin. */
typedef struct odam_sq_convergence {
    int patience;            /* 0 = never stop early; else stop after `patience` iterations without improvement   */
    float rel_tol;           /* finite, 0 <= rel_tol < 1                                                          */
    int keep_best;           /* 1: out_params = the parameters at which the lowest loss was evaluated               */
    int32_t *out_iters;      /* [n] iterations run (may be NULL)                                                  */
    int32_t *out_best_iter;  /* [n] iteration of the lowest finite loss, -1 if none (may be NULL)                  */
} odam_sq_convergence;

/* odam_sq_optimize_objective[_host] with the convergence rule above; conv == NULL is exactly that entry, and obj ==
 * NULL means the reference's objective.  out_iters and out_best_iter are device pointers for odam_sq_optimize_converge
 * and host pointers for the _host entry, as the other outputs.  Besides the checks of odam_sq_optimize_objective
 * [_host], ODAM_SQ_ERR_ARG (before any CUDA call) for patience < 0, a rel_tol that is not finite or outside [0, 1),
 * keep_best other than 0 or 1, and conv together with opt->out_pred, out_arg, out_eta_idx, out_grids or out_cycles:
 * those describe the last iteration, which the kernel only knows once it has run it. */
int odam_sq_optimize_converge(const float *init, const int32_t *cls, const int32_t *view_off,
                              const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                              int n, int n_iters, int representation, float lr, float lr_shape,
                              float *out_params, float *out_loss, int32_t *out_status,
                              const odam_sq_objective *obj, const odam_sq_convergence *conv,
                              const odam_sq_options *opt, void *stream);
int odam_sq_optimize_converge_host(const float *init, const int32_t *cls, const int32_t *view_off,
                                   const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                                   int n, int n_iters, int representation, float lr, float lr_shape,
                                   float *out_params, float *out_loss, int32_t *out_status,
                                   const odam_sq_objective *obj, const odam_sq_convergence *conv,
                                   const odam_sq_options *opt, int device);

/* Opt-in step reduction on a plateau for odam_sq_optimize_plateau[_host], as torch's ReduceLROnPlateau but per object:
 * when the rule of odam_sq_convergence runs out of patience, the object's learning rates shrink by `factor` and the
 * window restarts; only after R = max_reductions reductions does it stop.
 *
 * patience and rel_tol are those of odam_sq_convergence, keep as there, and all comparisons are in fp32:
 *
 *     best = +inf; b = -1; last = 0; r = 0
 *     for k in 0 .. n_iters-1:
 *         (iteration k at level r: loss L[k] at the current params, then the Adam step with both learning rates
 *          scaled by s_r[k])
 *         if isfinite(L[k]):
 *             if b < 0 or L[k] < best * keep:  last = k            # as odam_sq_convergence, fp32
 *             if b < 0 or L[k] < best:         best = L[k]; b = k
 *         if k - last >= patience:
 *             if r < R:  r += 1; last = k; reduce_iter[r-1] = k + 1   # the new level applies from iteration k+1
 *             else:      stop; iters = k + 1
 *
 * best is not reset by a reduction, and the Adam step count and moments carry on unchanged.  The scale of level r is
 * f_r = (float)pow((double)factor, r) (f_0 = 1), computed on the host, and s_r[k] = lr_scale[k] * f_r, an fp32
 * product rounded to nearest (f_r when obj->lr_scale is NULL).  Iteration k at level r takes the Adam step sizes that
 * odam_sq_optimize_objective takes for a schedule whose entry k is s_r[k]: an object re-run through that entry with
 * lr_scale'[k] = s_{r(k)}[k], the scale it actually saw, reproduces its run bit for bit.  With R = 0 this is the rule
 * of odam_sq_convergence.  The outputs of an object that stopped are those of odam_sq_convergence. */
typedef struct odam_sq_plateau {
    int max_reductions;         /* R: 1 .. 8                                                                       */
    float factor;               /* finite, 0 < factor < 1: each reduction multiplies both learning rates by it       */
    int32_t *out_reductions;    /* [n] reductions taken (may be NULL)                                              */
    int32_t *out_reduce_iter;   /* [n][R] k + 1 of each reduction taken (its first iteration at the new level), -1
                                   for those not taken (may be NULL)                                               */
} odam_sq_plateau;

/* odam_sq_optimize_converge[_host] with the step reduction above; plat == NULL is exactly that entry.  out_reductions
 * and out_reduce_iter are device pointers for odam_sq_optimize_plateau and host pointers for the _host entry.  Besides
 * the checks of odam_sq_optimize_converge[_host], ODAM_SQ_ERR_ARG (before any CUDA call) for plat with conv == NULL or
 * conv->patience == 0, max_reductions outside 1 .. 8, and a factor that is not finite or outside (0, 1). */
int odam_sq_optimize_plateau(const float *init, const int32_t *cls, const int32_t *view_off,
                             const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                             int n, int n_iters, int representation, float lr, float lr_shape,
                             float *out_params, float *out_loss, int32_t *out_status,
                             const odam_sq_objective *obj, const odam_sq_convergence *conv,
                             const odam_sq_plateau *plat, const odam_sq_options *opt, void *stream);
int odam_sq_optimize_plateau_host(const float *init, const int32_t *cls, const int32_t *view_off,
                                  const float *Ms, const float *box, const uint8_t *mask, const float *prior,
                                  int n, int n_iters, int representation, float lr, float lr_shape,
                                  float *out_params, float *out_loss, int32_t *out_status,
                                  const odam_sq_objective *obj, const odam_sq_convergence *conv,
                                  const odam_sq_plateau *plat, const odam_sq_options *opt, int device);

/* compute_ellipsoid_points (sq_libs.py:577-595): params[n][9] -> xyz[n][1000][3] world points. */
int odam_sq_sample_points(const float *params, int n, float *out_xyz, void *stream);
int odam_sq_sample_points_host(const float *params, int n, float *out_xyz, int device);

/* get_bbox (sq_libs.py:547-554) for every (object, view): out_box[SV][4] = x_min,x_max,y_min,y_max of the
 * projected samples (no validity test, plain division by z, as the reference does there). */
int odam_sq_project_boxes(const float *params, const int32_t *view_off, const float *Ms, int n,
                          float *out_box, void *stream);
int odam_sq_project_boxes_host(const float *params, const int32_t *view_off, const float *Ms, int n,
                               float *out_box, int device);

/* Differentiable ops (odam_b200/autograd.py): forward and vector-Jacobian products of the surface samples and of the
 * projected box sides, so that the optimiser's maths can be composed with other loss terms, optimisers or schedules.
 * Device pointers only.  Each kernel re-runs the sampler from params (nothing is saved between forward and backward);
 * every reduction has a fixed order, so results do not depend on the batch an object is launched in.  Each object's
 * views [view_off[i], view_off[i+1]) are clamped to [0, total_views] on the device.  odam_sq_box_sides_vjp treats the
 * camera matrices as constants; odam_sq_box_sides_vjp_cameras also returns the gradient with respect to Ms.
 *
 * odam_sq_sample_points_vjp: grad_xyz[n][1000][3] (dL/d of odam_sq_sample_points' output) -> out_grad_params[n][9].
 * odam_sq_box_sides: constraint_2d (sq_libs.py:397-413) for every (object, view): out_pred[SV][4] = x_min, x_max, y_min,
 *   y_max over the samples of valid ? q / (|q_z| + 1e-6) : +-1e6 with valid = q_z > 0.5 (first index on ties, NaN
 *   propagates as in torch.min/max); out_arg[SV][4] = the winning sample, -1 when a sentinel won.
 * odam_sq_box_sides_vjp: grad_pred[SV][4] and the arg of odam_sq_box_sides -> out_grad_params[n][9]; sides with
 *   arg < 0 contribute nothing.
 * odam_sq_box_sides_vjp_cameras: the same, plus out_grad_Ms[SV][12] = dL/dMs (row-major 3 x 4 per view), computed in the
 *   same launch.  out_grad_params may be NULL (camera-only refinement); out_grad_Ms is required.  A view's row sums its
 *   sides in the order x_min, x_max, y_min, y_max with one writer and no atomics, so it is bit-reproducible and
 *   independent of the batch; out_grad_params has the bits odam_sq_box_sides_vjp gives.  Rows that no object's clamped
 *   view range covers are not written (callers zero the buffer).  NaN or Inf in grad_pred reach only their own view's
 *   row. */
int odam_sq_sample_points_vjp(const float *params, const float *grad_xyz, int n, float *out_grad_params, void *stream);
int odam_sq_box_sides(const float *params, const int32_t *view_off, const float *Ms, int n, int total_views,
                      float *out_pred, int32_t *out_arg, void *stream);
int odam_sq_box_sides_vjp(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                          const float *grad_pred, int n, int total_views, float *out_grad_params, void *stream);
int odam_sq_box_sides_vjp_cameras(const float *params, const int32_t *view_off, const float *Ms, const int32_t *arg,
                                  const float *grad_pred, int n, int total_views, float *out_grad_params,
                                  float *out_grad_Ms, void *stream);

/* compute_ellipsoid_points + compute_oriented_bbox (src/scripts/run_multi_view.py:66-67, src/utils/box_utils.py:319-410):
 * params[n][9] -> out_corners[n][8][3] DOUBLE, the oriented box of each object's 1000 surface points: min-area rectangle
 * of the xy convex hull over the directions of the hull edges, upper four corners (z_max) first, then the same four at
 * z_min.  The reference takes its hull from scipy/Qhull and skips the hull's closing edge; the kernel builds the hull
 * itself (gift wrapping, exact orientation tests) and reproduces Qhull's vertex order (see csrc/sq_postproc.cuh).
 * out_flag[n] (may be NULL): 0 = ok, bit 0 = Qhull's vertex order could not be predicted with certainty (degenerate
 * extreme points), bit 1 = fewer than 3 hull vertices.  out_xyz (may be NULL): the surface points [n][1000][3] float. */
int odam_sq_oriented_boxes(const float *params, int n, double *out_corners, int32_t *out_flag, float *out_xyz,
                           void *stream);
int odam_sq_oriented_boxes_host(const float *params, int n, double *out_corners, int32_t *out_flag, float *out_xyz,
                                int device);
/* compute_oriented_bbox of arbitrary point sets: points[n][n_pts][3] float32 (n_pts <= 1024), HOST pointers. */
int odam_sq_oriented_boxes_of_points_host(const float *points, int n, int n_pts, double *out_corners,
                                          int32_t *out_flag, int device);

/* The pair costs of merge_process (src/scripts/run_merge.py:79-122) between the two optimisation passes:
 * boxes[n][8][3] double (bboxes_qc), cls[n] class ids (NULL = every pair may merge) ->
 * out_cost[n][n] = 1 - box3d_iou(box_i, box_j)[0] (src/utils/box_utils.py:97-120) where the classes allow a merge (equal,
 * or both in {4, 5}), else 1; symmetric, zero diagonal -- i.e. cost_mat after `cost_mat += cost_mat.T`.
 * out_iou3d / out_iou2d [n][n] (any may be NULL): the raw IoU values for i < j.  HOST pointers; one thread per pair.
 * Identical or edge-sharing rectangles make the reference's clipper divide by zero and raise; here such a pair
 * yields NaN. */
int odam_sq_merge_cost_host(const double *boxes, const int32_t *cls, int n, double *out_cost, double *out_iou3d,
                            double *out_iou2d, int device);

/* Drop-in for the reference's own native entry point, fast_sampler/sampling.hpp:5-15
 *   void sample_on_batch(float *shapes, float *epsilons, float *etas, float *omegas, int B, int M, int N,
 *                        int buffer_size, int seed)
 * as bound by _sampler.pyx:413-441 (N = 1000, buffer_size = 201, seed = 0 are the only values that path uses;
 * anything else is ODAM_SQ_ERR_ARG).  shapes[B][M][3], epsilons[B][M][2] -> etas, omegas [B][M][N]; HOST pointers.
 * As in the reference, ONE generator is seeded per call and keeps drawing across the B*M primitives
 * (sampling.cpp:169-214): primitive p sees uniforms [2000p, 2000p + 2000) of mt19937(seed). */
int odam_sq_sample_on_batch_host(const float *shapes, const float *epsilons, float *etas, float *omegas,
                                 int B, int M, int N, int buffer_size, int seed, int device);

/* Roofline probe: measured FP32 FMA throughput of `device` (dense independent FFMA chains, no memory traffic),
 * in TFLOP/s counting an FMA as 2 flop.  Best of 4 timed launches after one warm-up. */
int odam_sq_fma_peak(int device, double *tflops);

/* Device self-test: the kernels' split IEEE-754 division (one refined reciprocal shared by several quotients) against
 * the compiler's __fdiv_rn on n random operand pairs; *mismatches must come back 0. */
int odam_sq_selftest(int device, uint32_t seed, long long n, long long *mismatches);

/* The launch configuration odam_sq_optimize would use (for benchmarks/logging). */
int odam_sq_query_launch(const int32_t *view_off_host, int n, const odam_sq_options *opt,
                         int *threads, int *smem_bytes, int *ctas_per_sm, int *cluster, int *code_layout,
                         int *max_slices);

/* Host-side staging of the reference's call site (src/scripts/run_multi_view.py:31-58; load_pred_object,
 * src/utils/tracking_gt_utils.py:145-211, averaging_T_wos :59-66, the 20 px border rule of
 * src/super_quadric/quadric_helper.py:87-107) for all tracks of a call, in native code: no CUDA, callable without a GPU.
 * tracks[i] points to track i's rows (double, row_stride doubles apart, the 82-column layout of processor.py:98-108;
 * columns 0 frame id, 1 class, 2..5 box x_min y_min x_max y_max, 6..8 dims, 9..11 centre, 12 yaw are read),
 * rows_per[i] is its row count, frame_ids[n_frames] the frames of this call.  Per track: cls = int(median(class)),
 * t_wo[3] = mean centre over all rows, yaw = chordal mean of the yaws of the frames present (first row per frame),
 * dims[3] = their mean, n_present = their count; and CSR-packed per usable frame (at least one box side farther than
 * 20 px from the image border): view_off[n+1], frame_idx (index into frame_ids), box [.][4] / mask [.][4] in the
 * order x_min, x_max, y_min, y_max (absent sides 0) -- sized by the caller for sum(rows_per) entries. */
int odam_sq_stage_tracks_host(const double *const *tracks, const int64_t *rows_per, int n, int row_stride,
                              const int64_t *frame_ids, int n_frames, int img_h, int img_w,
                              int32_t *cls, double *t_wo, double *yaw, double *dims, int32_t *view_off,
                              int64_t *frame_idx, float *box, uint8_t *mask, int64_t *n_present);

/* How many objects can get a view-tiled cluster of `cluster` CTAs (2..4) with every CTA alone on its SM of `device`
 * (cudaOccupancyMaxActiveClusters; a cluster must fit one GPC, so this is less than SMs / cluster: 45 x 3 and 32 x 4
 * on a 148-SM B200).  The automatic launch configuration only picks a cluster size while the objects fit. */
int odam_sq_cluster_capacity(int device, int cluster, int *objects);

#ifdef __cplusplus
}
#endif
#endif /* ODAM_SQ_H_ */
