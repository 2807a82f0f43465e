"""A float32 numpy restatement of the fused optimiser's step reduction on a plateau (odam_sq_plateau,
include/odam_sq.h), for the tests to apply to a run's loss curve, and the schedule an object ran under, for the tests
to replay it.  The early-stopping rule it extends is tests/convergence_rule.py."""
import numpy as np

from convergence_rule import keep_factor


def plateau_rule(loss, patience, rel_tol, R):
    """(iters, b, reduce_iter) of the step-reduction rule (odam_sq_plateau) for one object whose losses before each
    step are loss[k]: stop_rule's answers, where the first R times the patience runs out the object reduces its step
    instead of stopping.  reduce_iter[j] = k + 1 of reduction j, -1 if not taken."""
    loss = np.asarray(loss, np.float32)
    keep = keep_factor(rel_tol)
    best, b, last, reduce_iter = np.float32(np.inf), -1, 0, []
    for k, L in enumerate(loss):
        if np.isfinite(L):
            if b < 0 or L < np.float32(best * keep):
                last = k
            if b < 0 or L < best:
                best, b = L, k
        if patience > 0 and k - last >= patience:
            if len(reduce_iter) < R:
                reduce_iter.append(k + 1)
                last = k
            else:
                return k + 1, b, reduce_iter + [-1] * (R - len(reduce_iter))
    return len(loss), b, reduce_iter + [-1] * (R - len(reduce_iter))


def lr_scale_seen(reduce_iter, factor, n_iters, lr_scale=None):
    """The schedule an object with these reductions actually ran under: s_r(k)[k] = lr_scale[k] * f_r(k) in float32,
    f_r = (float)factor^r, r(k) the reductions taken at or before iteration k (include/odam_sq.h)."""
    base = np.ones(n_iters, np.float32) if lr_scale is None else np.asarray(lr_scale, np.float32)
    r = np.zeros(n_iters, np.int64)
    for it in reduce_iter:
        if it >= 0:
            r[it:] += 1
    fd = float(np.float32(factor))   # the float the library is given, then pow in double as on the host
    f = np.array([np.float32(fd ** j) for j in range(int(r.max()) + 1)], np.float32)
    return (base * f[r]).astype(np.float32)
