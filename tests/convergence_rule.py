"""A float32 numpy restatement of the fused optimiser's early-stopping rule (odam_sq_convergence, include/odam_sq.h),
for the tests to apply to a full run's loss curve."""
import numpy as np


def keep_factor(rel_tol):
    """(float)(1.0 - (double)rel_tol), as the library computes it on the host."""
    return np.float32(1.0 - float(np.float32(rel_tol)))


def stop_rule(loss, patience, rel_tol):
    """(iters, b) of one object whose losses before each step are loss[k]: the iterations the rule runs, and the
    iteration of the lowest finite loss among them (-1 if none; the first on ties).  Comparisons in float32."""
    loss = np.asarray(loss, np.float32)
    keep = keep_factor(rel_tol)
    best, b, last = np.float32(np.inf), -1, 0
    for k, L in enumerate(loss):
        if np.isfinite(L):
            if b < 0 or L < np.float32(best * keep):
                last = k
            if b < 0 or L < best:
                best, b = L, k
        if patience > 0 and k - last >= patience:
            return k + 1, b
    return len(loss), b
