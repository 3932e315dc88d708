"""The outer Picard / Gauss-Newton loop every non-linear driver runs (control/control.py:630-800, 1203-1486,
3377-3590, 4886-5219): its stop rule and its output, written once."""

__all__ = ["picard"]


def picard(residual, step, history, *, max_iter, rel_tol, abs_tol, verbose):
    """Iterate until the residual norm falls to ``rel_tol`` times the first one or to ``abs_tol``, or ``max_iter``
    outer iterations ran.  ``residual()`` evaluates the residual at the current iterate and returns its norm;
    ``step()`` solves for one increment and updates the iterate.  Every norm is appended to ``history`` as it is
    computed, so a loop that raises part-way leaves what it reached there.  Returns the number of steps taken."""
    norm_0 = residual()
    history.append(norm_0)
    if verbose:
        print(f"Initial non-linear residual: {norm_0:.16e}")
    norm_k, k = norm_0, 0
    while norm_k > rel_tol * norm_0 and norm_k > abs_tol:
        step()
        norm_k = residual()
        k += 1
        history.append(norm_k)
        if verbose:
            print(f"Non-linear solver: iteration {k:d}, non-linear residual norm {norm_k:.16e}")
        if k + 1 > max_iter:
            break
    return k
