"""
numpy restatement of the across-member statistics kernels (xanthos_b200/csrc/ensemble_stats.cu), operation for
operation: the library is built without FMA contraction, so the kernels must equal these functions bit for bit.
Test infrastructure only - nothing under xanthos_b200/ imports it.

State: (sum, m2, min, max), float64 arrays of one shape.  `n` counts the members including the one being added.
"""

import numpy as np


def _nan_min(a, x):
    return np.where((x < a) | np.isnan(x), x, a)


def _nan_max(a, x):
    return np.where((x > a) | np.isnan(x), x, a)


def update(state, x, n):
    """Adds member number n (1-based) with values x; n == 1 initialises.  xan_ens_stats_update."""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(invalid='ignore'):
        if n == 1:
            return x.copy(), 0.0 * x, x.copy(), x.copy()
        s, m2, mn, mx = state
        mean_old = s / float(n - 1)
        s = s + x
        mean_new = s / float(n)
        m2 = m2 + (x - mean_old) * (x - mean_new)
        return s, m2, _nan_min(mn, x), _nan_max(mx, x)


def merge(a, na, b, nb):
    """Chan et al.: partial a of na members and partial b of nb members -> partial of na + nb.  xan_ens_stats_merge."""
    sa, m2a, mna, mxa = a
    sb, m2b, mnb, mxb = b
    na, nb = float(na), float(nb)
    n = na + nb
    with np.errstate(invalid='ignore'):
        d = sb / nb - sa / na
        return sa + sb, m2a + m2b + d * d * na * nb / n, _nan_min(mna, mnb), _nan_max(mxa, mxb)


def finalize(state, n, ddof=0):
    """{'mean', 'std', 'min', 'max'} over the n members.  xan_ens_stats_finalize (which also transposes)."""
    s, m2, mn, mx = state
    with np.errstate(invalid='ignore', divide='ignore'):
        return {'mean': s / float(n), 'std': np.sqrt(m2 / float(n - ddof)), 'min': mn.copy(), 'max': mx.copy()}


def run(members, ddof=0):
    """Statistics of a sequence of equally shaped arrays, folded in order."""
    state = None
    for k, x in enumerate(members):
        state = update(state, x, k + 1)
    return finalize(state, len(members), ddof)
