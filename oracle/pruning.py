"""Policy target pruning (Wu 2019, "Accelerating Self-Play Learning in Go",
section 3.2) in numpy.  TEST INFRASTRUCTURE ONLY: the reference that
``az_play_commit`` must reproduce bit for bit (az_engine_set_forced_playouts).

Every operation is one float32 operation with round-to-nearest, in the order
of the engine's k_select, so the results are exact, not approximate.
"""
import numpy as np

f32 = np.float32


def forced_visits(k, prior, sum_n):
    """n_forced = sqrt((k * P) * sum N), float32, one rounding per operation."""
    return np.sqrt((f32(k) * f32(prior)) * f32(sum_n))


def prune_score(n_real, w, prior, sq, coef, n):
    """The PUCT score of a root child with ``n`` visits: Q from its real
    visits ``n_real`` (0 when W is 0, as in k_select's shortcut) plus
    (coef * P) * (sqrt(sum N) / (1 + n))."""
    q = f32(0.0) if f32(w) == 0 else (-f32(w)) / max(f32(n_real), f32(1.0))
    return q + (f32(coef) * f32(prior)) * (f32(sq) / (f32(1.0) + f32(n)))


def prune_visits(visits, total_value, prior, coef, k):
    """Pruned visit counts of one root (float32 [k], as ``root_stats``).

    c* is the most-visited child (lowest ordinal on ties) and keeps its
    count.  Every other visited child keeps the fewest n whose score is still
    below score(c*, N*), but at least N - floor(n_forced) and at most N; a
    child left at 1 gets 0.  The score falls with n, so a scan from
    N - floor(n_forced) upwards finds the same n as the engine's bisection.
    """
    v = np.asarray(visits, dtype=f32)
    w = np.asarray(total_value, dtype=f32)
    p = np.asarray(prior, dtype=f32)
    out = v.copy()
    if len(v) == 0 or v.max() == 0:
        return out
    best = int(np.argmax(v))
    sum_n = f32(int(v.astype(np.int64).sum()))
    sq = np.sqrt(sum_n)
    s_best = prune_score(v[best], w[best], p[best], sq, coef, v[best])
    for j in range(len(v)):
        n = int(v[j])
        if j == best or n == 0:
            continue
        d = np.floor(forced_visits(k, p[j], sum_n))
        m = 0 if d >= n else n - int(d)
        while m < n and not prune_score(v[j], w[j], p[j], sq, coef, m) < s_best:
            m += 1
        out[j] = 0 if m == 1 else m
    return out
