"""Checks that a sample of root-noise vectors has the law of NumPy's
``RandomState.dirichlet(np.full(k, alpha))`` (mcts.py:126-127).  TEST
INFRASTRUCTURE ONLY.

The engine's sampler (az_dirichlet_noise) uses the approximate lg2 / ex2 of
the GPU and cannot be reproduced on the host, so its draws are compared with
NumPy's in law.  A sample is ``draws[S][G][k]``: S simulation counters times
G games, rows = S * G.  The statistics, and the thresholds they are held to:

- marginal: two-sample Kolmogorov-Smirnov over the components against 4x as
  many from ``RandomState(seed).dirichlet``;
- joint law: the same test on the per-row sums of the first m components,
  m = 32 and ceil(k / 2) (where m < k), against Beta(m alpha, (k - m) alpha),
  the law of such a sum by the aggregation property;
- independence: Pearson correlations, within 4 / sqrt(rows) of what
  independent draws give, of child j with child j + 32 (one Philox block)
  against -1 / (k - 1), of one child in games g and g + 1 at one counter
  against 0, and of one child at counters s and s + 1 against 0.

A KS test passes while D <= 1.95 sqrt((n + m) / (n m)).  Both sides are
clipped at 2^-100 first: the device flushes components below about 2^-126
times the row's largest to zero, and NumPy's float64 draws go far lower.
tests/test_root_noise_cpu.py holds these thresholds to a sample of the right
law (accepted), alpha off by 5 % (rejected) and children j and j + 32 sharing
one Gamma draw (rejected), at every (alpha, k) the GPU test uses.
"""
import math

import numpy as np

# (alpha, k) of the device test: production's 0.03 over a 11x11 and a 19x19
# root, the GS retry loop at work (alpha = 1), alpha > 1 with a fraction and
# integer (exponentials only), k < 32 and k = 33 (one child in the second slot)
CASES = ((0.03, 121), (0.03, 361), (0.3, 50), (1.0, 20), (2.5, 361), (2.0, 33), (0.5, 2))
GAMES = 4096
CLIP = 2.0 ** -100
KS_COEF = 1.95
CORR_COEF = 4.0
MIN_ROWS = 1 << 16
MIN_COMPONENTS = 1 << 19
MAX_COMPONENTS = 1 << 21        # marginal KS: a strided subsample beyond this


def num_sims(k, games=GAMES):
    """Simulation counters per game: at least MIN_ROWS rows and
    MIN_COMPONENTS components, an even number."""
    s = max(-(-MIN_ROWS // games), -(-MIN_COMPONENTS // (games * k)))
    return s + (s & 1)


def ks_distance(a, b):
    """Two-sample Kolmogorov-Smirnov statistic sup |F_a - F_b|."""
    a, b = np.sort(np.asarray(a, np.float64).ravel()), np.sort(np.asarray(b, np.float64).ravel())
    x = np.concatenate([a, b])
    fa = np.searchsorted(a, x, side='right') / len(a)
    fb = np.searchsorted(b, x, side='right') / len(b)
    return float(np.abs(fa - fb).max())


def ks_limit(n, m):
    return KS_COEF * math.sqrt((n + m) / (n * m))


def pearson(x, y):
    x = np.asarray(x, np.float64).ravel()
    y = np.asarray(y, np.float64).ravel()
    x, y = x - x.mean(), y - y.mean()
    return float((x * y).sum() / math.sqrt((x * x).sum() * (y * y).sum()))


def exact_failures(draws):
    """What no sample of a Dirichlet may show: a value that is not finite or
    negative, a row of zeros, or a row sum further than k 2^-23 from 1."""
    d = np.asarray(draws, np.float32)
    k = d.shape[-1]
    rows = d.reshape(-1, k)
    out = []
    if not np.isfinite(rows).all():
        out.append('non-finite values')
    elif (rows < 0).any():
        out.append('negative values')
    if not (rows > 0).any(axis=1).all():
        out.append('rows of zeros')
    err = np.abs(rows.astype(np.float64).sum(1) - 1.0).max()
    if not err <= k * 2.0 ** -23:
        out.append('row sum off by %g' % err)
    return out


def report(draws, alpha, seed=0):
    """Every statistic of the module docstring for ``draws[S][G][k]``:
    {name: (value, expected, limit)}; a check fails when
    |value - expected| > limit."""
    d = np.asarray(draws, np.float32)
    S, G, k = d.shape
    rows = S * G
    rs = np.random.RandomState(seed)
    out = {}
    flat = d.reshape(-1)
    step = -(-flat.size // MAX_COMPONENTS)
    dev = np.maximum(flat[::step].astype(np.float64), CLIP)
    m = 4 * dev.size
    ref = rs.dirichlet(np.full(k, alpha), size=-(-m // k)).reshape(-1)[:m]
    out['marginal KS'] = (ks_distance(dev, np.maximum(ref, CLIP)), 0.0, ks_limit(dev.size, m))
    for mm in sorted({32, -(-k // 2)}):
        if mm >= k:
            continue
        sums = np.maximum(d[..., :mm].astype(np.float64).sum(-1).ravel(), CLIP)
        ref = np.maximum(rs.beta(mm * alpha, (k - mm) * alpha, size=4 * rows), CLIP)
        out['KS of sum of first %d' % mm] = (ks_distance(sums, ref), 0.0, ks_limit(rows, 4 * rows))
    tol = CORR_COEF / math.sqrt(rows)
    js = np.array([j for j in range(k - 32) if (j // 32) % 2 == 0], np.int64)
    if len(js):
        out['corr(j, j + 32)'] = (pearson(d[..., js], d[..., js + 32]), -1.0 / (k - 1), tol)
    if k > 1:
        half = G // 2
        out['corr(game g, g + 1)'] = (pearson(d[:, 0:2 * half:2], d[:, 1:2 * half:2]), 0.0, tol)
        half = S // 2
        out['corr(sim s, s + 1)'] = (pearson(d[0:2 * half:2], d[1:2 * half:2]), 0.0, tol)
    return out


def failures(rep):
    """The checks of ``report`` that fail, with their numbers."""
    return ['%s: %.4g (expected %.4g, limit %.3g)' % (name, v, e, lim)
            for name, (v, e, lim) in rep.items() if not abs(v - e) <= lim]
