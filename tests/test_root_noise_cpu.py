"""Dirichlet root noise without a GPU: the oracle's noised select (forced.c)
against the plain oracle and against numpy's PUCT argmax, and the noise
statistics of oracle.dirichlet_stats held to samples of known law."""
import numpy as np
import pytest

import oracle
from oracle import dirichlet_stats as ds
from oracle import forced


def _state(tree):
    v, w, p = tree.root_stats()
    return v.tobytes(), w.tobytes(), p.tobytes(), tree.root_node(), tree.num_nodes


@pytest.mark.parametrize('n,sims,batch,mode', [(5, 60, 6, 2), (9, 100, 8, 1), (5, 30, 1, 0),
                                               (3, 20, 16, 2), (11, 80, 10, 2)])
def test_no_noise_is_the_oracle(n, sims, batch, mode):
    """eps = 0 with noise given, and noise None with eps != 0, are the
    oracle's own search, and forced.sample_paths_stub's at forced_k = 2,
    bit for bit, with tree reuse."""
    rng = np.random.default_rng(n * 1000 + sims)
    games = [oracle.Hex(n) for _ in range(6)]
    trees = [oracle.Tree(max_nodes=400_000) for _ in range(6)]
    rows = (sims // batch + 1) * batch
    for ply in range(5):
        k = n * n - ply
        eta = rng.dirichlet(np.full(k, 0.3), size=rows).astype(np.float32)
        sv = [trees[0].sample_paths_stub(games[0], sims, batch, 0.5, mode),
              forced.sample_paths_stub_noise(trees[1], games[1], sims, batch, 0.5, mode, 0.0, 0.0, eta),
              forced.sample_paths_stub_noise(trees[2], games[2], sims, batch, 0.5, mode, 0.0, 0.25, None),
              forced.sample_paths_stub(trees[3], games[3], sims, batch, 0.5, mode, 2.0),
              forced.sample_paths_stub_noise(trees[4], games[4], sims, batch, 0.5, mode, 2.0, 0.0, eta),
              forced.sample_paths_stub_noise(trees[5], games[5], sims, batch, 0.5, mode, 2.0, 0.25, None)]
        for a, b in ((0, 1), (0, 2), (3, 4), (3, 5)):
            assert _state(trees[a]) == _state(trees[b]) and sv[a] == sv[b], (ply, a, b)
        move_id = int(np.argmax(trees[0].root_stats()[0]))
        move = games[0].legal_moves()[move_id]
        for t, g in zip(trees, games):
            t.move(move_id)
            g.step(int(move))
    if n == 3:
        return                  # (2 x 16 descents visit a 3x3 tree alike whatever the priors)
    # and the noise does change the search
    g, t = oracle.Hex(n), oracle.Tree(max_nodes=400_000)
    eta = rng.dirichlet(np.full(n * n, 0.3), size=rows).astype(np.float32)
    forced.sample_paths_stub_noise(t, g, sims, batch, 0.5, mode, 0.0, 0.25, eta)
    ref = oracle.Tree(max_nodes=400_000)
    ref.sample_paths_stub(oracle.Hex(n), sims, batch, 0.5, mode)
    assert _state(t) != _state(ref)


def _random_root(n, rng):
    """An oracle tree of an empty n x n board whose root children carry
    random N, W and P."""
    game = oracle.Hex(n)
    tree = oracle.Tree(max_nodes=100_000)
    tree.root_leaf(game)
    k = n * n
    p = rng.dirichlet(np.full(k, rng.choice([0.1, 1.0]))).astype(np.float32)
    tree.expand_root(p)
    t = tree.t.contents
    fc = t.first_child[tree.root_id]
    nv = (rng.integers(0, 20, k) * (rng.random(k) < 0.6)).astype(np.float32)
    w = np.round((rng.random(k) * 2 - 1) * nv).astype(np.float32)
    for j in range(k):
        t.num_visits[fc + j] = nv[j]
        t.total_value[fc + j] = w[j]
    t.num_visits[tree.root_id] = float(nv.sum())
    return game, tree, fc, nv, w, p


def numpy_puct_argmax(nv, w, p_mixed, coef):
    """mcts.py:132-136 in float32, one rounding per operation, np.argmax."""
    f = np.float32
    sq = np.sqrt(f(nv.astype(np.float64).sum()))
    gap = sq / (f(1) + nv)
    u = (f(coef) * p_mixed) * gap
    q = (-w) / np.maximum(nv, f(1))
    return int(np.argmax(q + u))


def test_noised_root_descends_into_the_numpy_argmax():
    """Batch 1 on random small roots: the oracle descends into numpy's
    argmax of the fp32 PUCT score with P' = (float)((1 - eps) P + eps eta)
    mixed in float64; with noise dominant, the pick follows the noise."""
    rng = np.random.default_rng(3)
    differ = 0
    for trial in range(400):
        n = int(rng.integers(2, 6))
        eps = float(rng.choice([0.25, 0.5, 1.0, 0.1]))
        coef = float(rng.choice([0.5, 1.25, 2.0, 4.0]))
        game, tree, fc, nv, w, p = _random_root(n, rng)
        if nv.sum() == 0:
            continue
        eta = rng.dirichlet(np.full(len(p), float(rng.choice([0.03, 0.3, 1.0])))).astype(np.float32)
        pm = ((1.0 - eps) * p.astype(np.float64) + eps * eta.astype(np.float64)).astype(np.float32)
        want = numpy_puct_argmax(nv, w, pm, coef)
        got = forced.select_batch_noise(tree, game, 1, coef, 0.0, eps, eta[None])[0]['node'] - fc
        assert got == want, trial
        differ += want != numpy_puct_argmax(nv, w, p, coef)
    assert differ > 50, differ


def _root_2x2(prior, visits, values):
    game = oracle.Hex(2)
    tree = oracle.Tree(max_nodes=1000)
    tree.root_leaf(game)
    tree.expand_root(np.array(prior, np.float32))
    t = tree.t.contents
    fc = t.first_child[tree.root_id]
    for j in range(4):
        t.num_visits[fc + j] = visits[j]
        t.total_value[fc + j] = values[j]
    t.num_visits[tree.root_id] = float(sum(visits))
    return game, tree, fc


def test_forcing_uses_the_stored_prior():
    """n_forced = sqrt(k P sum N) takes the stored P, not the noised one
    (k = 2, sum N = 14, eps = 1, c = 0.01)."""
    # child 1: N = 2, Q = -1.  Stored P = 0.01: n_forced = 0.53, not forced, and PUCT
    # takes child 0; the noised P' = 1 would have forced it (n_forced = 5.3)
    game, tree, fc = _root_2x2([0.97, 0.01, 0.01, 0.01], [12, 2, 0, 0], [0, 2, 0, 0])
    eta = np.array([[0.0, 1.0, 0.0, 0.0]], np.float32)
    assert forced.select_batch_noise(tree, game, 1, 0.01, 2.0, 1.0, eta)[0]['node'] == fc
    # stored P = 0.5 forces child 1 (n_forced = 3.7 > 2), though P' = 0 would not and
    # PUCT alone takes child 0
    game, tree, fc = _root_2x2([0.4, 0.5, 0.05, 0.05], [12, 2, 0, 0], [0, 0, 0, 0])
    eta = np.array([[1.0, 0.0, 0.0, 0.0]], np.float32)
    assert forced.select_batch_noise(tree, game, 1, 0.01, 0.0, 1.0, eta)[0]['node'] == fc
    assert forced.select_batch_noise(tree, game, 1, 0.01, 2.0, 1.0, eta)[0]['node'] == fc + 1


def test_noise_rows_follow_the_descents():
    """Descent i of a batch uses row i: a batch whose rows each point at a
    different child visits exactly those children."""
    n = 3
    game = oracle.Hex(n)
    tree = oracle.Tree(max_nodes=1000)
    tree.root_leaf(game)
    tree.expand_root(np.full(9, 1 / 9, np.float32))
    t = tree.t.contents
    fc = t.first_child[tree.root_id]
    for j in range(9):
        t.num_visits[fc + j] = 1.0
    t.num_visits[tree.root_id] = 9.0
    order = [4, 7, 1, 8, 0]
    eta = np.zeros((5, 9), np.float32)
    eta[np.arange(5), order] = 1.0
    leaves = forced.select_batch_noise(tree, game, 5, 2.0, 0.0, 1.0, eta)
    assert [lv['node'] - fc for lv in leaves] == order


@pytest.mark.parametrize('alpha,k', ds.CASES)
def test_noise_statistics_self_check(alpha, k):
    """The statistics the device noise is held to, at the sizes the GPU test
    uses, accept RandomState.dirichlet(alpha) and reject dirichlet(1.05
    alpha) and, where there is a child j + 32, a sampler whose children j and
    j + 32 share one Gamma draw."""
    S, G = ds.num_sims(k), ds.GAMES
    rows = S * G
    assert rows >= ds.MIN_ROWS and rows * k >= ds.MIN_COMPONENTS

    def sample(seed, a):
        return np.random.RandomState(seed).dirichlet(np.full(k, a), size=rows).astype(np.float32)

    good = sample(7, alpha).reshape(S, G, k)
    assert ds.exact_failures(good) == []
    assert ds.failures(ds.report(good, alpha, seed=1)) == []
    bad = ds.failures(ds.report(sample(8, 1.05 * alpha).reshape(S, G, k), alpha, seed=1))
    assert any(f.startswith('marginal KS') for f in bad), bad
    js = np.array([j for j in range(k - 32) if (j // 32) % 2 == 0], np.int64)
    if len(js):
        g = np.random.RandomState(9).gamma(alpha, size=(rows, k))
        g[:, js + 32] = g[:, js]
        shared = (g / g.sum(1, keepdims=True)).astype(np.float32).reshape(S, G, k)
        bad = ds.failures(ds.report(shared, alpha, seed=1))
        assert any(f.startswith('corr(j, j + 32)') for f in bad), bad


def test_exact_checks():
    ok = np.random.RandomState(0).dirichlet(np.full(50, 0.3), size=100).astype(np.float32)
    assert ds.exact_failures(ok) == []
    nan, neg, off, zero = ok.copy(), ok.copy(), ok.copy(), ok.copy()
    nan[5, 7] = np.nan
    neg[5, 7] = -neg[5, 7]
    off[5] *= np.float32(1.0001)
    zero[3] = 0
    for bad in (nan, neg, off, zero):
        assert ds.exact_failures(bad) != []
