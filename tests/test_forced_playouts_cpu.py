"""Forced playouts and policy target pruning without a GPU: argument
validation, the oracle's forced rule on hand-built roots, the numpy pruning
reference, the C ABI surface and train()'s config plumbing."""
import math

import numpy as np
import pytest

import oracle
from oracle import forced
from oracle.pruning import forced_visits, prune_score, prune_visits

f32 = np.float32


def test_forced_playouts_setting():
    from azalea_b200.selfplay import forced_playouts_setting
    assert forced_playouts_setting(0, 0.5) == 0.0
    assert forced_playouts_setting(2, 0.5) == 2.0
    assert forced_playouts_setting(0.5, 0.0) == 0.5


@pytest.mark.parametrize('k,coef', [(-1.0, 0.5), (math.nan, 0.5), (math.inf, 0.5), (2.0, -0.1),
                                    (2.0, math.nan), (2.0, math.inf)])
def test_invalid_forced_playouts_arguments(k, coef):
    from azalea_b200.selfplay import LockstepSelfPlay, forced_playouts_setting
    with pytest.raises(ValueError):
        forced_playouts_setting(k, coef)
    # rejected before anything touches a device
    with pytest.raises(ValueError):
        LockstepSelfPlay(None, num_games=8, board_size=5, simulations=800, search_batch_size=10,
                         exploration_coef=coef, forced_playouts_k=k)


def test_random_play_ignores_forced_playouts():
    from azalea_b200.selfplay import LockstepSelfPlay
    try:
        LockstepSelfPlay(None, num_games=8, board_size=5, random_play=True, forced_playouts_k=-1.0)
    except ValueError:
        pytest.fail('random_play validated the forced-playouts setting')
    except Exception:
        pass                    # (no CUDA device here)


def test_abi_surface():
    from azalea_b200 import _cabi
    assert 'az_engine_set_forced_playouts' in _cabi.declared_symbols()
    assert len(_cabi.COUNTER_NAMES) == 16


# --------------------------------------------------------- the forced rule --

def _root_with_visits(n, visits, batch=4):
    """An oracle tree of an empty n x n board whose root children carry the
    given visits (W = 0), uniform priors."""
    game = oracle.Hex(n)
    tree = oracle.Tree(max_nodes=100_000)
    tree.root_leaf(game)
    k = n * n
    tree.expand_root(np.full(k, 1.0 / k, np.float32))
    t = tree.t.contents
    fc = t.first_child[tree.root_id]
    for j, v in enumerate(visits):
        t.num_visits[fc + j] = v
    t.num_visits[tree.root_id] = float(sum(visits))
    return game, tree, fc


def test_huge_k_forces_visited_children_in_ordinal_order():
    """With k huge every visited child is below n_forced and is descended
    into, lowest ordinal first (a virtual loss keeps it forced, so here one
    descent at a time, taking each forced child's visits away after it);
    unvisited children are never forced."""
    n = 3
    visits = [0, 5, 0, 1, 3, 0, 0, 2, 0]
    game, tree, fc = _root_with_visits(n, visits)
    order = []
    for _ in range(5):
        j = forced.select_batch(tree, game, 1, 0.5, 1e30)[0]['node'] - fc
        order.append(j)
        tree.t.contents.num_visits[fc + j] = 0.0
    assert order == [1, 3, 4, 7, 0]         # then nothing is visited: child 0 by np.argmax
    # without forcing, the same root descends into an unvisited child
    game, tree, fc = _root_with_visits(n, visits)
    assert visits[tree.select_batch(game, 1, 0.5)[0]['node'] - fc] == 0


def test_forced_k_zero_is_the_oracle():
    """With forced_k = 0 the forced search is the oracle's own, bit for bit:
    whole searches with tree reuse on 5x5 and 9x9, several batch sizes."""
    for n, sims, batch in ((5, 60, 6), (9, 100, 8), (5, 30, 1)):
        ga, gb = oracle.Hex(n), oracle.Hex(n)
        ta, tb = oracle.Tree(max_nodes=200_000), oracle.Tree(max_nodes=200_000)
        for ply in range(6):
            sa = ta.sample_paths_stub(ga, sims, batch, 0.5, 2)
            sb = forced.sample_paths_stub(tb, gb, sims, batch, 0.5, 2, 0.0)
            va, wa, pa = ta.root_stats()
            vb, wb, pb = tb.root_stats()
            assert (va.tobytes(), wa.tobytes(), pa.tobytes()) == (vb.tobytes(), wb.tobytes(), pb.tobytes())
            assert ta.num_nodes == tb.num_nodes and ta.root_node() == tb.root_node() and sa == sb
            move_id = int(np.argmax(va))
            move = ga.legal_moves()[move_id]
            for t, g in ((ta, ga), (tb, gb)):
                t.move(move_id)
                g.step(int(move))
    # and forcing does change the search
    g = oracle.Hex(5)
    ta, tb = oracle.Tree(max_nodes=200_000), oracle.Tree(max_nodes=200_000)
    ta.sample_paths_stub(g, 60, 6, 0.5, 2)
    forced.sample_paths_stub(tb, g, 60, 6, 0.5, 2, 2.0)
    assert ta.root_stats()[0].tobytes() != tb.root_stats()[0].tobytes()


def test_no_visits_no_forcing():
    n = 3
    game, tree, fc = _root_with_visits(n, [0] * 9)
    assert [lv['node'] for lv in forced.select_batch(tree, game, 1, 0.5, 1e30)] == [fc]


def test_forced_threshold_is_strict():
    """N == n_forced is not forced: uniform priors 1/4 and sum N = 8 give
    n_forced = sqrt(2 * 0.25 * 8) = 2 at k = 2."""
    n = 2
    assert forced_visits(2.0, f32(0.25), 8) == f32(2.0)
    game, tree, fc = _root_with_visits(n, [2, 2, 2, 2])
    picked = forced.select_batch(tree, game, 1, 0.5, 2.0)[0]['node'] - fc
    game, tree, fc = _root_with_visits(n, [2, 2, 2, 2])
    assert picked == tree.select_batch(game, 1, 0.5)[0]['node'] - fc
    # child 2 (N = 1 < 2) is forced, though plain PUCT prefers child 1
    game, tree, fc = _root_with_visits(n, [3, 1, 1, 3])
    assert forced.select_batch(tree, game, 1, 0.5, 2.0)[0]['node'] == fc + 1
    game, tree, fc = _root_with_visits(n, [3, 2, 1, 2])
    assert forced.select_batch(tree, game, 1, 0.5, 2.0)[0]['node'] == fc + 2


# ------------------------------------------------------------------ pruning --

def brute_force_prune(v, w, p, coef, k):
    """The definition: N' = max(N - floor(n_forced), min{N'' >= 0 : score <
    s*}), capped at N, by a scan of every N'' from 0; then 1 -> 0."""
    v, w, p = (np.asarray(a, np.float32) for a in (v, w, p))
    out = v.copy()
    if v.max() == 0:
        return out
    best = int(np.argmax(v))
    sum_n = int(v.sum())
    sq = np.sqrt(f32(sum_n))
    s_best = prune_score(v[best], w[best], p[best], sq, coef, v[best])
    for j in range(len(v)):
        n = int(v[j])
        if j == best or n == 0:
            continue
        below = [m for m in range(n + 1) if prune_score(v[j], w[j], p[j], sq, coef, m) < s_best]
        m_min = below[0] if below else n + 1
        d = int(np.floor(forced_visits(k, p[j], sum_n)))
        m = min(n, max(n - d, m_min))
        out[j] = 0 if m == 1 else m
    return out


def test_pruning_against_brute_force():
    rng = np.random.default_rng(0)
    for _ in range(300):
        kk = int(rng.integers(1, 30))
        v = rng.integers(0, 60, kk).astype(np.float32) * (rng.random(kk) < 0.7)
        w = (rng.random(kk).astype(np.float32) * 2 - 1) * v
        w = np.round(w).astype(np.float32)
        p = rng.dirichlet(np.ones(kk)).astype(np.float32)
        coef = float(rng.choice([0.5, 1.0, 2.0]))
        k = float(rng.choice([0.5, 2.0, 8.0]))
        got = prune_visits(v, w, p, coef, k)
        assert got.tobytes() == brute_force_prune(v, w, p, coef, k).tobytes()
        assert (got <= v).all()
        assert got[int(np.argmax(v))] == v.max()


def test_pruning_hand_worked():
    coef, k = 1.0, 2.0
    # c* = child 0 (N = 10, Q = 0): s* = 1 * 0.5 * sqrt(16) / 11 = 2/11.
    # child 1 (N = 6, P = 0.5, Q = 0): n_forced = sqrt(2 * 0.5 * 16) = 4, so at least 6 - 4 = 2;
    # score(n) = 2 / (1 + n) < 2/11 needs n >= 11 > 6: it keeps 6.
    v = np.array([10, 6], np.float32)
    w = np.zeros(2, np.float32)
    p = np.array([0.5, 0.5], np.float32)
    assert prune_visits(v, w, p, coef, k).tolist() == [10, 6]
    # a poor child: Q = -1 (W = +N, from the child's mover), P = 0.1, N = 3, sum N = 16:
    # score(n) = -1 + 0.4 / (1 + n) < 2/11 for every n >= 0, and n_forced =
    # sqrt(2 * 0.1 * 16) = 1.79 -> floor 1: N' = max(3 - 1, 0) = 2
    v = np.array([13, 3], np.float32)
    w = np.array([0, 3], np.float32)
    p = np.array([0.9, 0.1], np.float32)
    out = prune_visits(v, w, p, coef, k)
    assert out[0] == 13 and out[1] == 2
    # the same child with N = 2: N' = max(2 - 1, 0) = 1, and a child left at 1 becomes 0
    v = np.array([14, 2], np.float32)
    w = np.array([0, 2], np.float32)
    assert prune_visits(v, w, p, coef, k).tolist() == [14, 0]
    # a single visit is pruned even when nothing else was removed
    v = np.array([5, 1, 0], np.float32)
    w = np.array([0, 1, 0], np.float32)
    p = np.array([0.8, 0.1, 0.1], np.float32)
    assert prune_visits(v, w, p, 0.5, 1e-6).tolist() == [5, 0, 0]
    # ties with c*: the lowest ordinal keeps its count, an equal twin can be cut
    v = np.array([4, 4], np.float32)
    w = np.array([0, 4], np.float32)
    p = np.array([0.5, 0.5], np.float32)
    out = prune_visits(v, w, p, 0.5, 2.0)
    assert out[0] == 4 and out[1] < 4
    # no visits: nothing to do
    assert prune_visits(np.zeros(3, np.float32), np.zeros(3, np.float32),
                        np.full(3, 1 / 3, np.float32), 0.5, 2.0).tolist() == [0, 0, 0]


# ------------------------------------------------------------ train config --

def test_train_passes_forced_playouts_to_the_player(monkeypatch, tmp_path):
    """train() reads forced_playouts_k next to the other self-play settings
    and hands it to the player of every rank (here a rank > 0, stopped at the
    player's construction)."""
    from azalea_b200 import policy_trainer
    got = {}

    class Stop(Exception):
        pass

    def player(*a, **kw):
        got.update(kw)
        raise Stop

    class FakeDist:
        def get_rank(self):
            return 1

        def get_world_size(self):
            return 2

    class Net:
        def to(self, device):
            return self

    class Pol:
        net = Net()
        settings = {}

        def seed(self, s):
            pass

    monkeypatch.setattr(policy_trainer, 'Player', player)
    monkeypatch.setattr(policy_trainer, '_dist', lambda: FakeDist())
    monkeypatch.setattr(policy_trainer, 'AzaleaAgent', lambda *a, **kw: None)
    config = dict(seed=3, device='cuda', game='hex', board_size=5, replaybuf_oversampling=1,
                  batch_size=8, forced_playouts_k=2)
    with pytest.raises(Stop):
        policy_trainer.train(Pol(), config, str(tmp_path))
    assert got['forced_playouts_k'] == 2.0
    got.clear()
    del config['forced_playouts_k']
    with pytest.raises(Stop):
        policy_trainer.train(Pol(), config, str(tmp_path))
    assert got['forced_playouts_k'] == 0.0
