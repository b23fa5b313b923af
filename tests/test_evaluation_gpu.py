"""GPU tests of the tournament driver (azalea/evaluation.py:17-80 semantics):
two trees per game, per-policy evaluator routing, outcome bookkeeping."""
import numpy as np
import pytest
import torch

import oracle
from oracle.lockstep import bits

pytestmark = pytest.mark.gpu


def stub_agent(n, sims, mode=2, seed=0):
    import azalea_b200 as az
    p = az.Policy()
    p.net = az.StubEvaluator(mode)
    p.simulations, p.search_batch_size, p.exploration_coef = sims, 6, 0.5
    p.exploration_depth, p.exploration_temperature = 4, 1.0
    p.exploration_noise_alpha, p.exploration_noise_scale = 0.03, 0.25
    a = az.AzaleaAgent(lambda: az.HexGame(n), policy=p)
    a.settings['move_sampling'] = True
    return a


def net_agent(n, seed, sims=30):
    import azalea_b200 as az
    torch.manual_seed(seed)
    p = az.Policy()
    p.initialize(dict(device='cuda', network='HexNetwork', board_size=n,
                      num_blocks=1, base_chans=32, simulations=sims,
                      search_batch_size=5, exploration_coef=0.5,
                      exploration_depth=4, exploration_noise_alpha=0.03,
                      exploration_noise_scale=0.25, exploration_temperature=1.0))
    a = az.AzaleaAgent(lambda: az.HexGame(n), policy=p)
    a.settings['move_sampling'] = True
    return a


def test_matches_are_legal_games_with_correct_results():
    """Every game of play_matches replays through the oracle: all moves
    legal, alternating, and the reported winner is the oracle's."""
    import azalea_b200 as az
    n, G = 5, 16 + 64 + 64
    a, b = stub_agent(n, 120).policy, stub_agent(n, 100, mode=1).policy
    rnd = az.RandomPolicy()
    first = [a] * 16 + [b] * 64 + [rnd] * 64
    second = [b] * 16 + [rnd] * 64 + [a] * 64
    result, history = az.play_matches(first, second, n, seed=3)
    assert set(result.tolist()) <= {1, 3}
    for g in range(G):
        game = oracle.Hex(n)
        for ply in range(len(history)):
            mv = int(history[ply, g])
            if mv == 0:
                break
            assert mv in game.legal_moves()
            game.step(mv)
        assert game.result() == result[g]
    # even with a noise evaluator the search sees terminal positions, so the
    # searching side beats the random mover on balance (first = b vs random:
    # b moves first; first = random vs a: a moves second)
    wins = (result[16:80] == 3).sum() + (result[80:144] == 1).sum()
    assert wins > 0.55 * 128, wins


def test_evaluate_round_robin_bookkeeping():
    """evaluate(agents, rounds) -> {pair: [wins_i, draws, wins_j]} over all
    pairs i < j (evaluation.py:17-46), random anchor first as compare() does
    (compare_cli.py:57-82); two different networks are routed to their own
    trees."""
    import azalea_b200 as az
    n, rounds = 5, 12
    agents = [az.AzaleaAgent(lambda: az.HexGame(n)),      # RandomPolicy
              net_agent(n, 1), net_agent(n, 2), stub_agent(n, 50)]
    out = az.evaluate(agents, rounds)
    assert sorted(out) == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    for pair, (w, d, l) in out.items():
        assert w + d + l == rounds and d == 0      # Hex has no draws
    # the anchor loses to every searching policy on balance
    lost = sum(out[(0, j)][2] for j in (1, 2, 3))
    assert lost > 0.5 * 3 * rounds, out
    # first-move coin flips are the reference's: RandomState(10000*r + s)
    orders = [np.random.RandomState(10000 * r + s).choice([-1, 1])
              for r in range(rounds) for s in range(6)]
    assert 0.25 < np.mean(np.array(orders) == 1) < 0.75


def search_policy(sims, batch, coef, mode, sampling=False):
    import azalea_b200 as az
    p = az.Policy()
    p.net = az.StubEvaluator(mode)
    p.simulations, p.search_batch_size, p.exploration_coef = sims, batch, coef
    p.exploration_depth, p.exploration_temperature = 4, 1.0
    p.exploration_noise_alpha, p.exploration_noise_scale = 0.03, 0.25
    p.settings['move_sampling'] = sampling
    return p


def test_lockstep_seats_match_oracle_trees():
    """The two-seat lockstep path (play_game.py:46-54: both agents' trees are
    advanced on every move; search_tree.py:115-132: re-root or reset) pinned
    against the oracle: 64 games with mixed search configurations, stub
    evaluators and a random mover share two engines, groups of games are
    searched one configuration at a time with the others paused
    (AZ_ST_DISABLED), and after EVERY search the mover's root -- visit counts,
    total values, priors, root (N, W), reference node count -- equals a
    dedicated oracle tree of that (game, seat) bit for bit.  Moves are the
    engine's own (temperature 0): each must be a most-visited child in the
    oracle's tree; they are then played into both oracle trees."""
    import azalea_b200 as az
    from azalea_b200.evaluation import play_matches
    from oracle import stubs
    n, G = 5, 64
    A = search_policy(60, 6, 0.5, stubs.ROUGH)
    B = search_policy(45, 4, 1.0, stubs.DYADIC)
    C = search_policy(80, 8, 0.75, stubs.ROUGH)
    D = search_policy(60, 6, 0.5, stubs.DYADIC)     # A's search parameters, another evaluator
    R = az.RandomPolicy()
    combos = [(A, B), (B, A), (A, C), (C, R), (R, A), (B, C), (C, C), (D, A), (A, D), (R, B)]
    first = [combos[g % len(combos)][0] for g in range(G)]
    second = [combos[g % len(combos)][1] for g in range(G)]
    seen = {}           # (seat, game, ply) -> root statistics before the move

    def hook(seat, key, games):
        s = 0 if seat.eng.cfg.seed % 2 == 1 else 1      # play_matches: seeds 2k+1, 2k+2
        v, w, p, k, rnw, nodes = (x.cpu().numpy() for x in seat.eng.root_stats())
        ply = seat.eng.hex_state()[3].cpu().numpy()
        for g in games.cpu().numpy():
            seen[(s, int(g), int(ply[g]))] = (v[g, :max(k[g], 0)].copy(), w[g, :max(k[g], 0)].copy(),
                                              p[g, :max(k[g], 0)].copy(), rnw[g].copy(), int(nodes[g]))

    result, history = play_matches(first, second, n, seed=5, hook=hook)
    checked = 0
    for g in range(G):
        game = oracle.Hex(n)
        pols = (first[g], second[g])
        trees = [None if isinstance(p, az.RandomPolicy) else oracle.Tree(max_nodes=2_000_000)
                 for p in pols]
        for ply in range(len(history)):
            mv = int(history[ply, g])
            if mv == 0:
                break
            s = ply % 2
            legal = game.legal_moves()
            assert mv in legal
            mid = int(np.flatnonzero(legal == mv)[0])
            pol = pols[s]
            if trees[s] is not None:
                trees[s].sample_paths_stub(game, pol.simulations, pol.search_batch_size,
                                           pol.exploration_coef, pol.net.mode)
                ov, ow, op = trees[s].root_stats()
                v, w, p, rnw, nodes = seen[(s, g, ply)]
                where = (g, ply)
                assert bits(v) == bits(ov), where
                assert bits(w) == bits(ow), where
                assert bits(p) == bits(op), where
                assert bits(rnw) == bits(trees[s].root_node()), where
                assert nodes == trees[s].num_nodes, where
                assert ov[mid] == ov.max(), where       # temperature 0: an arg-max child
                checked += 1
            else:
                v = seen[(s, g, ply)][0]
                assert len(v) == len(legal) and (v == 1).all()     # uniform over the legal moves
            for t in trees:
                if t is not None:
                    t.move(mid)
            game.step(mv)
        assert game.result() == result[g] and result[g] in (1, 3)
    assert checked > 400


def test_evaluate_does_not_depend_on_world_size():
    """(round, pair) tasks are dealt round-robin to ranks and every game's
    random streams are keyed by its global task id: the two shares of a
    2-rank tournament add up to exactly the 1-rank tallies (SURVEY 8e)."""
    import azalea_b200 as az
    n, rounds = 5, 6
    agents = [az.AzaleaAgent(lambda: az.HexGame(n)),      # RandomPolicy anchor
              stub_agent(n, 50), stub_agent(n, 40, mode=1), stub_agent(n, 30)]
    whole = az.evaluate(agents, rounds)
    parts = [az.evaluate(agents, rounds, rank=r, world_size=2, reduce=False)
             for r in range(2)]
    assert sorted(whole) == sorted(parts[0]) == sorted(parts[1])
    for pair in whole:
        assert sum(whole[pair]) == rounds
        assert [a + b for a, b in zip(parts[0][pair], parts[1][pair])] == whole[pair], pair
    # and a share is not trivially empty
    assert sum(sum(v) for v in parts[0].values()) == rounds * 6 // 2
