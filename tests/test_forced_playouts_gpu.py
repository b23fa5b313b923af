"""Forced playouts and policy target pruning (az_engine_set_forced_playouts):
at the root of a full ply a visited child with N < sqrt(k P sum N) is searched
again, and the replay row gets the visits PUCT would have given without it;
the move is still drawn from the raw visits."""
import numpy as np
import pytest
import torch

import oracle
from oracle import forced, stubs
from oracle.lockstep import (assert_root_matches, assert_same_games, assert_streams_and_graphs_agree,
                             bits, check_replay_buffer, network, selfplay_fingerprint, selfplay_player,
                             stub_search, stub_selfplay, train_config)
from oracle.philox import full_ply, game_ids, move_at_temperature_1
from oracle.pruning import prune_visits

gpu = pytest.mark.gpu


def rows_by_game(rows, n):
    from azalea_b200.engine import decode_replay_rows
    h, _, vis = decode_replay_rows(rows, n)
    return h, vis, {(int(g), int(p)): i for i, (g, p) in enumerate(zip(h['game_id'], h['ply']))}


# ------------------------------------------------------------------ tests --

@gpu
@pytest.mark.parametrize('n', (5, 7))
def test_forced_playouts_off_is_byte_identical(n):
    """Never calling the setter, and calling it with k = 0, give the same
    chosen rows, replay bytes, counters and meta."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    out = []
    for off in (None, (0.0, 0.5), (0.0, 3.0)):
        sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=64, board_size=n, simulations=20,
                              search_batch_size=4, seed=3, cuda_graph=False)
        if off is not None:
            sp.eng.set_forced_playouts(*off)
        out.append(selfplay_fingerprint(sp, 30))
    assert len(out[0][1]) > 0
    assert all(o == out[0] for o in out[1:])


@gpu
@pytest.mark.parametrize('n,G,plies,cap', [(5, 64, 25, False), (13, 12, 8, False), (5, 64, 25, True)])
def test_forcing_matches_the_oracle(n, G, plies, cap):
    """Engine driven as _window_body drives it, noise off, k = 2, tree reuse:
    every ply's root (visits, W, priors, root N/W, node count) equals an
    oracle tree searched with forced_k = 2 -- or with forced_k = 0 on the
    fast plies of the playout cap -- bit for bit.  n = 5 runs k_select<4,.>,
    n = 13 k_select<12,.>.  Oracle trees without forcing, following the same
    moves, differ on most full plies, so the check is not vacuous."""
    from azalea_b200 import Engine
    sims, fast_sims, batch, coef, mode, seed, fk = 60, 10, 6, 0.5, stubs.ROUGH, 7, 2.0
    num_batches = sims // batch + 1
    eng = Engine(G, n, max_batch=batch, seed=seed, nodes_per_game=200_000)
    eng.set_forced_playouts(fk, coef)
    if cap:
        eng.set_playout_cap(0.5, (fast_sims // batch + 1) * batch)
    trees = [oracle.Tree(max_nodes=2_000_000) for _ in range(G)]
    plain = [oracle.Tree(max_nodes=2_000_000) for _ in range(G)]
    games = [oracle.Hex(n) for _ in range(G)]
    chosen = torch.zeros(G, 4, dtype=torch.int32, device='cuda')
    done = np.zeros(G, bool)
    full_plies = differ = fast_plies = 0
    for _ in range(plies):
        if done.all():
            break
        gid, ply = game_ids(eng)
        stub_search(eng, mode, batch, coef, num_batches)
        stats = [x.cpu().numpy() for x in eng.root_stats()]
        eng.play_commit(0.0, 0, False, False, False, chosen)
        ch = chosen.cpu().numpy()
        for g in np.flatnonzero(~done):
            full = not cap or full_ply(seed, int(gid[g]), int(ply[g]), 0.5)
            g_sims = sims if full else fast_sims
            forced.sample_paths_stub(trees[g], games[g], g_sims, batch, coef, mode, fk if full else 0.0)
            plain[g].sample_paths_stub(games[g], g_sims, batch, coef, mode)
            ov = assert_root_matches(stats, g, trees[g], (g, int(ply[g]), full))
            if full:
                full_plies += 1
                differ += bits(plain[g].root_stats()[0]) != bits(ov)
            else:
                fast_plies += 1
            mid = int(ch[g, 1])
            for t in (trees[g], plain[g]):
                t.move(mid)
            games[g].step(int(ch[g, 0]))
            if ch[g, 2] != 0:
                assert games[g].result() == ch[g, 2]
                done[g] = True
    assert full_plies > 0 and differ > full_plies // 2, (differ, full_plies)
    assert fast_plies > 0 if cap else fast_plies == 0
    assert (eng.status().cpu().numpy() == 0).all()


@gpu
@pytest.mark.parametrize('noise', (False, True))
def test_pruned_rows_match_numpy(noise):
    """Every replay row's visits equal the numpy pruning of root_stats()
    taken just before play_commit, bit for bit, matched by (game_id, ply) on
    temperature-1 and temperature-0 plies, with resignation on.  At
    temperature 1 numpy predicts move_id exactly from the raw visits and the
    commit's Philox draw: pruning does not change the move."""
    from azalea_b200 import Engine
    n, G, sims, batch, coef, mode, seed, fk, depth = 5, 64, 40, 4, 0.5, stubs.ROUGH, 9, 2.0, 6
    num_batches = sims // batch + 1
    eng = Engine(G, n, max_batch=batch, seed=seed, nodes_per_game=65536, replay_rows=2 * G * n * n)
    eng.set_forced_playouts(fk, coef)
    eng.set_resign(-0.05, 0.2)
    chosen = torch.zeros(G, 4, dtype=torch.int32, device='cuda')
    want, raw = {}, {}
    moves_checked = 0
    for _ in range(60):
        gid, ply = game_ids(eng)
        stub_search(eng, mode, batch, coef, num_batches, 0.25 if noise else 0.0, 0.03)
        v, w, p, k, _, _ = (x.cpu().numpy() for x in eng.root_stats())
        eng.play_commit(1.0, depth, True, True, True, chosen)
        ch = chosen.cpu().numpy()
        for g in range(G):
            kg = int(k[g])
            key = (int(gid[g]), int(ply[g]))
            want[key] = prune_visits(v[g, :kg], w[g, :kg], p[g, :kg], coef, fk)
            raw[key] = v[g, :kg].copy()
            if ch[g, 1] >= 0 and ply[g] < depth:
                assert ch[g, 1] == move_at_temperature_1(v[g, :kg], seed, *key), key
                moves_checked += 1
    assert (eng.status().cpu().numpy() == 0).all()
    h, vis, index = rows_by_game(eng.harvest_replay(), n)
    assert len(index) == len(h) > 0
    temps, pruned = set(), 0
    for key, i in index.items():
        kg = int(h['num_moves'][i])
        assert bits(vis[i, :kg]) == bits(want[key]), key
        assert not vis[i, kg:].any()
        assert h['move_id'][i] < kg and raw[key][h['move_id'][i]] > 0
        temps.add(float(h['temperature'][i]))
        pruned += bits(want[key]) != bits(raw[key])
    assert temps == {0.0, 1.0}
    assert pruned > len(h) // 4, (pruned, len(h))
    assert moves_checked > 0
    assert eng.resign_stats()['resigned_games'] > 0


@gpu
def test_random_play_and_preroll_rows_are_not_pruned():
    """RandomPolicy self-play and the preroll plies of a forced-playouts
    run record pi = 1/k exactly: one visit on every child, nothing pruned."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    from azalea_b200.selfplay import rows_to_dataframe
    n, G = 5, 64
    sp = LockstepSelfPlay(None, num_games=G, board_size=n, random_play=True, cuda_graph=False,
                          forced_playouts_k=2.0)
    assert sp.forced_playouts_k == 0.0
    for _ in range(30):
        sp.step_move()
    rows = sp.harvest()
    h, vis, _ = rows_by_game(rows, n)
    assert len(h) > 0
    for i in range(len(h)):
        kg = int(h['num_moves'][i])
        assert (vis[i, :kg] == 1.0).all()
    df = rows_to_dataframe(rows, n)
    for i in range(len(h)):
        probs = df[i].moves_prob
        assert np.array_equal(probs, np.full(len(probs), 1.0 / len(probs), np.float32))

    max_plies = 12
    sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=G, board_size=n, simulations=20,
                          search_batch_size=4, seed=3, cuda_graph=False, forced_playouts_k=2.0)
    sp.preroll(max_plies)
    for _ in range(30):
        sp.step_move()
    h, vis, index = rows_by_game(sp.harvest(), n)
    quota = [sum(1 for s in range(1, max_plies + 1) if -(-s * G // max_plies) <= g) for g in range(G)]
    seen = pruned = 0
    for (gid, ply), i in index.items():
        kg = int(h['num_moves'][i])
        if gid < G and ply < quota[gid]:
            assert (vis[i, :kg] == 1.0).all(), (gid, ply)
            seen += 1
        elif h['temperature'][i] == 1.0:
            pruned += int((vis[i, :kg] == 0).sum() > 0)
    assert seen > 0 and pruned > 0


@gpu
def test_forced_playouts_invariance():
    """Streams 1 and 2, eager and graphed, and 2 ranks x 32 games against
    1 rank x 64 leave the games and their rows unchanged."""
    kw = dict(forced_playouts_k=2.0, full_search_prob=0.5, fast_simulations=5)

    def play(streams, graph, **more):
        sp, _, _, chosen = stub_selfplay(40, streams=streams, graph=graph, **kw, **more)
        return chosen, sp.harvest(), sp.counters()
    r0 = assert_streams_and_graphs_agree(play)[1]
    assert len(r0) > 0
    assert_same_games(r0, [play(1, False, G=32, rank=r, world_size=2)[1] for r in range(2)])


@gpu
def test_forced_playouts_with_the_network():
    """6x64 network in the loop, packed leaves, two streams, a CUDA graph,
    preroll: rows go through rows_to_dataframe, DeviceReplayBuffer and
    Player.read, and every engine status stays 0."""
    from azalea_b200 import LockstepSelfPlay
    net = network(6)
    sp = LockstepSelfPlay(net, num_games=128, board_size=5, simulations=40, search_batch_size=8,
                          seed=5, streams=2, cuda_graph=True, forced_playouts_k=2.0)
    assert sp.pack_leaves and sp.streams == 2
    sp.preroll(8)
    for _ in range(40):
        sp.step_move()
    assert sp._graph is not None
    assert (sp.eng.status().cpu().numpy() == 0).all()
    rows = sp.harvest()
    assert len(rows) > 0
    check_replay_buffer(rows)

    player = selfplay_player(net, 40, 8, forced_playouts_k=2.0)
    assert player.sp.forced_playouts_k == 2.0
    examples, metrics = player.read(200)
    assert len(examples) >= 200


@gpu
def test_train_with_forced_playouts(tmp_path, monkeypatch):
    """train(...) with forced_playouts_k: 2: the self-play player gets the
    setting, training runs, and the checkpoint has no trace of it."""
    import azalea_b200 as az
    from azalea_b200 import policy_trainer
    from azalea_b200.parallel_player import Player
    made = []

    class Recording(Player):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            made.append(self)
    monkeypatch.setattr(policy_trainer, 'Player', Recording)
    config = train_config(forced_playouts_k=2)
    policy = az.Policy()
    policy.initialize(config)
    buf = policy_trainer.initialize_replay_buffer(None, lambda: az.HexGame(5), 256, num_games=32,
                                                  device='cuda', seed=3)
    policy_trainer.train(policy, config, str(tmp_path), replaybuf=buf)
    hist = policy_trainer.train.history
    assert len(hist) == 4 and all(np.isfinite(x['loss']) for x in hist)
    sp = [p for p in made if not p.sp.random_play][-1].sp
    assert sp.forced_playouts_k == 2.0 and sp.coef == 0.5
    assert 'forced_playouts_k' not in policy.state_dict()
