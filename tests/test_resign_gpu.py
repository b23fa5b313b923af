"""Resignation with calibration games (az_engine_set_resign): after the
search the player to move resigns when r = max(Q_root, Q_best) is below the
threshold, except in calibration games (one Philox coin per game id), which
never resign and record each colour's lowest r."""
import numpy as np
import pytest
import torch

import oracle
from oracle import stubs
from oracle.lockstep import (assert_root_matches, assert_same_games, assert_streams_and_graphs_agree,
                             bits, check_replay_buffer, network, selfplay_fingerprint, selfplay_player,
                             stub_search, stub_selfplay, train_config)
from oracle.philox import calibration_game, full_ply, game_ids

gpu = pytest.mark.gpu


def resign_value(v, w, k, root_nw):
    """r = max(Q_root, Q_best) in float32 from one game's root_stats()."""
    r = np.float32(root_nw[1]) / np.float32(root_nw[0])
    vis = v[:k]
    if k and vis.max() > 0:
        c = int(np.argmax(vis))
        r = max(r, -w[c] / vis[c])
    return np.float32(r)


def hist_bin(m):
    return min(64, max(0, int(np.floor((np.float32(m) + np.float32(1)) * np.float32(64)))))


# A deterministic stub's values sit close to 0 at these search sizes (the search averages
# hash-random leaf values), so the thresholds that trigger are just below 0.
STUB_THRESHOLD = -0.05


# ------------------------------------------------------------------ tests --

@gpu
@pytest.mark.parametrize('n', (5, 7))
def test_resign_off_is_byte_identical(n):
    """Never calling the setter, and calling it with the setting off, give
    the same moves, chosen rows, replay bytes, counters and meta."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    out = []
    for off in (None, (None, 0.1), (-1.0, 0.5), (-3.0, 1.0)):
        sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=64, board_size=n, simulations=20,
                              search_batch_size=4, seed=3, cuda_graph=False)
        if off is not None:
            sp.eng.set_resign(*off)
        out.append(selfplay_fingerprint(sp, 30))
        rs = sp.resign_stats()
        assert rs['resigned_games'] == rs['calibration_games'] == 0
    assert len(out[0][1]) > 0
    assert all(o == out[0] for o in out[1:])


@gpu
def test_resign_decisions_match_the_oracle():
    """Engine driven move by move, temperature 0, no auto reset, oracle trees
    with tree reuse.  At every ply r from numpy on root_stats() predicts
    exactly which games resign, and the numpy coin which games are
    calibration games.  Resigners get chosen = (0, -1, result, ply) and
    hex_state reports the opponent's win; every root is bit-equal to the
    oracle's.  The buffer's per-colour minima, resigned, calibration and
    false-positive counts and histogram equal the host's bookkeeping."""
    from azalea_b200 import Engine
    n, G, sims, batch, coef, mode, seed = 7, 128, 20, 4, 0.5, stubs.ROUGH, 11
    thr, disable = np.float32(-0.1), 0.25
    num_batches = sims // batch + 1
    eng = Engine(G, n, max_batch=batch, seed=seed, nodes_per_game=65536)
    eng.set_resign(float(thr), disable)
    trees = [oracle.Tree(max_nodes=200_000) for _ in range(G)]
    games = [oracle.Hex(n) for _ in range(G)]
    chosen = torch.zeros(G, 4, dtype=torch.int32, device='cuda')
    done = np.zeros(G, bool)
    gid0 = game_ids(eng)[0]
    calib = np.array([calibration_game(seed, int(gid0[g]), disable) for g in range(G)])
    mins = np.full((G, 2), np.inf, np.float32)
    want = np.zeros((G, 72), np.int64)
    winner_seen = set()
    plies = 0
    for _ in range(n * n):
        if done.all():
            break
        gid, ply = game_ids(eng)
        color = eng.meta[:, 2].cpu().numpy()          # the colour to move
        assert (gid == gid0).all()
        stub_search(eng, mode, batch, coef, num_batches)
        stats = [x.cpu().numpy() for x in eng.root_stats()]
        v, w, _, k, rnw, _ = stats
        eng.play_commit(0.0, 0, False, False, False, chosen)
        ch = chosen.cpu().numpy()
        _, _, result, hply = (x.cpu().numpy() for x in eng.hex_state())
        for g in np.flatnonzero(~done):
            where = (g, int(ply[g]))
            trees[g].sample_paths_stub(games[g], sims, batch, coef, mode)
            assert_root_matches(stats, g, trees[g], where)
            r = resign_value(v[g], w[g], int(k[g]), rnw[g])
            c = int(color[g])
            if calib[g]:
                mins[g, c - 1] = min(mins[g, c - 1], r)
            if not calib[g] and r < thr:
                res = 1 if c == 1 else 3
                assert tuple(ch[g]) == (0, -1, res, int(ply[g])), where
                assert result[g] == res and hply[g] == ply[g], where
                want[g, 2] += 1
                done[g] = True
                continue
            assert ch[g, 1] >= 0, where
            plies += 1
            trees[g].move(int(ch[g, 1]))
            games[g].step(int(ch[g, 0]))
            if ch[g, 2] != 0:
                assert games[g].result() == ch[g, 2] == result[g]
                done[g] = True
                if calib[g]:
                    m = mins[g, 0 if ch[g, 2] == 3 else 1]
                    want[g, 3] += 1
                    want[g, 4] += int(m < thr)
                    want[g, 5 + hist_bin(m)] += 1
                    winner_seen.add(hist_bin(m))
    assert done.all()
    buf = eng.resign.cpu().numpy()
    assert bits(buf[:, :2].view(np.float32)) == bits(mins)
    assert np.array_equal(buf[:, 2:70], want[:, 2:70])
    assert np.isinf(mins[~calib]).all()
    # every branch was taken: resignations, calibration games with and without a false positive
    assert want[:, 2].sum() > 0 and 0 < want[:, 4].sum() < want[:, 3].sum()
    assert len(winner_seen) > 1
    rs = eng.resign_stats()
    assert rs['resigned_games'] == want[:, 2].sum()
    assert rs['calibration_games'] == want[:, 3].sum() == rs['histogram'].sum()
    assert rs['false_positives'] == want[:, 4].sum()
    # a resigned game counts as a game; its resigning ply is no ply
    assert int(eng.counters[:, 6].sum()) == G
    assert int(eng.counters[:, 5].sum()) == plies
    assert (eng.status().cpu().numpy() == 0).all()


@gpu
def test_resign_value_sign_on_a_known_position():
    """X (to move) is one stone from connecting on 3x3 with no way for O to
    stop it: Q_root > 0 from X's view.  After X's winning move O is lost:
    a winning child shows a negative W (the node's own mover lost)."""
    from azalea_b200 import Engine
    n, G, B = 3, 1, 4
    board = np.zeros((G, n * n), np.int8)
    board[0, [0, 3]] = 1           # X: (0,0), (1,0); (2,0) wins, (2,1) too via (1,0)
    board[0, [1, 2]] = 2
    eng = Engine(G, n, max_batch=B, seed=1, nodes_per_game=4096)
    eng.hex_set_state(board, np.array([1], np.int32))
    stub_search(eng, stubs.UNIFORM, B, 0.5, 20)
    v, w, _, k, rnw, _ = (x.cpu().numpy() for x in eng.root_stats())
    kg = int(k[0])
    assert rnw[0, 1] / rnw[0, 0] > 0.3
    c = int(np.argmax(v[0, :kg]))
    assert -w[0, c] / v[0, c] > 0.9         # the most-visited child is a win for X


@gpu
@pytest.mark.parametrize('cap', (False, True))
def test_replay_of_resigned_games(cap):
    """A resigned game's rows are exactly plies 0 .. ply-1 (minus fast plies
    with the playout cap), with game_len = ply, the opponent's result,
    ply-parity rewards and reserved 0; natural endings are unchanged.  The
    rows go through rows_to_dataframe and DeviceReplayBuffer, and
    Player.read reports the resignation counts of its call."""
    from azalea_b200 import StubEvaluator
    from azalea_b200.engine import decode_replay_rows
    capkw = dict(full_search_prob=0.5, fast_simulations=5) if cap else {}
    # 40 moves of 64 games record at most 2560 rows: the replay output (2 * 64 * 25 rows) holds
    # every finished game's rows until the one harvest below
    sp, _, finished, _ = stub_selfplay(40, resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.2, **capkw)
    assert sp.counters()['replay_dropped'] == 0
    rows = sp.harvest()
    h, _, _ = decode_replay_rows(rows, 5)
    by_game = {}
    for i, gid in enumerate(h['game_id']):
        by_game.setdefault(int(gid), []).append(i)
    resigned = [gid for gid, f in finished.items() if f[2]]
    assert resigned and len(resigned) < len(finished)
    assert sp.resign_stats()['resigned_games'] == len(resigned)
    cnt = sp.counters()
    for gid, (length, result, _) in finished.items():
        plies = [p for p in range(length) if not cap or full_ply(3, gid, p, 0.5)]
        idx = by_game.get(gid, [])
        assert h['ply'][idx].tolist() == plies, gid
        for i in idx:
            assert h['game_len'][i] == length and h['result'][i] == result
            rw = np.float32(result - 2)
            assert h['reward'][i] == (-rw if h['ply'][i] % 2 else rw)
            assert h['reserved'][i] == 0
    assert set(by_game) <= set(finished)
    assert len(h) == cnt['replay_rows']
    assert cnt['games'] == len(finished)
    check_replay_buffer(rows)

    player = selfplay_player(StubEvaluator(stubs.ROUGH), 30, 4, cuda_graph=False,
                             resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.2, **capkw)
    assert player.resign
    for read in (player.read, player.read_device):
        rs0 = player.sp.resign_stats()
        _, metrics = read(200)
        rs1 = player.sp.resign_stats()
        assert metrics['resigned_games'] == rs1['resigned_games'] - rs0['resigned_games'] > 0
        assert metrics['resign_calibration_games'] == rs1['calibration_games'] - rs0['calibration_games']
        assert metrics['resign_false_positives'] == rs1['false_positives'] - rs0['false_positives']


@gpu
def test_resign_edge_settings():
    """disable_prob = 1 resigns nothing: the games are those of the setting
    off, and every game that ended is a calibration game with its winner's
    lowest r in the histogram.  disable_prob = 0 has no calibration game."""
    c_off = stub_selfplay(50)[3]
    sp, _, finished, c_all = stub_selfplay(50, resign_threshold=STUB_THRESHOLD, resign_disable_prob=1.0)
    assert np.array_equal(c_off, c_all)
    rs = sp.resign_stats()
    assert rs['resigned_games'] == 0 and not any(f[2] for f in finished.values())
    assert rs['calibration_games'] == sp.counters()['games'] == rs['histogram'].sum() > 0
    assert rs['false_positives'] <= rs['calibration_games']
    sp, _, finished, _ = stub_selfplay(50, resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.0)
    rs = sp.resign_stats()
    assert rs['calibration_games'] == rs['false_positives'] == rs['histogram'].sum() == 0
    assert rs['resigned_games'] == sum(f[2] for f in finished.values()) > 0


@gpu
def test_resign_invariance():
    """Streams 1 and 2, eager and graphed, and 2 ranks x 32 games against
    1 rank x 64 leave the games and the resignation state unchanged."""
    kw = dict(resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.3, full_search_prob=0.5,
              fast_simulations=5)

    def play(streams, graph, **more):
        sp, _, _, chosen = stub_selfplay(40, streams=streams, graph=graph, **kw, **more)
        return (chosen, sp.harvest(), sp.counters(), sp.eng.resign.cpu().numpy(),
                sp.resign_stats()['resigned_games'])
    _, r0, _, s0, resigned = assert_streams_and_graphs_agree(play)
    assert len(r0) > 0 and resigned > 0
    parts = [play(1, False, G=32, rank=r, world_size=2) for r in range(2)]
    # slot s of the 64-game run plays the games of rank s // 32's slot s % 32
    assert np.array_equal(np.concatenate([p[3] for p in parts]), s0)
    assert_same_games(r0, [p[1] for p in parts])


@gpu
def test_resign_with_the_network():
    """6x64 network in the loop, packed leaves, two streams, a CUDA graph:
    a measure-only run picks a threshold with resign_threshold_for, and a run
    with it resigns games and keeps every engine status at 0."""
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.selfplay import resign_threshold_for
    net = network(6)

    def play(threshold, disable):
        sp = LockstepSelfPlay(net, num_games=128, board_size=5, simulations=40, search_batch_size=8,
                              seed=5, streams=2, cuda_graph=True, resign_threshold=threshold,
                              resign_disable_prob=disable)
        assert sp.pack_leaves and sp.streams == 2
        sp.preroll(8)
        for _ in range(40):
            sp.step_move()
        assert sp._graph is not None
        assert (sp.eng.status().cpu().numpy() == 0).all()
        return sp.resign_stats(), sp.counters()
    rs, cnt = play(0.99, 1.0)
    assert rs['resigned_games'] == 0 and rs['calibration_games'] == cnt['games'] > 0
    thr = resign_threshold_for(rs['histogram'], rs['calibration_games'], 0.5)
    assert -1.0 < thr <= 0.0
    rs, cnt = play(thr, 0.1)
    assert rs['resigned_games'] > 0


@gpu
def test_train_with_resign(tmp_path, monkeypatch):
    """train(...) with resign_threshold / resign_disable_prob: the self-play
    player gets the setting, training runs, and the checkpoint has no trace
    of it."""
    import azalea_b200 as az
    from azalea_b200 import policy_trainer
    from azalea_b200.parallel_player import Player
    made = []

    class Recording(Player):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            made.append(self)
    monkeypatch.setattr(policy_trainer, 'Player', Recording)
    config = train_config(resign_threshold=-0.2, resign_disable_prob=0.3)
    policy = az.Policy()
    policy.initialize(config)
    buf = policy_trainer.initialize_replay_buffer(None, lambda: az.HexGame(5), 256, num_games=32,
                                                  device='cuda', seed=3)
    policy_trainer.train(policy, config, str(tmp_path), replaybuf=buf)
    hist = policy_trainer.train.history
    assert len(hist) == 4 and all(np.isfinite(x['loss']) for x in hist)
    sp = [p for p in made if not p.sp.random_play][-1].sp
    assert sp.resign_threshold == -0.2 and sp.resign_disable_prob == 0.3
    state = policy.state_dict()
    assert 'resign_threshold' not in state and 'resign_disable_prob' not in state
