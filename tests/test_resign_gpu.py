"""Resignation with calibration games (az_engine_set_resign): after the
search the player to move resigns when r = max(Q_root, Q_best) is below the
threshold, except in calibration games (one Philox coin per game id), which
never resign and record each colour's lowest r."""
import numpy as np
import pytest
import torch

import oracle
from oracle import stubs

gpu = pytest.mark.gpu
M32 = 0xFFFFFFFF
RESIGN_DOMAIN = 0x2E51C0A1
FULL_SEARCH_DOMAIN = 0xCA9F5EA7


def philox(c, k):
    """Philox4x32-10 as az_philox (az_common.cuh)."""
    c, k = list(c), list(k)
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & M32, p1 & M32, ((p0 >> 32) ^ c[3] ^ k[1]) & M32, p0 & M32]
        k = [(k[0] + 0x9E3779B9) & M32, (k[1] + 0xBB67AE85) & M32]
    return c


def _key(seed, game_id):
    return ((seed ^ game_id) & M32, ((seed >> 32) ^ (game_id >> 32)) & M32)


def _thresh(p):
    return np.ceil(np.float64(np.float32(p)) * 2.0 ** 32)


def calibration_game(seed, game_id, p):
    """The calibration coin of (seed, global game id)."""
    return philox((0, 0, 0, RESIGN_DOMAIN), _key(seed, game_id))[0] < _thresh(p)


def full_ply(seed, game_id, ply, p):
    return philox((ply, 0, 0, FULL_SEARCH_DOMAIN), _key(seed, game_id))[0] < _thresh(p)


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


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).tobytes()


def game_ids(eng):
    meta = eng.meta.cpu().numpy().astype(np.int64)
    return (meta[:, 10] & M32) | (meta[:, 11] << 32), meta[:, 4].copy(), meta[:, 2].copy()


def stub_selfplay(moves, G=64, n=5, seed=3, graph=False, streams=None, **kw):
    """Stub self-play recording per move and slot the game id and ply, the
    plies that were fast (playout cap), and the finished games with their
    length, result and whether they ended by resignation."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=G, board_size=n, simulations=30,
                          search_batch_size=4, seed=seed, cuda_graph=graph, exploration_depth=4,
                          streams=streams, **kw)
    finished, chosen = {}, []
    for _ in range(moves):
        gid, ply, _ = game_ids(sp.eng)
        sp.step_move()
        ch = sp.chosen.cpu().numpy().copy()
        chosen.append(ch)
        for g in range(G):
            if ch[g, 2] > 0:
                finished[int(gid[g])] = (int(ch[g, 3]), int(ch[g, 2]), bool(ch[g, 1] == -1))
                assert ch[g, 3] == ply[g] + (ch[g, 1] != -1)
    assert (sp.eng.status().cpu().numpy() == 0).all()
    return sp, finished, np.stack(chosen)


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
        chosen = []
        for _ in range(30):
            sp.step_move()
            chosen.append(sp.chosen.cpu().numpy().copy())
        out.append((np.stack(chosen).tobytes(), sp.harvest().tobytes(),
                    sp.eng.counters.cpu().numpy().tobytes(), sp.eng.meta.cpu().numpy().tobytes()))
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
        gid, ply, color = game_ids(eng)
        assert (gid == gid0).all()
        eng.select_root()
        eng.stub_eval(mode)
        eng.expand_root()
        for _ in range(num_batches):
            eng.select(batch, coef)
            eng.stub_eval(mode)
            eng.expand_backup()
        v, w, p, k, rnw, nodes = (x.cpu().numpy() for x in eng.root_stats())
        eng.play_commit(0.0, 0, False, False, False, chosen)
        ch = chosen.cpu().numpy()
        _, _, result, hply = (x.cpu().numpy() for x in eng.hex_state())
        for g in np.flatnonzero(~done):
            where = (g, int(ply[g]))
            trees[g].sample_paths_stub(games[g], sims, batch, coef, mode)
            ov, ow, op = trees[g].root_stats()
            kg = int(k[g])
            assert bits(v[g, :kg]) == bits(ov), where
            assert bits(w[g, :kg]) == bits(ow), where
            assert bits(rnw[g]) == bits(trees[g].root_node()), where
            r = resign_value(v[g], w[g], kg, rnw[g])
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
    eng.select_root()
    eng.stub_eval(stubs.UNIFORM)
    eng.expand_root()
    for _ in range(20):
        eng.select(B, 0.5)
        eng.stub_eval(stubs.UNIFORM)
        eng.expand_backup()
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
    from azalea_b200.engine import decode_replay_rows
    from azalea_b200.replay_device import DeviceReplayBuffer
    from azalea_b200.selfplay import rows_to_dataframe
    capkw = dict(full_search_prob=0.5, fast_simulations=5) if cap else {}
    # 40 moves of 64 games record at most 2560 rows: the replay output (2 * 64 * 25 rows) holds
    # every finished game's rows until the one harvest below
    sp, finished, _ = stub_selfplay(40, resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.2, **capkw)
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
    df = rows_to_dataframe(rows, 5)
    assert len(df) == len(h)
    buf = DeviceReplayBuffer(len(h) + 7, 5)
    buf.put(torch.from_numpy(rows).cuda())
    batch = buf.sample(64, generator=torch.Generator(device='cuda').manual_seed(4))
    idx = torch.randint(0, len(buf), (64,), device='cuda',
                        generator=torch.Generator(device='cuda').manual_seed(4)).cpu().numpy()
    assert np.array_equal(batch['reward'].cpu().numpy(), h['reward'][idx])
    assert np.allclose(batch['moves_prob'].sum(1).cpu().numpy(), 1.0, atol=1e-5)

    import azalea_b200 as az
    from azalea_b200.parallel_player import Player
    pol = az.Policy()
    pol.net = az.StubEvaluator(stubs.ROUGH)
    pol.simulations, pol.search_batch_size, pol.exploration_coef = 30, 4, 0.5
    pol.exploration_depth, pol.exploration_temperature = 4, 1.0
    pol.exploration_noise_alpha, pol.exploration_noise_scale = 0.03, 0.25
    agent = az.AzaleaAgent(lambda: az.HexGame(5), policy=pol)
    player = Player(None, [agent], num_games=64, seed=3, cuda_graph=False,
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
    _, _, c_off = stub_selfplay(50)
    sp, finished, c_all = stub_selfplay(50, resign_threshold=STUB_THRESHOLD, resign_disable_prob=1.0)
    assert np.array_equal(c_off, c_all)
    rs = sp.resign_stats()
    assert rs['resigned_games'] == 0 and not any(f[2] for f in finished.values())
    assert rs['calibration_games'] == sp.counters()['games'] == rs['histogram'].sum() > 0
    assert rs['false_positives'] <= rs['calibration_games']
    sp, finished, _ = stub_selfplay(50, resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.0)
    rs = sp.resign_stats()
    assert rs['calibration_games'] == rs['false_positives'] == rs['histogram'].sum() == 0
    assert rs['resigned_games'] == sum(f[2] for f in finished.values()) > 0


@gpu
def test_resign_invariance():
    """Streams 1 and 2, eager and graphed, and 2 ranks x 32 games against
    1 rank x 64 leave the games and the resignation state unchanged."""
    from azalea_b200.engine import decode_replay_rows
    kw = dict(resign_threshold=STUB_THRESHOLD, resign_disable_prob=0.3, full_search_prob=0.5,
              fast_simulations=5)

    def play(streams, graph, **more):
        sp, finished, chosen = stub_selfplay(40, streams=streams, graph=graph, **kw, **more)
        return sp, chosen, sp.harvest(), sp.counters(), sp.eng.resign.cpu().numpy()
    sp0, c0, r0, n0, s0 = play(1, False)
    assert len(r0) > 0 and sp0.resign_stats()['resigned_games'] > 0
    for streams, graph in ((2, False), (2, True), (1, True)):
        _, c1, r1, n1, s1 = play(streams, graph)
        assert np.array_equal(c0, c1) and r0.tobytes() == r1.tobytes() and n0 == n1
        assert np.array_equal(s0, s1)
    parts = [play(1, False, G=32, rank=r, world_size=2) for r in range(2)]
    # slot s of the 64-game run plays the games of rank s // 32's slot s % 32
    assert np.array_equal(np.concatenate([p[4] for p in parts]), s0)
    hw = decode_replay_rows(r0, 5)[0]
    by_id = {}
    for i, gid in enumerate(hw['game_id']):
        by_id.setdefault(int(gid), []).append(i)
    seen = 0
    for part in parts:
        hp = decode_replay_rows(part[2], 5)[0]
        games = {}
        for i, gid in enumerate(hp['game_id']):
            games.setdefault(int(gid), []).append(i)
        for gid, idx in games.items():
            assert r0[by_id[gid]].tobytes() == part[2][idx].tobytes()
            seen += 1
    assert seen == len(by_id) > 0


@gpu
def test_resign_with_the_network():
    """6x64 network in the loop, packed leaves, two streams, a CUDA graph:
    a measure-only run picks a threshold with resign_threshold_for, and a run
    with it resigns games and keeps every engine status at 0."""
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.network import HexNetwork
    from azalea_b200.selfplay import resign_threshold_for
    torch.manual_seed(0)
    net = HexNetwork(5, 6, 64).eval().cuda()
    net.prepare_inference(torch.bfloat16)

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
    config = dict(seed=3, device='cuda', game='hex', network='HexNetwork', board_size=5,
                  num_blocks=1, base_chans=64, simulations=10, search_batch_size=5,
                  exploration_coef=0.5, exploration_temperature=1.0, exploration_depth=15,
                  exploration_noise_alpha=0.03, exploration_noise_scale=0.25,
                  replaybuf_size=256, replaybuf_oversampling=1, batch_size=128, lr_initial=0.01,
                  lr_decay_steps=100, lr_decay=0.5, momentum=0.9, l2_regularization=1e-4,
                  total_steps=4, log_interval=0, model_checkpoint_interval=0,
                  num_selfplay_games=32, resign_threshold=-0.2, resign_disable_prob=0.3)
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
