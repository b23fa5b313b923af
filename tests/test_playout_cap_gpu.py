"""Playout cap randomization (az_engine_set_playout_cap): each ply of each
game is a full search with probability p (one Philox coin per game id and
ply), otherwise a fast search of fast_descents new descents without root
noise whose replay row is not flushed."""
import numpy as np
import pytest
import torch

import oracle
from oracle import stubs
from oracle.philox import full_ply, game_ids

gpu = pytest.mark.gpu
AZ_PRIOR_LOGITS = 1

def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).tobytes()


def random_positions(G, n, rng):
    """Mid-game positions that cannot be won yet (X has fewer than n stones)."""
    boards = np.zeros((G, n * n), np.int8)
    colors = np.zeros(G, np.int32)
    for g in range(G):
        p = rng.randint(1, 2 * (n - 1) + 1)
        tiles = rng.permutation(n * n)[:p]
        boards[g, tiles[0::2]] = 1
        boards[g, tiles[1::2]] = 2
        colors[g] = 1 if p % 2 == 0 else 2
    return boards, colors


def stub_selfplay(moves, G=64, n=5, seed=3, graph=False, **kw):
    """Stub self-play, recording per move and slot the game id, the ply and
    the descents of the move (simulations counter delta), and the games that
    finished with their length and result."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=G, board_size=n, simulations=30,
                          search_batch_size=4, seed=seed, cuda_graph=graph, exploration_depth=4, **kw)
    plies, finished, chosen = {}, {}, []
    for _ in range(moves):
        gid, ply = game_ids(sp.eng)
        sims0 = sp.eng.counters[:, 0].cpu().numpy().copy()
        sp.step_move()
        desc = sp.eng.counters[:, 0].cpu().numpy() - sims0
        ch = sp.chosen.cpu().numpy().copy()
        chosen.append(ch)
        for g in range(G):
            plies[(int(gid[g]), int(ply[g]))] = int(desc[g])
            if ch[g, 2] != 0:
                finished[int(gid[g])] = (int(ch[g, 3]), int(ch[g, 2]))
    assert (sp.eng.status().cpu().numpy() == 0).all()
    return sp, plies, finished, np.stack(chosen)


# ------------------------------------------------------------------ tests --

@gpu
@pytest.mark.parametrize('n', (5, 7))
def test_cap_off_is_byte_identical(n):
    """full_search_prob=1.0 (off) gives the moves, replay bytes, counters and
    meta of an engine that never heard of the cap."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    out = []
    for kw in ({}, dict(full_search_prob=1.0)):
        sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=64, board_size=n, simulations=20,
                              search_batch_size=4, seed=3, cuda_graph=False, **kw)
        chosen = []
        for _ in range(30):
            sp.step_move()
            chosen.append(sp.chosen.cpu().numpy().copy())
        out.append((np.stack(chosen).tobytes(), sp.harvest().tobytes(),
                    sp.eng.counters.cpu().numpy().tobytes(), sp.eng.meta.cpu().numpy().tobytes()))
    assert len(out[0][1]) > 0
    assert out[0] == out[1]


@gpu
def test_fast_and_full_plies_match_the_oracle():
    """Engine driven as _window_body drives it, cap on with p = 0.5: every
    ply's new descents are exactly fast_descents or the full count, as the
    coin says, and the root (visits, W, priors, root N/W, node count) equals a
    dedicated oracle tree searched with the matching simulation count, bit for
    bit, with tree reuse across plies.  Moves (temperature 0) are a
    most-visited child.  The fast share is within 5 sigma of 1 - p."""
    from azalea_b200 import Engine
    n, G, sims, fast_sims, batch, coef, mode, seed = 5, 64, 60, 10, 6, 0.5, stubs.ROUGH, 7
    num_batches = sims // batch + 1
    full_d, fast_d = num_batches * batch, (fast_sims // batch + 1) * batch
    eng = Engine(G, n, max_batch=batch, seed=seed, nodes_per_game=200_000)
    eng.set_playout_cap(0.5, fast_d)
    trees = [oracle.Tree(max_nodes=2_000_000) for _ in range(G)]
    games = [oracle.Hex(n) for _ in range(G)]
    chosen = torch.zeros(G, 4, dtype=torch.int32, device='cuda')
    done = np.zeros(G, bool)
    counts = {fast_d: 0, full_d: 0}
    for _ in range(n * n):
        if done.all():
            break
        gid, ply = game_ids(eng)
        sims0 = eng.counters[:, 0].cpu().numpy().copy()
        fast0 = int(eng.counters[:, 15].sum())
        eng.select_root()
        eng.stub_eval(mode)
        eng.expand_root()
        for _ in range(num_batches):
            eng.select(batch, coef)
            eng.stub_eval(mode)
            eng.expand_backup()
        desc = eng.counters[:, 0].cpu().numpy() - sims0
        v, w, p, k, rnw, nodes = (x.cpu().numpy() for x in eng.root_stats())
        eng.play_commit(0.0, 0, False, False, False, chosen)
        ch = chosen.cpu().numpy()
        fast_now = 0
        for g in np.flatnonzero(~done):
            full = full_ply(seed, int(gid[g]), int(ply[g]), 0.5)
            assert desc[g] == (full_d if full else fast_d), (g, desc[g])
            counts[int(desc[g])] += 1
            fast_now += not full
            trees[g].sample_paths_stub(games[g], sims if full else fast_sims, batch, coef, mode)
            ov, ow, op = trees[g].root_stats()
            kg = int(k[g])
            where = (g, int(ply[g]))
            assert bits(v[g, :kg]) == bits(ov), where
            assert bits(w[g, :kg]) == bits(ow), where
            assert bits(p[g, :kg]) == bits(op), where
            assert bits(rnw[g]) == bits(trees[g].root_node()), where
            assert int(nodes[g]) == trees[g].num_nodes, where
            mid = int(ch[g, 1])
            assert ov[mid] == ov.max(), where
            trees[g].move(mid)
            games[g].step(int(ch[g, 0]))
            if ch[g, 2] != 0:
                assert games[g].result() == ch[g, 2]
                done[g] = True
        assert int(eng.counters[:, 15].sum()) - fast0 == fast_now
    assert done.all()
    total = counts[fast_d] + counts[full_d]
    assert counts[fast_d] > 0 and counts[full_d] > 0
    assert abs(counts[fast_d] / total - 0.5) < 5 * 0.5 / np.sqrt(total), counts
    assert (eng.status().cpu().numpy() == 0).all()


@gpu
def test_fast_plies_draw_no_noise():
    """Twin engines on the same positions, root noise 0.25 vs 0: with every
    ply fast (p = 0) the trees are bit-equal, with the cap off they differ."""
    from azalea_b200 import Engine
    G, n, B, seed = 256, 7, 8, 13
    boards, colors = random_positions(G, n, np.random.RandomState(2))
    for p, equal in ((0.0, True), (1.0, False)):
        stats = []
        for eps in (0.25, 0.0):
            eng = Engine(G, n, max_batch=B, seed=seed, nodes_per_game=65536)
            eng.set_playout_cap(p, 3 * B)
            eng.hex_set_state(boards, colors)
            eng.select_root()
            eng.stub_eval(stubs.ROUGH)
            eng.expand_root()
            for _ in range(3):
                eng.select(B, 0.5, eps, 0.03)
                eng.stub_eval(stubs.ROUGH)
                eng.expand_backup()
            assert int(eng.counters[:, 0].sum()) == G * 3 * B
            stats.append([x.cpu().numpy() for x in eng.root_stats()])
        same = all(np.array_equal(a, b) for a, b in zip(*stats))
        assert same == equal, p


@gpu
def test_replay_holds_exactly_the_full_plies():
    """Stub self-play with the cap on: the harvested (game id, ply) set is
    exactly the full plies of the finished games, rewards follow the row's ply
    parity and the result, game_len is the true length, reserved is 0, and
    replay_rows + fast plies = plies over the finished games.  The rows go
    through rows_to_dataframe and DeviceReplayBuffer, and Player.read counts
    games and moves right when a game's first or last ply left no row."""
    from azalea_b200.engine import decode_replay_rows
    from azalea_b200.replay_device import DeviceReplayBuffer
    from azalea_b200.selfplay import rows_to_dataframe
    sp, plies, finished, _ = stub_selfplay(60, full_search_prob=0.5, fast_simulations=5)
    full_d, fast_d = 32, 8
    assert set(plies.values()) <= {0, fast_d, full_d}
    rows = sp.harvest()
    h, boards, visits = decode_replay_rows(rows, 5)
    got = set(zip(h['game_id'].tolist(), h['ply'].tolist()))
    want = {(gid, ply) for (gid, ply), d in plies.items() if gid in finished and d == full_d}
    assert got == want and len(got) == len(h)
    for (gid, ply), d in plies.items():
        if gid in finished and ply < finished[gid][0]:
            assert d == (full_d if full_ply(3, gid, ply, 0.5) else fast_d)
    fast_finished = sum(1 for (gid, ply), d in plies.items() if gid in finished and d == fast_d)
    assert len(h) + fast_finished == sum(length for length, _ in finished.values())
    assert sp.counters()['replay_rows'] == len(h)
    for i in range(len(h)):
        length, result = finished[int(h['game_id'][i])]
        assert h['game_len'][i] == length and h['result'][i] == result
        rw = np.float32(result - 2)
        assert h['reward'][i] == (-rw if h['ply'][i] % 2 else rw)
        assert h['reserved'][i] == 0
    # games whose first / last ply was fast are in the sample
    first = {gid for gid in finished if (gid, 0) not in got}
    last = {gid for gid, (length, _) in finished.items() if (gid, length - 1) not in got}
    assert first and last
    df = rows_to_dataframe(rows, 5)
    assert len(df) == len(h)
    buf = DeviceReplayBuffer(len(h) + 7, 5)
    buf.put(torch.from_numpy(rows).cuda())
    gen = torch.Generator(device='cuda').manual_seed(4)
    batch = buf.sample(64, generator=gen)
    idx = torch.randint(0, len(buf), (64,), device='cuda',
                        generator=torch.Generator(device='cuda').manual_seed(4)).cpu().numpy()
    assert np.array_equal(batch['reward'].cpu().numpy(), h['reward'][idx])
    assert np.array_equal(batch['color'].cpu().numpy(), h['color'][idx])
    assert np.allclose(batch['moves_prob'].sum(1).cpu().numpy(), 1.0, atol=1e-5)

    # Player.read: games by id, lengths from game_len
    import azalea_b200 as az
    from azalea_b200.parallel_player import Player
    pol = az.Policy()
    pol.net = az.StubEvaluator(stubs.ROUGH)
    pol.simulations, pol.search_batch_size, pol.exploration_coef = 30, 4, 0.5
    pol.exploration_depth, pol.exploration_temperature = 4, 1.0
    pol.exploration_noise_alpha, pol.exploration_noise_scale = 0.03, 0.25
    agent = az.AzaleaAgent(lambda: az.HexGame(5), policy=pol)
    player = Player(None, [agent], num_games=64, seed=3, cuda_graph=False,
                    full_search_prob=0.5, fast_simulations=5)
    assert player.sp.fast_descents == fast_d
    seen = []
    harvest = player.sp.harvest
    player.sp.harvest = lambda **kw: seen.append(harvest(**kw)) or seen[-1]
    examples, metrics = player.read(300)
    cnt = player.sp.counters()
    hr = decode_replay_rows(np.concatenate(seen), 5)[0]
    lengths = {int(g): int(L) for g, L in zip(hr['game_id'], hr['game_len'])}
    assert metrics['games'] == len(lengths) <= cnt['games']     # (a game of fast plies only has no rows)
    assert metrics['moves_per_game'] == sum(lengths.values())
    assert metrics['fast_plies'] == cnt['fast_plies'] > 0
    assert len(examples) == len(hr) == cnt['replay_rows']
    starts = {int(g) for g, p in zip(hr['game_id'], hr['ply']) if p == 0}
    assert len(starts) < len(lengths)           # (counting ply-0 rows would miss games)


@gpu
def test_cap_selfplay_invariance():
    """Cap on: with the network and packed leaves, one vs two streams and
    eager vs graphed give the same moves and replay bytes; with the stub,
    2 ranks x 32 games play the games 1 rank x 64 plays."""
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.engine import decode_replay_rows
    from azalea_b200.network import HexNetwork
    torch.manual_seed(0)
    net = HexNetwork(5, 2, 64).eval().cuda()
    net.prepare_inference(torch.bfloat16)

    def play(streams, graph):
        sp = LockstepSelfPlay(net, num_games=64, board_size=5, simulations=40, search_batch_size=8,
                              seed=5, streams=streams, cuda_graph=graph, full_search_prob=0.5,
                              fast_simulations=10)
        assert sp.pack_leaves and sp.fast_descents == 16
        chosen = []
        for _ in range(30):
            sp.step_move()
            chosen.append(sp.chosen.cpu().numpy().copy())
        assert (sp.eng.status().cpu().numpy() == 0).all()
        return np.stack(chosen), sp.harvest(), sp.counters()
    c0, r0, n0 = play(1, False)
    assert len(r0) > 0 and 0 < n0['fast_plies'] < n0['plies']
    for streams, graph in ((2, False), (2, True), (1, True)):
        c1, r1, n1 = play(streams, graph)
        assert np.array_equal(c0, c1) and r0.tobytes() == r1.tobytes() and n0 == n1

    whole = stub_selfplay(40, full_search_prob=0.5, fast_simulations=5)[0].harvest()
    parts = [stub_selfplay(40, G=32, rank=r, world_size=2, full_search_prob=0.5,
                           fast_simulations=5)[0].harvest() for r in range(2)]
    hw = decode_replay_rows(whole, 5)[0]
    by_id = {}
    for i, gid in enumerate(hw['game_id']):
        by_id.setdefault(int(gid), []).append(i)
    seen = 0
    for part in parts:
        hp = decode_replay_rows(part, 5)[0]
        games = {}
        for i, gid in enumerate(hp['game_id']):
            games.setdefault(int(gid), []).append(i)
        for gid, idx in games.items():
            assert whole[by_id[gid]].tobytes() == part[idx].tobytes()
            seen += 1
    assert seen == len(by_id) > 0


@gpu
def test_capped_games_cost_no_network_rows():
    """Packed leaves, every ply fast: once a move's fast budget is spent the
    games emit no leaves, the window's live row count is 0 and nn_rows stops
    growing; the next move searches again."""
    from azalea_b200 import Engine
    G, n, B = 128, 7, 8
    nn = n * n
    boards, colors = random_positions(G, n, np.random.RandomState(5))
    eng = Engine(G, n, max_batch=B, seed=1, nodes_per_game=65536, pack_leaves=True)
    eng.set_playout_cap(0.0, 2 * B)
    eng.hex_set_state(boards, colors)
    gen = torch.Generator(device='cuda').manual_seed(0)
    chosen = torch.zeros(G, 4, dtype=torch.int32, device='cuda')
    for move in range(2):
        eng.select_root()
        eng.prior[:, 0] = torch.randn(G, nn, device='cuda', generator=gen)
        eng.expand_root(None, AZ_PRIOR_LOGITS)
        for it in range(5):
            rows0 = int(eng.counters[:, 11].sum())
            eng.select(B, 0.5)
            live = int(eng.leaf_rows[0])
            grown = int(eng.counters[:, 11].sum()) - rows0
            assert live == grown
            if it < 2:
                assert live > 0
            else:
                assert live == 0 and (eng.leaf_info[..., 0] == -1).all()
            eng.value.view(-1).copy_(torch.rand(G * B, device='cuda', generator=gen) * 2 - 1)
            eng.prior.view(-1, nn).copy_(torch.randn(G * B, nn, device='cuda', generator=gen))
            eng.expand_backup(None, None, AZ_PRIOR_LOGITS)
        if move == 0:
            assert int(eng.counters[:, 0].sum()) == G * 2 * B
        eng.play_commit(1.0, 15, True, False, False, chosen)
    assert int(eng.counters[:, 15].sum()) == int(eng.counters[:, 5].sum()) >= G
    assert (eng.status().cpu().numpy() == 0).all()


@gpu
def test_train_with_playout_cap(tmp_path):
    """train(...) with full_search_prob / fast_simulations: the self-play
    refills put only rows of full-search plies into the replay buffer."""
    import azalea_b200 as az
    from azalea_b200 import policy_trainer
    from azalea_b200.engine import decode_replay_rows
    config = dict(seed=3, device='cuda', game='hex', network='HexNetwork', board_size=5,
                  num_blocks=1, base_chans=64, simulations=10, search_batch_size=5,
                  exploration_coef=0.5, exploration_temperature=1.0, exploration_depth=15,
                  exploration_noise_alpha=0.03, exploration_noise_scale=0.25,
                  replaybuf_size=256, replaybuf_oversampling=1, batch_size=128, lr_initial=0.01,
                  lr_decay_steps=100, lr_decay=0.5, momentum=0.9, l2_regularization=1e-4,
                  total_steps=4, log_interval=0, model_checkpoint_interval=0,
                  num_selfplay_games=32, full_search_prob=0.5, fast_simulations=2)
    policy = az.Policy()
    policy.initialize(config)
    buf = policy_trainer.initialize_replay_buffer(None, lambda: az.HexGame(5), 256, num_games=32,
                                                  device='cuda', seed=3)
    put, rows = buf.put, []
    buf.put = lambda r: rows.append(r.cpu().numpy()) or put(r)
    policy_trainer.train(policy, config, str(tmp_path), replaybuf=buf)
    hist = policy_trainer.train.history
    assert len(hist) == 4 and all(np.isfinite(x['loss']) for x in hist)
    assert rows
    h = decode_replay_rows(np.concatenate(rows), 5)[0]
    seed = 3 & 0x7fffffff
    assert all(full_ply(seed, int(g), int(p), 0.5) for g, p in zip(h['game_id'], h['ply']))
    assert (h['reserved'] == 0).all()
    # (a refill takes whole games: the fast plies are what is missing)
    assert len(h) < sum({int(g): int(L) for g, L in zip(h['game_id'], h['game_len'])}.values())
    assert 'full_search_prob' not in policy.state_dict()
