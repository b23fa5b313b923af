"""GPU tests of lockstep self-play: play_commit, replay rows, determinism,
world-size invariance, the network evaluator glue and the Player facade."""
import numpy as np
import pytest
import torch

import oracle
from oracle import stubs

pytestmark = pytest.mark.gpu


def run_selfplay(G=128, n=7, sims=60, batch=6, seed=3, rank=0, world=1,
                 moves=60, mode=stubs.ROUGH, graph=False, **kw):
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    sp = LockstepSelfPlay(StubEvaluator(mode), num_games=G, board_size=n,
                          simulations=sims, search_batch_size=batch,
                          exploration_depth=6, seed=seed, rank=rank,
                          world_size=world, cuda_graph=graph,
                          move_exploration=kw.pop('noise', False), **kw)
    rows = []
    for _ in range(moves):
        sp.step_move()
        if sp.eng.replay_count():
            rows.append(sp.harvest())
    assert (sp.eng.status().cpu().numpy() == 0).all()
    return sp, np.concatenate(rows)


def split_games(rows, n):
    from azalea_b200.engine import decode_replay_rows
    h, board, visits = decode_replay_rows(rows, n)
    games = {}
    for i in range(len(h)):
        games.setdefault(int(h['game_id'][i]), []).append(i)
    return h, board, visits, games


def test_replay_rows_are_consistent_games():
    """Every finished game: plies 0..L-1, each row's board is the previous
    one plus the recorded move, colours alternate, the visit vector belongs
    to that position, rewards follow play_game.py:63-67, and the oracle
    agrees on the winner."""
    n, sims, batch = 7, 60, 6
    sp, rows = run_selfplay(n=n, sims=sims, batch=batch)
    h, board, visits, games = split_games(rows, n)
    assert len(games) >= 100
    per_move = (sims // batch + 1) * batch
    for gid, idx in games.items():
        L = len(idx)
        assert list(h['ply'][idx]) == list(range(L))
        assert (h['game_len'][idx] == L).all()
        game = oracle.Hex(n)
        for r, i in enumerate(idx):
            assert (board[i] == game.board).all()
            assert h['color'][i] == game.color - 1 == r % 2
            legal = game.legal_moves()
            assert h['num_moves'][i] == len(legal)
            assert legal[h['move_id'][i]] == h['move'][i]
            v = visits[i]
            assert (v[len(legal):] == 0).all()
            assert v[h['move_id'][i]] > 0          # sampled moves were visited
            # every batch backs up at least one leaf; duplicates inside a
            # batch are backed up once (mcts.py:75)
            assert v.sum() >= sims // batch + 1
            assert h['temperature'][i] == (1.0 if r < 6 else 0.0)
            if r >= 6:
                assert v[h['move_id'][i]] == v.max()
            game.step(int(h['move'][i]))
        result = game.result()
        assert result in (1, 3) and (h['result'][idx] == result).all()
        want = np.full(L, result - 2.0, dtype=np.float32)
        want[1::2] *= -1
        assert (h['reward'][idx] == want).all()
    cnt = sp.counters()
    assert cnt['games'] >= len(games) and cnt['plies'] == 60 * 128
    assert cnt['simulations'] == 60 * 128 * per_move


def test_selfplay_is_deterministic_and_graph_equals_eager():
    _, a = run_selfplay(G=64, moves=40)
    _, b = run_selfplay(G=64, moves=40)
    _, c = run_selfplay(G=64, moves=40, graph=True)
    assert a.tobytes() == b.tobytes()
    assert a.tobytes() == c.tobytes()


def test_world_size_invariance():
    """Games are keyed by global game id: 2 ranks x 32 games play exactly the
    games one rank x 64 plays (first game of every slot)."""
    n = 7
    _, whole = run_selfplay(G=64, n=n, moves=45, world=1)
    parts = [run_selfplay(G=32, n=n, moves=45, rank=r, world=2)[1]
             for r in range(2)]
    hw, bw, vw, gw = split_games(whole, n)
    first = {gid: idx for gid, idx in gw.items() if gid < 64}
    assert len(first) == 64
    seen = 0
    for part in parts:
        hp, bp, vp, gp = split_games(part, n)
        for gid, idx in gp.items():
            if gid >= 64:
                continue
            ref = first[gid]
            assert len(ref) == len(idx)
            assert (hw['move'][ref] == hp['move'][idx]).all()
            assert vw[ref].tobytes() == vp[idx].tobytes()
            seen += 1
    assert seen == 64


def test_rows_to_dataframe_matches_reference_format():
    from azalea_b200.selfplay import rows_to_dataframe
    n = 5
    _, rows = run_selfplay(G=32, n=n, sims=40, batch=4, moves=30)
    df = rows_to_dataframe(rows, n)
    assert len(df) == len(rows)
    rec = df[0]
    assert rec.state.board.dtype == np.int32 and rec.state.board.shape == (n, n)
    assert rec.state.legal_moves.dtype == np.int32
    assert rec.moves_prob.dtype == np.float32
    assert abs(rec.moves_prob.sum() - 1) < 1e-5
    assert isinstance(rec.reward, np.float32) and rec.reward in (-1.0, 1.0)
    assert len(rec.moves_prob) == len(rec.state.legal_moves)


def test_logits_prior_path_matches_torch():
    """AZ_PRIOR_LOGITS (gather legal tiles -> log-softmax -> exp in the
    expand kernel, with the perspective flip) vs the same in torch fp32:
    priors within 1e-6 absolute."""
    from azalea_b200 import Engine, _cabi
    n, G = 11, 64
    eng = Engine(G, n, max_batch=10)
    rng = np.random.RandomState(0)
    # random positions, both colours to move
    boards = np.zeros((G, n * n), dtype=np.int8)
    colors = np.zeros(G, dtype=np.int32)
    for g in range(G):
        stones = rng.randint(0, 60)
        tiles = rng.choice(n * n, size=stones, replace=False)
        boards[g, tiles[0::2]] = 1
        boards[g, tiles[1::2]] = 2
        colors[g] = 1 + (stones % 2)
    eng.hex_set_state(boards, colors)
    eng.select_root()
    logits = torch.randn(G, 10, n * n, device=eng.device) * 3
    eng.expand_root(logits.contiguous(), _cabi.AZ_PRIOR_LOGITS)
    prior = eng.root_stats()[2].cpu().numpy()
    k = eng.root_stats()[3].cpu().numpy()
    info = eng.leaf_info.cpu().numpy()
    lg = logits[:, 0].cpu().numpy()
    for g in range(G):
        empt = np.flatnonzero(boards[g] == 0)
        assert k[g] == len(empt)
        assert (info[g, 0, 1] >> 8) & 1 == colors[g] - 1
        view = empt if colors[g] == 1 else \
            (n - 1 - empt % n) * n + (n - 1 - empt // n)
        want = torch.softmax(torch.tensor(lg[g, view]), 0).numpy()
        assert np.abs(prior[g, :len(empt)] - want).max() < 1e-6
    # and the network-view boards the evaluator sees are the reference's
    cells = eng.leaf_board.cpu().numpy()[:, 0, :n * n].reshape(G, n, n)
    from azalea_b200 import HexGame
    for g in range(G):
        b = boards[g].reshape(n, n).astype(np.int32)
        want = b if colors[g] == 1 else HexGame.flip_player_board(b)[0]
        assert (cells[g] == want).all()


def test_network_selfplay_runs_with_and_without_graph():
    """6x64 network in the loop (bf16, folded BN): moves are legal, games
    finish, replay rows come out; CUDA-graph replay gives the same games."""
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.network import HexNetwork
    outs = []
    for graph in (False, True):
        torch.manual_seed(0)
        net = HexNetwork(7, 2, 32).eval().cuda()
        sp = LockstepSelfPlay(net, num_games=32, board_size=7, simulations=40,
                              search_batch_size=8, seed=1, cuda_graph=graph,
                              move_exploration=False)
        rows = []
        for _ in range(55):
            sp.step_move()
            if sp.eng.replay_count():
                rows.append(sp.harvest())
        assert (sp.eng.status().cpu().numpy() == 0).all()
        rows = np.concatenate(rows)
        h, board, visits, games = split_games(rows, 7)
        assert len(games) >= 32
        for gid, idx in games.items():
            game = oracle.Hex(7)
            for i in idx:
                assert (board[i] == game.board).all()
                game.step(int(h['move'][i]))
            assert game.result() == h['result'][idx[0]]
        outs.append(h['move'][:64].copy())
    # bf16 cuDNN kernels may be picked differently under capture; the first
    # plies (identical inputs, deterministic kernels) must agree
    assert (outs[0][:8] == outs[1][:8]).all()


def test_player_facade():
    """Player(pool, agents).read(size) -> (ReplayDataFrame, metrics), the
    reference's call (parallel_player.py:17-28)."""
    import azalea_b200 as az
    p = az.Policy()
    torch.manual_seed(0)
    p.initialize(dict(device='cuda', network='HexNetwork', board_size=5,
                      num_blocks=1, base_chans=16, simulations=30,
                      search_batch_size=5, exploration_coef=0.5,
                      exploration_depth=4, exploration_noise_alpha=0.03,
                      exploration_noise_scale=0.25,
                      exploration_temperature=1.0, seed=7))
    agent = az.AzaleaAgent(lambda: az.HexGame(5), policy=p)
    agent.settings['move_sampling'] = True
    agent.settings['move_exploration'] = True
    player = az.Player(None, [agent], num_games=64)
    df, metrics = player.read(200)
    assert len(df) >= 200
    assert metrics['games'] > 0 and metrics['game_error'] == 0
    assert 5 <= metrics['moves_per_game'] / metrics['games'] <= 25


@pytest.mark.parametrize('n,chans', ((11, 64), (7, 32), (19, 64)))
def test_evaluator_glue_kernels_match_torch(n, chans):
    """az_nn_stem / az_nn_heads (csrc/az_nn_glue.cuh) against plain PyTorch
    fp32 of the same layers (network.py:68-85,138-142): one bf16 rounding of
    the output is the only difference allowed (rel 2^-8 + abs 1e-3)."""
    import ctypes
    import torch.nn.functional as F
    from azalea_b200 import _cabi
    from azalea_b200.network import HexNetwork, _fold
    torch.manual_seed(n)
    net = HexNetwork(n, 2, chans).eval().cuda()
    gen = torch.Generator(device='cuda').manual_seed(1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen, device='cuda') * 0.2)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen, device='cuda') + 0.5)
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=gen, device='cuda') + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen, device='cuda') * 0.2)
    net.prepare_inference(torch.bfloat16)
    f = net._fast
    N, nn = 257, n * n
    cs = (nn + 15) & ~15
    cells = torch.zeros(N, cs, dtype=torch.int8, device='cuda')
    cells[:, :nn] = torch.randint(0, 3, (N, nn), device='cuda', dtype=torch.int8)
    L = _cabi.lib()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    # stem
    out = torch.empty(N, n, n, chans, dtype=torch.bfloat16, device='cuda')
    _cabi.check(L.az_nn_stem(ctypes.c_void_p(cells.data_ptr()), cs, n, N,
                             ctypes.c_void_p(f['stem_table'].data_ptr()),
                             ctypes.c_void_p(f['stem_bias'].data_ptr()),
                             ctypes.c_void_p(out.data_ptr()), chans, 0, stream))
    with torch.no_grad():
        x = net.encoder(cells[:, :nn].long().view(N, n, n)).permute(0, 3, 1, 2)
        want = F.relu(net.bn1(net.conv1(x))).permute(0, 2, 3, 1)
    got = out.float()
    tol = want.abs() * 2 ** -6 + 2e-2       # table entries are bf16 too
    assert ((got - want).abs() <= tol).all(), float((got - want).abs().max())
    # heads
    xin = (torch.randn(N * nn, chans, device='cuda') * 0.7).to(torch.bfloat16)
    hout = torch.empty(N * nn, 6, dtype=torch.bfloat16, device='cuda')
    _cabi.check(L.az_nn_heads(ctypes.c_void_p(xin.data_ptr()), N * nn,
                              ctypes.c_void_p(f['heads_w32'].data_ptr()),
                              ctypes.c_void_p(f['heads_b32'].data_ptr()),
                              ctypes.c_void_p(hout.data_ptr()), 0, chans, 6, 0, stream))
    want = F.relu(xin.float() @ f['heads_w32'].t() + f['heads_b32'])
    got = hout.float()
    assert ((got - want).abs() <= want.abs() * 2 ** -7 + 1e-3).all()
    # whole evaluator: bf16 glue path vs the reference-interface fp32 path
    value, logits = net.evaluate_cells(cells)
    with torch.no_grad():
        moves = torch.arange(1, nn + 1, device='cuda', dtype=torch.int32).repeat(N, 1)
        ref = net.run(dict(board=cells[:, :nn].view(N, n, n).int(), legal_moves=moves))
    assert (value - ref['value']).abs().max() < 0.05
    want_lp = ref['moves_logprob']
    got_lp = torch.log_softmax(logits, 1)
    assert (got_lp - want_lp).abs().max() < 0.25
    assert (got_lp - want_lp).abs().mean() < 0.02


@pytest.mark.parametrize('n,N', ((11, 257), (19, 13), (7, 1000), (5, 3)))
def test_evaluator_glue_kernels_slab_layout(n, N):
    """The slab-layout stem and heads (k_nn_stem_slab / k_nn_heads_slab, the
    two ends of the tcgen05 tower) against the plain-layout kernels on the
    same inputs.  Summation order differs (and the slab stem pre-adds the
    three taps of a kernel row into one bf16 table entry), so outputs may
    differ by a bf16 rounding or two (rel 2^-6 + abs 1e-2 for the stem, rel
    2^-7 + abs 1e-3 for the heads); everything that is not a board cell stays
    zero."""
    import ctypes
    from azalea_b200 import _cabi, tower_layout as tl
    from azalea_b200.network import HexNetwork
    torch.manual_seed(n)
    net = HexNetwork(n, 1, 64).eval().cuda()
    net.prepare_inference(torch.bfloat16)
    f = net._fast
    nn = n * n
    cs = (nn + 15) & ~15
    cells = torch.zeros(N, cs, dtype=torch.int8, device='cuda')
    cells[:, :nn] = torch.randint(0, 3, (N, nn), device='cuda', dtype=torch.int8)
    L = _cabi.lib()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    plain = torch.empty(N, n, n, 64, dtype=torch.bfloat16, device='cuda')
    slab = torch.zeros(tl.buffer_rows(n, N), 64, dtype=torch.bfloat16, device='cuda')
    for out, padded in ((plain, 0), (slab, 1)):
        _cabi.check(L.az_nn_stem(p(cells), cs, n, N, p(f['stem_table']), p(f['stem_bias']),
                                 p(out), 64, padded, stream))
    got, rest = tl.from_slabs(slab, n, N)
    bpg = tl.boards_per_group(n)
    assert rest == 0.0
    assert ((got.float() - plain.float()).abs() <= plain.float().abs() * 2 ** -6 + 1e-2).all()
    # unused board slots of the last group are never written by the stem
    full = tl.from_slabs(slab, n, (N + bpg - 1) // bpg * bpg)[0]
    assert float(full[N:].float().abs().sum()) == 0.0
    # heads
    x = (torch.randn(N, n, n, 64, device='cuda') * 0.7).to(torch.bfloat16)
    h_plain = torch.empty(N * nn, 6, dtype=torch.bfloat16, device='cuda')
    h_slab = torch.full((N * nn + 7, 6), 7.0, dtype=torch.bfloat16, device='cuda')
    _cabi.check(L.az_nn_heads(p(x), N * nn, p(f['heads_w32']), p(f['heads_b32']), p(h_plain), 0, 64, 6, 0, stream))
    xs = tl.to_slabs(x)
    _cabi.check(L.az_nn_heads(p(xs), N * nn, p(f['heads_w32']), p(f['heads_b32']), p(h_slab),
                              0, 64, 6, n, stream))
    assert (h_slab[N * nn:] == 7.0).all()           # nothing written past the last board
    a, b = h_slab[:N * nn].float(), h_plain.float()
    assert ((a - b).abs() <= b.abs() * 2 ** -7 + 1e-3).all()
    # padded board rows (a GEMM-friendly K): the padding is left alone
    stride = (nn * 6 + 7) // 8 * 8 + 8
    h_pad = torch.full((N + 1, stride), 7.0, dtype=torch.bfloat16, device='cuda')
    _cabi.check(L.az_nn_heads(p(xs), N * nn, p(f['heads_w32']), p(f['heads_b32']), p(h_pad),
                              stride, 64, 6, n, stream))
    assert torch.equal(h_pad[:N, :nn * 6].reshape(N * nn, 6), h_slab[:N * nn])
    assert (h_pad[:N, nn * 6:] == 7.0).all() and (h_pad[N] == 7.0).all()


def test_device_replay_buffer_collate_matches_host_format():
    """DeviceReplayBuffer.sample == prep.torch_batch_replays over the same
    rows (prep.py:24-39,70-86): boards, ascending zero-padded legal moves,
    pi = as_distribution(visits, T) as float32 (1e-6), rewards; FIFO
    wraparound and the fresh-counter accounting of replay_buffer.py:121-149;
    a training step of the reference loss runs on the sampled batch."""
    import azalea_b200 as az
    from azalea_b200.selfplay import rows_to_dataframe
    n = 5
    _, rows = run_selfplay(G=64, n=n, sims=40, batch=4, moves=30)
    buf = az.DeviceReplayBuffer(len(rows) + 7, n)
    buf.put(torch.from_numpy(rows).cuda())
    assert len(buf) == len(rows) and buf.fresh_counter == len(rows)
    idx = torch.arange(len(rows))
    batch = buf.collate(idx)
    df = rows_to_dataframe(rows, n)
    K = max(len(s.legal_moves) for s in df.state)
    assert batch['legal_moves'].shape == (len(rows), K)
    assert batch['board'].dtype == torch.int32 and batch['color'].dtype == torch.int64
    lm = batch['legal_moves'].cpu().numpy()
    mp = batch['moves_prob'].cpu().numpy()
    bd = batch['board'].cpu().numpy()
    for i in range(len(rows)):
        k = len(df.state[i].legal_moves)
        assert (bd[i] == df.state[i].board).all()
        assert (lm[i, :k] == df.state[i].legal_moves).all() and (lm[i, k:] == 0).all()
        assert np.abs(mp[i, :k] - df.moves_prob[i]).max() < 1e-6
        assert (mp[i, k:] == 0).all()
    assert (batch['reward'].cpu().numpy() == np.array(df.reward)).all()
    assert (batch['color'].cpu().numpy() == [s.color for s in df.state]).all()
    assert (batch['result'].cpu().numpy() == 0).all()
    # wraparound keeps the newest rows (replay_buffer.py:134-149)
    buf.put(torch.from_numpy(rows[:10]).cuda())
    assert buf.write_idx == 3 and len(buf) == len(rows) + 7
    assert (buf.rows[:3].cpu().numpy() == rows[7:10]).all()
    # the reference's supervised step consumes the sampled batch
    torch.manual_seed(0)
    net = az.network.HexNetwork(n, 1, 16).cuda().train()
    out, loss = net.run(buf.sample(32), compute_loss=True)
    loss.backward()
    assert torch.isfinite(loss) and out['value'].shape == (32,)


def test_player_read_device_feeds_replay_buffer():
    import azalea_b200 as az
    p = az.Policy()
    torch.manual_seed(0)
    p.initialize(dict(device='cuda', network='HexNetwork', board_size=5,
                      num_blocks=1, base_chans=32, simulations=30,
                      search_batch_size=5, exploration_coef=0.5,
                      exploration_depth=4, exploration_noise_alpha=0.03,
                      exploration_noise_scale=0.25,
                      exploration_temperature=1.0, seed=7))
    agent = az.AzaleaAgent(lambda: az.HexGame(5), policy=p)
    agent.settings['move_sampling'] = True
    agent.settings['move_exploration'] = True
    player = az.Player(None, [agent], num_games=64)
    buf = az.DeviceReplayBuffer(500, 5)
    buf.consume(0, player)
    assert len(buf) == 0
    metrics = buf.consume(128, player)
    assert len(buf) >= 128 and metrics['games'] > 0
    assert buf.fresh_counter >= 0
    batch = buf.sample(64, trim=False)
    assert batch['legal_moves'].shape == (64, 25)
    assert torch.allclose(batch['moves_prob'].sum(1), torch.ones(64, device='cuda'), atol=1e-5)


@pytest.mark.parametrize('n,N', ((11, 64), (11, 1029), (19, 9), (7, 91), (5, 1), (11, 4100),
                                 (2, 1), (2, 300), (3, 33), (11, 1480), (11, 1490), (13, 2000)))
def test_tcgen05_conv3x3_matches_torch(n, N):
    """az_nn_conv3x3 (csrc/az_tower.cuh: tcgen05 implicit GEMM over the slab
    layout, N = 192 tap stacking, TMEM accumulator ring) against F.conv2d in
    fp32 on the same bf16 inputs: bias, ReLU, residual, in place; everything
    that is not a real cell stays zero.  Tolerance = one bf16 rounding of the
    output (2^-8 relative + 1e-2)."""
    import ctypes
    import torch.nn.functional as F
    from azalea_b200 import _cabi, tower_layout as tl
    L = _cabi.lib()
    assert L.az_nn_tower_rows(n, N) == tl.buffer_rows(n, N)
    assert L.az_nn_tower_group(n) == tl.boards_per_group(n)
    torch.manual_seed(n)
    x = (torch.randn(N, n, n, 64, device='cuda') * 0.5).to(torch.bfloat16)
    r = (torch.randn(N, n, n, 64, device='cuda') * 0.5).to(torch.bfloat16)
    w = (torch.randn(64, 64, 3, 3, device='cuda') * 0.05).to(torch.bfloat16)
    b = torch.randn(64, device='cuda') * 0.1
    xp, rp, wp = tl.to_slabs(x), tl.to_slabs(r), tl.pack_conv_weights(w)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    for use_res in (False, True):
        out = rp.clone() if use_res else torch.zeros_like(xp)     # residual case runs in place
        _cabi.check(L.az_nn_conv3x3(p(xp), p(wp), p(b), p(out) if use_res else None, p(out), n, N, stream))
        got, rest = tl.from_slabs(out, n, N)
        want = F.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), b, padding=1)
        if use_res:
            want = want + r.permute(0, 3, 1, 2).float()
        want = F.relu(want).permute(0, 2, 3, 1)
        assert ((got.float() - want).abs() <= want.abs() * 2 ** -8 + 1e-2).all()
        assert rest == 0.0


@pytest.mark.parametrize('n,N', ((11, 64), (11, 1029), (19, 9), (7, 91), (5, 1), (11, 4100),
                                 (2, 1), (2, 300), (3, 33), (11, 1480), (13, 2000), (11, 40960)))
def test_fused_resblock_equals_two_launches(n, N):
    """az_nn_resblock (csrc/az_block.cuh: conv1 and conv2 of a residual block on
    a cluster of two CTAs, the intermediate slabs handed over through
    distributed shared memory) is the SAME arithmetic as two az_nn_conv3x3
    launches -- same MMAs in the same order, same bf16 rounding of the
    intermediate -- so the outputs are bit-identical; and both match
    network.py:17-39 evaluated in fp32 within two bf16 roundings.  Two blocks
    back to back (different weights), in place, as the tower runs them."""
    import ctypes
    import torch.nn.functional as F
    from azalea_b200 import _cabi, tower_layout as tl
    L = _cabi.lib()
    torch.manual_seed(100 + n)
    x = (torch.randn(N, n, n, 64, device='cuda') * 0.5).to(torch.bfloat16)
    ws = [(torch.randn(64, 64, 3, 3, device='cuda') * 0.05).to(torch.bfloat16) for _ in range(4)]
    bs = [torch.randn(64, device='cuda') * 0.1 for _ in range(4)]
    wp = [tl.pack_conv_weights(w) for w in ws]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    # two launches per block
    xa, ya = tl.to_slabs(x), torch.zeros_like(tl.to_slabs(x))
    for blk in range(2):
        _cabi.check(L.az_nn_conv3x3(p(xa), p(wp[2 * blk]), p(bs[2 * blk]), None, p(ya), n, N, stream))
        _cabi.check(L.az_nn_conv3x3(p(ya), p(wp[2 * blk + 1]), p(bs[2 * blk + 1]), p(xa), p(xa), n, N, stream))
    # one launch per block
    xb = tl.to_slabs(x)
    scratch = torch.zeros(max(16, L.az_nn_resblock_scratch_bytes()), dtype=torch.uint8, device='cuda')
    for blk in range(2):
        w12 = torch.cat([wp[2 * blk], wp[2 * blk + 1]]).contiguous()
        b12 = torch.cat([bs[2 * blk], bs[2 * blk + 1]]).contiguous()
        _cabi.check(L.az_nn_resblock(p(xb), p(w12), p(b12), p(scratch), n, N, stream))
    torch.cuda.synchronize()
    assert torch.equal(xa.view(torch.int16), xb.view(torch.int16))
    got, rest = tl.from_slabs(xb, n, N)
    assert rest == 0.0
    # fp32 reference with the intermediate rounded to bf16 where the kernels round it
    t = x.permute(0, 3, 1, 2).float()
    for blk in range(2):
        y = F.relu(F.conv2d(t, ws[2 * blk].float(), bs[2 * blk], padding=1)).to(torch.bfloat16).float()
        t = F.relu(F.conv2d(y, ws[2 * blk + 1].float(), bs[2 * blk + 1], padding=1) + t)
        t = t.to(torch.bfloat16).float()
    want = t.permute(0, 2, 3, 1)
    assert ((got.float() - want).abs() <= want.abs() * 2 ** -7 + 2e-2).all()


def test_fused_resblock_concurrent_streams():
    """Two instances of the fused block running concurrently on two streams
    (what LockstepSelfPlay(streams=2) does) on their own buffers: results
    equal the single-stream ones.  (The two-launch kernel's first residual
    variant died in exactly this situation, DESIGN.md 3.5.)"""
    import ctypes
    from azalea_b200 import _cabi, tower_layout as tl
    L = _cabi.lib()
    n, N = 11, 10240
    torch.manual_seed(7)
    x = (torch.randn(N, n, n, 64, device='cuda') * 0.5).to(torch.bfloat16)
    w12 = torch.cat([tl.pack_conv_weights((torch.randn(64, 64, 3, 3, device='cuda') * 0.05).to(torch.bfloat16))
                     for _ in range(2)]).contiguous()
    b12 = (torch.randn(128, device='cuda') * 0.1).contiguous()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    ref = tl.to_slabs(x)
    # one hand-over ring per stream that launches concurrently
    scr = [torch.zeros(max(16, L.az_nn_resblock_scratch_bytes()), dtype=torch.uint8, device='cuda') for _ in range(2)]
    st0 = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    reps = 30
    for _ in range(reps):
        _cabi.check(L.az_nn_resblock(p(ref), p(w12), p(b12), p(scr[0]), n, N, st0))
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(2)]
    bufs = [tl.to_slabs(x) for _ in streams]
    torch.cuda.synchronize()
    for _ in range(reps):
        for s, b, sc in zip(streams, bufs, scr):
            _cabi.check(L.az_nn_resblock(p(b), p(w12), p(b12), p(sc), n, N, ctypes.c_void_p(s.cuda_stream)))
    torch.cuda.synchronize()
    for b in bufs:
        assert torch.equal(b.view(torch.int16), ref.view(torch.int16))


@pytest.mark.parametrize('n,N,K', ((11, 1, 6), (11, 64, 6), (11, 1029, 3), (19, 9, 6), (2, 1, 6), (2, 300, 2),
                                   (3, 33, 6), (7, 91, 6), (13, 2000, 6), (11, 4100, 10), (11, 40960, 6)))
def test_chained_tower_equals_block_launches(n, N, K):
    """az_nn_resblocks chains K residual blocks inside one launch (every
    cluster runs block b + 1 over its own range of board groups as soon as it
    has finished block b there; K > 8 continues in a second launch): bit-
    identical to K az_nn_resblock launches -- network.py:73, the tower is a
    plain nn.Sequential of Resblocks."""
    import ctypes
    from azalea_b200 import _cabi, tower_layout as tl
    L = _cabi.lib()
    torch.manual_seed(300 + n + K)
    x = (torch.randn(N, n, n, 64, device='cuda') * 0.5).to(torch.bfloat16)
    wall = torch.cat([tl.pack_conv_weights((torch.randn(64, 64, 3, 3, device='cuda') * 0.05).to(torch.bfloat16))
                      for _ in range(2 * K)]).contiguous()
    ball = (torch.randn(2 * K * 64, device='cuda') * 0.1).contiguous()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    scratch = torch.zeros(max(16, L.az_nn_resblock_scratch_bytes()), dtype=torch.uint8, device='cuda')
    xa, xb = tl.to_slabs(x), tl.to_slabs(x)
    wbytes = wall.numel() * wall.element_size() // K
    for b in range(K):
        _cabi.check(L.az_nn_resblock(p(xa), ctypes.c_void_p(wall.data_ptr() + b * wbytes),
                                     ctypes.cast(ball.data_ptr() + b * 128 * 4, ctypes.POINTER(ctypes.c_float)),
                                     p(scratch), n, N, stream))
    for _ in range(3 if N <= 4100 else 1):      # repeated: the hand-over between passes is a timing matter
        xb.copy_(tl.to_slabs(x))
        _cabi.check(L.az_nn_resblocks(p(xb), p(wall), ctypes.cast(ball.data_ptr(), ctypes.POINTER(ctypes.c_float)),
                                      p(scratch), n, N, K, stream))
        torch.cuda.synchronize()
        assert torch.equal(xa.view(torch.int16), xb.view(torch.int16))
    _, rest = tl.from_slabs(xb, n, N)
    assert rest == 0.0


def test_chained_tower_concurrent_streams():
    """Two chained towers in flight on two streams (LockstepSelfPlay(streams=2)
    evaluates its two windows like this), repeatedly, on their own buffers."""
    import ctypes
    from azalea_b200 import _cabi, tower_layout as tl
    L = _cabi.lib()
    n, N, K = 11, 10240, 6
    torch.manual_seed(8)
    x = (torch.randn(N, n, n, 64, device='cuda') * 0.5).to(torch.bfloat16)
    wall = torch.cat([tl.pack_conv_weights((torch.randn(64, 64, 3, 3, device='cuda') * 0.03).to(torch.bfloat16))
                      for _ in range(2 * K)]).contiguous()
    ball = (torch.randn(2 * K * 64, device='cuda') * 0.1).contiguous()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    fp = lambda t: ctypes.cast(t.data_ptr(), ctypes.POINTER(ctypes.c_float))
    ref = tl.to_slabs(x)
    reps = 8
    st0 = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for _ in range(reps):
        _cabi.check(L.az_nn_resblocks(p(ref), p(wall), fp(ball), None, n, N, K, st0))
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(2)]
    bufs = [tl.to_slabs(x) for _ in streams]
    torch.cuda.synchronize()
    for _ in range(reps):
        for s, b in zip(streams, bufs):
            _cabi.check(L.az_nn_resblocks(p(b), p(wall), fp(ball), None, n, N, K, ctypes.c_void_p(s.cuda_stream)))
    torch.cuda.synchronize()
    for b in bufs:
        assert torch.equal(b.view(torch.int16), ref.view(torch.int16))


def test_tcgen05_tower_matches_cudnn_tower():
    """The whole evaluator with the tcgen05 tower (AZALEA_B200_TOWER=tcgen05)
    against the default cuDNN tower on the same weights: both are bf16 with
    fp32 accumulation, so values agree to ~1e-2 and log-priors to ~0.1."""
    from azalea_b200.network import HexNetwork
    torch.manual_seed(3)
    net = HexNetwork(11, 6, 64).eval().cuda()
    net.prepare_inference(torch.bfloat16)
    cells = torch.zeros(1001, 128, dtype=torch.int8, device='cuda')
    cells[:, :121] = torch.randint(0, 3, (1001, 121), device='cuda', dtype=torch.int8)
    net.tower = 'cudnn'
    v0, l0 = net.evaluate_cells(cells)
    net.tower = 'tcgen05'
    v1, l1 = net.evaluate_cells(cells)
    v2, l2 = net.evaluate_cells(cells)          # buffers are reused: same answer again
    assert torch.equal(v1, v2) and torch.equal(l1, l2)
    assert (v0 - v1).abs().max() < 0.03
    lp0, lp1 = torch.log_softmax(l0, 1), torch.log_softmax(l1, 1)
    assert (lp0 - lp1).abs().max() < 0.15 and (lp0 - lp1).abs().mean() < 0.01


def test_random_policy_selfplay_rows():
    """Player over an AzaleaAgent without a policy (RandomPolicy,
    random_policy.py:25-41): uniform moves_prob = 1 / num_moves at every ply,
    whole games with rewards; the way the reference fills the replay buffer
    before training (policy_trainer.py:145-158)."""
    import azalea_b200 as az
    agent = az.AzaleaAgent(lambda: az.HexGame(5))
    player = az.Player(None, [agent], num_games=64, seed=3)
    df, metrics = player.read(300)
    assert len(df) >= 300 and metrics['games'] > 0 and metrics['game_error'] == 0
    first_moves = set()
    for state, probs, reward in zip(df.state, df.moves_prob, df.reward):
        k = len(state.legal_moves)
        assert probs.shape == (k,) and np.allclose(probs, 1.0 / k)
        assert reward in (-1.0, 1.0)
        if k == 25:
            first_moves.add(int(np.count_nonzero(state.board)))
    assert first_moves == {0}
    # moves are spread: many distinct second-ply boards among the games
    second = {s.board.tobytes() for s in df.state if len(s.legal_moves) == 24}
    assert len(second) >= 15


def test_policy_trainer_closes_the_loop(tmp_path):
    """policy_trainer.train (policy_trainer.py:24-120) with GPU self-play:
    random-policy buffer fill, SGD steps on device-collated minibatches,
    replay refills by the policy under training (weights refreshed in place),
    checkpoint in the reference's format."""
    import azalea_b200 as az
    from azalea_b200 import policy_trainer
    config = dict(seed=0xBAD5EED5, device='cuda', game='hex', network='HexNetwork', board_size=5,
                  num_blocks=1, base_chans=64, simulations=20, search_batch_size=5,
                  exploration_coef=0.5, exploration_temperature=1.0, exploration_depth=15,
                  exploration_noise_alpha=0.03, exploration_noise_scale=0.25,
                  replaybuf_size=2048, replaybuf_resample=2, batch_size=128, lr_initial=0.05,
                  lr_decay_steps=4, lr_decay=0.5, momentum=0.9, l2_regularization=1e-4,
                  total_steps=8, log_interval=4, model_checkpoint_interval=0,
                  num_selfplay_games=64)
    policy = az.Policy()
    policy.initialize(config)
    before = [p.detach().clone() for p in policy.net.parameters()]
    path = policy_trainer.train(policy, config, str(tmp_path))
    hist = policy_trainer.train.history
    assert len(hist) == 8 and all(np.isfinite(h['loss']) for h in hist)
    assert hist[0]['lr'] == 0.05 and hist[-1]['lr'] == pytest.approx(0.05 * 0.25)
    # 128 / 2 = 64 consumed per step against 2048 fresh random rows: refills by the network
    # start once those are used up -- force one more refill to see self-play with the trained net
    assert any(not torch.equal(a, b.detach()) for a, b in zip(before, policy.net.parameters()))
    loaded = az.Policy.load(path, device='cuda')
    assert loaded.simulations == 20 and loaded.board_size == 5
    for a, b in zip(loaded.net.parameters(), policy.net.parameters()):
        assert torch.equal(a.cpu(), b.detach().cpu())
    # the loss on uniform-random data starts near log(moves) + value variance
    assert 1.0 < hist[0]['loss'] < 6.0


def test_policy_trainer_refills_from_network_selfplay(tmp_path):
    """With a small buffer the fresh rows run out and the trainer refills from
    self-play by the current network (replay_buffer.py:121-132)."""
    import azalea_b200 as az
    from azalea_b200 import policy_trainer
    config = dict(seed=7, device='cuda', game='hex', network='HexNetwork', board_size=5,
                  num_blocks=1, base_chans=64, simulations=10, search_batch_size=5,
                  exploration_coef=0.5, exploration_temperature=1.0, exploration_depth=15,
                  exploration_noise_alpha=0.03, exploration_noise_scale=0.25,
                  replaybuf_size=256, replaybuf_oversampling=1, batch_size=128, lr_initial=0.01,
                  lr_decay_epochs=100, lr_decay=0.5, momentum=0.9, l2_regularization=1e-4,
                  total_epochs=3, log_interval=0, model_checkpoint_interval=0,
                  num_selfplay_games=32)
    policy = az.Policy()
    policy.initialize(config)
    policy_trainer.train(policy, config, str(tmp_path))
    hist = policy_trainer.train.history
    assert len(hist) == 6                       # 3 epochs x (256 // 128) steps
    assert sum(h.get('selfplay_games', 0) for h in hist) > 0
    assert not policy.net.training


def test_tcgen05_evaluator_against_reference_network_golden():
    """The whole bf16 evaluator on our kernels (stem, tcgen05 tower, heads)
    against the outputs of the REFERENCE's HexNetwork on the same seeded
    weights and boards (tests/golden/network.npz, generated by importing
    azalea.network): value within 2e-3, log-probabilities of the legal moves
    within 4e-3, about twice what a B200 measures (7.7e-4 / 1.9e-3; bf16
    activations through 13 layers).  A dropped bias of the FC layers or the
    stem moves these outputs by 0.013 or more."""
    import os
    from azalea_b200.network import HexNetwork
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'network.npz'))
    torch.manual_seed(0)
    net = HexNetwork(11, 6, 64).eval()
    gen = torch.Generator().manual_seed(1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen) + 0.5)
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
    net.cuda()
    net.prepare_inference(torch.bfloat16)
    assert net.tower == 'tcgen05' and net._fast['tower'] is not None
    board, moves = g['board'], g['legal_moves']
    B = len(board)
    cells = torch.zeros(B, 128, dtype=torch.int8, device='cuda')
    cells[:, :121] = torch.from_numpy(board.reshape(B, 121).astype(np.int8)).cuda()
    value, logits = net.evaluate_cells(cells)
    assert np.abs(value.cpu().numpy() - g['value']).max() < 2e-3
    for i in range(B):
        k = int((moves[i] > 0).sum())
        idx = torch.from_numpy(moves[i, :k].astype(np.int64) - 1).cuda()
        logp = torch.log_softmax(logits[i, idx], 0).cpu().numpy()
        assert np.abs(logp - g['moves_logprob'][i, :k]).max() < 4e-3, i


@pytest.mark.parametrize('streams', (2, 3))
def test_windowed_streams_do_not_change_the_games(streams):
    """LockstepSelfPlay(streams=k) drives k windows of the games on k streams
    (az_engine_set_window) so that tree kernels overlap the evaluator.  Games
    are independent, so moves, results and replay rows are identical to the
    single-stream run (stub evaluator: bit-exact), eager and graphed."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    from azalea_b200.engine import decode_replay_rows
    def play(streams, graph):
        sp = LockstepSelfPlay(StubEvaluator(2), num_games=50, board_size=5, simulations=40,
                              search_batch_size=8, seed=11, streams=streams, cuda_graph=graph)
        chosen = []
        for _ in range(30):
            sp.step_move()
            chosen.append(sp.chosen.cpu().numpy().copy())
        assert (sp.eng.status().cpu().numpy() == 0).all()
        return np.stack(chosen), sp.harvest(), sp.counters()
    c1, r1, n1 = play(1, False)
    for graph in (False, True):
        c2, r2, n2 = play(streams, graph)
        assert np.array_equal(c1, c2)
        assert r1.shape == r2.shape and np.array_equal(r1, r2)
        assert n1 == n2


@pytest.mark.parametrize('temperature', (1.0, 0.5))
def test_play_commit_samples_the_visit_distribution(temperature):
    """k_play_commit's move draw (policy.py:160 multinomial over
    as_distribution(visits, T), search_tree.py:327-344) on the device Philox
    streams: 4096 games at the same position have the same root visit counts
    N and independent streams, so the chosen moves must be a sample of
    p ~ N^(1/T): chi-square against the exact distribution, and never an
    unvisited child."""
    from azalea_b200 import Engine
    from azalea_b200.search_tree import as_distribution
    G, n, sims, batch = 4096, 5, 60, 6
    eng = Engine(G, n, max_batch=batch, seed=1234)
    eng.select_root()
    eng.stub_eval(stubs.ROUGH)
    eng.expand_root()
    for _ in range(sims // batch + 1):
        eng.select(batch, 0.5)
        eng.stub_eval(stubs.ROUGH)
        eng.expand_backup()
    v, _, _, k, _, _ = (x.cpu().numpy() for x in eng.root_stats())
    assert (k == n * n).all() and (v == v[0]).all()     # identical trees
    chosen = torch.zeros(G, 4, dtype=torch.int32, device=eng.device)
    eng.play_commit(temperature, 15, True, False, False, chosen)
    move_id = chosen[:, 1].cpu().numpy()
    p = as_distribution(v[0], temperature)
    obs = np.bincount(move_id, minlength=n * n).astype(np.float64)
    assert obs[p == 0].sum() == 0
    live = p > 0
    assert live.sum() >= 8
    chi2 = float((((obs - G * p) ** 2)[live] / (G * p[live])).sum())
    dof = int(live.sum()) - 1
    # P(chi2_dof > dof + 5 sqrt(2 dof)) < 1e-5; the streams are fixed, so this
    # either always passes or always fails
    assert chi2 < dof + 5 * np.sqrt(2 * dof), (chi2, dof)
    # and the games did not all draw the same number
    assert len(np.unique(move_id)) >= 5


def test_play_commit_temperature_zero_is_uniform_over_the_ties():
    """Temperature 0 (search_tree.py:338-339): uniform over the arg-max ties."""
    from azalea_b200 import Engine
    G, n = 2048, 5
    eng = Engine(G, n, max_batch=4, seed=99)
    eng.select_root()
    eng.stub_eval(stubs.UNIFORM)
    eng.expand_root()
    for _ in range(9):              # 36 descents over 25 children: visits 2 / 1
        eng.select(4, 0.5)
        eng.stub_eval(stubs.UNIFORM)
        eng.expand_backup()
    v = eng.root_stats()[0].cpu().numpy()
    top = np.flatnonzero(v[0] == v[0].max())
    assert 1 < len(top) < n * n
    chosen = torch.zeros(G, 4, dtype=torch.int32, device=eng.device)
    eng.play_commit(1.0, 0, True, False, False, chosen)     # ply 0 >= depth 0: T = 0
    move_id = chosen[:, 1].cpu().numpy()
    assert set(move_id) <= set(top)
    obs = np.bincount(move_id, minlength=n * n)[top].astype(np.float64)
    exp = G / len(top)
    chi2 = float(((obs - exp) ** 2 / exp).sum())
    dof = len(top) - 1
    assert chi2 < dof + 5 * np.sqrt(2 * dof), (chi2, dof)


@pytest.mark.parametrize('streams,graph', ((1, False), (2, False), (2, True)))
def test_packed_leaves_do_not_change_the_games(streams, graph):
    """LockstepSelfPlay packs the leaves by default when a network evaluates
    them (AZ_CFG_PACK_LEAVES: duplicates and terminal leaves cost no network
    time).  A row's evaluation does not depend on where in the batch it sits,
    so moves and replay rows are identical to the slot-indexed run -- 6x64
    network on our kernels, small searches near the end of 5x5 games (many
    duplicate and terminal leaves)."""
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.network import HexNetwork

    def play(pack, streams, graph):
        torch.manual_seed(0)
        net = HexNetwork(5, 2, 64).eval().cuda()
        net.prepare_inference(torch.bfloat16)
        assert net.tower == 'tcgen05'
        sp = LockstepSelfPlay(net, num_games=96, board_size=5, simulations=40,
                              search_batch_size=8, seed=5, streams=streams,
                              cuda_graph=graph, pack_leaves=pack)
        assert sp.pack_leaves == pack
        chosen = []
        for _ in range(30):
            sp.step_move()
            chosen.append(sp.chosen.cpu().numpy().copy())
        assert (sp.eng.status().cpu().numpy() == 0).all()
        return np.stack(chosen), sp.harvest(), sp.counters()
    c0, r0, n0 = play(False, 1, False)
    c1, r1, n1 = play(True, streams, graph)
    assert n1['nn_rows'] < n1['simulations']        # there was something to skip
    assert np.array_equal(c0, c1)
    assert r0.shape == r1.shape and np.array_equal(r0, r1)
    assert n0 == n1


def test_evaluator_live_rows():
    """az_nn_*_live: with a device-side row count the evaluator's outputs for
    the live rows equal the full evaluation's, the rows past the count are
    left alone, and a count of zero runs (clusters without a group)."""
    from azalea_b200.network import HexNetwork
    torch.manual_seed(1)
    n, N = 11, 700
    net = HexNetwork(n, 3, 64).eval().cuda()
    net.prepare_inference(torch.bfloat16)
    cells = torch.zeros(N, 128, dtype=torch.int8, device='cuda')
    cells[:, :n * n] = torch.randint(0, 3, (N, n * n), device='cuda', dtype=torch.int8)
    v0, l0 = net.evaluate_cells(cells)
    v0, l0 = v0.clone(), l0.clone()
    for live in (N, 699, 345, 10, 1, 0):
        cnt = torch.tensor([live], dtype=torch.int32, device='cuda')
        v = torch.full((N,), 7.0, device='cuda')
        lg = torch.full((N, n * n), 7.0, device='cuda')
        net.evaluate_cells(cells, value_out=v, logits_out=lg, logits_stride=n * n, live_rows=cnt)
        torch.cuda.synchronize()
        assert torch.equal(v[:live], v0[:live]) and torch.equal(lg[:live], l0[:live]), live
        assert (v[live:] == 7.0).all() and (lg[live:] == 7.0).all(), live


def test_pipelined_harvest_equals_harvest():
    """harvest_begin / harvest_end (count sync, copy to pinned memory and clear
    enqueued, the next move launched before the rows are waited for) return
    the same rows as harvest(), move by move."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    def make():
        return LockstepSelfPlay(StubEvaluator(2), num_games=64, board_size=5, simulations=30,
                                search_batch_size=6, seed=4, cuda_graph=False)
    a, b = make(), make()
    got, want = [], []
    b.step_move()
    for k in range(40):
        a.step_move()
        want.append(a.harvest())
        h = b.harvest_begin()
        b.step_move()                   # the next move is in flight while the rows come back
        got.append(b.harvest_end(h))
    assert sum(len(r) for r in want) > 200
    for r0, r1 in zip(want, got):
        assert r0.shape == r1.shape and np.array_equal(r0, r1)


def test_packed_leaves_19x19_do_not_change_the_games():
    """The same on the deep-search shape (19x19: six boards per tower group,
    k_select<12>): packed and slot-indexed network self-play play the same
    games."""
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.network import HexNetwork

    def play(pack):
        torch.manual_seed(0)
        net = HexNetwork(19, 2, 64).eval().cuda()
        net.prepare_inference(torch.bfloat16)
        sp = LockstepSelfPlay(net, num_games=10, board_size=19, simulations=60,
                              search_batch_size=10, seed=7, streams=2, cuda_graph=False,
                              pack_leaves=pack, nodes_per_game=200_000)
        chosen = []
        for _ in range(12):
            sp.step_move()
            chosen.append(sp.chosen.cpu().numpy().copy())
        assert (sp.eng.status().cpu().numpy() == 0).all()
        return np.stack(chosen), sp.counters()
    c0, n0 = play(False)
    c1, n1 = play(True)
    assert np.array_equal(c0, c1) and n0 == n1
