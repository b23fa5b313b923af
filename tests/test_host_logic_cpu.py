"""Host-side logic that needs no GPU: distribution maths, perspective flip,
network parity with the reference's architecture, replay row decoding,
multi-rank replay gather (gloo, world size 2)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

from azalea_b200 import as_distribution
from azalea_b200.game.hex import HexGame
from azalea_b200.network import HexNetwork


def test_as_distribution_golden(golden_formulas):
    f = golden_formulas
    for i in range(len(f['dist_k'])):
        k = int(f['dist_k'][i])
        got = as_distribution(f['dist_counts'][i][:k].copy(),
                              float(f['dist_temp'][i]))
        assert got.dtype == np.float64
        assert got.tobytes() == f['dist_out'][i][:k].tobytes()


@pytest.mark.parametrize('n', (3, 5, 11, 19))
def test_flip_golden(golden_hex, n):
    g = golden_hex
    fb, fm = HexGame.flip_player_board_moves(g[f'n{n}_flip_in_board'],
                                             g[f'n{n}_flip_in_moves'])
    assert (fb == g[f'n{n}_flip_out_board']).all()
    assert (fm == g[f'n{n}_flip_out_moves']).all()
    one_b, one_m = HexGame.flip_player_board_moves(
        g[f'n{n}_flip_in_board'][0], g[f'n{n}_flip_in_moves'][0])
    assert (one_b[0] == fb[0]).all() and (one_m[0] == fm[0]).all()


def test_network_matches_reference_architecture():
    """Golden: the reference's HexNetwork, given this module's seed-0
    state_dict, on fixed inputs (tests/golden/make_golden.py:gen_network)."""
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'network.npz'))
    torch.manual_seed(0)
    net = HexNetwork(11, 6, 64).eval()
    # give BatchNorm non-trivial statistics, deterministically
    gen = torch.Generator().manual_seed(1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen) + 0.5)
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
    board = torch.from_numpy(g['board'])
    moves = torch.from_numpy(g['legal_moves'])
    with torch.no_grad():
        out = net.run(dict(board=board, legal_moves=moves))
        assert np.allclose(out['value'].numpy(), g['value'], atol=1e-6)
        assert np.allclose(out['moves_logprob'].numpy(), g['moves_logprob'], atol=1e-5)
        # folded fp32 fast path == reference path
        net.prepare_inference(torch.float32)
        cells = torch.zeros(len(board), 128, dtype=torch.int8)
        cells[:, :121] = board.view(len(board), -1).to(torch.int8)
        value, logits = net.evaluate_cells(cells)
        lg = torch.gather(logits, 1, (moves - 1).clamp(min=0).long())
        lg = lg.masked_fill(moves == 0, -99)
        assert np.allclose(value.numpy(), g['value'], atol=1e-5)
        assert np.allclose(torch.log_softmax(lg, 1).numpy(), g['moves_logprob'], atol=1e-4)


def test_decode_replay_rows_layout():
    from azalea_b200.engine import (ROW_HEADER, decode_replay_rows,
                                    replay_row_bytes)
    n, nn, cs = 5, 25, 32
    hb = ROW_HEADER.itemsize
    assert hb == 48
    row_bytes = replay_row_bytes(n)
    rows = np.zeros((2, row_bytes), dtype=np.uint8)
    h = np.zeros(2, dtype=ROW_HEADER)
    h['game_id'] = [7, 1 << 40]
    h['ply'] = [3, 4]
    h['reward'] = [1.0, -1.0]
    rows[:, :hb] = h.view(np.uint8).reshape(2, hb)
    rows[0, hb:hb + nn] = np.arange(nn) % 3
    vis = np.arange(nn, dtype='<f4')
    rows[1, hb + cs:hb + cs + 4 * nn] = vis.view(np.uint8)
    hh, board, visits = decode_replay_rows(rows, n)
    assert list(hh['game_id']) == [7, 1 << 40] and list(hh['ply']) == [3, 4]
    assert (board[0].ravel() == np.arange(nn) % 3).all()
    assert (visits[1] == vis).all()


def test_bench_dump_outputs_dtypes_and_size_cap(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 files only; above the size
    limit a fixed seeded sample of the replay rows is written, the same
    sample for the same rows."""
    import bench
    from azalea_b200.engine import ROW_HEADER, replay_row_bytes
    n, nn, R = 5, 25, 60
    rows = np.zeros((R, replay_row_bytes(n)), dtype=np.uint8)
    h = rows[:, :48].view(ROW_HEADER).reshape(-1)
    h['game_id'] = np.arange(R) // 10 + (1 << 40)
    h['ply'] = np.arange(R) % 10
    rows[:, 48:48 + nn] = np.arange(nn) % 3
    rows[:, 48 + 32:48 + 32 + 4 * nn] = (np.arange(R * nn, dtype='<f4') % 7).reshape(R, nn).view(np.uint8)
    chosen = np.arange(32 * 4, dtype=np.int32).reshape(32, 4)

    def dump(d):
        bench.dump_outputs(str(d), chosen, rows, n)
        out = {f[:-4]: np.load(d / f) for f in os.listdir(d)}
        assert all(a.dtype in (np.float32, np.float64) for a in out.values())
        return out

    full = dump(tmp_path / 'full')
    assert (full['chosen_move_id'] == chosen[:, 1]).all()
    assert (full['replay_game_id'] == h['game_id']).all() and full['replay_visits'].shape == (R, nn)
    assert (full['replay_board'][3].ravel() == np.arange(nn) % 3).all()
    per_row = 8 * 10 + 4 * nn * 2
    monkeypatch.setattr(bench, 'DUMP_BYTES', full['chosen_ply'].nbytes * 4 + 17 * per_row)
    a, b = dump(tmp_path / 'a'), dump(tmp_path / 'b')
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_BYTES
    assert len(a['replay_ply']) == 17 and all((a[k] == b[k]).all() for k in a)
    idx = (a['replay_game_id'] - (1 << 40)) * 10 + a['replay_ply']
    assert (np.diff(idx) > 0).all() and (a['replay_visits'] == full['replay_visits'][idx.astype(int)]).all()


def _gather_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from azalea_b200.selfplay import gather_replay_rows
    dist.init_process_group('gloo', init_method=f'tcp://127.0.0.1:{port}',
                            rank=rank, world_size=world)
    # rank r contributes r + 2 rows whose bytes identify (rank, row)
    rows = torch.zeros(rank + 2, 48, dtype=torch.uint8)
    for i in range(rank + 2):
        rows[i] = 16 * rank + i
    out = gather_replay_rows(rows, dst=0)
    q.put((rank, None if out is None else out.numpy().copy()))
    dist.barrier()
    dist.destroy_process_group()


def test_replay_gather_two_ranks_gloo():
    """Replay rows of game shards reach rank 0 in rank order (SURVEY 8e)."""
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q))
             for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[1] is None
    assert got[0].shape == (5, 48)
    assert list(got[0][:, 0]) == [0, 1, 16, 17, 18]


def test_game_sharding_is_world_size_invariant():
    """Global game ids: rank r of W owns [r*G, (r+1)*G); a slot's successive
    games advance by W*G, so the id sets of different ranks never meet."""
    G, W = 4, 3
    seen = set()
    for rank in range(W):
        for slot in range(G):
            for serial in range(5):
                gid = rank * G + slot + serial * W * G
                assert gid not in seen
                seen.add(gid)
    assert seen == set(range(5 * W * G))


def test_tower_layout_helpers_roundtrip():
    """azalea_b200/tower_layout.py (the slab activation layout of the tcgen05
    tower, csrc/az_tower.cuh) on CPU tensors: the row formula, the 16-byte
    chunk swizzle, the weight packing order and the round trip."""
    import torch
    from azalea_b200 import tower_layout as tl
    for n, N in ((11, 23), (19, 7), (5, 1), (7, 33)):
        bpg = tl.boards_per_group(n)
        assert bpg == 128 // (n + 1)
        groups = (N + bpg - 1) // bpg
        assert tl.buffer_rows(n, N) == 8 + groups * n * 128 + 16
        x = torch.arange(N * n * n * 64, dtype=torch.float32).reshape(N, n, n, 64) % 251
        buf = tl.to_slabs(x)
        assert buf.shape == (tl.buffer_rows(n, N), 64)
        back, rest = tl.from_slabs(buf, n, N)
        assert torch.equal(back, x) and rest == 0.0
        # one cell by hand: board b, row y, column c -> row R, chunk j stored at j ^ (R & 7)
        b, y, c = N - 1, n - 1, n // 2
        R = 8 + ((b // bpg) * n + y) * 128 + (b % bpg) * (n + 1) + c
        for j in range(8):
            phys = j ^ (R & 7)
            assert torch.equal(buf[R, phys * 8:phys * 8 + 8], x[b, y, c, j * 8:j * 8 + 8])
        # the pad cell after each board row is zero
        assert float(buf[R - c + n].abs().sum()) == 0.0
    w = torch.arange(64 * 64 * 9, dtype=torch.float32).reshape(64, 64, 3, 3)
    wp = tl.pack_conv_weights(w)
    assert wp.shape == (576, 64)
    for kx, ky, co in ((0, 0, 0), (2, 1, 37), (1, 2, 63)):
        row = (kx * 3 + ky) * 64 + co
        for j in (0, 5):
            phys = j ^ (row & 7)
            assert torch.equal(wp[row, phys * 8:phys * 8 + 8], w[co, j * 8:j * 8 + 8, ky, kx])


def test_policy_trainer_config_helpers():
    """policy_trainer accepts both spellings of the reference's stale config
    keys (config/hex11_train_config.yml vs policy_trainer.py:38-66) and
    resolves the game class like the reference's import_and_get."""
    from azalea_b200 import policy_trainer as pt
    from azalea_b200.game.hex import HexGame
    assert pt._cfg({'replaybuf_resample': 10}, 'replaybuf_oversampling', 'replaybuf_resample') == 10
    assert pt._cfg({'replaybuf_oversampling': 4, 'replaybuf_resample': 10},
                   'replaybuf_oversampling', 'replaybuf_resample') == 4
    assert pt._cfg({}, 'a', 'b', default=7) == 7
    with pytest.raises(KeyError):
        pt._cfg({}, 'a', 'b')
    assert pt._game_class('hex') is HexGame
    assert pt._game_class('azalea.game.hex.HexGame') is HexGame
    assert pt._game_class('azalea_b200.game.hex.HexGame') is HexGame


class _FakeAgent:
    """An agent as far as evaluate() looks at one: .policy and .game.board_size."""

    class _Game:
        board_size = 5

    def __init__(self, tag):
        self.policy = tag
        self.game = self._Game()


def _fake_play(first, second, board_size, seed=0, device=None, game_ids=None, stats=None, **kw):
    """Stands in for play_matches on a GPU-less box: a game's result is a
    function of its global task id and of who moves first, nothing else."""
    res = [3 if (7 * gid + 3 * first[i] + second[i] + seed) % 3 else 1
           for i, gid in enumerate(game_ids)]
    return np.array(res, dtype=np.int64), np.zeros((0, len(res)), dtype=np.int32)


def _tournament_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from azalea_b200.evaluation import evaluate
    dist.init_process_group('gloo', init_method=f'tcp://127.0.0.1:{port}',
                            rank=rank, world_size=world)
    agents = [_FakeAgent(i) for i in range(5)]
    out = evaluate(agents, 7, _play=_fake_play)
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_tournament_sharding_and_reduce_two_ranks_gloo():
    """evaluate() under torch.distributed: (round, pair) tasks go round-robin
    to the ranks (evaluation.py:49-58 fans them over worker processes), the
    [pairs, 3] tallies are reduced onto rank 0, and the result equals the
    single-process tournament (SURVEY 8e)."""
    import torch.multiprocessing as mp
    from azalea_b200.evaluation import evaluate, gen_pairs, tournament_tasks
    agents = [_FakeAgent(i) for i in range(5)]
    whole = evaluate(agents, 7, _play=_fake_play)
    assert sorted(whole) == sorted(gen_pairs(5)) and len(whole) == 10
    assert all(sum(v) == 7 for v in whole.values())
    # the shares partition the task list, in the reference's order
    t0, t1 = tournament_tasks(5, 7, 0, 2), tournament_tasks(5, 7, 1, 2)
    assert sorted(t[0] for t in t0 + t1) == list(range(70))
    assert all(t[0] % 2 == 0 for t in t0) and all(t[0] % 2 == 1 for t in t1)
    for t, r, s, pair, order in t0 + t1:
        assert t == r * 10 + s and pair == gen_pairs(5)[s]
        assert order == np.random.RandomState(10000 * r + s).choice([-1, 1])
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_tournament_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0] == whole                      # rank 0: the whole tournament
    share1 = evaluate(agents, 7, rank=1, world_size=2, reduce=False, _play=_fake_play)
    assert got[1] == share1                     # rank 1 keeps its own share
    assert sum(sum(v) for v in share1.values()) == 35


class _FakePlayer:
    """read_device() of a self-play player, without a GPU: rows tagged with
    the rank and with a digest of the weights the rank played with."""

    def __init__(self, rank, net):
        self.rank, self.net, self.calls = rank, net, 0

    def read_device(self, size):
        self.calls += 1
        rows = torch.zeros(size, 48, dtype=torch.uint8)
        rows[:, 0] = self.rank
        rows[:, 1] = self.calls
        rows[:, 2] = int(round(float(self.net.weight.sum()))) % 251
        return rows, {'games': 1}

    def stop(self):
        pass


def _refill_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from azalea_b200.policy_trainer import DistributedSelfPlay
    dist.init_process_group('gloo', init_method=f'tcp://127.0.0.1:{port}',
                            rank=rank, world_size=world)
    torch.manual_seed(100 + rank)                   # the ranks start with different weights
    net = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.BatchNorm1d(3))
    sp = DistributedSelfPlay(_FakePlayer(rank, net[0]), net)
    if rank == 0:
        out = []
        for step in range(3):
            with torch.no_grad():
                net[0].weight.fill_(float(step + 1))        # "an optimizer step"
                net[1].running_mean.fill_(0.5 * step)
                net[1].num_batches_tracked.fill_(step)
            rows, _ = sp.read_device(7)
            out.append(rows.numpy().copy())
        sp.stop()
        q.put((rank, out, sp.bytes_broadcast))
    else:
        served = sp.serve()
        q.put((rank, (served, net[0].weight.detach().numpy().copy(),
                      net[1].running_mean.numpy().copy(), int(net[1].num_batches_tracked)), 0))
    dist.barrier()
    dist.destroy_process_group()


def test_distributed_refill_protocol_two_ranks_gloo():
    """SURVEY 8e, training hand-off: rank 0 trains and asks for replay rows;
    before every refill its weights (parameters AND BatchNorm buffers) are
    broadcast, every rank plays its share, rows are gathered to rank 0."""
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_refill_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {r: (a, b) for r, a, b in (q.get(timeout=120) for _ in range(2))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    refills, nbytes = got[0]
    assert nbytes == 3 * (4 * (12 + 3 + 3 + 3 + 3 + 3) + 8)      # float tensors + the int64 counter, 3 times
    for step, rows in enumerate(refills):
        assert rows.shape == (8, 48)                    # ceil(7 / 2) rows from each rank
        assert list(rows[:, 0]) == [0] * 4 + [1] * 4    # rank order
        assert (rows[:, 1] == step + 1).all()
        # both ranks played with the weights of this step: sum = 12 * (step + 1)
        assert (rows[:, 2] == (12 * (step + 1)) % 251).all()
    served, w, mean, tracked = got[1][0]
    assert served == 3 and (w == 3.0).all() and (mean == 1.0).all() and tracked == 2


def test_harvest_rows_are_sorted_by_game_and_ply():
    """Finished games append their rows in warp-scheduling order; every harvest
    path (harvest, harvest_begin / harvest_end, gathered) hands them out sorted
    by (game id, ply) through Engine._sort_rows."""
    import numpy as np
    from azalea_b200.engine import Engine, ROW_HEADER
    rng = np.random.RandomState(0)
    rows = np.zeros((200, 64), dtype=np.uint8)
    h = rows[:, :ROW_HEADER.itemsize].view(ROW_HEADER).reshape(-1)
    h['game_id'] = rng.randint(0, 7, size=200) + (1 << 33)
    h['ply'] = rng.randint(0, 50, size=200)
    rows[:, 60] = np.arange(200) % 251
    out = Engine._sort_rows(rows.copy())
    ho = out[:, :ROW_HEADER.itemsize].copy().view(ROW_HEADER).reshape(-1)
    key = list(zip(ho['game_id'].tolist(), ho['ply'].tolist()))
    assert key == sorted(key)
    assert sorted(map(bytes, out)) == sorted(map(bytes, rows))
    assert len(Engine._sort_rows(rows[:0])) == 0
