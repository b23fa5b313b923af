"""Drivers and checks the lockstep engine's GPU tests share.  TEST
INFRASTRUCTURE ONLY.

Plain functions over ``azalea_b200`` objects: a stub search of one ply, stub
self-play that records what the option tests read, the bit-for-bit root check
against an oracle tree, and the invariances every self-play option must keep
(streams, CUDA graphs, ranks).  ``azalea_b200`` and torch are imported inside
the functions, so importing this module needs neither.
"""
import numpy as np

from .philox import game_ids


def bits(a):
    """float32 bytes, for bit-equality asserts."""
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


def network(num_blocks):
    """A random-init 5x5 HexNetwork of num_blocks x 64 channels (torch seed 0)
    on the GPU, prepared for bf16 inference."""
    import torch
    from azalea_b200.network import HexNetwork
    torch.manual_seed(0)
    net = HexNetwork(5, num_blocks, 64).eval().cuda()
    net.prepare_inference(torch.bfloat16)
    return net


def stub_search(eng, mode, batch, coef, num_batches, eps=0.0, alpha=1.0):
    """One ply's search with the device stub evaluator: the root, then
    num_batches x (select, stub_eval, expand_backup)."""
    eng.select_root()
    eng.stub_eval(mode)
    eng.expand_root()
    for _ in range(num_batches):
        eng.select(batch, coef, eps, alpha)
        eng.stub_eval(mode)
        eng.expand_backup()


def assert_root_matches(stats, g, tree, where):
    """Game g's root in ``stats`` (Engine.root_stats() on the host) equals the
    oracle tree's bit for bit: visits, W, priors, root N/W and node count.
    Returns the oracle's visits."""
    v, w, p, k, rnw, nodes = stats
    ov, ow, op = tree.root_stats()
    kg = int(k[g])
    assert kg == len(ov), where
    assert bits(v[g, :kg]) == bits(ov), where
    assert bits(w[g, :kg]) == bits(ow), where
    assert bits(p[g, :kg]) == bits(op), where
    assert bits(rnw[g]) == bits(tree.root_node()), where
    assert int(nodes[g]) == tree.num_nodes, where
    return ov


def stub_selfplay(moves, G=64, n=5, seed=3, graph=False, streams=None, **kw):
    """``moves`` moves of ROUGH-stub self-play (30 simulations, batch 4,
    temperature 1 for 4 plies).  Returns the self-play, the descents of each
    (game id, ply) (the simulations counter's growth over the move), the
    finished games {game id: (length, result, resigned)} and the chosen rows
    of every move, stacked."""
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    from . import stubs
    sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=G, board_size=n, simulations=30,
                          search_batch_size=4, seed=seed, cuda_graph=graph, exploration_depth=4,
                          streams=streams, **kw)
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
                finished[int(gid[g])] = (int(ch[g, 3]), int(ch[g, 2]), bool(ch[g, 1] == -1))
                assert ch[g, 3] == ply[g] + (ch[g, 1] != -1)
    assert (sp.eng.status().cpu().numpy() == 0).all()
    return sp, plies, finished, np.stack(chosen)


def selfplay_fingerprint(sp, moves):
    """Play ``moves`` moves; the bytes of every move's chosen rows, of the
    replay rows, and of the counters and meta the engine ends with."""
    chosen = []
    for _ in range(moves):
        sp.step_move()
        chosen.append(sp.chosen.cpu().numpy().copy())
    return (np.stack(chosen).tobytes(), sp.harvest().tobytes(),
            sp.eng.counters.cpu().numpy().tobytes(), sp.eng.meta.cpu().numpy().tobytes())


def assert_streams_and_graphs_agree(play):
    """``play(streams, graph)`` returns (chosen, replay rows, counters, ...):
    two streams and a CUDA graph, apart or together, change none of it.
    Returns the one-stream eager run."""
    base = play(1, False)
    for streams, graph in ((2, False), (2, True), (1, True)):
        other = play(streams, graph)
        assert np.array_equal(base[0], other[0]) and base[1].tobytes() == other[1].tobytes()
        assert base[2] == other[2]
        for a, b in zip(base[3:], other[3:]):
            assert np.array_equal(a, b)
    return base


def assert_same_games(whole, parts, n=5):
    """The replay rows of 2 ranks x 32 games (``parts``) are those of 1 rank x
    64 games (``whole``), byte for byte, matched by (game id, ply)."""
    from azalea_b200.engine import decode_replay_rows

    def index(rows):
        h = decode_replay_rows(rows, n)[0]
        return {(int(g), int(p)): i for i, (g, p) in enumerate(zip(h['game_id'], h['ply']))}
    want = index(whole)
    seen = 0
    for part in parts:
        for key, i in index(part).items():
            assert whole[want[key]].tobytes() == part[i].tobytes(), key
            seen += 1
    assert seen == len(want) > 0


def check_replay_buffer(rows, n=5):
    """The rows go through rows_to_dataframe (one example each) and
    DeviceReplayBuffer: a sample draws with its generator the rows
    torch.randint draws, and each probability row sums to 1."""
    import torch
    from azalea_b200.engine import decode_replay_rows
    from azalea_b200.replay_device import DeviceReplayBuffer
    from azalea_b200.selfplay import rows_to_dataframe
    h = decode_replay_rows(rows, n)[0]
    assert len(rows_to_dataframe(rows, n)) == len(h)
    buf = DeviceReplayBuffer(len(h) + 7, n)
    buf.put(torch.from_numpy(rows).cuda())
    batch = buf.sample(64, generator=torch.Generator(device='cuda').manual_seed(4))
    idx = torch.randint(0, len(buf), (64,), device='cuda',
                        generator=torch.Generator(device='cuda').manual_seed(4)).cpu().numpy()
    assert np.array_equal(batch['reward'].cpu().numpy(), h['reward'][idx])
    assert np.array_equal(batch['color'].cpu().numpy(), h['color'][idx])
    assert np.allclose(batch['moves_prob'].sum(1).cpu().numpy(), 1.0, atol=1e-5)


def selfplay_player(net, simulations, search_batch_size, **kw):
    """A Player of 64 5x5 games, seed 3, whose policy searches with ``net``
    (c = 0.5, temperature 1 for 4 plies, root noise 0.25 / 0.03); ``kw`` goes
    to Player."""
    import azalea_b200 as az
    from azalea_b200.parallel_player import Player
    pol = az.Policy()
    pol.net = net
    pol.simulations, pol.search_batch_size, pol.exploration_coef = simulations, search_batch_size, 0.5
    pol.exploration_depth, pol.exploration_temperature = 4, 1.0
    pol.exploration_noise_alpha, pol.exploration_noise_scale = 0.03, 0.25
    agent = az.AzaleaAgent(lambda: az.HexGame(5), policy=pol)
    return Player(None, [agent], num_games=64, seed=3, **kw)


def train_config(**overrides):
    """A train() config of 4 steps on 5x5 Hex: a 1 x 64 network, 32 self-play
    games of 10 simulations, a replay buffer of 256."""
    return dict(seed=3, device='cuda', game='hex', network='HexNetwork', board_size=5,
                num_blocks=1, base_chans=64, simulations=10, search_batch_size=5,
                exploration_coef=0.5, exploration_temperature=1.0, exploration_depth=15,
                exploration_noise_alpha=0.03, exploration_noise_scale=0.25,
                replaybuf_size=256, replaybuf_oversampling=1, batch_size=128, lr_initial=0.01,
                lr_decay_steps=100, lr_decay=0.5, momentum=0.9, l2_regularization=1e-4,
                total_steps=4, log_interval=0, model_checkpoint_interval=0,
                num_selfplay_games=32, **overrides)
