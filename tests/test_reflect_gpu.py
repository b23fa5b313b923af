"""random_reflect: Hex's one rule-preserving symmetry, the 180-degree rotation
tile t -> n*n-1-t, in the search (k_select writes a network row rotated when
its coin says so, k_expand_backup reads its logits back rotated), in the host
evaluator path of SearchTree and on training batches (az_batch_reflect)."""
import numpy as np
import pytest
import torch

import oracle
from azalea_b200._cabi import AZ_PRIOR_LOGITS
from oracle import stubs
from oracle.lockstep import (assert_same_games, assert_streams_and_graphs_agree, network, random_positions,
                             train_config)

gpu = pytest.mark.gpu


def flip_tile(t, n):
    r, c = t // n, t % n
    return (n - 1 - c) * n + (n - 1 - r)


# ------------------------------------------------------------------- CPU --

@pytest.mark.parametrize('n', (3, 5, 7, 11))
def test_rotation_keeps_the_winner(golden_hex, n):
    """check_win on recorded games and on random boards equals check_win on
    their rotation (the winning edges of each player map onto themselves)."""
    g = golden_hex
    nn = n * n
    for moves, plies in zip(g[f'n{n}_moves'], g[f'n{n}_plies']):
        game = oracle.Hex(n)
        for m in moves[:plies]:
            game.step(int(m))
            b = game.board
            t = int(m) - 1
            assert oracle.check_win(b, t) == oracle.check_win(b[::-1, ::-1], nn - 1 - t)
    rng = np.random.RandomState(n)
    wins = 0
    for _ in range(300):
        b = rng.randint(0, 3, size=(n, n)).astype(np.int32)
        for t in np.flatnonzero(b.ravel()):
            w = oracle.check_win(b, int(t))
            wins += bool(w)
            assert w == oracle.check_win(b[::-1, ::-1], nn - 1 - int(t))
    assert wins > 0


def test_host_rotation_helper():
    """HexGame.rotate_board_moves: the board reversed on both axes, the k
    moves m -> n*n+1-m in ascending order, padding zero; its own inverse."""
    from azalea_b200.game.hex import HexGame
    rng = np.random.RandomState(0)
    n, B, nn = 5, 64, 25
    board = rng.randint(0, 3, size=(B, n, n)).astype(np.int32)
    board[0] = 0
    board[1] = 1
    K = int((board.reshape(B, -1) == 0).sum(1).max())
    moves = np.zeros((B, K), np.int32)
    for i in range(B):
        legal = np.flatnonzero(board[i].ravel() == 0) + 1
        moves[i, :len(legal)] = legal
    rb, rm = HexGame.rotate_board_moves(board, moves)
    for i in range(B):
        assert (rb[i] == board[i][::-1, ::-1]).all()
        legal = np.flatnonzero(rb[i].ravel() == 0) + 1
        assert (rm[i, :len(legal)] == legal).all() and (rm[i, len(legal):] == 0).all()
    bb, mm = HexGame.rotate_board_moves(rb, rm)
    assert (bb == board).all() and (mm == moves).all()


# ------------------------------------------------------------------- GPU --

def leaf_rows(eng, root):
    """{(g, b): (network row bytes, leaf_info)} of the rows the evaluator reads."""
    info = eng.leaf_info.cpu().numpy()
    cells = eng.leaf_board.cpu().numpy().reshape(-1, eng.cell_stride)
    G, B = info.shape[:2]
    out = {}
    for g, b in zip(*np.nonzero((info[..., 0] >= 0) & ((info[..., 1] & 0xff) == 0))):
        if root:
            r = g * B
        elif eng.pack_leaves:
            r = info[g, b, 3] >> 10
        else:
            r = g * B + b
        out[(g, b)] = (r, cells[r, :eng.nn], info[g, b])
    return out


def node_pool(eng):
    G, C = eng.num_games, eng.nodes_per_game
    nodes = eng.mem[:G * 2 * C * 16].view(torch.int32).view(G, 2, C, 4)
    half = eng.meta[:, 0].long()
    return nodes[torch.arange(G, device=eng.device), half].cpu().numpy()


def engine_state(eng):
    """The buffers the ABI exposes and every node in use, as bytes (the rest
    of the device block is scratch that no kernel reads before writing)."""
    pool, tail = node_pool(eng), eng.meta[:, 1].cpu().numpy()
    out = [pool[g, :tail[g]].tobytes() for g in range(eng.num_games)]
    for t in (eng.leaf_board, eng.leaf_info, eng.value, eng.prior, eng.meta, eng.counters,
              eng.globals, eng.leaf_rows):
        out.append(t.cpu().numpy().tobytes())
    return out


def softmax64(x):
    x = np.asarray(x, np.float64)
    e = np.exp(x - x.max())
    return e / e.sum()


def check_children(pool, g, node, view_off, rotated, color, logits, n):
    """Priors of the children of an expanded leaf == softmax over its legal
    tiles t of logits[rot(view(t))] (rotated row) or logits[view(t)]."""
    nn = n * n
    link = int(pool[g, node, 3]) & 0xffffffff
    k, fc = link & 511, link >> 9
    idx = []
    for t in range(nn):
        u = flip_tile(t, n) if color else t
        if view_off[u] == 0:
            idx.append(nn - 1 - u if rotated else u)
    assert k == len(idx)
    prior = pool[g, fc:fc + k, 2].view(np.float32)
    assert np.abs(prior - softmax64(logits[idx])).max() < 1e-6


@gpu
@pytest.mark.parametrize('pack', (False, True))
def test_select_writes_rotated_rows_and_expand_gathers_them_back(pack):
    """Twin engines, same seed and positions, reflect on and off: descents do
    not depend on the orientation, so both produce the same leaves, and every
    row of the reflect-on engine equals the twin's, rotated exactly when
    AZ_LEAF_REFLECTED is set (root mode, slot-indexed and packed leaves).
    Logits are fed to the reflect-on engine rotated where the twin's are not:
    the children's priors (expand_root and expand_backup) are a softmax over
    logits[rot(view(t))] within 1e-6, and both trees stay bit-identical.  The
    rotated fraction is within 5 sigma of 1/2 and equals the counter; with
    reflect off the engine is byte-equal to a default one."""
    from azalea_b200 import Engine
    G, n, B = 300, 11, 8
    nn = n * n
    boards, colors = random_positions(G, n, np.random.RandomState(4))
    engs = []
    for reflect in (True, False, None):
        eng = Engine(G, n, max_batch=B, seed=21, nodes_per_game=16384, pack_leaves=pack)
        if reflect is not None:
            eng.set_reflect(reflect)
        eng.hex_set_state(boards, colors)
        engs.append(eng)
    on, off, default = engs
    gen = torch.Generator(device='cuda').manual_seed(3)
    total = rotated_total = 0
    for it in range(6):
        root = it == 0
        for eng in engs:
            if root:
                eng.select_root()
            else:
                eng.select(B, 0.5)
        ron, roff = leaf_rows(on, root), leaf_rows(off, root)
        assert ron.keys() == roff.keys() and len(ron) > 0
        logits_off = torch.randn(G * B, nn, device='cuda', generator=gen)
        value = torch.rand(G * B, device='cuda', generator=gen) * 2 - 1
        logits_on = logits_off.clone()
        rotated = {}
        for key, (r1, c1, i1) in ron.items():
            r0, c0, i0 = roff[key]
            rot = bool((i1[1] >> 9) & 1)
            rotated[key] = rot
            assert i1[0] == i0[0] and i1[2] == i0[2] and (i1[1] & ~512) == i0[1]
            assert (i1[3] & 1023) == (i0[3] & 1023)
            assert (c1 == (c0[::-1] if rot else c0)).all(), key
            g, b = key
            slot = g * B + b
            logits_on[r1] = logits_off[slot].flip(0) if rot else logits_off[slot]
        total += len(ron)
        rotated_total += sum(rotated.values())
        for eng in engs:
            # the evaluation of leaf (g, b) goes to that engine's row of it
            lg, vals = logits_off.clone(), value.clone()
            for key, (r, _, _) in leaf_rows(eng, root).items():
                slot = key[0] * B + key[1]
                lg[r] = logits_on[ron[key][0]] if eng is on else logits_off[slot]
                vals[r] = value[slot]
            if root:
                eng.prior[:, 0] = lg.view(G, B, nn)[:, 0]
                eng.expand_root(None, AZ_PRIOR_LOGITS)
            else:
                eng.value.view(-1).copy_(vals)
                eng.prior.view(-1, nn).copy_(lg)
                eng.expand_backup(None, None, AZ_PRIOR_LOGITS)
        pool = node_pool(on)
        lo = logits_on.cpu().numpy()
        for key, (r1, _, i1) in ron.items():
            check_children(pool, key[0], int(i1[0]), roff[key][1], rotated[key],
                           (i1[1] >> 8) & 1, lo[r1], n)
        for a, b in zip(on.root_stats(), off.root_stats()):
            assert torch.equal(a, b)
        if not pack:
            assert engine_state(off) == engine_state(default)
    frac = rotated_total / total
    assert abs(frac - 0.5) < 5 * 0.5 / np.sqrt(total), (frac, total)
    assert on.counter_totals()['reflected_rows'] == rotated_total
    assert off.counter_totals()['reflected_rows'] == 0
    assert (on.status().cpu().numpy() == 0).all()


class EquivariantEvaluator:
    """Test evaluator whose value and logits are exactly rotation-equivariant
    in fp32: integer sums over cell pairs {t, rot t} with symmetric weights,
    so an orientation bug anywhere shows up as a difference."""
    _fast = True

    def __init__(self, n):
        self.n = n
        nn = n * n
        u = np.arange(nn)
        w = (np.minimum(u, nn - 1 - u) * 37) % 11 + 1
        self.w = torch.from_numpy(w).cuda()

    def evaluate_cells(self, cells, value_out=None, logits_out=None,
                       logits_stride=None, want_value=True, live_rows=None):
        nn = self.n * self.n
        N = cells.shape[0]
        c = cells[:, :nn].long()
        h = (c * self.w).sum(1, keepdim=True)
        logits = ((3 * c + 5 * c.flip(1) + self.w * h) % 13).float()
        value = ((h[:, 0] % 17) - 8).float() / 8
        if value_out is not None and want_value:
            value_out.copy_(value)
        if logits_out is not None:
            torch.as_strided(logits_out, (N, nn), (int(logits_stride or nn), 1)).copy_(logits)
        return value, logits


def play(evaluator, reflect, streams, graph, G=64, n=5, moves=30, seed=5, **kw):
    from azalea_b200 import LockstepSelfPlay
    sp = LockstepSelfPlay(evaluator, num_games=G, board_size=n, simulations=40,
                          search_batch_size=8, seed=seed, streams=streams,
                          cuda_graph=graph, random_reflect=reflect, **kw)
    assert sp.eng.reflect == reflect
    chosen = []
    for _ in range(moves):
        sp.step_move()
        chosen.append(sp.chosen.cpu().numpy().copy())
    assert (sp.eng.status().cpu().numpy() == 0).all()
    return np.stack(chosen), sp.harvest(), sp.counters()


@gpu
@pytest.mark.parametrize('streams,graph', ((1, False), (2, False), (1, True), (2, True)))
def test_equivariant_evaluator_cancels_the_orientation(streams, graph):
    """With an exactly equivariant evaluator the orientation must cancel:
    packed-leaf self-play with reflect on gives moves and replay rows
    byte-identical to reflect off, while about half the rows were rotated."""
    ev = EquivariantEvaluator(5)
    c0, r0, n0 = play(ev, False, 1, False)
    c1, r1, n1 = play(ev, True, streams, graph)
    assert np.array_equal(c0, c1)
    assert r0.shape == r1.shape and r0.tobytes() == r1.tobytes()
    assert n1['nn_rows'] < n1['simulations']            # packed leaves did skip rows
    assert n0['reflected_rows'] == 0
    # (root rows come on top of nn_rows: at most one per game and move)
    assert 0.45 * n1['nn_rows'] < n1['reflected_rows'] < 0.55 * (n1['nn_rows'] + n1['plies'])
    n1 = dict(n1, reflected_rows=0)
    assert n0 == n1


@gpu
def test_reflect_selfplay_invariance_with_network():
    """Reflect on, random-init HexNetwork: the coins follow the game's Philox
    stream, so one vs two streams and eager vs graphed are bit-identical, and
    2 ranks x 32 games play the games 1 rank x 64 plays."""
    net = network(2)
    _, r0, n0 = assert_streams_and_graphs_agree(lambda streams, graph: play(net, True, streams, graph))
    assert n0['reflected_rows'] > 0
    # and the orientation matters for a real network
    _, r_off, _ = play(net, False, 1, False)
    assert r_off.tobytes() != r0.tobytes()
    whole = play(net, True, 1, False, G=64, moves=25)[1]
    parts = [play(net, True, 1, False, G=32, moves=25, rank=r, world_size=2)[1] for r in range(2)]
    assert_same_games(whole, parts)


class RecordingHostNet:
    """Host evaluator (the reference's network.run interface) that records its
    batches; value and log-priors are exactly equivariant and do not depend
    on the order of the moves (log(w / sum w) with integer weights)."""

    def __init__(self, n):
        self.n, self.batches = n, []
        self.device = torch.device('cpu')

    def eval(self):
        return self

    def run(self, batch):
        b = batch['board'].numpy().reshape(len(batch['board']), -1).astype(np.int64)
        m = batch['legal_moves'].numpy()
        self.batches.append((b.copy(), m.copy()))
        nn = self.n * self.n
        u = np.arange(nn)
        w = (np.minimum(u, nn - 1 - u) * 37) % 11 + 1
        h = (b * w).sum(1)
        t = np.clip(m - 1, 0, None)
        pairs = np.take_along_axis(b, t, 1) + np.take_along_axis(b, nn - 1 - t, 1)
        wt = np.where(m > 0, 1 + (pairs + w[t] * h[:, None]) % 7, 0).astype(np.float64)
        logp = np.where(m > 0, np.log(np.maximum(wt, 1) / wt.sum(1, keepdims=True)), -99.0)
        value = (((h % 17) - 8) / 8).astype(np.float32)
        return {'value': torch.from_numpy(value),
                'moves_logprob': torch.from_numpy(logp.astype(np.float32))}


@gpu
def test_host_evaluator_sees_rotated_batches():
    """SearchTree's host path: one coin per position from the policy's
    RandomState; the evaluator sees those boards rotated with ascending
    rotated moves, and with an equivariant evaluator Policy.choose_action at
    temperature 0 returns the same probabilities (float64 bits) and value as
    with the setting off."""
    from azalea_b200 import HexGame, Policy
    from azalea_b200.search_tree import SearchTree
    n = 5
    results = {}
    for reflect in (False, True):
        p = Policy()
        p.net = RecordingHostNet(n)
        p.simulations, p.search_batch_size, p.exploration_coef = 40, 8, 0.5
        p.exploration_depth, p.exploration_noise_alpha = 15, 0.03
        p.exploration_noise_scale, p.exploration_temperature = 0.25, 1.0
        p.random_reflect = reflect
        p.seed(11)
        p.tree = SearchTree()
        p.ply = 0
        game = HexGame(n)
        for m in (7, 13, 19):
            game.step(m)
        move, info = p.choose_action(game)
        results[reflect] = (info['moves_prob'], info['value'], p.net.batches)
    (p0, v0, b0), (p1, v1, b1) = results[False], results[True]
    assert p0.dtype == np.float64 and p0.tobytes() == p1.tobytes()
    assert np.float32(v0) == np.float32(v1)
    coins_rng = np.random.RandomState(11)
    assert len(b0) == len(b1)
    flips = 0
    for (bo, mo), (br, mr) in zip(b0, b1):
        coins = coins_rng.randint(2, size=len(bo)).astype(bool)
        for i in range(len(bo)):
            k = int((mo[i] > 0).sum())
            if coins[i]:
                flips += 1
                assert (br[i] == bo[i][::-1]).all()
                assert (mr[i, :k] == n * n + 1 - mo[i, k - 1::-1]).all()
                assert (mr[i, k:] == 0).all()
                if (np.diff(mo[i, :k]) > 0).all():      # (the second player's view is not sorted)
                    assert (np.diff(mr[i, :k]) > 0).all()
            else:
                assert (br[i] == bo[i]).all() and (mr[i] == mo[i]).all()
    assert flips > 0


def stub_rows(n=5, G=64):
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    sp = LockstepSelfPlay(StubEvaluator(stubs.ROUGH), num_games=G, board_size=n, simulations=20,
                          search_batch_size=4, seed=2, cuda_graph=False, exploration_depth=4)
    chunks = []
    while sum(len(c) for c in chunks) < 400:
        sp.step_move()
        if sp.eng.replay_count():
            chunks.append(sp.harvest())
    return torch.from_numpy(np.concatenate(chunks)).cuda()


@gpu
def test_batch_reflect_matches_numpy():
    """az_batch_reflect on a collated batch equals a numpy rotation with the
    same coins, applying it twice is the identity, padding stays zero and
    every probability row keeps its sum; sample(reflect=True) draws its coins
    from the generator right after the row indices."""
    from azalea_b200.game.hex import HexGame
    from azalea_b200.replay_device import DeviceReplayBuffer, reflect_batch
    n, B = 5, 256
    buf = DeviceReplayBuffer(1024, n)
    buf.put(stub_rows(n))
    idx = torch.randint(0, len(buf), (B,), device='cuda', generator=torch.Generator(device='cuda').manual_seed(1))
    coins = torch.randint(0, 2, (B,), device='cuda', dtype=torch.uint8,
                          generator=torch.Generator(device='cuda').manual_seed(2))
    for trim in (False, True):
        ref = buf.collate(idx, trim=trim)
        got = buf.collate(idx, trim=trim)
        reflect_batch(got, coins)
        c = coins.cpu().numpy().astype(bool)
        b0, m0, p0 = (ref[k].cpu().numpy() for k in ('board', 'legal_moves', 'moves_prob'))
        b1, m1, p1 = (got[k].cpu().numpy() for k in ('board', 'legal_moves', 'moves_prob'))
        rb, rm = HexGame.rotate_board_moves(b0, m0)
        assert (b1[c] == rb[c]).all() and (b1[~c] == b0[~c]).all()
        assert (m1[c] == rm[c]).all() and (m1[~c] == m0[~c]).all()
        for i in range(B):
            k = int((m0[i] > 0).sum())
            want = p0[i, k - 1::-1] if c[i] else p0[i, :k]
            assert p1[i, :k].tobytes() == want.tobytes()
            assert (p1[i, k:] == 0).all() and (m1[i, k:] == 0).all()
        assert np.allclose(p1.sum(1, dtype=np.float64), p0.sum(1, dtype=np.float64), atol=1e-6)
        reflect_batch(got, coins)
        for k in ('board', 'legal_moves', 'moves_prob'):
            assert torch.equal(got[k], ref[k])
    g1 = torch.Generator(device='cuda').manual_seed(9)
    s = buf.sample(B, generator=g1, reflect=True)
    g2 = torch.Generator(device='cuda').manual_seed(9)
    idx2 = torch.randint(0, len(buf), (B,), device='cuda', generator=g2, dtype=torch.int64)
    coins2 = torch.randint(0, 2, (B,), device='cuda', generator=g2, dtype=torch.uint8)
    want = buf.collate(idx2)
    reflect_batch(want, coins2)
    assert 0 < int(coins2.sum()) < B
    for k in want:
        assert torch.equal(s[k], want[k])


@gpu
def test_train_with_reflect_and_checkpoint_key(tmp_path):
    """train(...) runs with random_reflect on; the saved policy keeps the
    setting and a checkpoint without the key (like the shipped
    hex11-20180712-3362.policy.pth) loads with it off."""
    import azalea_b200 as az
    from azalea_b200 import policy_trainer
    config = train_config(random_reflect=True)
    policy = az.Policy()
    policy.initialize(config)
    assert policy.random_reflect
    path = policy_trainer.train(policy, config, str(tmp_path))
    hist = policy_trainer.train.history
    assert len(hist) == 4 and all(np.isfinite(h['loss']) for h in hist)
    assert sum(h.get('selfplay_games', 0) for h in hist) > 0
    loaded = az.Policy.load(path, device='cuda')
    assert loaded.random_reflect is True
    state = torch.load(path, weights_only=False)
    del state['policy']['random_reflect']
    old = str(tmp_path / 'old.policy.pth')
    torch.save(state, old)
    assert az.Policy.load(old, device='cuda').random_reflect is False
    assert az.Policy().random_reflect is False


@gpu
def test_tournament_reflects_only_the_reflecting_policy():
    """A tournament seat holds games of both policies: only the games whose
    searching policy reflects count rotated rows."""
    from azalea_b200 import Policy
    from azalea_b200.evaluation import play_matches
    from azalea_b200.selfplay import StubEvaluator

    def policy(reflect):
        p = Policy()
        p.net = StubEvaluator(stubs.ROUGH)
        p.simulations, p.search_batch_size, p.exploration_coef = 20, 4, 0.5
        p.exploration_depth, p.exploration_noise_alpha = 15, 0.03
        p.exploration_noise_scale, p.exploration_temperature = 0.0, 1.0
        p.random_reflect = reflect
        return p
    A, Bp = policy(True), policy(False)
    G = 16
    first = [A] * (G // 2) + [Bp] * (G // 2)
    second = [Bp] * (G // 2) + [A] * (G // 2)
    seats = {}

    def hook(seat, key, games):
        seats[id(seat)] = seat
    result, history = play_matches(first, second, 5, seed=1, hook=hook)
    assert len(seats) == 2 and history.shape[0] >= 4
    for s in seats.values():
        refl = s.eng.counters[:, 14].cpu().numpy()
        mine = np.array([p is A for p in s.policies])
        assert (refl[mine] > 0).all() and (refl[~mine] == 0).all()
