"""Generate golden fixtures from the UNMODIFIED Python reference.

Run in the build container (the reference lives at /root/reference there and
does not travel to the GPU box):

    OMP_NUM_THREADS=1 python tests/golden/make_golden.py

It imports the reference with the one-line Numba shim (hex.py:6 imports
``numba.jitclass``, which moved to ``numba.experimental``), drives its Hex
rules, ``Policy``/``AzaleaAgent``/``SearchTree``/``mcts`` with the stub
evaluators of oracle/stubs.py and writes small ``.npz`` files next to this
script.  Nothing here is used at test time except the files it wrote.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get('AZALEA_REFERENCE', '/root/reference')

import numba  # noqa: E402
import numba.experimental  # noqa: E402
numba.jitclass = numba.experimental.jitclass
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import azalea as az  # noqa: E402
from azalea import mcts, search_tree  # noqa: E402
from azalea.game import hex as refhex  # noqa: E402
from azalea.game.hex import HexGame  # noqa: E402
from oracle import crc, stubs  # noqa: E402

_REAL_EVALUATE_BATCH = mcts.evaluate_batch


# ------------------------------------------------------------------ hex ----

def gen_hex_rules():
    out = {}
    rng = np.random.RandomState(1234)
    for n, games in ((2, 8), (3, 40), (4, 40), (5, 40), (7, 30), (9, 20),
                     (11, 40), (13, 10), (19, 8)):
        nn = n * n
        moves = np.zeros((games, nn), dtype=np.int16)
        results = np.zeros((games, nn), dtype=np.int8)
        colors = np.zeros((games, nn), dtype=np.int8)
        legal_crc = np.zeros((games, nn + 1), dtype=np.uint32)
        legal_len = np.zeros((games, nn + 1), dtype=np.int16)
        plies = np.zeros(games, dtype=np.int16)
        boards = np.zeros((games, n, n), dtype=np.int8)
        for g in range(games):
            game = HexGame(n)
            ply = 0
            while True:
                st = game.state
                legal_crc[g, ply] = crc(st.legal_moves)
                legal_len[g, ply] = len(st.legal_moves)
                if st.result:
                    break
                move = int(rng.choice(st.legal_moves))
                game.step(move)
                moves[g, ply] = move
                results[g, ply] = game.state.result
                colors[g, ply] = game.state.color
                ply += 1
            plies[g] = ply
            boards[g] = game.state.board
        out[f'n{n}_moves'] = moves
        out[f'n{n}_results'] = results
        out[f'n{n}_colors'] = colors
        out[f'n{n}_legal_crc'] = legal_crc
        out[f'n{n}_legal_len'] = legal_len
        out[f'n{n}_plies'] = plies
        out[f'n{n}_boards'] = boards
    for n in (2, 3, 5, 11, 19):
        neigh = -np.ones((n * n, 6), dtype=np.int16)
        for t in range(n * n):
            v = refhex.neighbors(np.int32(t), (n, n))
            neigh[t, :len(v)] = v
        out[f'n{n}_neighbors'] = neigh
    for n in (3, 5, 11, 19):
        b = rng.randint(0, 3, size=(6, n, n)).astype(np.int32)
        k = n * n // 2
        mv = np.zeros((6, k + 3), dtype=np.int32)
        for i in range(6):
            sel = np.sort(rng.choice(n * n, size=k, replace=False)) + 1
            m = max(1, k - i)
            mv[i, :m] = sel[:m]             # ragged rows, zero padded
        fb, fm = HexGame.flip_player_board_moves(b, mv)
        out[f'n{n}_flip_in_board'] = b
        out[f'n{n}_flip_in_moves'] = mv
        out[f'n{n}_flip_out_board'] = fb.astype(np.int32)
        out[f'n{n}_flip_out_moves'] = fm.astype(np.int32)
    # check_win called directly on random full-ish boards
    for n in (3, 5, 11):
        b = rng.randint(0, 3, size=(200, n, n)).astype(np.int32)
        tiles = np.zeros(200, dtype=np.int32)
        wins = np.zeros(200, dtype=np.int32)
        for i in range(200):
            nz = np.flatnonzero(b[i])
            tiles[i] = rng.choice(nz)
            wins[i] = refhex.check_win(b[i], np.int32(tiles[i]))
        out[f'n{n}_cw_boards'] = b.astype(np.int8)
        out[f'n{n}_cw_tiles'] = tiles
        out[f'n{n}_cw_wins'] = wins
    np.savez_compressed(os.path.join(HERE, 'hex_rules.npz'), **out)
    print('hex_rules.npz', len(out), 'arrays')


# ----------------------------------------------------------------- mcts ----

def make_policy(sims, batch, coef, net, depth=15, temperature=1.0):
    p = az.Policy()
    p.net = net
    p.simulations = sims
    p.search_batch_size = batch
    p.exploration_coef = coef
    p.exploration_depth = depth
    p.exploration_noise_alpha = 0.03
    p.exploration_noise_scale = 0.25
    p.exploration_temperature = temperature
    return p


def record_search(agent, rec, n):
    """Snapshot the searched root after choose_action()."""
    nn = n * n
    tree = agent.policy.tree
    st = tree.root.move_stats
    k = len(st.num_visits)
    row = dict(
        k=k,
        visits=np.zeros(nn, np.float32), total_value=np.zeros(nn, np.float32),
        prior=np.zeros(nn, np.float32), probs=np.zeros(nn, np.float64))
    row['visits'][:k] = st.num_visits
    row['total_value'][:k] = -st.total_value     # back to the stored sign
    row['prior'][:k] = st.prior_prob
    row['probs'][:k] = agent.info['moves_prob']
    row['root_visits'] = np.float32(tree.root.num_visits)
    row['root_value'] = np.float32(tree.root.total_value)
    row['num_nodes'] = tree.num_nodes
    row['move'] = agent.info['moves'][agent.info['move_id']]
    row['move_id'] = agent.info['move_id']
    row['value'] = np.float32(agent.info['value'])
    row['search_value'] = np.float32(agent.info['metrics']['search_value'])
    for key, v in row.items():
        rec.setdefault(key, []).append(v)


def trace_selfplay(name, n, sims, batch, coef, mode, seed, iface,
                   sampling=False, depth=15, max_plies=10 ** 6):
    """One agent on both sides, one tree reused across plies
    (policy_trainer.py:72-75, play_game.py:46-54)."""
    if iface == 'run':
        mcts.evaluate_batch = _REAL_EVALUATE_BATCH
        net = stubs.StubNet(mode)
    else:
        mcts.evaluate_batch = stubs.make_evaluate_batch(mode)
        net = stubs.StubNet(mode)   # unused by the patched evaluate_batch
    policy = make_policy(sims, batch, coef, net, depth=depth)
    agent = az.AzaleaAgent(lambda: HexGame(n), policy=policy)
    agent.reset()
    agent.seed(seed)
    agent.settings['move_sampling'] = sampling
    rec = {}
    ply = 0
    result = 0
    while ply < max_plies:
        agent.choose_action()
        record_search(agent, rec, n)
        result = agent.execute_action(rec['move'][-1])
        ply += 1
        if result:
            break
    out = {k: np.array(v) for k, v in rec.items()}
    out['result'] = np.int32(result)
    out['config'] = np.array([n, sims, batch, mode, seed, int(sampling),
                              depth], dtype=np.int64)
    out['coef'] = np.float64(coef)
    out['iface'] = np.array(iface)
    mcts.evaluate_batch = _REAL_EVALUATE_BATCH
    print(name, 'plies', ply, 'result', result, 'nodes', out['num_nodes'][-1])
    return {f'{name}/{k}': v for k, v in out.items()}


def trace_match(name, n, sims, batch, coef, modes, seed):
    """Two agents, two trees; every move is pushed into both trees
    (play_game.py:47-48), so opponent moves exercise SearchTree.move's
    reset branch (search_tree.py:122-130)."""
    agents = []
    for i, mode in enumerate(modes):
        # both agents share the patched evaluate_batch, so give both the
        # same stub mode through it and differ in search parameters instead
        policy = make_policy(sims[i], batch[i], coef[i], stubs.StubNet(mode))
        agent = az.AzaleaAgent(lambda: HexGame(n), policy=policy)
        agent.reset()
        agent.seed(seed + 10 * i)
        agents.append(agent)
    mcts.evaluate_batch = stubs.make_evaluate_batch(modes[0])
    rec = {}
    ply = 0
    order = list(agents)
    while True:
        order[0].choose_action()
        record_search(order[0], rec, n)
        move = rec['move'][-1]
        res = [a.execute_action(move) for a in order]
        ply += 1
        if res[0]:
            break
        order = order[::-1]
    out = {k: np.array(v) for k, v in rec.items()}
    out['result'] = np.int32(res[0])
    out['config'] = np.array([n, sims[0], batch[0], sims[1], batch[1],
                              modes[0], seed], dtype=np.int64)
    out['coef'] = np.array(coef, dtype=np.float64)
    mcts.evaluate_batch = _REAL_EVALUATE_BATCH
    print(name, 'plies', ply, 'result', res[0])
    return {f'{name}/{k}': v for k, v in out.items()}


def gen_mcts():
    out = {}
    # SURVEY 8c known answers: uniform stub through the .run interface
    out.update(trace_selfplay('uniform11_run', 11, 800, 10, 0.5, stubs.UNIFORM,
                              7, 'run', max_plies=3))
    # exact-prior traces, whole games
    out.update(trace_selfplay('dyadic11', 11, 800, 10, 0.5, stubs.DYADIC, 3,
                              'patch'))
    out.update(trace_selfplay('rough11', 11, 800, 10, 0.5, stubs.ROUGH, 5,
                              'patch', sampling=True))
    out.update(trace_selfplay('rough11_c075', 11, 200, 10, 0.75, stubs.ROUGH,
                              11, 'patch', max_plies=30))
    for i, (n, sims, batch, coef, mode) in enumerate((
            (3, 50, 4, 1.0, stubs.ROUGH),
            (4, 64, 1, 0.5, stubs.DYADIC),
            (5, 100, 3, 0.75, stubs.ROUGH),
            (5, 200, 16, 1.5, stubs.DYADIC),
            (7, 150, 10, 0.5, stubs.ROUGH),
            (7, 90, 7, 0.3, stubs.ROUGH),
            (9, 120, 10, 0.5, stubs.DYADIC))):
        out.update(trace_selfplay(f'small{i}', n, sims, batch, coef, mode,
                                  100 + i, 'patch', sampling=(i % 2 == 0),
                                  depth=6))
    # the drop-in interface: priors through log -> np.exp
    out.update(trace_selfplay('rough7_run', 7, 100, 10, 0.5, stubs.ROUGH, 21,
                              'run'))
    out.update(trace_selfplay('dyadic11_run', 11, 200, 10, 0.5, stubs.DYADIC,
                              22, 'run', max_plies=12))
    # big board, a few plies
    out.update(trace_selfplay('rough19', 19, 200, 10, 0.5, stubs.ROUGH, 9,
                              'patch', max_plies=6))
    # two trees per game
    out.update(trace_match('match7', 7, (100, 60), (10, 4), (0.5, 1.0),
                           (stubs.ROUGH, stubs.ROUGH), 31))
    out.update(trace_match('match5', 5, (40, 80), (3, 8), (0.75, 0.5),
                           (stubs.DYADIC, stubs.DYADIC), 32))
    np.savez_compressed(os.path.join(HERE, 'mcts_traces.npz'), **out)
    print('mcts_traces.npz', len(out), 'arrays')


def gen_formulas():
    out = {}
    rng = np.random.RandomState(99)
    # score_actions, mcts.py:119-136 (noise off)
    cases = []
    for i in range(64):
        k = int(rng.randint(1, 122))
        nv = rng.randint(0, 40, size=k).astype(np.float32)
        if i % 4 == 0:
            nv[:] = 0
        tv = (rng.uniform(-1, 1, size=k) * nv).astype(np.float32)
        pr = rng.dirichlet(np.ones(k)).astype(np.float32)
        coef = [0.5, 0.75, 0.3, 1.5][i % 4]
        st = search_tree.SearchStats(nv, -tv, pr)
        sc = mcts.score_actions(st, coef, 0.0, 0.03, rng)
        assert sc.dtype == np.float32
        row = np.zeros((4, 121), dtype=np.float32)
        row[0, :k], row[1, :k], row[2, :k], row[3, :k] = nv, tv, pr, sc
        cases.append((k, coef, row))
    out['score_k'] = np.array([c[0] for c in cases], dtype=np.int32)
    out['score_coef'] = np.array([c[1] for c in cases], dtype=np.float64)
    out['score_rows'] = np.stack([c[2] for c in cases])
    # as_distribution, search_tree.py:327-344
    cnt, temps, dist, ks = [], [], [], []
    for i in range(32):
        k = int(rng.randint(1, 60))
        c = rng.randint(0, 30, size=k).astype(np.float32)
        c[rng.randint(k)] += 1
        if i % 3 == 0:
            c[rng.randint(k)] = c.max()     # force a tie at the top
        t = [1.0, 0.0, 0.5, 2.0][i % 4]
        d = search_tree.as_distribution(c, t)
        row = np.zeros(64, np.float32)
        row[:k] = c
        drow = np.zeros(64, np.float64)
        drow[:k] = d
        cnt.append(row)
        ks.append(k)
        temps.append(t)
        dist.append(drow)
    out['dist_k'] = np.array(ks, dtype=np.int32)
    out['dist_counts'] = np.stack(cnt)
    out['dist_temp'] = np.array(temps)
    out['dist_out'] = np.stack(dist)
    # stub evaluator values themselves
    boards = rng.randint(0, 3, size=(12, 5, 5)).astype(np.int32)
    hashes, vals, pris = [], [], []
    for b in boards:
        mv = np.flatnonzero(b.ravel() == 0).astype(np.int32) + 1
        hashes.append(stubs.board_hash(b))
        for mode in (0, 1, 2):
            v, p = stubs.stub_eval(mode, b, mv)
            row = np.zeros(25, np.float32)
            row[:len(p)] = p
            vals.append(v)
            pris.append(row)
    out['stub_boards'] = boards
    out['stub_hash'] = np.array(hashes, dtype=np.uint32)
    out['stub_value'] = np.array(vals, dtype=np.float32)
    out['stub_prior'] = np.stack(pris)
    np.savez_compressed(os.path.join(HERE, 'formulas.npz'), **out)
    print('formulas.npz', len(out), 'arrays')


def gen_network():
    """The reference's HexNetwork (with the torch>=2 contiguity shim, SURVEY
    8c) loaded with azalea_b200's seed-0 state_dict, on fixed inputs."""
    import torch
    import torch.nn.functional as F
    from azalea.network import HexNetwork as RefNet, Network as RefBase
    from azalea_b200.network import HexNetwork
    torch.manual_seed(0)
    mine = HexNetwork(11, 6, 64).eval()
    gen = torch.Generator().manual_seed(1)
    for m in mine.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen) + 0.5)
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
    ref = RefNet(11, 6, 64)
    ref.load_state_dict(mine.state_dict())
    ref.eval()
    rng = np.random.RandomState(5)
    B = 9
    board = rng.randint(0, 3, size=(B, 11, 11)).astype(np.int32)
    lm = np.zeros((B, 121), np.int32)
    for i in range(B):
        e = np.flatnonzero(board[i].ravel() == 0) + 1
        lm[i, :len(e)] = e
    lm = lm[:, :(lm > 0).sum(1).max()]
    with torch.no_grad():
        x = ref.encoder(torch.tensor(board).long()).permute(0, 3, 1, 2).contiguous()
        value, p = RefBase.forward(ref, x)
        logit = ref.move_fc(p)
        tl = torch.tensor(lm)
        logit = torch.gather(logit, 1, (tl - 1).clamp(min=0).long())
        logit.masked_fill_(tl == 0, -99)
        logp = F.log_softmax(logit, dim=1)
    np.savez_compressed(os.path.join(HERE, 'network.npz'), board=board,
                        legal_moves=lm, value=value.numpy(),
                        moves_logprob=logp.numpy())
    print('network.npz')


if __name__ == '__main__':
    which = sys.argv[1:] or ['hex', 'formulas', 'mcts', 'network']
    if 'network' in which:
        gen_network()
    if 'hex' in which:
        gen_hex_rules()
    if 'formulas' in which:
        gen_formulas()
    if 'mcts' in which:
        gen_mcts()
