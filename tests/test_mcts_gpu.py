"""GPU parity: the search kernels vs golden traces of the Python reference
and vs the C oracle.  Visit counts, total values, priors, node counts and
root statistics are compared bit for bit; chosen moves follow."""
import numpy as np
import pytest
import torch

import oracle
from oracle import dirichlet_stats as ds
from oracle import stubs
from oracle.lockstep import assert_root_matches, bits, stub_search

pytestmark = pytest.mark.gpu


class GpuTree:
    """One-game engine driven with the device stub evaluator."""

    def __init__(self, n, batch, mode, **kw):
        from azalea_b200 import Engine
        self.eng = Engine(1, n, max_batch=batch, **kw)
        self.batch, self.mode = batch, mode

    def search(self, sims, coef):
        e = self.eng
        if int(e.root_stats()[3].item()) < 0:
            e.select_root()
            e.stub_eval(self.mode)
            e.expand_root()
        for _ in range(sims // self.batch + 1):
            e.select(self.batch, coef)
            e.stub_eval(self.mode)
            e.expand_backup()

    def stats(self):
        v, w, p, k, rnw, nodes = self.eng.root_stats()
        k = int(k.item())
        return (v[0, :k].cpu().numpy(), w[0, :k].cpu().numpy(),
                p[0, :k].cpu().numpy(), rnw[0].cpu().numpy(),
                int(nodes.item()))


def trace_names(g, iface):
    names = sorted({k.split('/')[0] for k in g.files})
    return [nm for nm in names if not nm.startswith('match')
            and str(g[f'{nm}/iface']) == iface]


def test_golden_traces_device_stub(golden_mcts):
    """Exact-prior traces (whole games on 3x3 .. 19x19, batch sizes 1..16,
    four c_puct values): after every search the root matches the reference
    bit for bit; the recorded moves are then played."""
    g = golden_mcts
    names = trace_names(g, 'patch')
    assert len(names) >= 10
    for name in names:
        n, sims, batch, mode = (int(x) for x in g[f'{name}/config'][:4])
        coef = float(g[f'{name}/coef'])
        t = GpuTree(n, batch, mode)
        for ply in range(len(g[f'{name}/move'])):
            t.search(sims, coef)
            k = int(g[f'{name}/k'][ply])
            v, w, p, rnw, nodes = t.stats()
            where = (name, ply)
            assert len(v) == k, where
            assert bits(v) == bits(g[f'{name}/visits'][ply][:k]), where
            assert bits(w) == bits(g[f'{name}/total_value'][ply][:k]), where
            assert bits(p) == bits(g[f'{name}/prior'][ply][:k]), where
            assert bits(rnw[0]) == bits(g[f'{name}/root_visits'][ply]), where
            assert bits(rnw[1]) == bits(g[f'{name}/root_value'][ply]), where
            assert nodes == g[f'{name}/num_nodes'][ply], where
            move_id = int(g[f'{name}/move_id'][ply])
            t.eng.tree_move([move_id])
            res = int(t.eng.hex_step([int(g[f'{name}/move'][ply])]).item())
            assert int(t.eng.status().item()) == 0, where
        assert res == int(g[f'{name}/result'])


def make_agent(n, sims, batch, coef, mode, depth=15):
    import azalea_b200 as az
    p = az.Policy()
    p.net = stubs.StubNet(mode)
    p.simulations, p.search_batch_size, p.exploration_coef = sims, batch, coef
    p.exploration_depth = depth
    p.exploration_noise_alpha, p.exploration_noise_scale = 0.03, 0.25
    p.exploration_temperature = 1.0
    return az.AzaleaAgent(lambda: az.HexGame(n), policy=p)


def test_dropin_agent_reproduces_reference_games(golden_mcts):
    """The reference's own calling sequence -- AzaleaAgent.seed /
    choose_action / execute_action with an evaluator object plugged into
    Policy.net -- reproduces the reference's moves, probabilities, value,
    metrics and tree statistics."""
    g = golden_mcts
    for name in trace_names(g, 'run'):
        n, sims, batch, mode, seed, sampling, depth = \
            (int(x) for x in g[f'{name}/config'])
        agent = make_agent(n, sims, batch, float(g[f'{name}/coef']), mode, depth)
        agent.reset()
        agent.seed(seed)
        agent.settings['move_sampling'] = bool(sampling)
        for ply in range(len(g[f'{name}/move'])):
            move = agent.choose_action()
            where = (name, ply)
            k = int(g[f'{name}/k'][ply])
            v, w, p, rn, rw = agent.policy.tree.root_stats()
            assert bits(v) == bits(g[f'{name}/visits'][ply][:k]), where
            assert bits(w) == bits(g[f'{name}/total_value'][ply][:k]), where
            assert bits(p) == bits(g[f'{name}/prior'][ply][:k]), where
            assert move == g[f'{name}/move'][ply], where
            info = agent.info
            assert info['move_id'] == g[f'{name}/move_id'][ply]
            assert info['moves_prob'].tobytes() == g[f'{name}/probs'][ply][:k].tobytes()
            assert bits(info['value']) == bits(g[f'{name}/value'][ply])
            m = info['metrics']
            assert m['search_tree_nodes'] == g[f'{name}/num_nodes'][ply], where
            assert np.isclose(m['search_value'], g[f'{name}/search_value'][ply], atol=1e-6)
            assert m['search_root_children'] == k
            result = agent.execute_action(move)
        if len(g[f'{name}/move']) > 20:
            assert result == int(g[f'{name}/result'])


def test_survey_known_answers_dropin():
    """SURVEY 8c: uniform stub, 11x11, 800 sims, batch 10, c 0.5, seed 7."""
    agent = make_agent(11, 800, 10, 0.5, stubs.UNIFORM)
    agent.reset()
    agent.seed(7)
    moves, nodes = [], []
    for ply in range(3):
        moves.append(int(agent.choose_action()))
        nodes.append(int(agent.info['metrics']['search_tree_nodes']))
        if ply == 0:
            v = agent.policy.tree.root_stats()[0]
            assert (v[:84] == 7).all() and (v[84:] == 6).all()
        agent.execute_action(moves[-1])
    assert moves == [30, 17, 57]
    assert nodes == [96633, 192327, 287210]


@pytest.mark.parametrize('name', ('match7', 'match5'))
def test_two_tree_match(golden_mcts, name):
    """Two trees per game: opponent moves re-root or reset the other tree
    (search_tree.py:115-132, play_game.py:47-48)."""
    g = golden_mcts
    cfg = g[f'{name}/config']
    n, mode = int(cfg[0]), int(cfg[5])
    sims, batch = (int(cfg[1]), int(cfg[3])), (int(cfg[2]), int(cfg[4]))
    coef = [float(x) for x in g[f'{name}/coef']]
    trees = [GpuTree(n, batch[0], mode), GpuTree(n, batch[1], mode)]
    for ply in range(len(g[f'{name}/move'])):
        a = ply % 2
        trees[a].search(sims[a], coef[a])
        k = int(g[f'{name}/k'][ply])
        v, w, p, rnw, nodes = trees[a].stats()
        assert bits(v) == bits(g[f'{name}/visits'][ply][:k]), ply
        assert bits(w) == bits(g[f'{name}/total_value'][ply][:k]), ply
        assert nodes == g[f'{name}/num_nodes'][ply], ply
        for t in trees:
            t.eng.tree_move([int(g[f'{name}/move_id'][ply])])
            res = int(t.eng.hex_step([int(g[f'{name}/move'][ply])]).item())
    assert res == int(g[f'{name}/result'])


@pytest.mark.parametrize('n,G,sims,batch,coef,mode,plies', (
    (11, 256, 800, 10, 0.5, stubs.ROUGH, 12),
    (11, 64, 320, 32, 1.25, stubs.DYADIC, 40),
    (7, 512, 200, 8, 0.5, stubs.ROUGH, 49),
    (19, 16, 400, 10, 0.5, stubs.ROUGH, 6),
    (5, 256, 60, 5, 2.0, stubs.ROUGH, 25),
))
def test_lockstep_games_vs_oracle(n, G, sims, batch, coef, mode, plies):
    """Many different games searched in lockstep on the GPU against the C
    oracle, one oracle tree per game.  Each game follows its own line (the
    g-th most visited move, ties to the lowest index), so the trees differ."""
    from azalea_b200 import Engine
    eng = Engine(G, n, max_batch=batch)
    games = [oracle.Hex(n) for _ in range(G)]
    trees = [oracle.Tree(max_nodes=3_000_000) for _ in range(G)]
    alive = np.ones(G, dtype=bool)
    for ply in range(plies):
        stub_search(eng, mode, batch, coef, sims // batch + 1)
        stats = [x.cpu().numpy() for x in eng.root_stats()]
        assert (eng.status().cpu().numpy()[alive] == 0).all()
        move_ids = -np.ones(G, dtype=np.int32)
        moves = np.zeros(G, dtype=np.int32)
        for gi in np.flatnonzero(alive):
            trees[gi].sample_paths_stub(games[gi], sims, batch, coef, mode)
            ov = assert_root_matches(stats, gi, trees[gi], (ply, gi))
            order = np.argsort(-ov, kind='stable')
            mid = int(order[(gi + ply) % min(len(ov), 3)])
            move_ids[gi] = mid
            moves[gi] = games[gi].legal_moves()[mid]
            trees[gi].move(mid)
            games[gi].step(int(moves[gi]))
        eng.tree_move(move_ids)
        res = eng.hex_step(moves).cpu().numpy()
        for gi in np.flatnonzero(alive):
            assert res[gi] == games[gi].result()
            if res[gi]:
                alive[gi] = False
        if not alive.any():
            break
    cnt = eng.counter_totals()
    assert cnt['simulations'] > 0 and cnt['sum_depth'] >= cnt['simulations']


def test_search_tree_full_is_raised():
    """search_tree.MAX_NODES emulation: SearchTreeFull (search_tree.py:258)."""
    import azalea_b200 as az
    from azalea_b200 import search_tree
    old = search_tree.MAX_NODES
    search_tree.MAX_NODES = 5000
    try:
        agent = make_agent(11, 800, 10, 0.5, stubs.UNIFORM)
        agent.reset()
        agent.seed(1)
        with pytest.raises(az.SearchTreeFull):
            agent.choose_action()
    finally:
        search_tree.MAX_NODES = old
    # the oracle raises at the same limit
    t = oracle.Tree(max_nodes=5000)
    with pytest.raises(oracle.SearchTreeFull):
        t.sample_paths_stub(oracle.Hex(11), 800, 10, 0.5, 0)


def test_pool_overflow_is_flagged_not_corrupting():
    from azalea_b200 import Engine, _cabi
    eng = Engine(4, 11, max_batch=10, nodes_per_game=2000)
    stub_search(eng, 0, 10, 0.5, 40)
    st = eng.status().cpu().numpy()
    assert (st == _cabi.AZ_ST_POOL_FULL).all()
    v, _, _, k, _, _ = eng.root_stats()
    assert (k.cpu().numpy() == 121).all()
    assert float(v.sum()) > 0


def test_soft_pool_full_skips_expansions_and_keeps_the_game():
    """AZ_CFG_SOFT_POOL_FULL (the lockstep drivers' mode): when a game's pool
    half is exhausted the expansion is skipped and counted, no status bit is
    set, visits keep accumulating (every descent is still backed up), and the
    game goes on: after the move the re-root compacts the pool and expansion
    resumes.  Whole games finish with games_failed == 0."""
    from azalea_b200 import Engine, LockstepSelfPlay, StubEvaluator
    eng = Engine(4, 11, max_batch=10, nodes_per_game=2000, soft_pool_full=True)
    stub_search(eng, 2, 10, 0.5, 40)
    assert (eng.status().cpu().numpy() == 0).all()
    cnt = eng.counter_totals()
    assert cnt['pool_skipped_expansions'] > 0
    v, _, _, k, rnw, _ = eng.root_stats()
    assert (k.cpu().numpy() == 121).all()
    # 400 descents per game, duplicates inside a batch backed up once
    assert (rnw[:, 0].cpu().numpy() >= 40).all() and (rnw[:, 0].cpu().numpy() <= 400).all()
    # whole games on a pool far too small for a move's growth
    sp = LockstepSelfPlay(StubEvaluator(2), num_games=32, board_size=7, simulations=120,
                          search_batch_size=6, nodes_per_game=1500, cuda_graph=False)
    for _ in range(60):
        sp.step_move()
    c = sp.counters()
    assert c['pool_skipped_expansions'] > 0 and c['games_failed'] == 0 and c['games'] >= 32
    assert (sp.eng.status().cpu().numpy() == 0).all()
    rows = sp.harvest()
    from azalea_b200.engine import decode_replay_rows
    h, board, _ = decode_replay_rows(rows, 7)
    game = oracle.Hex(7)
    first = [i for i in range(len(h)) if h['game_id'][i] == h['game_id'][0]]
    for i in first:                                 # a finished game is a legal game
        assert (board[i] == game.board).all()
        game.step(int(h['move'][i]))
    assert game.result() == h['result'][first[0]]


def test_reroot_compaction_preserves_subtree():
    """Re-rooting copies the kept subtree; searching on from it gives the
    same statistics as the reference, which keeps everything in place
    (covered ply by ply by the golden traces); here: the kept child's own
    N/W survive the move."""
    t = GpuTree(7, 10, stubs.ROUGH)
    t.search(300, 0.5)
    v, w, p, rnw, _ = t.stats()
    mid = int(np.argmax(v))
    t.eng.tree_move([mid])
    v2, w2, p2, rnw2, _ = t.stats()
    assert bits(rnw2[0]) == bits(v[mid]) and bits(rnw2[1]) == bits(w[mid])
    assert v2.sum() <= v[mid]


def test_dirichlet_noise_statistics():
    """Root noise (mcts.py:126-131) is only statistically comparable: with
    epsilon = 1 the prior is pure Dirichlet(alpha) noise redrawn per
    simulation, so visits spread over many more children than without."""
    from azalea_b200 import Engine
    G = 64
    eng = Engine(G, 11, max_batch=10, seed=5)
    stub_search(eng, 0, 10, 2.0, 30, eps=0.25, alpha=0.03)
    v = eng.root_stats()[0].cpu().numpy()
    # duplicate leaves inside a batch are backed up once (mcts.py:75)
    assert (v.sum(1) <= 300).all() and (v.sum(1) >= 280).all()
    assert (eng.status().cpu().numpy() == 0).all()
    # different games draw different noise
    assert len({v[g].tobytes() for g in range(G)}) > G // 2


@pytest.mark.parametrize('alpha,k', ds.CASES + ((0.03, 1), (2.5, 1)))
def test_dirichlet_noise_distribution(alpha, k):
    """The device noise (Engine.noise_sample, the vectors k_select draws:
    test_root_noise_gpu.py) has the law of RandomState.dirichlet(np.full(k,
    alpha)) (mcts.py:126-127).  Exact: k = 1 gives 1.0; values finite and
    >= 0, no row of zeros, rows sum to 1 within k 2^-23.  Statistical, on
    4096 games x several simulation counters (oracle.dirichlet_stats, whose
    thresholds test_root_noise_cpu.py holds to samples of known law):
    two-sample KS of the components and of the sums of the first 32 and
    ceil(k/2) components against NumPy, and the correlations of child j with
    j + 32, of one child across neighbouring games and across neighbouring
    counters."""
    from azalea_b200 import Engine
    G = ds.GAMES
    eng = Engine(G, 19, max_batch=1, nodes_per_game=4, seed=11)
    if k == 1:
        for s in (0, 1, 12345):
            assert (eng.noise_sample(alpha, 1, sim=s) == 1.0).all()
        return
    S = ds.num_sims(k)
    draws = torch.stack([eng.noise_sample(alpha, k, sim=s) for s in range(S)]).cpu().numpy()
    assert draws.shape == (S, G, k)
    assert ds.exact_failures(draws) == []
    rep = ds.report(draws, alpha, seed=0)
    assert ds.failures(rep) == [], rep
    # moments and the largest component (the mean of all components is 1/k for any sampler
    # whose rows sum to 1: not a check)
    rows = draws.reshape(-1, k).astype(np.float64)
    want_var = (k - 1) / (k * k * (k * alpha + 1))
    assert abs(rows.var() / want_var - 1) < 0.05, (rows.var(), want_var)
    ref = np.random.RandomState(0).dirichlet(np.full(k, alpha), size=len(rows))
    q = [0.1, 0.25, 0.5, 0.75, 0.9]
    got_q, ref_q = np.quantile(rows.max(1), q), np.quantile(ref.max(1), q)
    assert np.abs(got_q - ref_q).max() < 0.02, (got_q, ref_q)
    # different simulations and different games draw different vectors
    assert len({rows[i].tobytes() for i in range(0, len(rows), 97)}) > 300


def test_deep_search_19x19_vs_oracle():
    """Config 5 shape: 19x19, thousands of simulations per move, a node pool
    of millions per game -- still bit-exact against the oracle."""
    from azalea_b200 import Engine
    n, G, sims, batch, coef, mode = 19, 2, 4000, 10, 0.5, stubs.ROUGH
    eng = Engine(G, n, max_batch=batch, nodes_per_game=3_500_000)
    games = [oracle.Hex(n) for _ in range(G)]
    trees = [oracle.Tree(max_nodes=8_000_000) for _ in range(G)]
    for ply in range(3):
        stub_search(eng, mode, batch, coef, sims // batch + 1)
        v, w, p, k, rnw, nodes = (x.cpu().numpy() for x in eng.root_stats())
        assert (eng.status().cpu().numpy() == 0).all()
        move_ids = np.zeros(G, dtype=np.int32)
        moves = np.zeros(G, dtype=np.int32)
        for gi in range(G):
            trees[gi].sample_paths_stub(games[gi], sims, batch, coef, mode)
            ov, ow, op = trees[gi].root_stats()
            assert bits(v[gi, :len(ov)]) == bits(ov), (ply, gi)
            assert bits(w[gi, :len(ov)]) == bits(ow), (ply, gi)
            assert nodes[gi] == trees[gi].num_nodes
            move_ids[gi] = int(np.argsort(-ov, kind='stable')[gi])
            moves[gi] = games[gi].legal_moves()[move_ids[gi]]
            trees[gi].move(int(move_ids[gi]))
            games[gi].step(int(moves[gi]))
        eng.tree_move(move_ids)
        eng.hex_step(moves)
    assert nodes.max() > 3_000_000


@pytest.mark.parametrize('name', ('rough7_run', 'dyadic11_run'))
def test_play_game_reproduces_reference_game(golden_mcts, name):
    """azalea_b200.play_game (azalea/play_game.py:18-78) with one self-play
    agent on both sides, as policy_trainer.py:72-75 plays it: the moves, the
    result, the recorded states / move distributions and the alternating
    rewards (play_game.py:63-67) are those of the reference's game."""
    import azalea_b200 as az
    g = golden_mcts
    n, sims, batch, mode, seed, sampling, depth = (int(x) for x in g[f'{name}/config'])
    moves = [int(m) for m in g[f'{name}/move']]
    agent = make_agent(n, sims, batch, float(g[f'{name}/coef']), mode, depth)
    agent.seed(seed)
    agent.settings['move_sampling'] = bool(sampling)
    whole = int(g[f'{name}/result']) != 0       # the trace is a finished game
    result, data, metrics = az.play_game([agent], collect_data=True,
                                         game_max_length=300 if whole else len(moves))
    assert len(data) == len(moves)
    board = np.zeros((n, n), dtype=np.int32)
    for ply, rec_move in enumerate(moves):
        st = data.state[ply]
        assert st.color == ply % 2 and st.result == 0
        assert (st.board == board).all(), ply
        k = int(g[f'{name}/k'][ply])
        assert len(st.legal_moves) == k
        want = g[f'{name}/probs'][ply][:k].astype(np.float32)
        assert data.moves_prob[ply].dtype == np.float32
        assert data.moves_prob[ply].tobytes() == want.tobytes(), ply
        board.flat[rec_move - 1] = 1 + ply % 2
    if whole:
        assert result == int(g[f'{name}/result'])
        assert (agent.game.state.board == board).all()
    else:
        assert result == 2                      # game_max_length reached: a draw (play_game.py:57-61)
    want_reward = np.full(len(moves), result - 2.0, dtype=np.float32)
    want_reward[1::2] *= -1
    assert np.array_equal(np.asarray(data.reward, dtype=np.float32), want_reward)
    assert metrics['moves_per_game'] == len(moves) and metrics['games'] == 1
    assert metrics['reward'] == float(want_reward[-1])
    nodes = np.asarray(g[f'{name}/num_nodes'], dtype=np.float64)
    assert np.isclose(metrics['search_tree_nodes'], nodes.mean())
    assert np.isclose(metrics['search_value'], np.mean(g[f'{name}/search_value']), atol=1e-5)


@pytest.mark.parametrize('G,n,B', ((48, 5, 8), (6, 19, 10), (1, 11, 10), (33, 3, 16)))
def test_packed_leaves_engine_level(G, n, B):
    """AZ_CFG_PACK_LEAVES: az_mcts_select writes the leaves that need the
    evaluator (unique, not terminal; mcts.py:75,139-152,192-200) as consecutive
    rows of the window, leaf_info[..][3] = depth | row << 10, the count in
    AZ_BUF_LEAF_ROWS[g0]; az_mcts_expand_backup reads value / prior at the row
    and resets the count.  Same searches as the slot-indexed engine, bit for
    bit, on full-board and windowed launches."""
    from azalea_b200 import Engine
    coef = 0.5
    nn = n * n
    a = Engine(G, n, max_batch=B, seed=9)
    b = Engine(G, n, max_batch=B, seed=9, pack_leaves=True)
    gen = torch.Generator(device='cuda').manual_seed(1)
    # whole engine, then two windows
    windows = [(0, 0), (0, G // 2), (G // 2, G - G // 2)] if G >= 4 else [(0, 0)] * 3
    for eng in (a, b):
        eng.select_root(); eng.stub_eval(stubs.ROUGH); eng.expand_root()
    for it in range(40):
        w = windows[it % 3] if it >= 10 else (0, 0)
        g0, cnt = w if w[1] else (0, G)
        for eng in (a, b):
            eng.set_window(*w)
            eng.select(B, coef)
        ia = a.leaf_info.cpu().numpy()[g0:g0 + cnt]
        ib = b.leaf_info.cpu().numpy()[g0:g0 + cnt]
        live = int(b.leaf_rows[g0].item())
        need = (ia[..., 0] >= 0) & ((ia[..., 1] & 0xff) == 0)
        assert live == int(need.sum()) and (live > 0 or n == 3)     # (3x3 games end within the search)
        assert (ia[..., :3] == ib[..., :3]).all()
        assert ((ib[..., 3] & 1023) == ia[..., 3]).all()
        rows = (ib[..., 3] >> 10)[need]
        assert sorted(rows.tolist()) == list(range(live))       # dense, every row used once
        # a game's leaves sit in consecutive rows, in slot order
        ca = a.leaf_board.cpu().numpy()[g0:g0 + cnt].reshape(cnt * B, -1)
        cb = b.leaf_board.cpu().numpy()[g0:g0 + cnt].reshape(cnt * B, -1)
        assert (cb[rows] == ca[need.reshape(-1)]).all()
        # evaluator outputs: slot-indexed for a, row-indexed for b
        value = torch.rand(cnt * B, device='cuda', generator=gen) * 2 - 1
        prior = torch.randn(cnt * B, nn, device='cuda', generator=gen)
        a.value[g0:g0 + cnt].view(-1).copy_(value)
        a.prior[g0:g0 + cnt].view(-1, nn).copy_(prior)
        idx = torch.from_numpy(np.flatnonzero(need.reshape(-1))).cuda()
        rt = torch.from_numpy(rows.astype(np.int64)).cuda()
        b.value[g0:g0 + cnt].view(-1)[rt] = value[idx]
        b.prior[g0:g0 + cnt].view(-1, nn)[rt] = prior[idx]
        for eng in (a, b):
            eng.expand_backup(None, None, 1)
        assert int(b.leaf_rows[g0].item()) == 0
        for eng in (a, b):
            eng.set_window(0, 0)
        sa, sb = a.root_stats(), b.root_stats()
        for x, y in zip(sa, sb):
            assert torch.equal(x, y)
    assert (a.status().cpu().numpy() == 0).all() and (b.status().cpu().numpy() == 0).all()
    assert a.counter_totals() == b.counter_totals()
