"""Pin the C oracle against fixtures generated from the Python reference
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

import oracle
from oracle import HEX_SIZES, crc, stubs


@pytest.mark.parametrize('n', HEX_SIZES)
def test_hex_games(golden_hex, n):
    """legal_moves / step / result / colour at every ply of random games
    (hex.py:151-179)."""
    g = golden_hex
    for gi in range(len(g[f'n{n}_plies'])):
        game = oracle.Hex(n)
        plies = int(g[f'n{n}_plies'][gi])
        for ply in range(plies + 1):
            legal = game.legal_moves()
            assert len(legal) == g[f'n{n}_legal_len'][gi, ply]
            assert crc(legal) == g[f'n{n}_legal_crc'][gi, ply]
            if ply == plies:
                break
            game.step(int(g[f'n{n}_moves'][gi, ply]))
            assert game.result() == g[f'n{n}_results'][gi, ply]
            assert game.color - 1 == g[f'n{n}_colors'][gi, ply]
        assert game.result() in (1, 3)
        assert len(game.legal_moves()) == 0
        assert (game.board == g[f'n{n}_boards'][gi]).all()


@pytest.mark.parametrize('n', (2, 3, 5, 11, 19))
def test_neighbors(golden_hex, n):
    want = golden_hex[f'n{n}_neighbors']
    for t in range(n * n):
        got = oracle.neighbors(t, n)
        assert list(got) == [x for x in want[t] if x >= 0]


def test_neighbors_survey_known_answers():
    # SURVEY 8c
    assert list(oracle.neighbors(0, 11)) == [1, 11]
    assert list(oracle.neighbors(10, 11)) == [9, 20, 21]
    assert list(oracle.neighbors(110, 11)) == [99, 100, 111]
    assert list(oracle.neighbors(120, 11)) == [109, 119]
    assert list(oracle.neighbors(60, 11)) == [49, 50, 59, 61, 70, 71]


def test_win_known_answers():
    # SURVEY 8c: 3x3 X column 0, O row 1
    g = oracle.Hex(3)
    for m, r in zip((1, 2, 4, 3, 7), (0, 0, 0, 0, 3)):
        g.step(m)
        assert g.result() == r
    assert len(g.legal_moves()) == 0
    g = oracle.Hex(3)
    for m, r in zip((1, 4, 2, 5, 9, 6), (0, 0, 0, 0, 0, 1)):
        g.step(m)
        assert g.result() == r
    with pytest.raises(AssertionError):
        g.step(3)


@pytest.mark.parametrize('n', (3, 5, 11))
def test_check_win_random_boards(golden_hex, n):
    b = golden_hex[f'n{n}_cw_boards'].astype(np.int32)
    for i in range(len(b)):
        assert oracle.check_win(b[i], golden_hex[f'n{n}_cw_tiles'][i]) == \
            golden_hex[f'n{n}_cw_wins'][i]


@pytest.mark.parametrize('n', (3, 5, 11, 19))
def test_flip(golden_hex, n):
    bi, mi = golden_hex[f'n{n}_flip_in_board'], golden_hex[f'n{n}_flip_in_moves']
    bo, mo = golden_hex[f'n{n}_flip_out_board'], golden_hex[f'n{n}_flip_out_moves']
    for i in range(len(bi)):
        assert (oracle.flip_board(bi[i]) == bo[i]).all()
        assert (oracle.flip_moves(mi[i], n) == mo[i]).all()


def test_score_actions(golden_formulas):
    f = golden_formulas
    for i in range(len(f['score_k'])):
        k = int(f['score_k'][i])
        nv, tv, pr, want = f['score_rows'][i][:, :k]
        got = oracle.score_actions(nv, -tv, pr, float(f['score_coef'][i]))
        assert got.tobytes() == want.tobytes()


def test_stub_evaluators_agree(golden_formulas):
    """C stub == numpy stub == golden (bit for bit)."""
    f = golden_formulas
    row = 0
    for bi, b in enumerate(f['stub_boards']):
        mv = np.flatnonzero(b.ravel() == 0).astype(np.int32) + 1
        assert oracle.board_hash(b) == f['stub_hash'][bi] == stubs.board_hash(b)
        for mode in (0, 1, 2):
            v, p = oracle.stub_eval(mode, b, mv)
            v2, p2 = stubs.stub_eval(mode, b, mv)
            assert np.float32(v).tobytes() == f['stub_value'][row].tobytes()
            assert p.tobytes() == f['stub_prior'][row][:len(p)].tobytes()
            assert np.float32(v2).tobytes() == np.float32(v).tobytes()
            assert p2.tobytes() == p.tobytes()
            row += 1


# ------------------------------------------------------------------ mcts ---

def trace_names(g):
    return sorted({k.split('/')[0] for k in g.files})


def replay_trace(g, name, check):
    """Re-run a recorded self-play trace through the oracle, forcing the
    recorded moves, and hand every searched root to `check`."""
    cfg = g[f'{name}/config']
    n, sims, batch, mode = (int(x) for x in cfg[:4])
    coef = float(g[f'{name}/coef'])
    iface = str(g[f'{name}/iface'])
    game = oracle.Hex(n)
    tree = oracle.Tree()
    plies = len(g[f'{name}/move'])
    for ply in range(plies):
        if iface == 'patch':
            tree.sample_paths_stub(game, sims, batch, coef, mode)
        else:
            run_interface_search(tree, game, sims, batch, coef, mode)
        check(ply, tree)
        legal = game.legal_moves()
        move_id = int(g[f'{name}/move_id'][ply])
        assert legal[move_id] == g[f'{name}/move'][ply]
        tree.move(move_id)
        game.step(int(legal[move_id]))
    assert game.result() == int(g[f'{name}/result'])


def run_interface_search(tree, game, sims, batch, coef, mode):
    """The reference's evaluator interface: priors arrive as
    np.exp(float32 log-probabilities) (mcts.py:210)."""
    def priors(leaves):
        K = max([len(lv['legal_moves']) for lv in leaves] + [1])
        value = np.zeros(len(leaves), np.float32)
        prior = np.zeros((len(leaves), K), np.float32)
        for i, lv in enumerate(leaves):
            if lv['result']:
                continue
            v, p = stubs.stub_eval(mode, lv['board'], lv['legal_moves'])
            value[i] = v
            prior[i, :len(p)] = np.exp(np.log(p))
        return value, prior
    if not tree.root_evaluated():
        _, prior = priors(tree.root_leaf(game))
        tree.expand_root(prior[0])
    for _ in range(sims // batch + 1):
        leaves = tree.select_batch(game, batch, coef)
        value, prior = priors(leaves)
        tree.expand_backup(value, prior)


def test_mcts_traces(golden_mcts):
    """Visit counts, total values, priors, node counts and root statistics
    after every search of every recorded game: bit-exact."""
    g = golden_mcts
    names = [nm for nm in trace_names(g) if not nm.startswith('match')]
    assert len(names) >= 10
    for name in names:
        def check(ply, tree, name=name):
            k = int(g[f'{name}/k'][ply])
            v, w, p = tree.root_stats()
            assert len(v) == k, (name, ply)
            assert v.tobytes() == g[f'{name}/visits'][ply][:k].tobytes(), (name, ply)
            assert w.tobytes() == g[f'{name}/total_value'][ply][:k].tobytes(), (name, ply)
            assert p.tobytes() == g[f'{name}/prior'][ply][:k].tobytes(), (name, ply)
            rn, rw = tree.root_node()
            assert np.float32(rn) == g[f'{name}/root_visits'][ply]
            assert np.float32(rw).tobytes() == g[f'{name}/root_value'][ply].tobytes()
            assert tree.num_nodes == g[f'{name}/num_nodes'][ply], (name, ply)
        replay_trace(g, name, check)


def test_survey_known_answers(golden_mcts):
    """SURVEY 8c: uniform stub, 11x11, 800 sims, batch 10, seed 7."""
    g = golden_mcts
    v = g['uniform11_run/visits'][0]
    assert (v[:84] == 7).all() and (v[84:121] == 6).all()
    assert list(g['uniform11_run/move']) == [30, 17, 57]
    assert list(g['uniform11_run/num_nodes']) == [96633, 192327, 287210]
    assert g['uniform11_run/root_visits'][0] == 810
    assert g['uniform11_run/root_visits'][1] == 817


@pytest.mark.parametrize('name', ('match7', 'match5'))
def test_mcts_match_traces(golden_mcts, name):
    """Two trees per game; opponent moves re-root or reset
    (search_tree.py:115-132)."""
    g = golden_mcts
    cfg = g[f'{name}/config']
    n = int(cfg[0])
    sims, batch = (int(cfg[1]), int(cfg[3])), (int(cfg[2]), int(cfg[4]))
    mode = int(cfg[5])
    coef = [float(x) for x in g[f'{name}/coef']]
    game = oracle.Hex(n)
    trees = [oracle.Tree(), oracle.Tree()]
    for ply in range(len(g[f'{name}/move'])):
        a = ply % 2
        trees[a].sample_paths_stub(game, sims[a], batch[a], coef[a], mode)
        k = int(g[f'{name}/k'][ply])
        v, w, p = trees[a].root_stats()
        assert v.tobytes() == g[f'{name}/visits'][ply][:k].tobytes(), ply
        assert w.tobytes() == g[f'{name}/total_value'][ply][:k].tobytes(), ply
        assert trees[a].num_nodes == g[f'{name}/num_nodes'][ply]
        move_id = int(g[f'{name}/move_id'][ply])
        legal = game.legal_moves()
        for t in trees:
            t.move(move_id)
        game.step(int(legal[move_id]))
    assert game.result() == int(g[f'{name}/result'])
