"""GPU parity: Hex rules in the CUDA engine vs the reference's golden vectors
and vs the C oracle.  Everything goes through the C ABI (Engine)."""
import numpy as np
import pytest
import torch

import oracle
from oracle import HEX_SIZES, crc

pytestmark = pytest.mark.gpu


def make_engine(G, n, **kw):
    from azalea_b200 import Engine
    return Engine(G, n, max_batch=kw.pop('max_batch', 1),
                  nodes_per_game=kw.pop('nodes_per_game', 4), **kw)


@pytest.mark.parametrize('n', HEX_SIZES)
def test_golden_games_lockstep(golden_hex, n):
    """All recorded games of one size advance in lockstep; results, colour to
    move, legal-move lists and final boards match the reference at every ply
    (hex.py:151-179)."""
    g = golden_hex
    moves = g[f'n{n}_moves'].astype(np.int32)
    G = len(moves)
    eng = make_engine(G, n)
    plies = g[f'n{n}_plies']
    for ply in range(int(plies.max()) + 1):
        legal, count = eng.hex_legal_moves()
        legal, count = legal.cpu().numpy(), count.cpu().numpy()
        for gi in range(G):
            if ply <= plies[gi]:
                assert count[gi] == g[f'n{n}_legal_len'][gi, ply]
                assert crc(legal[gi, :count[gi]]) == g[f'n{n}_legal_crc'][gi, ply]
                assert (legal[gi, count[gi]:] == 0).all()
        if ply == plies.max():
            break
        mv = np.where(ply < plies, moves[:, min(ply, moves.shape[1] - 1)], 0)
        res = eng.hex_step(mv).cpu().numpy()
        _, color, result, _ = eng.hex_state()
        live = ply < plies
        assert (res[live] == g[f'n{n}_results'][live, ply]).all()
        assert (result.cpu().numpy() == res).all()
        assert (color.cpu().numpy()[live] == g[f'n{n}_colors'][live, ply]).all()
    board, _, result, plyc = eng.hex_state()
    assert (board.cpu().numpy() == g[f'n{n}_boards']).all()
    assert (plyc.cpu().numpy() == plies).all()
    assert set(result.cpu().numpy().tolist()) <= {1, 3}
    assert (eng.status().cpu().numpy() == 0).all()


@pytest.mark.parametrize('n', (3, 5, 11))
def test_check_win_golden_boards(golden_hex, n):
    """check_win on arbitrary boards (hex.py:204-231)."""
    g = golden_hex
    boards = g[f'n{n}_cw_boards']
    tiles = g[f'n{n}_cw_tiles']
    eng = make_engine(len(boards), n)
    eng.hex_set_state(boards.reshape(len(boards), -1),
                      np.ones(len(boards)), tiles)
    _, _, result, _ = eng.hex_state()
    winner = {0: 0, 3: 1, 1: 2}
    got = np.array([winner[r] for r in result.cpu().numpy().tolist()])
    assert (got == g[f'n{n}_cw_wins']).all()


@pytest.mark.parametrize('n,G', ((11, 4096), (19, 512), (6, 1024)))
def test_random_games_vs_oracle(n, G):
    """Thousands of random games: every ply's result matches the oracle and
    the game ends exactly when the oracle says so."""
    rng = np.random.RandomState(n)
    nn = n * n
    # random permutations played until somebody wins
    perms = np.stack([rng.permutation(nn) + 1 for _ in range(G)]).astype(np.int32)
    want = np.zeros((G, nn), dtype=np.int32)
    length = np.zeros(G, dtype=np.int32)
    for gi in range(G):
        game = oracle.Hex(n)
        for ply in range(nn):
            game.step(int(perms[gi, ply]))
            want[gi, ply] = game.result()
            if want[gi, ply]:
                length[gi] = ply + 1
                break
    eng = make_engine(G, n)
    for ply in range(int(length.max())):
        mv = np.where(ply < length, perms[:, ply], 0)
        res = eng.hex_step(mv).cpu().numpy()
        live = ply < length
        assert (res[live] == want[live, ply]).all(), ply
    board, _, result, plyc = eng.hex_state()
    assert (plyc.cpu().numpy() == length).all()
    assert (result.cpu().numpy() != 0).all()
    _, count = eng.hex_legal_moves()
    assert (count.cpu().numpy() == 0).all()        # hex.py:152-153
    assert (eng.status().cpu().numpy() == 0).all()


def test_full_board_always_has_a_winner():
    """Size-independent property: Hex has no draws."""
    n, G = 11, 2048
    rng = np.random.RandomState(3)
    perms = np.stack([rng.permutation(n * n) + 1 for _ in range(G)]).astype(np.int32)
    eng = make_engine(G, n)
    done = np.zeros(G, dtype=bool)
    for ply in range(n * n):
        res = eng.hex_step(np.where(done, 0, perms[:, ply])).cpu().numpy()
        done |= res != 0
    assert done.all()
    # winner's stones really span the board (checked by the oracle)
    board = eng.hex_state()[0].cpu().numpy()
    for gi in range(0, G, 64):
        b = board[gi].astype(np.int32)
        res = int(eng.hex_state()[2][gi].item())
        color = 1 if res == 3 else 2
        tiles = np.flatnonzero(b.ravel() == color)
        assert any(oracle.check_win(b, t) == color for t in tiles)


def test_dropin_hexgame_interface():
    """HexGame keeps the reference's SearchableEnv behaviour."""
    from azalea_b200 import HexGame
    g = HexGame(3)
    st = g.state
    assert st.color == 0 and st.result == 0 and isinstance(st.color, int)
    assert st.board.dtype == np.int32 and st.legal_moves.dtype == np.int32
    assert list(st.legal_moves) == list(range(1, 10))
    # SURVEY 8c known answers
    for m, r in zip((1, 2, 4, 3, 7), (0, 0, 0, 0, 3)):
        g.step(m)
        assert g.state.result == r
    assert len(g.state.legal_moves) == 0
    with pytest.raises(AssertionError):
        g.step(5)
    g.reset()
    for m, r in zip((1, 4, 2, 5, 9, 6), (0, 0, 0, 0, 0, 1)):
        g.step(m)
        assert g.state.result == r
    g.reset()
    g.step(5)
    g.snapshot()
    g.step(1)
    g.step(9)
    g.restore()
    st = g.state
    assert st.color == 1 and list(st.legal_moves) == [1, 2, 3, 4, 6, 7, 8, 9]
    with pytest.raises(AssertionError):
        g.step(5)
    import pickle
    g2 = pickle.loads(pickle.dumps(g))
    assert (g2.state.board == st.board).all() and g2.state.color == st.color
