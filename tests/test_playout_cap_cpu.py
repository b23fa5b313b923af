"""Playout cap randomization without a GPU: argument validation, the
fast_descents arithmetic, the C ABI surface and Player.read's bookkeeping
when a game's first or last ply left no replay row."""
import math

import numpy as np
import pytest


def test_fast_descents_follow_the_num_batches_rule():
    from azalea_b200.selfplay import playout_cap_descents
    # mcts.py:268 num_batches = sims // batch + 1, applied to the fast count
    assert playout_cap_descents(0.25, 100, 800, 10) == 110
    assert playout_cap_descents(0.5, 10, 60, 6) == 12
    assert playout_cap_descents(0.0, 0, 30, 4) == 4
    assert playout_cap_descents(0.5, 5, 30, 4) == 8
    # off: the fast count is not looked at
    assert playout_cap_descents(1.0, None, 800, 10) == 0
    assert playout_cap_descents(2.0, 10_000, 800, 10) == 0


@pytest.mark.parametrize('p,fast', [(0.5, None), (0.25, 800), (0.25, 809), (0.0, 10_000), (0.5, -1),
                                    (-0.1, 100), (math.nan, 100)])
def test_invalid_playout_cap_arguments(p, fast):
    from azalea_b200.selfplay import LockstepSelfPlay, playout_cap_descents
    with pytest.raises(ValueError):
        playout_cap_descents(p, fast, 800, 10)
    # rejected before anything touches a device
    with pytest.raises(ValueError):
        LockstepSelfPlay(None, num_games=8, board_size=5, simulations=800, search_batch_size=10,
                         full_search_prob=p, fast_simulations=fast)


def test_random_play_ignores_the_cap():
    """RandomPolicy self-play has no search to cap: the arguments are not
    even validated (the device is only needed after that)."""
    from azalea_b200.selfplay import LockstepSelfPlay
    try:
        LockstepSelfPlay(None, num_games=8, board_size=5, random_play=True, full_search_prob=0.5)
    except ValueError:
        pytest.fail('random_play validated the playout cap')
    except Exception:
        pass                    # (no CUDA device here)


def test_abi_surface():
    from azalea_b200 import _cabi
    assert 'az_engine_set_playout_cap' in _cabi.declared_symbols()
    assert _cabi.COUNTER_NAMES[15] == 'fast_plies' and len(_cabi.COUNTER_NAMES) == 16


def make_rows(games, n=3):
    """Replay rows of finished games {game_id: (game_len, [plies kept])},
    sorted by (game id, ply), on an empty n x n board."""
    from azalea_b200.engine import ROW_HEADER, replay_row_bytes
    nn = n * n
    rb = replay_row_bytes(n)
    out = []
    for gid, (length, plies) in sorted(games.items()):
        for ply in plies:
            row = np.zeros(rb, np.uint8)
            h = np.zeros(1, ROW_HEADER)
            h['game_id'], h['ply'], h['color'], h['num_moves'] = gid, ply, ply % 2, nn
            h['reward'], h['result'], h['temperature'] = (-1.0 if ply % 2 else 1.0), 3, 1.0
            h['move'], h['game_len'] = 1, length
            row[:ROW_HEADER.itemsize] = h.view(np.uint8)
            vis = np.ones(nn, np.float32)
            off = ROW_HEADER.itemsize + ((nn + 15) & ~15)
            row[off:off + 4 * nn] = vis.view(np.uint8)
            out.append(row)
    return np.stack(out)


class FakeSelfPlay:
    """One harvest of canned rows; counters as the engine would report."""

    def __init__(self, rows, fast):
        self.rows, self.fast, self.moves = rows, fast, 0
        outer = self

        class Eng:
            def replay_count(self):
                return len(outer.rows) if outer.moves else 0
        self.eng = Eng()

    def step_move(self):
        self.moves += 1

    def harvest(self):
        return self.rows

    def counters(self):
        return {'fast_plies': self.fast if self.moves else 0, 'games_failed': 0,
                'pool_skipped_expansions': 0}


def test_player_read_counts_games_by_id():
    """Game 7 lost its ply 0 row and game 8 its last row to fast plies: the
    metrics still count three games and their true lengths."""
    from azalea_b200.parallel_player import Player
    games = {5: (5, [0, 1, 2, 3, 4]), 7: (6, [1, 2, 4, 5]), 8: (7, [0, 3, 5])}
    rows = make_rows(games)
    player = Player.__new__(Player)
    player.board_size = 3
    player.sp = FakeSelfPlay(rows, fast=6)
    examples, metrics = player.read(1)
    assert len(examples) == len(rows) == 12
    assert metrics['games'] == 3
    assert metrics['moves_per_game'] == 5 + 6 + 7
    assert metrics['fast_plies'] == 6
    assert metrics['reward'] == 1.0 - 1.0 - 1.0      # each game's last row
