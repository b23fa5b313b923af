"""Resignation without a GPU: argument validation, resign_threshold_for on
hand-made histograms, the C ABI surface and Player.read's bookkeeping."""
import logging
import math

import numpy as np
import pytest


def test_resign_setting():
    from azalea_b200.selfplay import resign_setting
    assert resign_setting(None, 0.1) is None
    assert resign_setting(-1.0, 0.1) is None          # <= -1: off
    assert resign_setting(-5, 0.0) is None
    assert resign_setting(-0.8, 0.1) == -0.8
    assert resign_setting(1.0, 1.0) == 1.0
    assert resign_setting(0, 0) == 0.0


@pytest.mark.parametrize('t,p', [(math.nan, 0.1), (1.5, 0.1), (-0.5, -0.1), (-0.5, 1.1),
                                 (-0.5, math.nan), (None, 2.0)])
def test_invalid_resign_arguments(t, p):
    from azalea_b200.selfplay import LockstepSelfPlay, resign_setting
    with pytest.raises(ValueError):
        resign_setting(t, p)
    # rejected before anything touches a device
    with pytest.raises(ValueError):
        LockstepSelfPlay(None, num_games=8, board_size=5, simulations=800, search_batch_size=10,
                         resign_threshold=t, resign_disable_prob=p)


def test_random_play_ignores_resign():
    """RandomPolicy self-play has no search values to resign on: the
    arguments are not even validated (the device is only needed after that)."""
    from azalea_b200.selfplay import LockstepSelfPlay
    try:
        LockstepSelfPlay(None, num_games=8, board_size=5, random_play=True, resign_threshold=math.nan)
    except ValueError:
        pytest.fail('random_play validated the resign setting')
    except Exception:
        pass                    # (no CUDA device here)


def test_abi_surface():
    from azalea_b200 import _cabi
    assert 'az_engine_set_resign' in _cabi.declared_symbols()
    assert _cabi.AZ_BUF_RESIGN == 10
    assert _cabi.AZ_RS_HIST + _cabi.AZ_RS_BINS <= 72


def test_resign_threshold_for():
    from azalea_b200.selfplay import resign_threshold_for
    hist = np.zeros(65, np.int64)
    # 100 calibration games: winners' lowest values in bins 10 (x2), 32 (x3), 64 (the rest)
    hist[10], hist[32], hist[64] = 2, 3, 95
    # edge j counts the games in bins < j: 0 up to edge 10, 2 up to edge 32, 5 after it
    assert resign_threshold_for(hist, 100, 0.0) == -1.0 + 10 / 64
    assert resign_threshold_for(hist, 100, 0.02) == -1.0 + 32 / 64
    assert resign_threshold_for(hist, 100, 0.049) == -1.0 + 32 / 64
    assert resign_threshold_for(hist, 100, 0.05) == 0.0
    assert resign_threshold_for(hist, 100, 1.0) == 0.0
    # no safe edge above -1: -1 turns resignation off
    hist = np.zeros(65, np.int64)
    hist[0] = 10
    assert resign_threshold_for(hist, 10, 0.5) == -1.0
    # edges are exact binary fractions: the bin rule of the kernel puts r = edge in bin j
    for j in range(65):
        r = np.float32(-1.0 + j / 64)
        assert min(64, max(0, int(np.floor((r + np.float32(1)) * np.float32(64))))) == j
    with pytest.raises(ValueError):
        resign_threshold_for(np.zeros(64), 10, 0.05)
    with pytest.raises(ValueError):
        resign_threshold_for(np.zeros(65), 0, 0.05)


def test_player_read_reports_resignation(caplog):
    from azalea_b200.parallel_player import Player
    from test_playout_cap_cpu import FakeSelfPlay, make_rows
    rows = make_rows({5: (3, [0, 1, 2]), 7: (2, [0, 1])})
    player = Player.__new__(Player)
    player.board_size = 3
    player.resign = True
    player.sp = FakeSelfPlay(rows, resign=dict(resigned_games=4, calibration_games=20, false_positives=1))
    with caplog.at_level(logging.WARNING):
        _, metrics = player.read(1)
    assert metrics['resigned_games'] == 4
    assert metrics['resign_calibration_games'] == 20 and metrics['resign_false_positives'] == 1
    assert 'calibration games' not in caplog.text          # 5 %: not above the limit
    player.sp = FakeSelfPlay(rows, resign=dict(resigned_games=4, calibration_games=20, false_positives=2))
    with caplog.at_level(logging.WARNING):
        _, metrics = player.read(1)
    assert metrics['resign_false_positives'] == 2
    assert 'calibration games' in caplog.text              # 10 %
    # off: no resignation metrics
    player.resign = False
    _, metrics = player.read(1)
    assert 'resigned_games' not in metrics
