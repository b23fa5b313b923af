"""The engine's counter-based coins on the host.  TEST INFRASTRUCTURE ONLY.

Philox4x32-10 as az_philox (az_common.cuh), keyed like the engine: the key of
a game is (seed, global game id), so a test can predict each game's coins
from its id and ply alone.
"""
import numpy as np

M32 = 0xFFFFFFFF
FULL_SEARCH_DOMAIN = 0xCA9F5EA7
RESIGN_DOMAIN = 0x2E51C0A1
MOVE_DOMAIN = 0xC0111700


def philox(c, k):
    """Philox4x32-10 as az_philox (az_common.cuh)."""
    c, k = list(c), list(k)
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & M32, p1 & M32, ((p0 >> 32) ^ c[3] ^ k[1]) & M32, p0 & M32]
        k = [(k[0] + 0x9E3779B9) & M32, (k[1] + 0xBB67AE85) & M32]
    return c


def philox_key(seed, game_id):
    """The Philox key of (seed, global game id)."""
    return ((seed ^ game_id) & M32, ((seed >> 32) ^ (game_id >> 32)) & M32)


def threshold(p):
    """coin < p * 2^32 for an integer coin is coin < ceil(p * 2^32)."""
    return np.ceil(np.float64(np.float32(p)) * 2.0 ** 32)


def full_ply(seed, game_id, ply, p):
    """The playout cap's full-search coin of (seed, global game id, ply)."""
    return philox((ply, 0, 0, FULL_SEARCH_DOMAIN), philox_key(seed, game_id))[0] < threshold(p)


def calibration_game(seed, game_id, p):
    """The resignation calibration coin of (seed, global game id)."""
    return philox((0, 0, 0, RESIGN_DOMAIN), philox_key(seed, game_id))[0] < threshold(p)


def move_at_temperature_1(v, seed, game_id, ply):
    """k_play_commit's inverse CDF over integer weights: exact in any order."""
    x = philox((0, 0, ply, MOVE_DOMAIN), philox_key(seed, game_id))[0]
    w = v.astype(np.float64)
    tot = w.sum()
    target = tot * ((x + 0.5) * (1.0 / 4294967296.0))
    hit = np.flatnonzero((w > 0) & (np.cumsum(w) > target))
    if len(hit):
        return int(hit[0])
    return int(np.flatnonzero(w > 0)[-1])


def game_ids(eng):
    """Each slot's global game id and ply, from the engine's meta."""
    meta = eng.meta.cpu().numpy().astype(np.int64)
    return (meta[:, 10] & M32) | (meta[:, 11] << 32), meta[:, 4].copy()
