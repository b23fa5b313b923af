"""CPU oracle for the Azalea self-play search hot path.  TEST INFRASTRUCTURE ONLY.

ctypes wrapper over ``oracle/build/libazalea_oracle.so`` (built from
azalea_oracle.c by ``make -C oracle`` / ``__graft_entry__.build()``).  Only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs
may import this package; ``azalea_b200`` never does.

Parity status: pinned against fixtures generated from the unmodified Python
reference (tests/golden/make_golden.py, tests/test_oracle_golden.py).
"""
import ctypes as C
import os
import subprocess
import zlib

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, 'build', 'libazalea_oracle.so')

MAXT = 19 * 19
OMAX_BATCH = 64
# the board sizes of tests/golden/hex_rules.npz
HEX_SIZES = (2, 3, 4, 5, 7, 9, 11, 13, 19)


def crc(a):
    """The checksum tests/golden/hex_rules.npz records legal-move lists by."""
    return zlib.crc32(np.ascontiguousarray(a, dtype=np.int32).tobytes())


class OHex(C.Structure):
    _fields_ = [('n', C.c_int32), ('color', C.c_int32), ('winner', C.c_int32),
                ('board', C.c_int32 * MAXT)]


class OTree(C.Structure):
    _fields_ = [('max_nodes', C.c_int64), ('num_nodes', C.c_int64),
                ('root_id', C.c_int32),
                ('parent', C.POINTER(C.c_int32)),
                ('first_child', C.POINTER(C.c_int32)),
                ('num_children', C.POINTER(C.c_int32)),
                ('num_visits', C.POINTER(C.c_float)),
                ('total_value', C.POINTER(C.c_float)),
                ('prior_prob', C.POINTER(C.c_float))]


class OLeaves(C.Structure):
    _fields_ = [('count', C.c_int32),
                ('node', C.c_int32 * OMAX_BATCH),
                ('color', C.c_int32 * OMAX_BATCH),
                ('result', C.c_int32 * OMAX_BATCH),
                ('num_moves', C.c_int32 * OMAX_BATCH),
                ('board_view', (C.c_int32 * MAXT) * OMAX_BATCH),
                ('moves_view', (C.c_int32 * MAXT) * OMAX_BATCH),
                ('sum_children', C.c_int64),
                ('sum_depth', C.c_int64)]


def build(force=False):
    """Compile the oracle with gcc (idempotent)."""
    src = os.path.join(_HERE, 'azalea_oracle.c')
    hdr = os.path.join(_HERE, 'azalea_oracle.h')
    if (not force and os.path.exists(_LIB_PATH)
            and os.path.getmtime(_LIB_PATH) >= max(os.path.getmtime(src),
                                                   os.path.getmtime(hdr))):
        return _LIB_PATH
    subprocess.check_call(['make', '-C', _HERE, '-B'],
                          stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        build()
    L = C.CDLL(_LIB_PATH)
    i32p, f32p = C.POINTER(C.c_int32), C.POINTER(C.c_float)
    i64p = C.POINTER(C.c_int64)
    L.ohex_init.argtypes = [C.POINTER(OHex), C.c_int]
    L.ohex_legal_moves.argtypes = [C.POINTER(OHex), i32p]
    L.ohex_result.argtypes = [C.POINTER(OHex)]
    L.ohex_step.argtypes = [C.POINTER(OHex), C.c_int]
    L.ohex_neighbors.argtypes = [C.c_int, C.c_int, i32p]
    L.ohex_check_win.argtypes = [i32p, C.c_int, C.c_int]
    L.ohex_flip_board.argtypes = [i32p, C.c_int, i32p]
    L.ohex_flip_moves.argtypes = [i32p, C.c_int, C.c_int, i32p]
    L.ostub_board_hash.argtypes = [i32p, C.c_int]
    L.ostub_board_hash.restype = C.c_uint32
    L.ostub_eval.argtypes = [C.c_int, i32p, C.c_int, i32p, C.c_int, f32p, f32p]
    L.otree_new.argtypes = [C.c_int64]
    L.otree_new.restype = C.POINTER(OTree)
    L.otree_free.argtypes = [C.POINTER(OTree)]
    L.otree_reset.argtypes = [C.POINTER(OTree)]
    L.otree_move.argtypes = [C.POINTER(OTree), C.c_int]
    L.otree_root_stats.argtypes = [C.POINTER(OTree), f32p, f32p, f32p]
    L.omcts_score_actions.argtypes = [f32p, f32p, f32p, C.c_int, C.c_float,
                                      f32p]
    L.omcts_select_batch.argtypes = [C.POINTER(OTree), C.POINTER(OHex),
                                     C.c_int, C.c_float, C.POINTER(OLeaves)]
    L.omcts_expand_backup.argtypes = [C.POINTER(OTree), C.POINTER(OLeaves),
                                      f32p, f32p, C.c_int, f32p]
    L.omcts_root_leaf.argtypes = [C.POINTER(OTree), C.POINTER(OHex),
                                  C.POINTER(OLeaves)]
    L.omcts_expand_root.argtypes = [C.POINTER(OTree), C.POINTER(OLeaves), f32p]
    L.omcts_sample_paths_stub.argtypes = [C.POINTER(OTree), C.POINTER(OHex),
                                          C.c_int, C.c_int, C.c_float, C.c_int,
                                          f32p]
    L.obench_selfplay_stub.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_float, C.c_int, C.c_int,
                                       C.c_int64, C.c_uint64, i64p,
                                       C.POINTER(C.c_double), i64p, i64p, i64p]
    L.obench_selfplay_stub.restype = C.c_int64
    _lib = L
    return L


def _i32(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _f32(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


class SearchTreeFull(Exception):
    pass


class Hex:
    """HexGameImpl (game/hex.py:144-179) through the C oracle."""

    def __init__(self, n=11):
        self.g = OHex()
        lib().ohex_init(C.byref(self.g), n)

    @property
    def n(self):
        return self.g.n

    @property
    def color(self):
        return self.g.color

    @property
    def board(self):
        n = self.g.n
        return np.array(self.g.board[:n * n], dtype=np.int32).reshape(n, n)

    def legal_moves(self):
        out = np.zeros(MAXT, dtype=np.int32)
        k = lib().ohex_legal_moves(C.byref(self.g), _i32(out))
        return out[:k].copy()

    def result(self):
        return lib().ohex_result(C.byref(self.g))

    def step(self, move):
        if lib().ohex_step(C.byref(self.g), int(move)) != 0:
            raise AssertionError('illegal move')

    def copy(self):
        h = Hex.__new__(Hex)
        h.g = OHex()
        C.memmove(C.byref(h.g), C.byref(self.g), C.sizeof(OHex))
        return h


def neighbors(tile, n):
    out = np.zeros(6, dtype=np.int32)
    k = lib().ohex_neighbors(int(tile), int(n), _i32(out))
    return out[:k].copy()


def check_win(board, tile):
    b = np.ascontiguousarray(board, dtype=np.int32)
    return lib().ohex_check_win(_i32(b), b.shape[0], int(tile))


def flip_board(board):
    b = np.ascontiguousarray(board, dtype=np.int32)
    out = np.zeros_like(b)
    lib().ohex_flip_board(_i32(b), b.shape[0], _i32(out))
    return out


def flip_moves(moves, n):
    m = np.ascontiguousarray(moves, dtype=np.int32)
    out = np.zeros_like(m)
    lib().ohex_flip_moves(_i32(m), len(m), int(n), _i32(out))
    return out


def stub_eval(mode, board_view, moves_view):
    b = np.ascontiguousarray(board_view, dtype=np.int32)
    m = np.ascontiguousarray(moves_view, dtype=np.int32)
    value = C.c_float()
    prior = np.zeros(max(len(m), 1), dtype=np.float32)
    lib().ostub_eval(int(mode), _i32(b), b.shape[0], _i32(m), len(m),
                     C.byref(value), _f32(prior))
    return np.float32(value.value), prior[:len(m)]


def board_hash(board_view):
    b = np.ascontiguousarray(board_view, dtype=np.int32)
    return int(lib().ostub_board_hash(_i32(b), b.shape[0]))


def score_actions(num_visits, neg_total_value, prior, coef):
    nv = np.ascontiguousarray(num_visits, dtype=np.float32)
    tv = np.ascontiguousarray(neg_total_value, dtype=np.float32)
    pr = np.ascontiguousarray(prior, dtype=np.float32)
    out = np.zeros_like(nv)
    lib().omcts_score_actions(_f32(nv), _f32(tv), _f32(pr), len(nv),
                              C.c_float(coef), _f32(out))
    return out


class Tree:
    """SearchTree (search_tree.py:24-132) + mcts.py through the C oracle."""

    def __init__(self, max_nodes=10_000_000):
        self.t = lib().otree_new(max_nodes)
        if not self.t:
            raise MemoryError
        self._lv = OLeaves()

    def __del__(self):
        if getattr(self, 't', None):
            lib().otree_free(self.t)
            self.t = None

    @property
    def num_nodes(self):
        return self.t.contents.num_nodes

    @property
    def root_id(self):
        return self.t.contents.root_id

    def reset(self):
        lib().otree_reset(self.t)

    def move(self, move_id):
        rc = lib().otree_move(self.t, int(move_id))
        if rc < 0:
            raise AssertionError('illegal child')
        return rc

    def root_evaluated(self):
        return self.t.contents.num_children[self.root_id] >= 0

    def root_stats(self):
        """(visits, total_value, prior) of the root's children."""
        v = np.zeros(MAXT, dtype=np.float32)
        w = np.zeros(MAXT, dtype=np.float32)
        p = np.zeros(MAXT, dtype=np.float32)
        k = lib().otree_root_stats(self.t, _f32(v), _f32(w), _f32(p))
        if k < 0:
            raise AssertionError('unevaluated root')
        return v[:k].copy(), w[:k].copy(), p[:k].copy()

    def root_node(self):
        t = self.t.contents
        return float(t.num_visits[t.root_id]), float(t.total_value[t.root_id])

    def sample_paths_stub(self, game, num_simulations, batch_size, coef,
                          stub_mode):
        sv = C.c_float()
        rc = lib().omcts_sample_paths_stub(self.t, C.byref(game.g),
                                           num_simulations, batch_size,
                                           C.c_float(coef), stub_mode,
                                           C.byref(sv))
        if rc == -1:
            raise SearchTreeFull('too many nodes')
        if rc < 0:
            raise AssertionError('oracle search failed: %d' % rc)
        return float(sv.value)

    # split interface: select -> (external evaluator) -> expand/backup
    def _leaves(self, n):
        lv = self._lv
        out = []
        for i in range(lv.count):
            k = lv.num_moves[i]
            out.append(dict(
                node=lv.node[i], color=lv.color[i], result=lv.result[i],
                board=np.array(lv.board_view[i][:n * n],
                               dtype=np.int32).reshape(n, n),
                legal_moves=np.array(lv.moves_view[i][:k], dtype=np.int32)))
        return out

    def select_batch(self, game, batch_size, coef):
        rc = lib().omcts_select_batch(self.t, C.byref(game.g), batch_size,
                                      C.c_float(coef), C.byref(self._lv))
        if rc < 0:
            raise AssertionError('oracle select failed: %d' % rc)
        return self._leaves(game.n)

    def expand_backup(self, value, prior):
        value = np.ascontiguousarray(value, dtype=np.float32)
        prior = np.ascontiguousarray(prior, dtype=np.float32)
        stride = prior.shape[1] if prior.ndim == 2 else 0
        sv = C.c_float()
        rc = lib().omcts_expand_backup(self.t, C.byref(self._lv), _f32(value),
                                       _f32(prior), stride, C.byref(sv))
        if rc == -1:
            raise SearchTreeFull('too many nodes')
        if rc < 0:
            raise AssertionError('oracle expand failed: %d' % rc)
        return float(sv.value)

    def root_leaf(self, game):
        lib().omcts_root_leaf(self.t, C.byref(game.g), C.byref(self._lv))
        return self._leaves(game.n)

    def expand_root(self, prior):
        prior = np.ascontiguousarray(prior, dtype=np.float32)
        if lib().omcts_expand_root(self.t, C.byref(self._lv), _f32(prior)):
            raise SearchTreeFull('too many nodes')


def bench_selfplay_stub(n=11, num_games=8, threads=1, num_simulations=800,
                        batch_size=10, coef=0.5, stub_mode=0,
                        exploration_depth=15, max_nodes=10_000_000, seed=0):
    """Time whole stub-evaluator self-play games on host threads."""
    sims = C.c_int64()
    secs = C.c_double()
    sc, sd, ul = C.c_int64(), C.c_int64(), C.c_int64()
    plies = lib().obench_selfplay_stub(
        n, num_games, threads, num_simulations, batch_size, C.c_float(coef),
        stub_mode, exploration_depth, max_nodes, seed, C.byref(sims),
        C.byref(secs), C.byref(sc), C.byref(sd), C.byref(ul))
    return dict(plies=int(plies), simulations=sims.value, seconds=secs.value,
                sum_children=sc.value, sum_depth=sd.value,
                unique_leaves=ul.value)
