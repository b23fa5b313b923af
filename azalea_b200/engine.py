"""Device engine: G games (boards + search trees) resident in HBM.

Thin host wrapper over the C ABI (include/azalea_b200.h).  PyTorch is used
for what it is good at here -- device memory, streams -- and nothing else:
the engine's memory is one ``torch.uint8`` block, the buffers the caller
touches are views into it, and every op enqueues sm_100a kernels on torch's
current CUDA stream without synchronising.
"""
import ctypes as C

import numpy as np
import torch

from . import _cabi
from ._cabi import (AZ_BUF_COUNTERS, AZ_BUF_GLOBALS, AZ_BUF_LEAF_BOARD, AZ_BUF_LEAF_INFO,
                    AZ_BUF_LEAF_MOVES, AZ_BUF_META, AZ_BUF_PRIOR,
                    AZ_BUF_REPLAY, AZ_BUF_VALUE,
                    AZ_PRIOR_PROBS, COUNTER_NAMES, check)

_DTYPES = {1: torch.int8, 4: torch.int32, 8: torch.int64}


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class Engine:
    """G Hex games and their MCTS trees on one GPU.

    :param num_games: games resident on this GPU (one warp each)
    :param board_size: n (2..19)
    :param max_batch: upper bound for search_batch_size (<= 32)
    :param nodes_per_game: capacity of each half of a game's node pool
    :param max_nodes_ref: the reference's ``search_tree.MAX_NODES``; a tree
        whose reference node count would exceed it is flagged
        ``AZ_ST_TREE_FULL`` (raised as ``SearchTreeFull`` by the front ends)
    :param soft_pool_full: when a game's pool half is exhausted, skip the
        expansion (counted in ``pool_skipped_expansions``) instead of
        flagging ``AZ_ST_POOL_FULL``
    """

    def __init__(self, num_games, board_size=11, max_batch=10,
                 nodes_per_game=None, max_nodes_ref=10_000_000, replay_rows=0,
                 max_plies=300, seed=0, first_game_id=0, game_id_stride=0,
                 device=None, soft_pool_full=False, pack_leaves=False):
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError('azalea_b200.Engine needs a CUDA device '
                               '(there is no CPU fallback)')
        self.lib = _cabi.lib()
        self.device = device
        self.num_games = int(num_games)
        self.n = int(board_size)
        self.nn = self.n * self.n
        self.max_batch = int(max_batch)
        if nodes_per_game is None:
            nodes_per_game = 2 * 811 * self.nn
        nodes_per_game = int(min(nodes_per_game, (1 << 23) - 1))
        self.nodes_per_game = nodes_per_game
        self.cfg = _cabi.AzConfig(
            num_games=self.num_games, board_size=self.n,
            max_batch=self.max_batch, nodes_per_game=nodes_per_game,
            max_nodes_ref=int(max_nodes_ref), replay_rows=int(replay_rows),
            max_plies=int(max_plies), seed=int(seed) & (2 ** 64 - 1),
            first_game_id=int(first_game_id),
            game_id_stride=int(game_id_stride),
            flags=(_cabi.AZ_CFG_SOFT_POOL_FULL if soft_pool_full else 0)
            | (_cabi.AZ_CFG_PACK_LEAVES if pack_leaves else 0))
        self.pack_leaves = bool(pack_leaves)
        nbytes = self.lib.az_engine_device_bytes(C.byref(self.cfg))
        if nbytes == 0:
            raise ValueError('invalid engine configuration')
        self.mem = torch.empty(nbytes, dtype=torch.uint8, device=device)
        self._h = C.c_void_p()
        with torch.cuda.device(device):
            torch.cuda.synchronize()
            check(self.lib.az_engine_create(
                C.byref(self._h), C.byref(self.cfg), _ptr(self.mem), nbytes,
                device.index or 0))
        self.row_bytes = self.lib.az_replay_row_bytes(self._h)
        self.leaf_board = self._view(AZ_BUF_LEAF_BOARD)
        self.leaf_info = self._view(AZ_BUF_LEAF_INFO)
        self.value = self._view(AZ_BUF_VALUE, torch.float32)
        self.prior = self._view(AZ_BUF_PRIOR, torch.float32)
        self.meta = self._view(AZ_BUF_META)
        self.counters = self._view(AZ_BUF_COUNTERS)
        self.leaf_moves = self._view(AZ_BUF_LEAF_MOVES)
        self.globals = self._view(AZ_BUF_GLOBALS)
        # AZ_CFG_PACK_LEAVES: [g0] = live leaf rows of the window that starts at game g0
        self.leaf_rows = self._view(_cabi.AZ_BUF_LEAF_ROWS)
        # per-slot resignation state and counts (az_engine_set_resign)
        self.resign = self._view(_cabi.AZ_BUF_RESIGN)
        self.replay = self._view(AZ_BUF_REPLAY, torch.uint8) \
            if replay_rows else None
        self.cell_stride = self.leaf_board.shape[-1]
        self._spans = {}
        self.reflect = False

    def span(self, first, last):
        """One contiguous uint8 view of the device block covering the buffers
        from ``first`` to ``last`` (AZ_BUF_* ids, ``first`` before ``last`` in the
        block) with everything between them, and each one's byte offset inside it: lets a host front end move
        several small buffers with ONE copy."""
        key = (first, last)
        if key not in self._spans:
            descs = {}
            for which in range(_cabi.AZ_BUF_GLOBALS + 1):
                d = _cabi.AzBufferDesc()
                check(self.lib.az_engine_buffer(self._h, which, C.byref(d)))
                descs[which] = (d.offset, d.bytes)
            lo, hi = descs[first][0], descs[last][0] + descs[last][1]
            assert lo < hi
            inside = {w: (o - lo, b) for w, (o, b) in descs.items() if lo <= o and o + b <= hi}
            self._spans[key] = (self.mem[lo:hi], inside)
        return self._spans[key]

    def __del__(self):
        h = getattr(self, '_h', None)
        if h:
            self.lib.az_engine_destroy(h)
            self._h = None

    def _view(self, which, dtype=None):
        d = _cabi.AzBufferDesc()
        check(self.lib.az_engine_buffer(self._h, which, C.byref(d)))
        dtype = dtype or _DTYPES[d.elem_bytes]
        flat = self.mem[d.offset:d.offset + d.bytes].view(dtype)
        return flat.view(*[d.shape[i] for i in range(d.ndim)])

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _new(self, *shape, dtype=torch.int32):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    # ------------------------------------------------------------- games --
    def reset(self, mask=None):
        """HexGame.reset + Policy.reset for masked games (all if None)."""
        if mask is not None:
            mask = mask.to(self.device, torch.uint8).contiguous()
        check(self.lib.az_games_reset(self._h, _ptr(mask), self._stream))

    def hex_step(self, moves):
        """HexGameImpl.step (hex.py:172-179); moves 1-based, 0 = skip."""
        moves = torch.as_tensor(moves, dtype=torch.int32).to(self.device).contiguous()
        results = self._new(self.num_games)
        check(self.lib.az_hex_step(self._h, _ptr(moves), _ptr(results),
                                   self._stream))
        return results

    def hex_state(self):
        """HexGame.state (hex.py:55-60): board int8[G,n,n], color, result, ply."""
        board = self._new(self.num_games, self.n, self.n, dtype=torch.int8)
        color, result, ply = (self._new(self.num_games) for _ in range(3))
        check(self.lib.az_hex_state(self._h, _ptr(board), _ptr(color),
                                    _ptr(result), _ptr(ply), self._stream))
        return board, color, result, ply

    def hex_legal_moves(self):
        """HexGameImpl.legal_moves (hex.py:151-159): int32[G,n*n] 0-padded."""
        moves = self._new(self.num_games, self.nn)
        count = self._new(self.num_games)
        check(self.lib.az_hex_legal_moves(self._h, _ptr(moves), _ptr(count),
                                          self._stream))
        return moves, count

    def hex_set_state(self, board, color, last_tile=None, reset_trees=True):
        board = torch.as_tensor(board).to(self.device, torch.int8).contiguous()
        color = torch.as_tensor(color).to(self.device, torch.int32).contiguous()
        if last_tile is not None:
            last_tile = torch.as_tensor(last_tile).to(
                self.device, torch.int32).contiguous()
        check(self.lib.az_hex_set_state(self._h, _ptr(board), _ptr(color),
                                        _ptr(last_tile), int(reset_trees),
                                        self._stream))

    # ------------------------------------------------------------ search --
    def select_root(self):
        check(self.lib.az_mcts_select_root(self._h, self._stream))

    def select(self, batch_size, exploration_coef, noise_scale=0.0,
               noise_alpha=1.0):
        p = _cabi.AzSearchParams(int(batch_size), float(exploration_coef),
                                 float(noise_scale), float(noise_alpha))
        check(self.lib.az_mcts_select(self._h, C.byref(p), self._stream))

    def compute_leaf_moves(self):
        check(self.lib.az_leaf_moves(self._h, self._stream))
        return self.leaf_moves

    def expand_backup(self, value=None, prior=None, prior_kind=AZ_PRIOR_PROBS):
        check(self.lib.az_mcts_expand_backup(self._h, _ptr(value), _ptr(prior),
                                             prior_kind, self._stream))

    def expand_root(self, prior=None, prior_kind=AZ_PRIOR_PROBS):
        check(self.lib.az_mcts_expand_root(self._h, _ptr(prior), prior_kind,
                                           self._stream))

    def root_stats(self):
        """visits, total_value, prior f32[G,n*n]; k int32[G]; root (N,W)
        f32[G,2]; reference node count int64[G]."""
        G, nn = self.num_games, self.nn
        visits = self._new(G, nn, dtype=torch.float32)
        total = self._new(G, nn, dtype=torch.float32)
        prior = self._new(G, nn, dtype=torch.float32)
        k = self._new(G)
        root_nw = self._new(G, 2, dtype=torch.float32)
        num_nodes = self._new(G, dtype=torch.int64)
        check(self.lib.az_root_stats(self._h, _ptr(visits), _ptr(total),
                                     _ptr(prior), _ptr(k), _ptr(root_nw),
                                     _ptr(num_nodes), self._stream))
        return visits, total, prior, k, root_nw, num_nodes

    def set_window(self, first_game=0, num_games=0):
        """Restrict the per-game kernels to games [first, first + num)
        (0, 0: all games).  Read at launch time: see az_engine_set_window."""
        check(self.lib.az_engine_set_window(self._h, int(first_game), int(num_games)))
        self.window = (int(first_game), int(num_games) or self.num_games)

    def set_reflect(self, on=True):
        """Random orientation of the network rows (az_engine_set_reflect):
        each leaf that goes to the evaluator is written rotated by 180 degrees
        with probability 1/2, and the logits of such a row are read back
        rotated.  Read at launch time: set it before capturing a graph."""
        check(self.lib.az_engine_set_reflect(self._h, int(bool(on))))
        self.reflect = bool(on)

    def set_playout_cap(self, full_search_prob=1.0, fast_descents=0):
        """Playout cap randomization (az_engine_set_playout_cap): each ply of
        each game is a full search with probability ``full_search_prob``
        (one coin per game id and ply); otherwise ``select`` stops after
        ``fast_descents`` new descents this move, with no root noise, and the
        ply's replay row is not flushed.  ``full_search_prob >= 1`` is off.
        Every move must begin with ``select_root``.  Read at launch time: set
        it before capturing a graph."""
        check(self.lib.az_engine_set_playout_cap(self._h, float(full_search_prob),
                                                 int(fast_descents)))

    def set_resign(self, threshold=None, disable_prob=0.1):
        """Resignation with calibration games (az_engine_set_resign): after
        the search, the player to move resigns when r = max(Q_root, Q_best)
        is below ``threshold``, except in calibration games (probability
        ``disable_prob``, one coin per game id), which never resign and
        record how often the eventual winner's value fell below it
        (``resign_stats``).  ``threshold=None`` (or <= -1) is off;
        ``disable_prob=1`` only measures.  Read at launch time: set it before
        capturing a graph."""
        t = -1.0 if threshold is None else float(threshold)
        check(self.lib.az_engine_set_resign(self._h, t, float(disable_prob)))

    def set_forced_playouts(self, k=0.0, exploration_coef=0.5):
        """Forced playouts and policy target pruning (Wu 2019, section 3.2;
        az_engine_set_forced_playouts): on full plies a visited root child
        with fewer than sqrt(k * P * sum N) visits is descended into first,
        and the replay row's visits are pruned back to what PUCT with
        ``exploration_coef`` would have given; the move is still drawn from
        the raw visits.  ``k=0`` is off.  Read at launch time: set it before
        capturing a graph."""
        check(self.lib.az_engine_set_forced_playouts(self._h, float(k), float(exploration_coef)))

    def resign_stats(self):
        """Resignation counts summed over the slots (one D2H copy):
        ``resigned_games``, ``calibration_games`` (calibration games that
        ended with a winner), ``false_positives`` (those whose winner's lowest
        r was below the threshold) and ``histogram`` (int64[65], the winner's
        lowest r: bin i < 64 holds [-1 + i/64, -1 + (i+1)/64), bin 64 r >= 0)."""
        tot = self.resign.to(torch.int64).sum(0).cpu().numpy()
        return dict(resigned_games=int(tot[_cabi.AZ_RS_RESIGNED]),
                    calibration_games=int(tot[_cabi.AZ_RS_CALIB]),
                    false_positives=int(tot[_cabi.AZ_RS_FALSE_POS]),
                    histogram=tot[_cabi.AZ_RS_HIST:_cabi.AZ_RS_HIST + _cabi.AZ_RS_BINS].copy())

    def root_uniform(self):
        """One visit on every child of every expanded root: the RandomPolicy
        seat (random_policy.py:25-41) in terms of the tree."""
        check(self.lib.az_mcts_root_uniform(self._h, self._stream))

    def tree_move(self, move_ids):
        """SearchTree.move (search_tree.py:115-132); -1 = skip."""
        move_ids = torch.as_tensor(move_ids, dtype=torch.int32).to(
            self.device).contiguous()
        check(self.lib.az_tree_move(self._h, _ptr(move_ids), self._stream))

    def status(self):
        st = self._new(self.num_games)
        check(self.lib.az_status(self._h, _ptr(st), self._stream))
        return st

    def stub_eval(self, mode):
        """Device stub evaluator (test/bench aid) -> engine value/prior."""
        check(self.lib.az_stub_eval(self._h, int(mode), self._stream))

    def noise_sample(self, alpha, k, sim=0):
        """Test aid: the Dirichlet(alpha) root-noise vector each game would
        draw for simulation `sim` of its current ply, f32[G, k]."""
        out = self._new(self.num_games, k, dtype=torch.float32)
        check(self.lib.az_noise_sample(self._h, float(alpha), int(k), int(sim),
                                       _ptr(out), self._stream))
        return out

    # ------------------------------------------------------ lockstep play --
    def play_commit(self, temperature=1.0, exploration_depth=15,
                    move_sampling=True, collect_replay=False, auto_reset=True,
                    chosen=None):
        p = _cabi.AzPlayParams(float(temperature), int(exploration_depth),
                               int(move_sampling), int(collect_replay),
                               int(auto_reset))
        check(self.lib.az_play_commit(self._h, C.byref(p), _ptr(chosen),
                                      self._stream))

    def replay_clear(self):
        check(self.lib.az_replay_clear(self._h, self._stream))

    def counter_totals(self):
        """Sum the per-game counters (one D2H copy)."""
        tot = self.counters.sum(0).cpu().numpy()
        return {name: int(tot[i]) for i, name in enumerate(COUNTER_NAMES)}

    def replay_count(self):
        """Rows waiting in the replay buffer (syncs)."""
        return int(self.globals[0].item())

    @staticmethod
    def _sort_rows(rows):
        # finished games append in warp-scheduling order: sort by
        # (game id, ply) so the output is deterministic
        if len(rows):
            key = rows[:, :12].copy().view([('g', '<i8'), ('p', '<i4')]).reshape(-1)
            rows = rows[np.argsort(key, order=('g', 'p'), kind='stable')]
        return rows

    def harvest_begin(self, pinned_bytes=64 << 20):
        """First half of a pipelined harvest: read the row count (the only
        sync), enqueue the rows' copy into pinned host memory and the clear,
        and return a handle.  The caller may enqueue the next move before
        ``harvest_end(handle)`` waits for the copy, so the host's share of the
        harvest runs under that move."""
        if self.replay is None:
            raise RuntimeError('engine was created with replay_rows=0')
        count = min(self.replay_count(), self.replay.shape[0])
        cap = max(1, int(pinned_bytes) // self.row_bytes)
        if count > cap:
            return ('sync', self.harvest_replay())
        if getattr(self, '_pinned_rows', None) is None or self._pinned_rows.shape[0] < cap:
            self._pinned_rows = torch.empty(cap, self.row_bytes, dtype=torch.uint8).pin_memory()
        self._pinned_rows[:count].copy_(self.replay[:count], non_blocking=True)
        self.replay_clear()
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(self.device))
        return ('async', count, done)

    def harvest_end(self, handle):
        """Second half: the rows of ``harvest_begin`` (host, sorted)."""
        if handle[0] == 'sync':
            return handle[1]
        _, count, done = handle
        done.synchronize()
        return self._sort_rows(self._pinned_rows[:count].numpy().copy())

    def harvest_replay(self):
        """Copy the finished games' rows to the host and clear the buffer."""
        if self.replay is None:
            raise RuntimeError('engine was created with replay_rows=0')
        count = min(self.replay_count(), self.replay.shape[0])
        rows = self.replay[:count].cpu().numpy()
        self.replay_clear()
        return self._sort_rows(rows)


def decode_replay_rows(rows, board_size):
    """Split raw replay rows (uint8 [R, row_bytes], host) into arrays.

    Row layout (az_common.cuh: az_row_header, 48 bytes): int64 game_id,
    int32 ply, color, num_moves, f32 reward, int32 result, f32 temperature,
    int32 move, move_id, game_len, reserved; then int8 board[cell_stride]
    (absolute view, before the move), then f32 visits[n*n] by move ordinal.
    With the playout cap on (``Engine.set_playout_cap``) the rows of fast
    plies never reach the output: a game's rows may skip plies, while
    ``game_len`` and ``result`` are still the whole game's and ``reward``
    follows the row's own ply.  A game that ended by resignation
    (``Engine.set_resign``) has no row for its last ply, the one at which
    the mover resigned: its rows are plies ``0 .. game_len - 1``.
    """
    rows = np.ascontiguousarray(rows)
    n, nn = board_size, board_size * board_size
    cs = (nn + 15) & ~15
    hb = ROW_HEADER.itemsize
    h = rows[:, :hb].copy().view(ROW_HEADER).reshape(-1)
    board = rows[:, hb:hb + nn].copy().view(np.int8).reshape(-1, n, n)
    visits = rows[:, hb + cs:hb + cs + 4 * nn].copy().view('<f4').reshape(-1, nn)
    return h, board, visits


ROW_HEADER = np.dtype([('game_id', '<i8'), ('ply', '<i4'), ('color', '<i4'),
                       ('num_moves', '<i4'), ('reward', '<f4'),
                       ('result', '<i4'), ('temperature', '<f4'),
                       ('move', '<i4'), ('move_id', '<i4'),
                       ('game_len', '<i4'), ('reserved', '<i4')])


def replay_row_bytes(board_size):
    nn = board_size * board_size
    return (ROW_HEADER.itemsize + ((nn + 15) & ~15) + 4 * nn + 15) & ~15
