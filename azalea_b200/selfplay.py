"""Lockstep self-play: thousands of games advance one move at a time on one
GPU, sharded by game index across GPUs.

Replaces the reference's process-per-game data parallelism
(azalea/parallel_player.py:17-76, azalea/process_pool.py:15-47,
azalea/play_game.py:18-78) for the self-play path.  One ``step_move()`` is
what ``AzaleaAgent.choose_action`` + ``execute_action`` do for one game
(azalea_agent.py:54-64), done for every resident game:

    select_root -> evaluate -> expand_root          (mcts.evaluate_root)
    num_batches x [ select -> evaluate -> expand_backup ]   (mcts.sample_paths)
    play_commit                                      (policy.py:160-176, play_game.py:46-67)

Everything between two host calls stays on the device; with
``cuda_graph=True`` the whole move is one CUDA graph launch.  Games are
independent: rank r of W owns global games [r*G, (r+1)*G), each game's
Philox stream is keyed by its global id, so results do not depend on the
world size.  The only exchange is the replay gather to rank 0.
"""

import numpy as np
import torch

from . import _cabi
from .engine import Engine, decode_replay_rows
from .replay_buffer import ReplayDataFrame
from .search_tree import as_distribution
from .typing import GameState


def default_nodes_per_game(num_games, num_tiles, sims_per_move, device=None,
                           keep_factor=4, memory_fraction=0.45):
    """Capacity of each half of a game's node pool.

    One move grows a tree by at most ``growth = (sims_per_move + 1) * n*n``
    nodes (the reference materialises every child of an expanded leaf,
    search_tree.py:254-274).  Re-rooting copies the kept subtree into the
    other half, so the steady-state size is ``growth / (1 - f)`` with ``f``
    the chosen child's share of the tree: ``keep_factor`` = 4 covers shares
    up to 0.75, which peaked searches of a trained network reach at
    temperature 0.  Capped so that all pools together use at most
    ``memory_fraction`` of the device's free memory, and by the 23-bit node id.
    """
    growth = (sims_per_move + 1) * num_tiles
    want = keep_factor * growth
    try:
        free, _ = torch.cuda.mem_get_info(device)
        cap = int(memory_fraction * free) // (num_games * 2 * 16)
        want = min(want, max(cap, growth + num_tiles + 1))
    except Exception:
        pass
    return int(min(want, (1 << 23) - 1))


class StubEvaluator:
    """Deterministic device stub (test / bench aid; modes as in
    oracle/azalea_oracle.h): 0 uniform, 1 dyadic, 2 rough."""

    def __init__(self, mode=0):
        self.mode = int(mode)


class LockstepSelfPlay:
    def __init__(self, evaluator, *, num_games=4096, board_size=11,
                 simulations=800, search_batch_size=10, exploration_coef=0.5,
                 exploration_depth=15, exploration_noise_alpha=0.03,
                 exploration_noise_scale=0.25, exploration_temperature=1.0,
                 move_sampling=True, move_exploration=True, seed=0,
                 device=None, rank=0, world_size=1, nodes_per_game=None,
                 replay_rows=None, collect_replay=True, cuda_graph=True,
                 max_plies=300, random_play=False, streams=None, pack_leaves=None,
                 random_reflect=False):
        # random_play: RandomPolicy self-play (random_policy.py:25-41) -- no
        # search, uniform move choice and uniform moves_prob at every ply;
        # how the reference fills the replay buffer before training
        # (policy_trainer.py:145-158)
        self.random_play = bool(random_play)
        if self.random_play:
            evaluator = StubEvaluator(0)
            simulations, exploration_depth = 0, 1 << 30
            exploration_temperature, move_sampling = 1.0, True
        self.evaluator = evaluator
        self.G = int(num_games)
        self.n = int(board_size)
        self.nn = self.n * self.n
        self.batch = int(search_batch_size)
        # mcts.py:268: num_batches = sims // batch + 1
        self.num_batches = int(simulations) // self.batch + 1
        self.sims_per_move = self.num_batches * self.batch
        self.coef = float(exploration_coef)
        self.depth = int(exploration_depth)
        self.temperature = float(exploration_temperature)
        self.move_sampling = bool(move_sampling)
        # policy.py:142-147: noise only when sampling and exploring
        self.noise_scale = float(exploration_noise_scale) \
            if (move_sampling and move_exploration) else 0.0
        self.noise_alpha = float(exploration_noise_alpha)
        self.collect_replay = bool(collect_replay)
        if replay_rows is None:
            replay_rows = 2 * self.G * min(self.nn, max_plies) if collect_replay else 0
        if nodes_per_game is None:
            nodes_per_game = default_nodes_per_game(
                self.G, self.nn, self.sims_per_move, device)
        # a full pool half never kills a game here: the expansion is skipped and
        # counted (AZ_CFG_SOFT_POOL_FULL); see counters()['pool_skipped_expansions']
        # packed leaves (AZ_CFG_PACK_LEAVES): with a network in the loop the select kernel
        # writes only the leaves that need it (unique, not terminal; mcts.py:75,192-200) as
        # consecutive rows, and the evaluator works on that many -- default whenever the
        # evaluator can take a device-side row count
        self.is_stub = isinstance(evaluator, StubEvaluator)
        if pack_leaves is None:
            pack_leaves = not self.is_stub and hasattr(evaluator, 'evaluate_cells')
        self.pack_leaves = bool(pack_leaves) and not self.is_stub
        self.eng = Engine(self.G, self.n, max_batch=self.batch,
                          nodes_per_game=nodes_per_game,
                          replay_rows=replay_rows, max_plies=max_plies,
                          seed=seed, first_game_id=rank * self.G,
                          game_id_stride=world_size * self.G, device=device,
                          soft_pool_full=True, pack_leaves=self.pack_leaves)
        # random_reflect: every leaf the network evaluates is shown in a random one of
        # Hex's two rule-preserving orientations (az_engine_set_reflect); part of the
        # captured graph, so it is fixed for the life of this object
        self.random_reflect = bool(random_reflect) and not self.random_play
        if self.random_reflect:
            self.eng.set_reflect(True)
        self.device = self.eng.device
        self.chosen = torch.zeros(self.G, 4, dtype=torch.int32,
                                  device=self.device)
        if not self.is_stub:
            if getattr(evaluator, '_fast', None) is None:
                evaluator.eval()
                evaluator.to(self.device)
                evaluator.prepare_inference()
            torch.backends.cudnn.benchmark = True
        # streams > 1: the games are split into that many windows driven on separate streams,
        # so the tree kernels of one window run under the evaluator of another
        # (az_engine_set_window); results do not depend on it (tested bit for bit).  With a
        # network in the loop two windows are 6 % faster than one (DESIGN.md 5) and the
        # default; the stub evaluator has nothing to overlap with.
        if streams is None:
            streams = 1 if (self.is_stub or self.G < 64) else 2
        self.streams = max(1, min(int(streams), self.G))
        self._side = [torch.cuda.Stream(device=self.device) for _ in range(self.streams - 1)]
        self.moves_done = 0
        self._graph = None
        self._want_graph = bool(cuda_graph)
        # kernels of ours launched per move (for bench.py's gpu_launches)
        self.launches_per_move = 3 + self.num_batches * (3 if self.is_stub else 2) \
            + (1 if self.is_stub else 0)

    # ------------------------------------------------------------ one move --
    def _evaluate(self, root, g0=0, g1=None):
        """Leaves of games [g0, g1) -> (value, prior/logits, kind)."""
        eng = self.eng
        g1 = self.G if g1 is None else g1
        if self.is_stub:
            eng.stub_eval(self.evaluator.mode)
            return None, None, _cabi.AZ_PRIOR_PROBS
        # the evaluator's tail kernel writes fp32 value / logits straight into the
        # engine's own value / prior rows of this window: nothing to copy, and
        # expand_backup(None, None) reads them in place
        if root:
            # leaf slot 0 of every game; the root's value is discarded (mcts.py:25-26)
            self.evaluator.evaluate_cells(
                eng.leaf_board[g0:g1, 0], logits_out=eng.prior[g0:g1, 0],
                logits_stride=eng.max_batch * eng.nn, want_value=False)
            return None, None, _cabi.AZ_PRIOR_LOGITS
        cells = eng.leaf_board[g0:g1].view((g1 - g0) * eng.max_batch, eng.cell_stride)
        kw = {'live_rows': eng.leaf_rows[g0:g0 + 1]} if self.pack_leaves else {}
        self.evaluator.evaluate_cells(
            cells, value_out=eng.value[g0:g1].view(-1),
            logits_out=eng.prior[g0:g1].view(-1, eng.nn), logits_stride=eng.nn, **kw)
        return None, None, _cabi.AZ_PRIOR_LOGITS

    def _window_body(self, g0, g1):
        """One move of games [g0, g1) on the current stream (the engine's
        window must be set to it)."""
        eng = self.eng
        eng.select_root()
        _, _, kind = self._evaluate(True, g0, g1)
        eng.expand_root(None, kind)
        if self.random_play:
            eng.root_uniform()
        for _ in range(0 if self.random_play else self.num_batches):
            eng.select(self.batch, self.coef, self.noise_scale,
                       self.noise_alpha)
            value, prior, kind = self._evaluate(False, g0, g1)
            eng.expand_backup(value, prior, kind)
            # keep evaluator outputs alive until the kernel that reads them
            # has been enqueued (same stream: safe to drop afterwards)
        eng.play_commit(self.temperature, self.depth, self.move_sampling,
                        self.collect_replay, True, self.chosen)

    def _move_body(self):
        if self.streams == 1:
            return self._window_body(0, self.G)
        eng = self.eng
        main = torch.cuda.current_stream(self.device)
        bounds = [self.G * i // self.streams for i in range(self.streams + 1)]
        fork = torch.cuda.Event()
        fork.record(main)
        joins = []
        try:
            for i in range(1, self.streams):
                side = self._side[i - 1]
                side.wait_event(fork)
                with torch.cuda.stream(side):
                    eng.set_window(bounds[i], bounds[i + 1] - bounds[i])
                    self._window_body(bounds[i], bounds[i + 1])
                    done = torch.cuda.Event()
                    done.record(side)
                    joins.append(done)
            eng.set_window(bounds[0], bounds[1] - bounds[0])
            self._window_body(bounds[0], bounds[1])
        finally:
            eng.set_window(0, 0)        # the window is engine state: never leave it narrowed
            for done in joins:
                main.wait_event(done)

    def preroll(self, max_plies):
        """Stagger the games: slot g is advanced by ``g * max_plies // G``
        uniformly random plies (RandomPolicy moves, random_policy.py:25-41;
        recorded as such in the replay rows), so that a lockstep run no longer
        has every game at the same ply -- games end, restart, and reuse
        subtrees at different times, as in steady-state self-play.  Eager;
        call it before the move graph is captured or between replays."""
        eng, G = self.eng, self.G
        max_plies = int(max_plies)
        try:
            for s in range(1, max_plies + 1):
                g0 = -(-s * G // max_plies)         # slots with quota >= s
                if g0 >= G:
                    break
                eng.set_window(g0, G - g0)
                eng.select_root()
                eng.stub_eval(0)
                eng.expand_root()
                eng.root_uniform()
                eng.play_commit(1.0, 1 << 30, True, self.collect_replay, True,
                                self.chosen)
        finally:
            eng.set_window(0, 0)

    def capture(self):
        """Capture one move as a CUDA graph (capturing does not execute)."""
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._move_body()
        self._graph = graph

    def step_move(self):
        """One move of every game (enqueue only; no host sync).  The first
        two moves run eagerly (cuDNN autotune, allocator warm-up), the third
        call captures the move as a CUDA graph, later calls replay it."""
        if self._want_graph and self._graph is None and self.moves_done >= 2:
            self.capture()
        if self._graph is not None:
            self._graph.replay()
        else:
            self._move_body()
        self.moves_done += 1

    # -------------------------------------------------------------- output --
    def harvest(self, gather=False):
        """Finished games' replay rows (host, raw uint8 [R, row_bytes]).

        With ``gather=True`` under torch.distributed, every rank's rows are
        gathered to rank 0 over NCCL (the path's only exchange, SURVEY 8e):
        rank 0 returns all rows, the other ranks an empty array."""
        if not gather:
            return self.eng.harvest_replay()
        import torch.distributed as dist
        eng = self.eng
        count = min(eng.replay_count(), eng.replay.shape[0])
        rows = gather_replay_rows(eng.replay[:count])
        eng.replay_clear()
        if rows is None or (dist.is_initialized() and dist.get_rank() != 0):
            return np.zeros((0, eng.row_bytes), dtype=np.uint8)
        rows = rows.cpu().numpy()
        if len(rows):
            key = rows[:, :12].copy().view([('g', '<i8'), ('p', '<i4')]).reshape(-1)
            rows = rows[np.argsort(key, order=('g', 'p'), kind='stable')]
        return rows

    def harvest_begin(self, gather=False):
        """Pipelined harvest, first half: sync on the row count(s), enqueue
        the exchange (``gather=True``: every rank's rows to rank 0 over NCCL),
        the copy to pinned memory and the clear.  Enqueue the next
        ``step_move()`` before calling ``harvest_end``, so the host's share of
        the harvest runs under that move."""
        if not gather:
            return self.eng.harvest_begin()
        import torch.distributed as dist
        eng = self.eng
        count = min(eng.replay_count(), eng.replay.shape[0])
        rows = gather_replay_rows(eng.replay[:count])
        eng.replay_clear()
        if rows is None or (dist.is_initialized() and dist.get_rank() != 0):
            return ('sync', np.zeros((0, eng.row_bytes), dtype=np.uint8))
        n = rows.shape[0]
        pinned = getattr(self, '_pinned_gather', None)
        if pinned is None or pinned.shape[0] < n:
            # (a first call may find everything the warm-up left behind: grow by a quarter, not by two)
            pinned = torch.empty(max(n + n // 4, 1 << 15), eng.row_bytes, dtype=torch.uint8).pin_memory()
            self._pinned_gather = pinned
        pinned[:n].copy_(rows, non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(self.device))
        return ('gathered', n, done, rows)      # (rows: kept alive until the copy has run)

    def harvest_end(self, handle):
        if handle[0] == 'gathered':
            _, n, done, _ = handle
            done.synchronize()
            return Engine._sort_rows(self._pinned_gather[:n].numpy().copy())
        return self.eng.harvest_end(handle)

    def counters(self):
        return self.eng.counter_totals()


def rows_to_dataframe(rows, board_size) -> ReplayDataFrame:
    """Raw replay rows -> the reference's ``ReplayDataFrame``
    (replay_buffer.py:25-104, play_game.py:63-67,90-96): state before the
    move, pi = as_distribution(visits, temperature) as float32, reward."""
    h, boards, visits = decode_replay_rows(rows, board_size)
    df = ReplayDataFrame()
    for i in range(len(h)):
        board = boards[i].astype(np.int32)
        legal = np.flatnonzero(board.ravel() == 0).astype(np.int32) + 1
        k = int(h['num_moves'][i])
        assert k == len(legal)
        df.state.append(GameState(int(h['color'][i]), legal, 0, board))
        df.moves_prob.append(
            as_distribution(visits[i, :k], float(h['temperature'][i]))
            .astype(np.float32))
        df.reward.append(np.float32(h['reward'][i]))
    return df


def gather_replay_rows(rows: torch.Tensor, dst: int = 0, group=None):
    """The path's only exchange: variable-length row blocks to rank ``dst``
    (NCCL on device tensors, gloo on host tensors).  Returns the
    concatenated rows on ``dst`` and None elsewhere."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized():
        return rows
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    count = torch.tensor([rows.shape[0]], dtype=torch.int64, device=rows.device)
    counts = [torch.zeros_like(count) for _ in range(world)]
    dist.all_gather(counts, count, group=group)
    counts = [int(c.item()) for c in counts]
    cap = max(max(counts), 1)
    padded = torch.zeros(cap, rows.shape[1], dtype=rows.dtype,
                         device=rows.device)
    padded[:rows.shape[0]] = rows
    bufs = [torch.zeros_like(padded) for _ in range(world)] \
        if rank == dst else None
    dist.gather(padded, bufs, dst=dst, group=group)
    if rank != dst:
        return None
    return torch.cat([b[:c] for b, c in zip(bufs, counts)])
