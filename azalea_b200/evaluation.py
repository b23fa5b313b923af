"""Round-robin tournament on the GPU (the compare / evaluation path).

Same call and result as the reference's ``evaluate(agents, num_rounds,
num_workers)`` (azalea/evaluation.py:17-80): every pair ``(i, j), i < j``
plays ``num_rounds`` games, the first mover of each game is a coin flip from
``RandomState(10000 * round + s)``, and the result is ``{pair: [wins of i,
draws, wins of j]}``.  The reference plays one game per worker process with
two agents, two trees and two networks, and pushes every move into both trees
(azalea/play_game.py:46-54).  Here all of a rank's ``(round, pair)`` games run
in lockstep: one engine holds the first movers' trees, another the second
movers'; at each ply the mover's engine searches, commits, and the move is
replayed into the other engine (``tree_move`` + ``hex_step``).  Leaves are
routed to the network of the policy that owns the tree.

Sharding (SURVEY 8e, the reference's ``parallel_compare`` fans the same tasks
over worker processes, evaluation.py:49-58): task ``t = round * pairs + s``
goes to rank ``t % world``; there is no exchange while the games run, and the
``[pairs, 3]`` tallies are summed onto rank 0 with one ``reduce``.  Every
game's random streams are keyed by its global task index, so the tallies do
not depend on the world size.

Moves are drawn on the device (per-game Philox streams) instead of from each
agent's NumPy ``RandomState``: outcomes are statistically, not bitwise,
comparable with the reference's; the searches themselves are bit-exact
(tests/test_evaluation_gpu.py compares every tree with the oracle's).
``RandomPolicy`` agents move uniformly at random without search
(azalea/random_policy.py:25-41).
"""
from collections import defaultdict
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _cabi
from .engine import Engine
from .random_policy import RandomPolicy
from .selfplay import StubEvaluator, default_nodes_per_game

Pair = Tuple[int, int]
M_STATUS, M_GID_LO, M_GID_HI = 5, 10, 11


def gen_pairs(num_players: int) -> List[Pair]:
    """Round robin pair ordering (evaluation.py:41-46)."""
    return [(i, j) for j in range(num_players) for i in range(j)]


def _policy_key(policy):
    if isinstance(policy, RandomPolicy):
        return ('random',)
    net = policy.net
    kind = ('stub', net.mode) if isinstance(net, StubEvaluator) else ('net',)
    sampling = bool(policy.settings.get('move_sampling', False))
    noise = policy.exploration_noise_scale \
        if (sampling and policy.settings.get('move_exploration', False)) else 0.0
    return (policy.simulations, policy.search_batch_size,
            float(policy.exploration_coef), float(policy.exploration_temperature),
            int(policy.exploration_depth), sampling, float(noise),
            float(policy.exploration_noise_alpha),
            bool(getattr(policy, 'random_reflect', False))) + kind


class _Seat:
    """One engine = the trees of all games' first (or second) movers."""

    def __init__(self, policies, board_size, seed, device, nodes_per_game,
                 game_ids=None):
        self.policies = policies                # policy object per game
        G = len(policies)
        batch = max([p.search_batch_size for p in policies
                     if not isinstance(p, RandomPolicy)] + [1])
        sims = max([p.simulations for p in policies
                    if not isinstance(p, RandomPolicy)] + [1])
        if nodes_per_game is None:
            per_move = (sims // batch + 1) * batch
            nodes_per_game = default_nodes_per_game(G, board_size ** 2, per_move, device)
        self.eng = Engine(G, board_size, max_batch=batch,
                          nodes_per_game=nodes_per_game, seed=seed,
                          device=device, soft_pool_full=True)
        self.device = self.eng.device
        if game_ids is not None:
            # the Philox streams follow the game's global id, not its slot
            ids = torch.as_tensor(np.asarray(game_ids, dtype=np.int64), device=self.device)
            self.eng.meta[:, M_GID_LO] = (ids & 0xffffffff).to(torch.int32)
            self.eng.meta[:, M_GID_HI] = (ids >> 32).to(torch.int32)
        self.chosen = torch.zeros(G, 4, dtype=torch.int32, device=self.device)
        # games grouped by search configuration, then by evaluator object
        self.groups = defaultdict(lambda: defaultdict(list))
        for g, p in enumerate(policies):
            key = _policy_key(p)
            self.groups[key][id(None if key[0] == 'random' else p.net)].append(g)
        self.nets = {id(p.net): p.net for p in policies
                     if not isinstance(p, RandomPolicy)}
        for net in self.nets.values():
            if not isinstance(net, StubEvaluator):
                net.eval()
                net.to(self.device)
                if getattr(net, '_fast', None) is None:
                    net.prepare_inference()
        self.index = {k: {nid: torch.tensor(gs, device=self.device)
                          for nid, gs in by_net.items()}
                      for k, by_net in self.groups.items()}
        # test hook: called as on_search_done(seat, key, games) after a group's
        # search and before its moves are committed
        self.on_search_done: Optional[Callable] = None

    def _pause_all_but(self, games):
        pause = torch.full((self.eng.num_games,), _cabi.AZ_ST_DISABLED,
                           dtype=torch.int32, device=self.device)
        pause[games] = 0
        status = self.eng.meta[:, M_STATUS]
        self.eng.meta[:, M_STATUS] = (status & ~_cabi.AZ_ST_DISABLED) | pause

    def _resume_all(self):
        status = self.eng.meta[:, M_STATUS]
        self.eng.meta[:, M_STATUS] = status & ~_cabi.AZ_ST_DISABLED

    def _evaluate(self, key, by_net, root):
        eng = self.eng
        if key[-2] == 'stub':
            eng.stub_eval(key[-1])
            return _cabi.AZ_PRIOR_PROBS
        B = 1 if root else eng.max_batch
        for nid, idx in by_net.items():
            cells = eng.leaf_board[idx, :B].reshape(-1, eng.cell_stride)
            value, logits = self.nets[nid].evaluate_cells(cells)
            eng.value[idx, :B] = value.view(len(idx), B)
            eng.prior[idx, :B] = logits.view(len(idx), B, eng.nn)
        return _cabi.AZ_PRIOR_LOGITS

    def play_ply(self):
        """Every unfinished game's mover (this seat) searches and moves.
        Returns (move, move_id) int32[G] tensors (0 / -1 for finished games)."""
        eng = self.eng
        self.chosen.zero_()
        self.chosen[:, 1] = -1
        for key, by_net in self.index.items():
            games = torch.cat(list(by_net.values()))
            self._pause_all_but(games)
            # the orientation of this group's network rows (az_engine_set_reflect)
            eng.set_reflect(key[0] != 'random' and key[8])
            if key[0] == 'random':
                # RandomPolicy.choose_action (random_policy.py:25-41) in terms of the
                # tree: one visit on every child of the expanded root, then the
                # temperature-1 draw of play_commit is uniform over the legal moves
                eng.select_root()
                eng.stub_eval(0)
                eng.expand_root()
                eng.root_uniform()
                if self.on_search_done is not None:
                    self.on_search_done(self, key, games)
                eng.play_commit(1.0, 1 << 30, True, False, False, self.chosen)
                continue
            sims, batch, coef, temp, depth, sampling, noise, alpha = key[:8]
            eng.select_root()
            kind = self._evaluate(key, by_net, True)
            eng.expand_root(None, kind)
            for _ in range(sims // batch + 1):
                eng.select(batch, coef, noise, alpha)
                kind = self._evaluate(key, by_net, False)
                eng.expand_backup(None, None, kind)
            if self.on_search_done is not None:
                self.on_search_done(self, key, games)
            eng.play_commit(temp, depth, sampling, False, False, self.chosen)
        self._resume_all()
        return self.chosen[:, 0].clone(), self.chosen[:, 1].clone()

    def apply_opponent(self, moves, move_ids):
        """AzaleaAgent.execute_action for the opponent's move
        (azalea_agent.py:60-64): tree first, then game."""
        self.eng.tree_move(move_ids)
        self.eng.hex_step(moves)


def play_matches(first: List, second: List, board_size: int, seed: int = 0,
                 device=None, nodes_per_game: Optional[int] = None,
                 game_max_length: int = 300, game_ids=None, hook=None,
                 stats: Optional[dict] = None):
    """Play len(first) games in lockstep; game g is first[g] (moves first)
    against second[g].  Returns (results int array: 3 first mover won, 1
    second mover won, 2 draw; move history int32 [plies, G]).

    ``game_ids``: global id of every game (default: its index); a game's
    random streams depend on (seed, id) only, not on which other games share
    the engine.  ``hook``: test aid, see ``_Seat.on_search_done``.
    ``stats``: optional dict that receives ``plies`` and ``simulations``."""
    assert len(first) == len(second)
    G = len(first)
    if G == 0:
        return np.zeros(0, dtype=np.int64), np.zeros((0, 0), dtype=np.int32)
    seats = [_Seat(first, board_size, 2 * seed + 1, device, nodes_per_game, game_ids),
             _Seat(second, board_size, 2 * seed + 2, device, nodes_per_game, game_ids)]
    for s in seats:
        s.on_search_done = hook
    history = []
    result = np.zeros(G, dtype=np.int64)
    for ply in range(min(game_max_length, board_size ** 2)):
        mover, other = seats[ply % 2], seats[1 - ply % 2]
        moves, move_ids = mover.play_ply()
        other.apply_opponent(moves, move_ids)
        history.append(moves.cpu().numpy())
        res = mover.eng.hex_state()[2].cpu().numpy()
        result = res
        bad = (mover.eng.status() | other.eng.status()).cpu().numpy()
        assert not (bad & _cabi.AZ_ST_ILLEGAL).any(), 'inconsistent game state'
        if (res != 0).all():
            break
    if stats is not None:
        tot = [s.eng.counter_totals() for s in seats]
        stats['plies'] = int(sum(int((h != 0).sum()) for h in history))
        stats['simulations'] = sum(t['simulations'] for t in tot)
        stats['pool_skipped_expansions'] = sum(t['pool_skipped_expansions'] for t in tot)
    result = np.where(result == 0, 2, result)       # play_game.py:57-61
    return result, np.stack(history)


def tournament_tasks(num_agents: int, num_rounds: int, rank: int = 0, world: int = 1):
    """This rank's share of the tournament: [(task id, round, pair index,
    pair, order)], task ``t = round * num_pairs + s`` on rank ``t % world``.
    ``order`` is the reference's coin flip for the first move
    (evaluation.py:67-76): +1 = pair[0] moves first."""
    pairs = gen_pairs(num_agents)
    out = []
    for r in range(num_rounds):
        for s, pair in enumerate(pairs):
            t = r * len(pairs) + s
            if t % world != rank:
                continue
            order = int(np.random.RandomState(10000 * r + s).choice([-1, 1]))
            out.append((t, r, s, pair, order))
    return out


def _dist_info(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def evaluate(agents: List, num_rounds: int, num_workers: Optional[int] = None,
             device=None, *, group=None, rank: Optional[int] = None,
             world_size: Optional[int] = None, reduce: bool = True,
             stats: Optional[dict] = None, _play=None) -> Dict[Pair, List[int]]:
    """Round robin tournament between agents (evaluation.py:17-38).

    ``num_workers`` is accepted for compatibility and ignored: under
    ``torch.distributed`` the ranks take the role of the reference's worker
    processes.  With a process group, rank 0 returns the tallies of the whole
    tournament (one ``reduce`` of a ``[pairs, 3]`` tensor) and the other
    ranks return their own share; ``rank`` / ``world_size`` override the
    group's (``reduce=False``: no collective, this rank's share only).
    """
    r0, w0 = _dist_info(group)
    rank = r0 if rank is None else rank
    world = w0 if world_size is None else world_size
    pairs = gen_pairs(len(agents))
    tasks = tournament_tasks(len(agents), num_rounds, rank, world)
    first, second = [], []
    for _, _, _, pair, order in tasks:
        pa, pb = agents[pair[0]].policy, agents[pair[1]].policy
        first.append(pa if order == 1 else pb)
        second.append(pb if order == 1 else pa)
    board_size = agents[0].game.board_size
    seed = int(np.random.RandomState(num_rounds).randint(1 << 30))
    play = _play or play_matches
    result, _ = play(first, second, board_size, seed=seed, device=device,
                     game_ids=[t for t, *_ in tasks], stats=stats)
    tally = np.zeros((len(pairs), 3), dtype=np.int64)
    for (_, _, s, _, order), res in zip(tasks, result):
        outcome = order * (int(res) - 2)            # evaluation.py:78-80
        tally[s, 0 if outcome > 0 else (1 if outcome == 0 else 2)] += 1
    if reduce and world > 1:
        total = reduce_tallies(tally.copy(), group=group, device=device)
        if rank == 0:
            tally = total       # the other ranks keep (and return) their own share
    return {pair: [int(x) for x in tally[s]] for s, pair in enumerate(pairs)}


def reduce_tallies(tally: np.ndarray, dst: int = 0, group=None, device=None) -> np.ndarray:
    """Sum the ranks' ``[pairs, 3]`` tallies onto rank ``dst`` (the path's
    only exchange).  NCCL groups reduce a device tensor, gloo a host tensor."""
    import torch.distributed as dist
    backend = dist.get_backend(group)
    t = torch.from_numpy(np.ascontiguousarray(tally))
    if 'nccl' in str(backend):
        t = t.to(device if device is not None else
                 torch.device('cuda', torch.cuda.current_device()))
    dist.reduce(t, dst=dst, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()
