"""``SearchTree`` with the reference's interface, tree resident in HBM.

Drop-in for azalea/search_tree.py:24-154,327-344 + azalea/mcts.py:258-293:
``search(game, network, ...) -> (move_probs, value, metrics)``, ``move``,
``reset``, ``SearchTreeFull``.  The tree is one row of a 1-game device
``Engine``; selection, virtual loss, dedup, expansion and backup run in the
CUDA kernels (csrc/az_kernels.cuh).  What stays on the host is exactly what
the reference also does on the host around an evaluator call
(mcts.py:155-217): build the padded batch dict, call ``network.run``,
exponentiate the log-probabilities with NumPy, so any evaluator object that
works with the reference works here and sees the same inputs.

The many-games path (``azalea_b200.selfplay``) uses the same kernels without
any of this host traffic.
"""
from typing import Any, Dict, Optional, Tuple

import numpy as np
import torch
from numpy.random import RandomState

from . import _cabi
from .engine import Engine
from .game.hex import HexGame, default_device

# search_tree.py:17-18
MAX_NODES = 10000000

# nodes per half of the device pool for a single-game tree: the kept subtree
# plus one move's growth must fit (the reference keeps everything, up to
# MAX_NODES, in 240 MB of host memory)
DEVICE_NODES = 4_000_000


class SearchTreeFull(Exception):
    pass


def as_distribution(counts: np.ndarray, temperature: float = 1.0) \
        -> np.ndarray:
    """Visit counts -> move distribution (search_tree.py:327-344).

    Same operation order as the reference so the float64 result is
    bit-identical: log of the clipped counts in float32, temperature in
    float32, logaddexp-normalise in float64.  Temperature 0 = uniform over
    the arg-max ties.
    """
    assert all(counts >= 0)
    log_pi = np.log(counts.clip(min=1))
    log_pi[counts == 0] = -np.inf
    if temperature:
        log_pi = log_pi / temperature
    else:
        log_pi[log_pi < log_pi.max()] = -np.inf
    log_pi = log_pi.astype(np.float64)
    return np.exp(log_pi - np.logaddexp.reduce(log_pi))


class SearchTree:
    """Explored game tree + MCTS statistics of one game, on the GPU."""

    def __init__(self, device=None, device_nodes: Optional[int] = None):
        self.device = torch.device(device) if device else None
        self._device_nodes = device_nodes
        self._eng = None
        self._max_nodes = MAX_NODES      # read at construction, like the
        # reference reads search_tree.MAX_NODES in __init__ (:48-55)

    # ---------------------------------------------------------- plumbing --
    def _engine(self, board_size, batch_size) -> Engine:
        eng = self._eng
        if eng is None or eng.n != board_size or eng.max_batch < batch_size:
            if eng is not None and self.root_is_evaluated():
                raise RuntimeError('board size / batch size changed '
                                   'under a live search tree')
            dev = self.device or default_device()
            nodes = self._device_nodes or min(
                DEVICE_NODES, max(1024, self._max_nodes + 2))
            self._eng = Engine(1, board_size, max_batch=max(batch_size, 10),
                               nodes_per_game=nodes,
                               max_nodes_ref=self._max_nodes, device=dev)
        return self._eng

    def _raise_if_full(self):
        st = int(self._eng.status().item())
        if st & (_cabi.AZ_ST_POOL_FULL | _cabi.AZ_ST_TREE_FULL):
            raise SearchTreeFull('too many nodes')
        assert not (st & _cabi.AZ_ST_ILLEGAL), 'inconsistent search state'

    @property
    def num_nodes(self) -> int:
        """The reference's ``tree.num_nodes`` (never shrinks on re-root)."""
        if self._eng is None:
            return 1
        return int(self._eng.root_stats()[5].item())

    def root_is_evaluated(self) -> bool:
        return self._eng is not None and int(self._eng.root_stats()[3].item()) >= 0

    def root_stats(self):
        """(num_visits, total_value, prior_prob) of the root's children, and
        (N, W) of the root -- total_value in the stored sign
        (search_tree.py:37-40)."""
        v, w, p, k, rnw, _ = self._eng.root_stats()
        k = int(k.item())
        assert k >= 0, 'unevaluated nodes have no stats'
        rnw = rnw.cpu().numpy()
        return (v[0, :k].cpu().numpy(), w[0, :k].cpu().numpy(),
                p[0, :k].cpu().numpy(), np.float32(rnw[0, 0]),
                np.float32(rnw[0, 1]))

    # ------------------------------------------------------------- API ---
    def reset(self):
        """Clear tree (search_tree.py:59-71)."""
        if self._eng is not None:
            self._eng.reset()

    def move(self, move_id: int) -> None:
        """Commit move and pick new root node (search_tree.py:115-132)."""
        if self._eng is None:
            return      # unevaluated root: "step to the unknown"
        self._eng.tree_move([int(move_id)])
        st = int(self._eng.status().item())
        assert not (st & _cabi.AZ_ST_ILLEGAL), 'illegal child'

    def search(self, game, network, *,
               num_simulations: int = 100,
               temperature: float = 1.0,
               exploration_coef: float = 1.0,
               exploration_noise_scale: float = 1.0,
               exploration_noise_alpha: float = 1.0,
               batch_size: int = 10,
               rng: Optional[RandomState] = None,
               random_reflect: bool = False) \
            -> Tuple[np.ndarray, float, Dict[str, Any]]:
        """Plan next moves with batched MCTS (search_tree.py:73-113).

        ``random_reflect``: every position handed to ``network.run`` is
        rotated by 180 degrees with probability 1/2 (one ``rng`` draw per
        position, so the later move draws differ from a run without it).

        :return: next move probabilities, game value, debug metrics
        """
        if rng is None:
            rng = RandomState(0)
        state = game.state
        check_game_state(state)
        assert not state.result, 'terminal root'
        n = state.board.shape[0]
        eng = self._engine(n, batch_size)
        # the tree's root position is the game's current position
        eng.hex_set_state(state.board.reshape(1, -1), [state.color + 1],
                          None, reset_trees=False)
        if exploration_noise_scale:
            # device Philox streams instead of RandomState.dirichlet
            # (statistical parity only; noise is off in deterministic play)
            eng.meta[0, 10] = int(rng.randint(1 << 31))

        with torch.no_grad():
            network.eval()
            metrics = self._sample_paths(
                eng, game, network, num_simulations, batch_size,
                exploration_coef, exploration_noise_scale,
                exploration_noise_alpha, rng, random_reflect)

        visits, _, _, root_n, root_w = self.root_stats()
        move_probs = as_distribution(visits, temperature)
        value = root_w / root_n
        metrics['search_root_width'] = np.sum(visits > 0)
        metrics['search_root_visits'] = np.mean(visits)
        metrics['search_root_children'] = len(visits)
        metrics['search_tree_nodes'] = self.num_nodes
        return move_probs, value, metrics

    # ------------------------------------------------------ mcts.py glue --
    def _sample_paths(self, eng, game, net, num_simulations, batch_size,
                      coef, noise_scale, noise_alpha, rng, reflect=False):
        """mcts.sample_paths (mcts.py:258-293) around the device kernels."""
        num_batches = num_simulations // batch_size + 1
        search_value = 0
        if not self.root_is_evaluated():
            # evaluate_root, mcts.py:18-27 (value discarded)
            eng.select_root()
            self._evaluate(eng, game, net, rng, reflect)
            eng.expand_root()
            self._raise_if_full()
        for _ in range(num_batches):
            eng.select(batch_size, coef, noise_scale, noise_alpha)
            values = self._evaluate(eng, game, net, rng, reflect)
            eng.expand_backup()
            search_value += np.sum(values)
        self._raise_if_full()
        return {'search_value': search_value / (num_batches * batch_size)}

    def _host_buffers(self, eng):
        """Persistent pinned staging for the two copies of a search batch:
        leaf info + boards + legal moves come down in ONE device-to-host copy
        (the three buffers are neighbours in the engine's block), values +
        priors go up in ONE host-to-device copy."""
        hb = getattr(self, '_hb', None)
        if hb is None or hb['eng'] is not eng:
            down, d_off = eng.span(_cabi.AZ_BUF_LEAF_INFO, _cabi.AZ_BUF_LEAF_MOVES)
            up, u_off = eng.span(_cabi.AZ_BUF_VALUE, _cabi.AZ_BUF_PRIOR)
            pin_down = torch.empty(down.numel(), dtype=torch.uint8).pin_memory()
            pin_up = torch.zeros(up.numel(), dtype=torch.uint8).pin_memory()
            B, nn, cs = eng.max_batch, eng.nn, eng.cell_stride
            nd, nu = pin_down.numpy(), pin_up.numpy()

            def view(buf, offs, which, dtype, shape):
                o, b = offs[which]
                return buf[o:o + b].view(dtype).reshape(shape)
            hb = dict(eng=eng, down=down, up=up, pin_down=pin_down, pin_up=pin_up,
                      info=view(nd, d_off, _cabi.AZ_BUF_LEAF_INFO, np.int32, (-1, B, 4))[0],
                      board=view(nd, d_off, _cabi.AZ_BUF_LEAF_BOARD, np.int8, (-1, B, cs))[0],
                      moves=view(nd, d_off, _cabi.AZ_BUF_LEAF_MOVES, np.int32, (-1, B, nn))[0],
                      value=view(nu, u_off, _cabi.AZ_BUF_VALUE, np.float32, (-1, B))[0],
                      prior=view(nu, u_off, _cabi.AZ_BUF_PRIOR, np.float32, (-1, B, nn))[0])
            self._hb = hb
        return hb

    def _evaluate(self, eng, game, net, rng, reflect=False):
        """mcts.evaluate_batch (mcts.py:155-217) for the leaves the select
        kernel just produced.  Returns the values in leaf-list order
        (terminal rows included).  One device-to-host copy + sync and one
        host-to-device copy per search batch."""
        hb = self._host_buffers(eng)
        eng.compute_leaf_moves()
        hb['pin_down'].copy_(hb['down'], non_blocking=True)
        torch.cuda.current_stream(eng.device).synchronize()
        info = hb['info']
        slots = np.flatnonzero(info[:, 0] >= 0)
        flags = info[slots, 1] & 0xff
        color = (info[slots, 1] >> 8) & 1
        values = np.zeros(len(slots), dtype=np.float32)
        term = flags != 0
        # terminal positions: -1 for the player to move (mcts.py:192-195)
        values[term] = -1.0
        if np.any(~term):
            live = slots[~term]
            n, nn = eng.n, eng.nn
            boards = hb['board'][live, :nn]
            moves = hb['moves'][live]
            # prep.pad (prep.py:70-86): K = longest legal-move list in the
            # whole batch (terminal rows have none)
            K = int(info[slots, 2].max())
            batch = {
                'color': color[~term].astype(np.int64),
                'legal_moves': moves[:, :K].astype(np.int32),
                'result': np.zeros(len(live), dtype=np.int64),
                'board': boards.reshape(-1, n, n).astype(np.int32),
            }
            # the reference's random_reflect is a no-op and takes no random
            # numbers (hex.py:124-134); with `reflect` a coin per position
            # rotates it, and its priors (by move ordinal) are turned back below
            coins = rng.randint(2, size=len(live)).astype(bool) if reflect else None
            if coins is not None and coins.any():
                batch['board'][coins], batch['legal_moves'][coins] = \
                    HexGame.rotate_board_moves(batch['board'][coins],
                                               batch['legal_moves'][coins])
            tbatch = {}
            for k in batch:
                tbatch[k] = torch.from_numpy(batch[k])
                if net.device.type == 'cuda':
                    tbatch[k] = tbatch[k].pin_memory().to(net.device)
            output = net.run(tbatch)
            nonterm_value = output['value'].cpu().numpy()
            prior = np.exp(output['moves_logprob'].cpu().numpy())
            assert (prior >= 0.0).all(), 'negative prior prob'
            assert (np.abs(prior.sum(1) - 1.0) < 1e-4).all(), \
                'prior probs normalized incorrectly'
            if coins is not None:
                for i in np.flatnonzero(coins):
                    k = int(info[live[i], 2])
                    prior[i, :k] = prior[i, k - 1::-1].copy()
            values[~term] = nonterm_value
            hb['value'][live] = nonterm_value
            hb['prior'][live, :prior.shape[1]] = prior
            # stream-ordered: the pinned buffer is next written after the next
            # batch's synchronize, i.e. after this copy has completed
            hb['up'].copy_(hb['pin_up'], non_blocking=True)
        return values


def check_game_state(state):
    """mcts.check_game_state (mcts.py:30-43)."""
    assert isinstance(state.board, np.ndarray), 'board type error'
    assert state.board.dtype == np.int32, 'board type error'
    assert len(state.board.shape) == 2, 'board type error'
    assert isinstance(state.legal_moves, np.ndarray), 'moves type error'
    assert state.legal_moves.dtype == np.int32, 'moves type error'
    assert len(state.legal_moves.shape) == 1, 'moves type error'
    assert all(state.legal_moves > 0), 'moves value error'
    assert isinstance(state.color, int), 'color type error'
    assert isinstance(state.result, int), 'result type error'
    assert len(state.legal_moves) or state.result, \
        'no legal moves but game is continuing'
    assert not (len(state.legal_moves) and state.result), \
        'legal moves but game ended'
