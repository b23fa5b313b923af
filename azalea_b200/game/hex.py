"""Game of Hex with the reference's ``HexGame`` interface, rules on the GPU.

Drop-in for azalea/game/hex.py:19-134 (``SearchableEnv``): same methods, same
``HexGameState`` fields and dtypes, same assertion behaviour.  The rules
themselves (legal moves, step, winner) run in the CUDA engine
(csrc/az_engine.cu: k_hex_step / k_hex_legal / az_hex_wins) on bit-packed
boards; this class only moves one game's state across the PCIe bus.  The
throughput path never touches this class -- thousands of games live in one
``Engine`` -- it exists so that reference-style single-game code keeps working.
"""
from typing import Optional, Tuple

import numpy as np
import torch

from ..engine import Engine
from ..typing import GameState

HexGameState = GameState


def default_device():
    if not torch.cuda.is_available():
        raise RuntimeError('azalea_b200 needs a CUDA device '
                           '(there is no CPU fallback)')
    return torch.device('cuda', torch.cuda.current_device())


class HexGame:
    """hex.py:19-70.  One game = one row of a 1-game device engine."""

    def __init__(self, board_size: int = 11, device=None) -> None:
        self.board_size = board_size
        self.device = torch.device(device) if device else default_device()
        self._eng = Engine(1, board_size, max_batch=1, nodes_per_game=2,
                           device=self.device)
        self._game_snapshot = None
        self._last_tile = -1

    # pickling support, hex.py:33-45
    def __getstate__(self):
        st = self.state
        return (st.board, st.color + 1, self._winner(), self._last_tile,
                str(self.device))

    def __setstate__(self, state):
        board, color, winner, last_tile, device = state
        self.__init__(board.shape[0], device=device)
        self._load(board, color, last_tile)

    def _load(self, board, color, last_tile):
        self._eng.hex_set_state(board.reshape(1, -1), [color], [last_tile])
        self._last_tile = last_tile

    def _winner(self):
        return {0: 0, 1: 2, 3: 1}[self.state.result]

    def reset(self):
        self._eng.reset()
        self._game_snapshot = None
        self._last_tile = -1

    def seed(self, seed: Optional[int] = None) -> None:
        pass

    @property
    def state(self) -> HexGameState:
        board, color, result, _ = self._eng.hex_state()
        moves, count = self._eng.hex_legal_moves()
        k = int(count.item())
        return HexGameState(int(color.item()),
                            moves[0, :k].cpu().numpy().astype(np.int32),
                            int(result.item()),
                            board[0].cpu().numpy().astype(np.int32))

    def step(self, move: int) -> None:
        self._eng.hex_step([int(move)])
        if int(self._eng.status().item()) & 4:
            # hex.py:174-176: occupied tile, out of range, or game over
            self._eng.meta[0, 5] = 0
            raise AssertionError('illegal move')
        self._last_tile = int(move) - 1

    def snapshot(self) -> None:
        st = self.state
        self._game_snapshot = (st.board, st.color + 1, self._last_tile)

    def restore(self) -> None:
        assert self._game_snapshot
        self._load(*self._game_snapshot)

    # perspective flip: host-side array utility of the data format
    # (hex.py:72-134); the search path does this inside k_select
    @staticmethod
    def flip_player_board(board: np.ndarray) -> np.ndarray:
        assert isinstance(board, np.ndarray)
        if board.ndim == 2:
            return HexGame.flip_player_board(board[None])
        assert board.ndim == 3, 'expecting batch of boards'
        assert board.shape[-2] == board.shape[-1], 'board must be square'
        swapped = np.where(board > 0, 3 - board, 0).astype(board.dtype)
        # out[i, j] = in[n-1-j, n-1-i]
        return swapped[:, ::-1, ::-1].transpose(0, 2, 1)

    @staticmethod
    def flip_player_board_moves(board: np.ndarray, moves: np.ndarray) \
            -> Tuple[np.ndarray, np.ndarray]:
        assert isinstance(board, np.ndarray) and isinstance(moves, np.ndarray)
        if board.ndim == 2:
            assert moves.ndim == 1, 'expecting 1D moves array'
            return HexGame.flip_player_board_moves(board[None], moves[None])
        board = HexGame.flip_player_board(board)
        assert moves.ndim == 2, 'expecting batch of moves'
        assert len(moves) == len(board), 'board and moves batch sizes differ'
        n = board.shape[-1]
        tiles = moves - 1
        flipped = (n - 1 - tiles % n) * n + (n - 1 - tiles // n) + 1
        return board, np.where(moves > 0, flipped, 0).astype(moves.dtype)

    @staticmethod
    def rotate_board_moves(board: np.ndarray, moves: np.ndarray) \
            -> Tuple[np.ndarray, np.ndarray]:
        """Hex's rule-preserving symmetry, the 180-degree rotation
        (i, j) -> (n-1-i, n-1-j), of a batch of boards [B, n, n] and their
        ascending, zero-padded moves [B, K]: the board is reversed on both
        axes, the k non-zero moves m of a row become n*n+1-m and are reversed
        so that they stay ascending.  Its own inverse."""
        assert isinstance(board, np.ndarray) and isinstance(moves, np.ndarray)
        assert board.ndim == 3 and moves.ndim == 2 and len(board) == len(moves)
        nn = board.shape[-1] * board.shape[-2]
        out = np.zeros_like(moves)
        for i, k in enumerate(np.count_nonzero(moves, axis=1)):
            out[i, :k] = nn + 1 - moves[i, k - 1::-1] if k else 0
        return np.ascontiguousarray(board[:, ::-1, ::-1]), out

    @staticmethod
    def random_reflect(board, moves=None, rng=None):
        """hex.py:124-134: a no-op in the reference (consumes no RNG)."""
        if moves is not None:
            return board, moves
        return board
