"""GPU-resident replay buffer: the step right after the self-play path.

Reference: ``ReplayBuffer`` (azalea/replay_buffer.py:107-149) is a circular
list of Python objects that a ``DataLoader`` collates on the host with
``prep.torch_batch_replays`` (azalea/prep.py:24-39).  Here the rows that
``k_play_commit`` wrote stay on the device: ``put`` is a (wrapping) device
copy, ``sample`` draws row indices on the device and ``az_replay_collate``
turns them into the padded training tensors the network's ``run(batch,
compute_loss=True)`` consumes (azalea/network.py:87-102) -- no host round
trip between self-play and the optimiser.
"""
import ctypes as C
from typing import Dict, Optional

import torch

from . import _cabi
from .engine import replay_row_bytes


class DeviceReplayBuffer:
    def __init__(self, capacity: int, board_size: int, device=None):
        self.n = int(board_size)
        self.nn = self.n * self.n
        self.row_bytes = replay_row_bytes(self.n)
        self.device = torch.device(device or 'cuda')
        if self.device.type != 'cuda':
            raise RuntimeError('DeviceReplayBuffer needs a CUDA device')
        self.rows = torch.zeros(capacity, self.row_bytes, dtype=torch.uint8,
                                device=self.device)
        self.capacity = int(capacity)
        self.size = 0               # rows filled so far (<= capacity)
        self.write_idx = 0          # replay_buffer.py:117
        self.fresh_counter = 0      # replay_buffer.py:118

    def __len__(self) -> int:
        return self.size

    def put(self, new_rows: torch.Tensor) -> None:
        """FIFO write with wraparound (replay_buffer.py:134-149)."""
        new_rows = new_rows.to(self.device)
        count = new_rows.shape[0]
        if count > self.capacity:
            new_rows, count = new_rows[-self.capacity:], self.capacity
        first = min(count, self.capacity - self.write_idx)
        self.rows[self.write_idx:self.write_idx + first] = new_rows[:first]
        if count > first:
            self.rows[:count - first] = new_rows[first:]
        self.write_idx = (self.write_idx + count) % self.capacity
        self.size = min(self.capacity, self.size + count)
        self.fresh_counter += count

    def consume(self, num_examples: int, player) -> Dict[str, float]:
        """Account for consumed examples and refill from self-play when the
        fresh ones run out (replay_buffer.py:121-132)."""
        self.fresh_counter -= num_examples
        refill = max(0, num_examples - self.fresh_counter)
        if not refill:
            return {}
        rows, metrics = player.read_device(refill)
        self.put(rows)
        return metrics

    def state_dict(self) -> Dict:
        """replay_buffer.py:151-158, with the rows as one uint8 tensor."""
        return {'rows': self.rows[:self.size].cpu(), 'board_size': self.n,
                'capacity': self.capacity, 'write_idx': self.write_idx,
                'fresh_counter': self.fresh_counter}

    def load_state_dict(self, state: Dict) -> None:
        assert state['board_size'] == self.n and state['capacity'] == self.capacity
        rows = state['rows']
        self.rows[:rows.shape[0]] = rows.to(self.device)
        self.size = rows.shape[0]
        self.write_idx = state['write_idx']
        self.fresh_counter = state['fresh_counter']

    def sample(self, batch_size: int, generator: Optional[torch.Generator] = None,
               trim: bool = True, reflect: bool = False) -> Dict[str, torch.Tensor]:
        """A uniformly sampled minibatch as the reference's collated dict:
        ``board`` int32 [B,n,n], ``legal_moves`` int32 [B,K], ``moves_prob``
        f32 [B,K], ``reward`` f32 [B], ``color``/``result`` int64 [B].  With
        ``trim`` K is the longest legal-move list in the batch (prep.pad,
        one host sync); otherwise K = n*n.  With ``reflect`` each sample is
        rotated by 180 degrees with probability 1/2 (``reflect_batch``; the
        coins come from ``generator`` after the row indices)."""
        if self.size == 0:
            raise RuntimeError('replay buffer is empty')
        idx = torch.randint(0, self.size, (batch_size,), device=self.device,
                            generator=generator, dtype=torch.int64)
        batch = self.collate(idx, trim=trim)
        if reflect:
            coins = torch.randint(0, 2, (batch_size,), device=self.device,
                                  generator=generator, dtype=torch.uint8)
            reflect_batch(batch, coins)
        return batch

    def collate(self, idx: torch.Tensor, trim: bool = True):
        B, nn, dev = idx.numel(), self.nn, self.device
        idx = idx.to(dev, torch.int64).contiguous()
        board = torch.empty(B, self.n, self.n, dtype=torch.int32, device=dev)
        moves = torch.empty(B, nn, dtype=torch.int32, device=dev)
        probs = torch.empty(B, nn, dtype=torch.float32, device=dev)
        reward = torch.empty(B, dtype=torch.float32, device=dev)
        color = torch.empty(B, dtype=torch.int64, device=dev)
        result = torch.empty(B, dtype=torch.int64, device=dev)
        k = torch.empty(B, dtype=torch.int32, device=dev)
        p = lambda t: C.c_void_p(t.data_ptr())
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().az_replay_collate(
            p(self.rows), self.row_bytes, p(idx), B, self.n, p(board), p(moves),
            p(probs), p(reward), p(color), p(result), p(k), stream))
        if trim:
            K = int(k.max().item())
            moves, probs = moves[:, :K], probs[:, :K]
        return dict(color=color, legal_moves=moves, result=result, board=board,
                    moves_prob=probs, reward=reward)


def reflect_batch(batch: Dict[str, torch.Tensor], coins: torch.Tensor) -> None:
    """Hex's 180-degree rotation of the collated samples whose coin (uint8 [B],
    device) is non-zero, in place (az_batch_reflect): ``board`` is reversed on
    both axes, the k legal moves m become n*n+1-m and, like their
    ``moves_prob``, are reversed so that they stay ascending; padding stays
    zero.  Its own inverse for the same coins."""
    board, moves, probs = batch['board'], batch['legal_moves'], batch['moves_prob']
    B, n = board.shape[0], board.shape[-1]
    assert board.dtype == torch.int32 and board.is_contiguous()
    assert moves.dtype == torch.int32 and probs.dtype == torch.float32
    assert moves.shape == probs.shape and moves.stride() == probs.stride() and moves.stride(1) == 1
    coins = coins.to(board.device, torch.uint8).contiguous()
    assert coins.numel() == B
    p = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(board.device).cuda_stream)
    _cabi.check(_cabi.lib().az_batch_reflect(
        p(board), p(moves), p(probs), p(coins), B, n, moves.shape[1], moves.stride(0), stream))
