"""``Player.read(size)`` facade over lockstep GPU self-play.

Same call as the reference's (azalea/parallel_player.py:17-52): hand it the
self-play agent, ask for ``size`` positions, get ``(ReplayDataFrame,
metrics)`` back.  The reference's process pool argument is accepted and
ignored -- the games run in lockstep on the GPU instead of one per worker
process.
"""
from collections import defaultdict
from typing import Dict, Sequence, Tuple

import numpy as np

from .engine import decode_replay_rows
from .random_policy import RandomPolicy
from .replay_buffer import ReplayDataFrame
from .selfplay import LockstepSelfPlay, rows_to_dataframe

Metrics = Dict[str, float]


class Player:
    def __init__(self, pool, agents: Sequence, num_games: int = 4096,
                 seed: int = 0, **kwargs):
        self.agents = agents
        policy = agents[0].policy
        board_size = agents[0].game.board_size
        settings = policy.settings
        self.board_size = board_size
        if isinstance(policy, RandomPolicy):
            # AzaleaAgent(game_factory) without a policy: random self-play
            self.sp = LockstepSelfPlay(None, num_games=num_games, board_size=board_size,
                                       random_play=True, seed=seed, **kwargs)
            self.running = True
            return
        self.sp = LockstepSelfPlay(
            policy.net, num_games=num_games, board_size=board_size,
            simulations=policy.simulations,
            search_batch_size=policy.search_batch_size,
            exploration_coef=policy.exploration_coef,
            exploration_depth=policy.exploration_depth,
            exploration_noise_alpha=policy.exploration_noise_alpha,
            exploration_noise_scale=policy.exploration_noise_scale,
            exploration_temperature=policy.exploration_temperature,
            move_sampling=settings.get('move_sampling', True),
            move_exploration=settings.get('move_exploration', True),
            random_reflect=getattr(policy, 'random_reflect', False),
            seed=seed, **kwargs)
        self.running = True

    def read(self, size: int) -> Tuple[ReplayDataFrame, Metrics]:
        """Play self-play games until ``size`` positions are available."""
        examples = ReplayDataFrame()
        metrics: Metrics = defaultdict(int)
        while len(examples) < size:
            self.sp.step_move()
            if self.sp.eng.replay_count() == 0:
                continue
            rows = self.sp.harvest()
            h, _, _ = decode_replay_rows(rows, self.board_size)
            last = np.flatnonzero(np.r_[h['ply'][1:] == 0, True])
            metrics['games'] += len(last)
            metrics['moves_per_game'] += float(np.sum(h['ply'][last] + 1))
            metrics['reward'] += float(np.sum(h['reward'][last]))
            examples.append(rows_to_dataframe(rows, self.board_size))
        self._report(metrics)
        return examples, metrics

    def _report(self, metrics) -> None:
        """Games dropped on SearchTreeFull (parallel_player.py:71-76) and
        expansions skipped on a full pool half are never silent."""
        import logging
        cnt = self.sp.counters()
        metrics['game_error'] = cnt['games_failed']
        metrics['pool_skipped_expansions'] = cnt['pool_skipped_expansions']
        if cnt['games_failed'] or cnt['pool_skipped_expansions']:
            logging.warning('self-play: %d games dropped (tree full), %d expansions skipped on a full '
                            'node pool -- raise nodes_per_game', cnt['games_failed'],
                            cnt['pool_skipped_expansions'])

    def read_device(self, size: int):
        """Like ``read`` but the rows stay on the device (uint8
        [R, row_bytes] tensor) for ``DeviceReplayBuffer.put``."""
        import torch
        eng = self.sp.eng
        chunks, total = [], 0
        metrics: Metrics = defaultdict(int)
        games0 = self.sp.counters()['games']
        while total < size:
            self.sp.step_move()
            count = min(eng.replay_count(), eng.replay.shape[0])
            if count:
                chunks.append(eng.replay[:count].clone())
                eng.replay_clear()
                total += count
        metrics['games'] = self.sp.counters()['games'] - games0
        metrics['moves_per_game'] = float(total)
        self._report(metrics)
        return torch.cat(chunks), metrics

    def stop(self) -> None:
        """parallel_player.py:49-52; nothing to shut down here."""
        self.running = False
