"""Training loop around GPU self-play (azalea/policy_trainer.py:24-181).

Same entry points and the same flow as the reference -- fill the replay buffer
with random-policy games, then alternate SGD steps on minibatches with replay
refills from self-play by the policy being trained -- but the whole loop stays
on the device: ``Player`` plays the games in lockstep on the GPU, the
``DeviceReplayBuffer`` keeps their rows in HBM and collates minibatches with
``az_replay_collate``, and the evaluator's folded inference weights are
refreshed in place after the optimizer steps, so the captured self-play graph
keeps running.

Deviations from the reference, all on purpose:

* minibatches are drawn uniformly with replacement from the device buffer
  instead of a shuffled ``DataLoader`` epoch (no host round trip);
* the shipped config (config/hex11_train_config.yml) and the code disagree on
  key names: both spellings are accepted (``replaybuf_resample`` /
  ``replaybuf_oversampling``, ``total_steps`` / ``total_epochs``,
  ``lr_decay_steps`` / ``lr_decay_epochs``); ``num_player_workers`` and
  ``num_dataloader_workers`` are ignored, ``num_selfplay_games`` (default
  1024) sets how many games are resident on the GPU;
* ``game`` may be ``'hex'`` or a dotted class path;
* tensorboard monitoring is out of scope: scalars go to ``logging``;
* ``random_reflect`` (default off) is honoured: each minibatch sample is
  rotated by 180 degrees with probability 1/2 (``DeviceReplayBuffer.sample``,
  coins from the seeded device generator), and the self-play search shows the
  network its leaves in random orientations (the policy's setting).
"""
import logging
import os
import time
from functools import partial
from typing import Callable, Dict, Optional

import numpy as np
import torch
from torch import optim
from torch.optim import lr_scheduler

from .azalea_agent import AzaleaAgent
from .parallel_player import Player
from .replay_device import DeviceReplayBuffer
from .utils import import_and_get


def _game_class(name: str):
    if name in ('hex', 'HexGame'):
        from .game.hex import HexGame
        return HexGame
    if name.startswith('azalea.'):
        name = 'azalea_b200.' + name[len('azalea.'):]
    return import_and_get(name)


def _cfg(config, *names, default=None):
    for name in names:
        if name in config:
            return config[name]
    if default is None:
        raise KeyError(names[0])
    return default


class _TrainingPlayer:
    """Self-play by the policy under training: switches the network to eval
    mode and refreshes the folded inference weights (in place) around every
    refill."""

    def __init__(self, player: Player, net):
        self.player, self.net = player, net

    def read_device(self, size: int):
        was_training = self.net.training
        self.net.eval()
        self.net.prepare_inference()
        try:
            return self.player.read_device(size)
        finally:
            self.net.train(was_training)

    def stop(self):
        self.player.stop()


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


def _comm_device(net_device, group=None):
    """NCCL moves device tensors, gloo host tensors."""
    import torch.distributed as dist
    return net_device if 'nccl' in str(dist.get_backend(group)) else torch.device('cpu')


def broadcast_policy_weights(net, src: int = 0, group=None) -> int:
    """The trainer's network to every self-play rank (SURVEY 8e: "weight
    broadcast rank 0 -> all when the trainer updates the net"; the reference
    gets the same effect by pickling the agent into every game it dispatches,
    parallel_player.py:36-38).  Parameters and buffers (BatchNorm statistics)
    travel as one flat tensor per dtype; returns the bytes sent.  No-op
    without a process group."""
    dist = _dist()
    if dist is None:
        return 0
    tensors = [p.data for p in net.parameters()] + list(net.buffers())
    by_dtype: Dict = {}
    for t in tensors:
        by_dtype.setdefault(t.dtype, []).append(t)
    nbytes = 0
    for ts in by_dtype.values():
        dev = _comm_device(ts[0].device, group)
        flat = torch.cat([t.reshape(-1) for t in ts]).to(dev)
        dist.broadcast(flat, src=src, group=group)
        off = 0
        for t in ts:
            n = t.numel()
            t.copy_(flat[off:off + n].view_as(t))
            off += n
        nbytes += flat.numel() * flat.element_size()
    return nbytes


class DistributedSelfPlay:
    """Replay refills played by ALL ranks of the process group for the one
    rank that trains (SURVEY 8e).  Rank 0 calls ``read_device(size)`` wherever
    the single-GPU loop calls its player; the other ranks sit in ``serve()``.
    Per refill: one broadcast of the request, one broadcast of the weights
    (~2 MB), every rank plays ``ceil(size / world)`` positions with its own
    games, and the rows are gathered to rank 0 (``gather_replay_rows``, the
    path's only data exchange).  ``stop()`` on rank 0 releases the servers."""

    def __init__(self, player, net, group=None):
        self.player, self.net, self.group = player, net, group
        self.bytes_broadcast = 0

    def _header(self, value=0):
        import torch.distributed as dist
        dev = _comm_device(next(self.net.parameters()).device, self.group)
        h = torch.tensor([int(value)], dtype=torch.int64, device=dev)
        dist.broadcast(h, src=0, group=self.group)
        return int(h.item())

    def _play_and_gather(self, size):
        import torch.distributed as dist
        from .selfplay import gather_replay_rows
        world = dist.get_world_size(self.group)
        self.bytes_broadcast += broadcast_policy_weights(self.net, 0, self.group)
        rows, metrics = self.player.read_device(-(-size // world))
        rows = rows.to(_comm_device(rows.device, self.group))
        return gather_replay_rows(rows, dst=0, group=self.group), metrics

    def read_device(self, size: int):
        """Rank 0: ask every rank for its share and collect the rows."""
        self._header(size)
        rows, metrics = self._play_and_gather(int(size))
        return rows, metrics

    def serve(self) -> int:
        """Ranks > 0: play refills until rank 0 stops.  Returns how many."""
        served = 0
        while True:
            size = self._header()
            if size < 0:
                return served
            self._play_and_gather(size)
            served += 1

    def stop(self):
        import torch.distributed as dist
        if dist.get_rank(self.group) == 0:
            self._header(-1)
        self.player.stop()


def train(policy, config, rundir, *,
          replaybuf: Optional[DeviceReplayBuffer] = None,
          max_steps: Optional[int] = None) -> str:
    """Train model (policy_trainer.py:24-120).  Returns the final checkpoint path."""
    os.makedirs(rundir, exist_ok=True)
    os.makedirs(f'{rundir}/checkpoints', exist_ok=True)

    seed = int(config['seed'])
    np.random.seed(seed % (1 << 32))
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
    policy.seed(seed % (1 << 32))

    device = config['device']
    if device == 'auto':
        device = 'cuda' if torch.cuda.is_available() else 'cpu'
    device = torch.device(device)
    if device.type != 'cuda':
        raise RuntimeError('GPU self-play needs a CUDA device')
    oversampling = _cfg(config, 'replaybuf_oversampling', 'replaybuf_resample')
    batch_size = config['batch_size']
    num_games = int(config.get('num_selfplay_games', 1024))

    game_class = _game_class(config['game'])
    game_factory = partial(game_class, board_size=config['board_size'])

    # Under torch.distributed (one process per GPU): rank 0 trains, every rank plays
    # self-play for its refills with its own block of game ids (SURVEY 8e)
    dist = _dist()
    rank = dist.get_rank() if dist else 0
    world = dist.get_world_size() if dist else 1
    if rank > 0:
        policy.net.to(device)
        policy.settings['move_exploration'] = True
        policy.settings['move_sampling'] = True
        agent = AzaleaAgent(game_factory, policy=policy, device=str(device))
        worker = DistributedSelfPlay(
            _TrainingPlayer(Player(None, [agent], num_games=num_games, seed=seed & 0x7fffffff,
                                   device=device, rank=rank, world_size=world), policy.net),
            policy.net)
        served = worker.serve()
        logging.info(f'rank {rank}: served {served} replay refills')
        return ''

    # initialize replay buffer with random policy
    if replaybuf is None:
        replaybuf = initialize_replay_buffer(None, game_factory, config['replaybuf_size'],
                                             num_games=num_games, device=device, seed=seed)

    optimizer = optim.SGD(policy.net.parameters(),
                          lr=config['lr_initial'],
                          momentum=config['momentum'],
                          weight_decay=config['l2_regularization'])
    steps_per_epoch = max(1, len(replaybuf) // batch_size)
    if 'total_steps' in config:
        total_steps = int(config['total_steps'])
    else:
        total_steps = int(config['total_epochs']) * steps_per_epoch
    if max_steps is not None:
        total_steps = min(total_steps, int(max_steps))
    if 'lr_decay_steps' in config:
        decay_steps = int(config['lr_decay_steps'])
    else:
        decay_steps = int(config['lr_decay_epochs']) * steps_per_epoch
    scheduler = lr_scheduler.StepLR(optimizer, step_size=max(1, decay_steps),
                                    gamma=config['lr_decay'])

    policy.net.to(device)
    policy.net.train()
    policy.settings['move_exploration'] = True
    policy.settings['move_sampling'] = True

    # instantiate game and wrap it together with policy
    agent = AzaleaAgent(game_factory, policy=policy, device=str(device))
    player = _TrainingPlayer(Player(None, [agent], num_games=num_games, seed=seed & 0x7fffffff,
                                    device=device, rank=rank, world_size=world), policy.net)
    if dist:
        player = DistributedSelfPlay(player, policy.net)
    sampler = torch.Generator(device=device)
    sampler.manual_seed(seed)
    reflect = bool(config.get('random_reflect', False))

    log_interval = config.get('log_interval', 0)
    ckpt_interval = config.get('model_checkpoint_interval', 0)
    loss = 0.0
    start_time = time.time()
    history = []
    for step in range(total_steps):
        batch = replaybuf.sample(batch_size, generator=sampler, reflect=reflect)
        batch = game_class.random_reflect(batch)
        output, loss_ = supervised_step(policy.net, batch, train=True,
                                        optimizer=optimizer, device=device)
        scheduler.step()
        loss += loss_
        history.append(dict(loss=loss_, value_loss=output['value_loss'],
                            moves_loss=output['moves_loss'],
                            lr=optimizer.param_groups[0]['lr']))

        # update replay buffer
        metrics = replaybuf.consume(batch_size / oversampling, player)
        if metrics:
            history[-1]['selfplay_games'] = metrics.get('games', 0)

        if log_interval and step % log_interval == 0:
            sps = log_interval / max(1e-9, time.time() - start_time)
            logging.info(f'step {step} loss {loss / log_interval:.4f} steps/sec {sps:.2f}')
            loss = 0.0
            start_time = time.time()

        if ckpt_interval and step % ckpt_interval == 0:
            save_checkpoint(policy, f'{rundir}/checkpoints/checkpoint.{step}',
                            optimizer=optimizer)

    player.stop()
    policy.net.eval()
    path = save_checkpoint(policy, f'{rundir}/checkpoints/final')
    train.history = history         # last run's scalars (the reference sends them to tensorboard)
    return path


def supervised_step(model, batch, *, train=False, optimizer=None, device='cpu'):
    """Process one batch (policy_trainer.py:123-142)."""
    if train:
        model.train()
    else:
        model.eval()
    with torch.set_grad_enabled(train):
        if train:
            optimizer.zero_grad()
        for k in batch:
            batch[k] = batch[k].to(device)
        output, loss = model.run(batch, compute_loss=True)
        if train:
            loss.backward()
            optimizer.step()
    return output, loss.item()


def initialize_replay_buffer(pool, game_factory: Callable, size: int, *,
                             num_games: int = 1024, device=None, seed: int = 0) \
        -> DeviceReplayBuffer:
    """Fill a fresh replay buffer with random-policy games
    (policy_trainer.py:145-158); ``pool`` is accepted and ignored."""
    agent = AzaleaAgent(game_factory)                   # RandomPolicy
    player = Player(pool, [agent], num_games=num_games, seed=seed & 0x7fffffff, device=device)
    rows, metrics = player.read_device(size)
    player.stop()
    buf = DeviceReplayBuffer(size, agent.game.board_size, device=rows.device)
    buf.put(rows[:size])
    # ReplayBuffer(examples) starts with fresh_counter = 0 (replay_buffer.py:118):
    # the initial rows do not count as fresh, so consume() asks the player for new
    # self-play from the first training step on
    buf.fresh_counter = 0
    logging.info(f'replaybuf initialized with {metrics["games"]} games '
                 f'and {len(buf)} examples')
    return buf


def save_checkpoint(policy, name, *, optimizer=None, replaybuf=None) -> str:
    """Save model (and replay buffer) checkpoint (policy_trainer.py:161-181)."""
    state: Dict = {'policy': policy.state_dict()}
    if optimizer:
        state['optimizer'] = optimizer.state_dict()
    path = f'{name}.policy.pth'
    torch.save(state, path)
    logging.info(f'saved policy checkpoint to {path}')
    if replaybuf is not None:
        rpath = f'{name}.replaybuf.pth'
        torch.save(replaybuf.state_dict(), rpath)
        logging.info(f'saved replay buffer checkpoint to {rpath}')
    return path
