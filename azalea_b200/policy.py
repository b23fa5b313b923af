"""``Policy`` with the reference's interface (azalea/policy.py:21-208).

Search runs on the GPU through ``SearchTree``; everything the reference's
callers rely on is kept: the attribute names, ``settings``, ``initialize``
with the reference's config keys, ``state_dict`` / ``load_state_dict`` /
``load`` with the reference's checkpoint format (the shipped
``hex11-20180712-3362.policy.pth`` loads), and the host ``RandomState`` that
draws the move, so seeded deterministic play reproduces the reference's.

``random_reflect`` (config key, default off) shows every position the network
evaluates in a random one of Hex's two rule-preserving orientations (the
180-degree rotation), in the search and in training.  It is saved with the
policy; checkpoints without the key load with it off.  In
``choose_action`` the orientation coins come from the policy's
``RandomState``, so with it on the sampled moves differ from a run with it off.
"""
from typing import Any, Dict, Optional, Tuple

import numpy as np
import torch

from .search_tree import SearchTree
from .utils import import_and_get


def create_network(network_type, board_size, num_blocks, base_chans):
    # policy.py:12-18: checkpoints and configs name the reference's classes;
    # map them onto this package's network
    if network_type in ('HexNetwork', 'azalea.network.HexNetwork'):
        network_type = 'azalea_b200.network.HexNetwork'
    Net = import_and_get(network_type)
    return Net(board_size=board_size, num_blocks=num_blocks,
               base_chans=base_chans)


class Policy:
    """Game playing policy, combination of MCTS and network."""

    SEARCH_KEYS = ('simulations', 'search_batch_size', 'exploration_coef',
                   'exploration_depth', 'exploration_noise_alpha',
                   'exploration_noise_scale', 'exploration_temperature')
    NET_KEYS = ('network_type', 'board_size', 'num_blocks', 'base_chans')

    def __init__(self):
        # greedy & deterministic inference by default (policy.py:27-31)
        self.settings = {
            'move_sampling': False,
            'move_exploration': False,
        }
        self.rng = np.random.RandomState()
        self.seed()
        self.random_reflect = False

    def initialize(self, config):
        """Initialize policy for training (policy.py:36-63)."""
        device = config['device']
        if device == 'auto':
            device = 'cuda' if torch.cuda.is_available() else 'cpu'
        device = torch.device(device)
        self.net = create_network(config['network'], config['board_size'],
                                  config['num_blocks'], config['base_chans'])
        self.net.to(device)
        self.net.eval()
        self.network_type = config['network']
        self.board_size = config['board_size']
        self.num_blocks = config['num_blocks']
        self.base_chans = config['base_chans']
        self.simulations = config['simulations']
        self.search_batch_size = config['search_batch_size']
        self.exploration_coef = config['exploration_coef']
        self.exploration_depth = config['exploration_depth']
        self.exploration_noise_alpha = config['exploration_noise_alpha']
        self.exploration_noise_scale = config['exploration_noise_scale']
        self.exploration_temperature = config['exploration_temperature']
        self.random_reflect = bool(config.get('random_reflect', False))
        if 'seed' in config:
            self.seed(config['seed'])

    @property
    def net(self):
        try:
            return self._net
        except AttributeError:
            raise RuntimeError('Policy must be initialized or loaded before use')

    @net.setter
    def net(self, net):
        self._net = net

    def reset(self):
        """Start new game (policy.py:72-76)."""
        tree = getattr(self, 'tree', None)
        if tree is not None:
            tree.reset()        # keep the device pool, clear the tree
        else:
            self.tree = SearchTree()
        self.ply = 0

    def seed(self, seed: Optional[int] = None) -> None:
        self.rng.seed(seed)

    def load_state_dict(self, state):
        """Load model state (policy.py:85-111)."""
        for key in self.NET_KEYS:
            setattr(self, key, state[key])
        self.net = create_network(self.network_type, self.board_size,
                                  self.num_blocks, self.base_chans)
        self.net.load_state_dict(state['net'])
        for key in self.SEARCH_KEYS:
            setattr(self, key, state[key])
        self.random_reflect = bool(state.get('random_reflect', False))
        if 'rng' in state:
            self.rng.__setstate__(state['rng'])

    def state_dict(self):
        """(Hyper)parameters only, not the ongoing game (policy.py:113-130)."""
        state = {'net': self.net.state_dict(),
                 'rng': self.rng.__getstate__()}
        for key in self.NET_KEYS + self.SEARCH_KEYS:
            state[key] = getattr(self, key)
        state['random_reflect'] = self.random_reflect
        return state

    def choose_action(self, game) -> Tuple[int, Dict[str, Any]]:
        """Choose next move; can raise SearchTreeFull (policy.py:132-168)."""
        assert not game.state.result

        temperature = 0.0
        noise_scale = 0.0
        if self.settings['move_sampling']:
            temperature = self.exploration_temperature
            if self.settings['move_exploration']:
                noise_scale = self.exploration_noise_scale
        if self.ply >= self.exploration_depth:
            temperature = 0.

        probs, value, metrics = self.tree.search(
            game, self.net,
            temperature=temperature,
            exploration_noise_scale=noise_scale,
            num_simulations=self.simulations,
            batch_size=self.search_batch_size,
            exploration_coef=self.exploration_coef,
            exploration_noise_alpha=self.exploration_noise_alpha,
            random_reflect=self.random_reflect,
            rng=self.rng)
        move_id = np.argmax(self.rng.multinomial(1, probs))
        legal_moves = game.state.legal_moves
        move = legal_moves[move_id]
        info = dict(prob=probs[move_id],
                    value=value,
                    moves=legal_moves,
                    moves_prob=probs,
                    move_id=move_id,
                    metrics=metrics)
        return move, info

    def execute_action(self, move: int, legal_moves: np.ndarray) -> None:
        """Update search tree with own or opponent action (policy.py:170-176)."""
        move_id = legal_moves.tolist().index(move)
        self.tree.move(move_id)
        self.ply += 1

    @classmethod
    def load(cls, path: str, device: Optional[str] = None) -> 'Policy':
        """Create policy and load weights from a reference checkpoint
        (policy.py:181-208)."""
        policy = cls()
        location = None
        if device:
            device = torch.device(device)
            location = device.type
            if location == 'cuda':
                location += f':{device.index or 0}'
        if path.startswith('s3://'):
            import smart_open   # optional, as in the reference
            with smart_open.smart_open(path) as f:
                state = torch.load(f, map_location=location, weights_only=False)
        else:
            state = torch.load(path, map_location=location, weights_only=False)
        policy.load_state_dict(state['policy'])
        policy.net.eval()
        if device:
            policy.net.to(device)
        return policy
