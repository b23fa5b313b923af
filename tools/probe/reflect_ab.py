"""A/B of random_reflect on the flagship step: 4096 games of 11x11 self-play with the 6x64
network in the loop (bench.py's search settings, packed leaves, two streams, CUDA graph), one
LockstepSelfPlay with the setting off and one with it on, timed in alternating rounds in one
process so that both see the same box.  Prints simulations/s per round and arm, with the card's
name and power limit.

    python tools/probe/reflect_ab.py [--games 4096] [--rounds 4] [--moves 5]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SEARCH = dict(simulations=800, search_batch_size=10, exploration_coef=0.5,
              exploration_depth=15, exploration_noise_alpha=0.03,
              exploration_noise_scale=0.25, exploration_temperature=1.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--games', type=int, default=4096)
    ap.add_argument('--board', type=int, default=11)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--moves', type=int, default=5, help='timed moves per arm and round')
    args = ap.parse_args()
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.network import HexNetwork
    from azalea_b200.selfplay import default_nodes_per_game
    assert torch.cuda.is_available(), 'needs a GPU'
    dev = torch.device('cuda', 0)
    smi = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                          '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    print(f'card: {torch.cuda.get_device_name(dev)} | nvidia-smi: {smi}', flush=True)
    torch.manual_seed(0)
    net = HexNetwork(args.board, 6, 64).eval().to(dev)
    net.prepare_inference(torch.bfloat16)
    G, nn = args.games, args.board ** 2
    per_move = (SEARCH['simulations'] // SEARCH['search_batch_size'] + 1) * SEARCH['search_batch_size']
    # both arms resident at once: each gets a fifth of the free memory for its node pools
    npg = default_nodes_per_game(G, nn, per_move, dev, memory_fraction=0.2)
    arms = {}
    for name, reflect in (('off', False), ('on', True)):
        arms[name] = LockstepSelfPlay(net, num_games=G, board_size=args.board, seed=1, device=dev,
                                      cuda_graph=True, collect_replay=False, nodes_per_game=npg,
                                      random_reflect=reflect, **SEARCH)
        for _ in range(3):                      # two eager moves, then the graph is captured
            arms[name].step_move()
    torch.cuda.synchronize(dev)
    totals = {name: [0.0, 0] for name in arms}
    for r in range(args.rounds):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for name in order:
            sp = arms[name]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.moves):
                sp.step_move()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            sims = G * per_move * args.moves
            totals[name][0] += ms
            totals[name][1] += sims
            print(f'round {r} {name:3s}: {sims / (ms * 1e-3):.4e} simulations/s '
                  f'({ms / args.moves:.2f} ms/move)', flush=True)
    for name, sp in arms.items():
        ms, sims = totals[name]
        cnt = sp.counters()
        print(f'{name:3s} overall: {sims / (ms * 1e-3):.4e} simulations/s; rows rotated '
              f'{cnt["reflected_rows"]} of {cnt["nn_rows"]} search rows', flush=True)
    off = totals['off'][1] / totals['off'][0]
    on = totals['on'][1] / totals['on'][0]
    print(f'on / off: {on / off:.4f}', flush=True)


if __name__ == '__main__':
    main()
