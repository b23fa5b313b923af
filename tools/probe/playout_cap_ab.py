"""A/B of playout cap randomization on the flagship step: 4096 games of 11x11 self-play with the
6x64 network in the loop (bench.py's search settings with root noise, packed leaves, two streams,
CUDA graph), one LockstepSelfPlay with the cap off and one with full_search_prob=0.25,
fast_simulations=100, timed in alternating rounds in one process so that both see the same box.
Each arm is prerolled 110 random plies first, so the timed window is the steady state with games
ending and restarting, not the opening.  Prints per arm simulations/s, moves/s, finished games/s,
full-search plies/s (the training rows: plies - fast_plies) and network rows per move, with the
card's name and power limit.

    python tools/probe/playout_cap_ab.py [--games 4096] [--rounds 4] [--moves 10]
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
KEYS = ('simulations', 'plies', 'games', 'fast_plies', 'nn_rows')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--games', type=int, default=4096)
    ap.add_argument('--board', type=int, default=11)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--moves', type=int, default=10, help='timed moves per arm and round')
    ap.add_argument('--full-search-prob', type=float, default=0.25)
    ap.add_argument('--fast-simulations', type=int, default=100)
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
    for name, cap in (('off', {}), ('on', dict(full_search_prob=args.full_search_prob,
                                               fast_simulations=args.fast_simulations))):
        sp = LockstepSelfPlay(net, num_games=G, board_size=args.board, seed=1, device=dev,
                              cuda_graph=True, collect_replay=False, nodes_per_game=npg,
                              **SEARCH, **cap)
        sp.preroll(110)
        for _ in range(3):                      # two eager moves, then the graph is captured
            sp.step_move()
        arms[name] = sp
    torch.cuda.synchronize(dev)
    totals = {name: dict(ms=0.0, **{k: 0 for k in KEYS}) for name in arms}
    for r in range(args.rounds):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for name in order:
            sp = arms[name]
            c0 = sp.counters()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.moves):
                sp.step_move()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            c1 = sp.counters()
            d = {k: c1[k] - c0[k] for k in KEYS}
            t = totals[name]
            t['ms'] += ms
            for k in KEYS:
                t[k] += d[k]
            s = ms * 1e-3
            print(f'round {r} {name:3s}: {d["simulations"] / s:.4e} simulations/s, '
                  f'{d["plies"] / s:.4e} moves/s, {d["games"] / s:.1f} games/s, '
                  f'{(d["plies"] - d["fast_plies"]) / s:.4e} full-search plies/s '
                  f'({ms / args.moves:.2f} ms/move)', flush=True)
    for name, t in totals.items():
        s = t['ms'] * 1e-3
        print(f'{name:3s} overall: {t["simulations"] / s:.4e} simulations/s, {t["plies"] / s:.4e} moves/s, '
              f'{t["games"] / s:.1f} games/s, {(t["plies"] - t["fast_plies"]) / s:.4e} full-search plies/s, '
              f'{t["nn_rows"] / max(t["plies"], 1):.1f} network rows per move '
              f'(fast plies {t["fast_plies"]} of {t["plies"]})', flush=True)
    off, on = totals['off'], totals['on']

    def rate(t, k):
        return (t['plies'] - t['fast_plies'] if k == 'full' else t[k]) / t['ms']
    print('on / off: ' + ', '.join(f'{k} {rate(on, k) / rate(off, k):.3f}'
                                   for k in ('simulations', 'plies', 'games', 'full')) +
          f', network rows per move {on["nn_rows"] / on["plies"] / (off["nn_rows"] / off["plies"]):.3f}',
          flush=True)


if __name__ == '__main__':
    main()
