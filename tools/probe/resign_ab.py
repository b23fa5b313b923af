"""A/B of resignation on the flagship step: 4096 games of 11x11 self-play with the 6x64 network in
the loop (bench.py's search settings with root noise, packed leaves, two streams, CUDA graph), one
LockstepSelfPlay with resignation off and one per threshold (default -0.95, -0.8, -0.5, each with
resign_disable_prob=0.1), timed in alternating rounds in one process so that all see the same box.
Each arm is prerolled 110 random plies first (nobody resigns there), so the timed window is the
steady state with games ending and restarting, not the opening.  Prints per arm moves/s, finished
games/s, plies per finished game, the resigned share of finished games, the calibration games'
false-positive rate and simulations/s, with the card's name and power limit.

    python tools/probe/resign_ab.py [--games 4096] [--rounds 4] [--moves 10] [--thresholds ...]
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
KEYS = ('simulations', 'plies', 'games')
RS_KEYS = ('resigned_games', 'calibration_games', 'false_positives')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--games', type=int, default=4096)
    ap.add_argument('--board', type=int, default=11)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--moves', type=int, default=10, help='timed moves per arm and round')
    ap.add_argument('--thresholds', type=float, nargs='+', default=[-0.95, -0.8, -0.5])
    ap.add_argument('--disable-prob', type=float, default=0.1)
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
    settings = [('off', None)] + [(f'{t:+.2f}', t) for t in args.thresholds]
    # every arm resident at once: they share 45 % of the free memory for their node pools
    npg = default_nodes_per_game(G, nn, per_move, dev, memory_fraction=0.45 / len(settings))
    arms = {}
    for name, thr in settings:
        sp = LockstepSelfPlay(net, num_games=G, board_size=args.board, seed=1, device=dev,
                              cuda_graph=True, collect_replay=False, nodes_per_game=npg,
                              resign_threshold=thr, resign_disable_prob=args.disable_prob, **SEARCH)
        sp.preroll(110)
        for _ in range(3):                      # two eager moves, then the graph is captured
            sp.step_move()
        arms[name] = sp
    torch.cuda.synchronize(dev)
    totals = {name: dict(ms=0.0, **{k: 0 for k in KEYS + RS_KEYS}) for name in arms}
    for r in range(args.rounds):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for name in order:
            sp = arms[name]
            c0, s0 = sp.counters(), sp.resign_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.moves):
                sp.step_move()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            c1, s1 = sp.counters(), sp.resign_stats()
            d = {k: c1[k] - c0[k] for k in KEYS}
            d.update({k: s1[k] - s0[k] for k in RS_KEYS})
            t = totals[name]
            t['ms'] += ms
            for k in KEYS + RS_KEYS:
                t[k] += d[k]
            s = ms * 1e-3
            print(f'round {r} {name:5s}: {d["plies"] / s:.4e} moves/s, {d["games"] / s:.1f} games/s, '
                  f'{d["simulations"] / s:.4e} simulations/s ({ms / args.moves:.2f} ms/move)', flush=True)
    for name, t in totals.items():
        s = t['ms'] * 1e-3
        fp = t['false_positives'] / t['calibration_games'] if t['calibration_games'] else float('nan')
        print(f'{name:5s} overall: {t["plies"] / s:.4e} moves/s, {t["games"] / s:.1f} games/s, '
              f'{t["plies"] / max(t["games"], 1):.1f} plies per finished game, '
              f'resigned {t["resigned_games"] / max(t["games"], 1):.3f} of {t["games"]} games, '
              f'false positives {t["false_positives"]} of {t["calibration_games"]} calibration games '
              f'({fp:.3f}), {t["simulations"] / s:.4e} simulations/s', flush=True)
    off = totals['off']
    for name, t in totals.items():
        if name == 'off':
            continue
        print(f'{name} / off: ' + ', '.join(f'{k} {t[k] / t["ms"] / (off[k] / off["ms"]):.3f}'
                                            for k in ('plies', 'games', 'simulations')), flush=True)


if __name__ == '__main__':
    main()
