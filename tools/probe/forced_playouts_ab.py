"""A/B of forced playouts and policy target pruning on the flagship step: 4096 games of 11x11
self-play with the 6x64 network in the loop (bench.py's search settings with root noise, packed
leaves, two streams, CUDA graph), one LockstepSelfPlay with the setting off and one with
forced_playouts_k = 2, timed in alternating rounds in one process so that both see the same box.
Each arm is prerolled 110 random plies first, so the timed window is the steady state with games
ending and restarting, not the opening.  Prints per arm simulations/s, moves/s and network rows per
move, with the card's name and power limit.  Then, untimed, each arm plays --target-moves more
moves, so that games begun after the preroll finish and flush their rows; over the temperature-1
rows (plies < exploration_depth; the preroll's uniform rows left out) it prints the mean number of
non-zero visit entries and the mean entropy of pi.

    python tools/probe/forced_playouts_ab.py [--games 4096] [--rounds 4] [--moves 10] [--k 2]
                                             [--target-moves 130]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SEARCH = dict(simulations=800, search_batch_size=10, exploration_coef=0.5,
              exploration_depth=15, exploration_noise_alpha=0.03,
              exploration_noise_scale=0.25, exploration_temperature=1.0)
KEYS = ('simulations', 'plies', 'games', 'nn_rows')


def target_stats(rows, n):
    """(rows, non-zero entries, entropy of pi in nats) summed over the temperature-1 rows
    that are not uniform preroll rows."""
    from azalea_b200.engine import decode_replay_rows
    if len(rows) == 0:
        return 0, 0.0, 0.0
    h, _, vis = decode_replay_rows(rows, n)
    cnt, nz, ent = 0, 0.0, 0.0
    for i in np.flatnonzero(h['temperature'] == 1.0):
        v = vis[i, :int(h['num_moves'][i])].astype(np.float64)
        if (v == 1.0).all():
            continue
        pi = v[v > 0] / v.sum()
        cnt += 1
        nz += len(pi)
        ent -= float((pi * np.log(pi)).sum())
    return cnt, nz, ent


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--games', type=int, default=4096)
    ap.add_argument('--board', type=int, default=11)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--moves', type=int, default=10, help='timed moves per arm and round')
    ap.add_argument('--k', type=float, default=2.0)
    ap.add_argument('--target-moves', type=int, default=130,
                    help='untimed moves per arm for the policy-target statistics')
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
    settings = [('off', 0.0), (f'k={args.k:g}', args.k)]
    # both arms resident at once: they share 45 % of the free memory for their node pools
    npg = default_nodes_per_game(G, nn, per_move, dev, memory_fraction=0.45 / len(settings))
    arms = {}
    for name, k in settings:
        sp = LockstepSelfPlay(net, num_games=G, board_size=args.board, seed=1, device=dev,
                              cuda_graph=True, nodes_per_game=npg, forced_playouts_k=k, **SEARCH)
        sp.preroll(110)
        for _ in range(3):                      # two eager moves, then the graph is captured
            sp.step_move()
        sp.harvest()
        arms[name] = sp
    torch.cuda.synchronize(dev)
    totals = {name: dict(ms=0.0, rows=0, nz=0.0, ent=0.0, **{k: 0 for k in KEYS}) for name in arms}
    # (rows are harvested after every window, outside the timing, so the replay output never fills)
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
            sp.harvest()
            t = totals[name]
            t['ms'] += ms
            for k in KEYS:
                t[k] += d[k]
            s = ms * 1e-3
            print(f'round {r} {name:5s}: {d["simulations"] / s:.4e} simulations/s, '
                  f'{d["plies"] / s:.4e} moves/s, {d["nn_rows"] / max(d["plies"], 1):.1f} network rows/move '
                  f'({ms / args.moves:.2f} ms/move)', flush=True)
    for name, sp in arms.items():
        t = totals[name]
        for m in range(args.target_moves):
            sp.step_move()
            if m % 10 == 9 or m == args.target_moves - 1:
                rows, nz, ent = target_stats(sp.harvest(), args.board)
                t['rows'] += rows
                t['nz'] += nz
                t['ent'] += ent
    for name, t in totals.items():
        s = t['ms'] * 1e-3
        print(f'{name:5s} overall: {t["simulations"] / s:.4e} simulations/s, {t["plies"] / s:.4e} moves/s, '
              f'{t["nn_rows"] / max(t["plies"], 1):.1f} network rows/move; temperature-1 rows: {t["rows"]}, '
              f'non-zero visit entries {t["nz"] / max(t["rows"], 1):.2f}, '
              f'pi entropy {t["ent"] / max(t["rows"], 1):.3f} nats', flush=True)
    off = totals['off']
    for name, t in totals.items():
        if name != 'off':
            print(f'{name} / off: ' + ', '.join(f'{k} {t[k] / t["ms"] / (off[k] / off["ms"]):.3f}'
                                                for k in ('simulations', 'plies')), flush=True)


if __name__ == '__main__':
    main()
