#!/usr/bin/env python
"""Benchmark of the self-play search hot path (BASELINE.json metric:
MCTS simulations/sec and self-play moves/sec, Hex 11x11).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One *step* = one lockstep move of every resident game: evaluate_root +
81 x (select, evaluate, expand/backup) + move commit = 810 root-to-leaf
descents per game (mcts.py:268).  Default workload = BASELINE.json
configs[1]: 4096 concurrent games per GPU, 6x64 resnet random-init in bf16,
self-play settings (temperature sampling + Dirichlet root noise), search
parameters of config/hex11_train_config.yml.  Games shard by index over
ranks (no collective on the path): scaling is weak.

Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = 'mcts_simulations_per_sec'
UNIT = 'simulations/s'
SEARCH = dict(simulations=800, search_batch_size=10, exploration_coef=0.5,
              exploration_depth=15, exploration_noise_alpha=0.03,
              exploration_noise_scale=0.25, exploration_temperature=1.0)
NN_FLOP_PER_LEAF = {11: 107.852e6, 19: 322.466e6}     # SURVEY 8d


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=4)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=('ours', 'reference'))
    ap.add_argument('--games', type=int, default=4096, help='games per GPU')
    ap.add_argument('--board', type=int, default=11)
    ap.add_argument('--evaluator', default='net', choices=('net', 'stub'))
    ap.add_argument('--stub-mode', type=int, default=2)
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-games', type=int, default=0)
    ap.add_argument('--skip-tree-only', action='store_true')
    ap.add_argument('--sims', type=int, default=800, help='simulations per move')
    ap.add_argument('--nodes-per-game', type=int, default=0)
    ap.add_argument('--streams', type=int, default=2,
                    help='windows of the games driven on separate streams (network evaluator; DESIGN.md 5)')
    ap.add_argument('--pack-leaves', type=int, default=1,
                    help='1: the evaluator runs on the packed unique non-terminal leaves (default); '
                         '0: on every leaf slot (A/B)')
    ap.add_argument('--preroll', type=int, default=110,
                    help='stagger the games before the steady-state window: slot g is advanced by '
                         'g * PREROLL / G random plies (0 = time the opening only)')
    ap.add_argument('--skip-configs', action='store_true',
                    help='skip the config 1 / 4 / 5 legs (BASELINE.json configs[0], [3], [4])')
    ap.add_argument('--c5-games', type=int, default=512)
    ap.add_argument('--c5-sims', type=int, default=4000)
    ap.add_argument('--c4-rounds', type=int, default=64, help='tournament rounds per GPU')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="write what the last timed end-to-end step returned (rank 0's chosen "
                         'moves and the replay rows of the games it finished) as DIR/<name>.npy; '
                         'git ignores bench_outputs/')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    SEARCH['simulations'] = args.sims
    return args


def workload_name(args):
    ev = '6x64 resnet random-init bf16' if args.evaluator == 'net' \
        else f'stub evaluator mode {args.stub_mode}'
    return (f'Hex {args.board}x{args.board} lockstep self-play, {args.games} '
            f'concurrent games/GPU, {ev}, {args.sims} sims batch 10')


def shared_config(args):
    """`config` of the JSON line: identical for both arms (--impl ours / reference)."""
    per_move = (args.sims // SEARCH['search_batch_size'] + 1) * SEARCH['search_batch_size']
    return {'workload': workload_name(args), 'board_size': args.board,
            'games_per_gpu': args.games, 'sims_per_move': per_move, **SEARCH}


# ------------------------------------------------------------------ clocks --

class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(
                    ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                     '--format=csv,noheader,nounits'], capture_output=True,
                    text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unsampled']}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                 'sw_power_cap')
        reasons = [nm for i, nm in enumerate(names)
                   if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.rows[0][1]),
                'power_w_max': max(float(r[2]) for r in self.rows),
                'samples': len(self.rows), 'reasons': reasons}


# ---------------------------------------------------------- CPU baseline ----

def cpu_selfplay_sample(board, evaluator, stub_mode, games, moves, threads):
    """The oracle (C port of the reference's search + rules) timed on host
    cores on a bounded sample of the workload: `games` whole-tree searches
    advanced `moves` plies.  With the network evaluator the leaves of all
    sampled games are batched into one fp32 PyTorch-CPU forward per search
    batch (the reference evaluates <= 10 leaves per call; batching across
    games only helps the baseline)."""
    import oracle
    sims, batch, coef = SEARCH['simulations'], SEARCH['search_batch_size'], \
        SEARCH['exploration_coef']
    per_move = (sims // batch + 1) * batch
    if evaluator == 'stub':
        t0 = time.time()
        # whole games on C threads; bounded by the number of games
        r = oracle.bench_selfplay_stub(n=board, num_games=games, threads=threads,
                                       num_simulations=sims, batch_size=batch,
                                       coef=coef, stub_mode=stub_mode,
                                       exploration_depth=SEARCH['exploration_depth'],
                                       max_nodes=10_000_000, seed=1)
        secs = r['seconds']
        return dict(sims=r['simulations'], plies=r['plies'], seconds=secs,
                    sample=f'{games} whole games, {r["plies"]} plies, '
                           f'{threads} C threads, stub evaluator')
    import torch
    from azalea_b200.network import HexNetwork
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    net = HexNetwork(board, 6, 64).eval()
    nn = board * board
    hexes = [oracle.Hex(board) for _ in range(games)]
    trees = [oracle.Tree(max_nodes=2_000_000) for _ in range(games)]
    rng = np.random.RandomState(0)

    def evaluate(all_leaves):
        rows = [(g, i) for g, lv in enumerate(all_leaves)
                for i, leaf in enumerate(lv) if not leaf['result']]
        value = [np.zeros(len(lv), np.float32) for lv in all_leaves]
        prior = [np.zeros((len(lv), nn), np.float32) for lv in all_leaves]
        if rows:
            boards = np.stack([all_leaves[g][i]['board'] for g, i in rows])
            K = max(len(all_leaves[g][i]['legal_moves']) for g, i in rows)
            moves_ = np.zeros((len(rows), K), np.int32)
            for r, (g, i) in enumerate(rows):
                lm = all_leaves[g][i]['legal_moves']
                moves_[r, :len(lm)] = lm
            with torch.no_grad():
                out = net.run(dict(board=torch.from_numpy(boards),
                                   legal_moves=torch.from_numpy(moves_)))
            v = out['value'].numpy()
            p = np.exp(out['moves_logprob'].numpy())
            for r, (g, i) in enumerate(rows):
                value[g][i] = v[r]
                prior[g][i, :K] = p[r]
        return value, prior

    def one_move():
        need = [g for g in range(games) if not trees[g].root_evaluated()]
        if need:
            leaves = [trees[g].root_leaf(hexes[g]) for g in need]
            _, prior = evaluate(leaves)
            for j, g in enumerate(need):
                trees[g].expand_root(prior[j][0])
        for _ in range(sims // batch + 1):
            # select for all games, one network call, expand/backup for all
            leaves = [trees[g].select_batch(hexes[g], batch, coef)
                      for g in range(games)]
            value, prior = evaluate(leaves)
            for g in range(games):
                trees[g].expand_backup(value[g], prior[g])
        for g in range(games):
            v, _, _ = trees[g].root_stats()
            mid = int(rng.choice(len(v), p=v / v.sum()))
            mv = hexes[g].legal_moves()[mid]
            trees[g].move(mid)
            hexes[g].step(int(mv))
            if hexes[g].result():
                hexes[g] = oracle.Hex(board)
                trees[g].reset()

    one_move()      # warm-up (allocations, torch thread pool)
    t0 = time.time()
    for _ in range(moves):
        one_move()
    secs = time.time() - t0
    return dict(sims=games * moves * per_move, plies=games * moves, seconds=secs,
                sample=f'{games} games x {moves} plies, C oracle tree + fp32 '
                       f'PyTorch-CPU 6x64 net ({threads} threads), leaves of all '
                       f'sampled games batched per search batch')


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path.
    The Python/Numba reference does not travel to the GPU box, so this is the
    oracle port (kind = 'port'), on all host cores."""
    cores = os.cpu_count() or 1
    threads = max(1, cores)
    games = args.cpu_games or (4 * threads if args.evaluator == 'net'
                               else 16 * threads)
    tot_sims = tot_plies = 0
    tot_secs = 0.0
    sample = ''
    for step in range(args.warmup + args.steps):
        if args.evaluator == 'net':
            r = cpu_selfplay_sample(args.board, 'net', args.stub_mode, games, 1, threads)
        else:
            r = cpu_selfplay_sample(args.board, 'stub', args.stub_mode, games, 0, threads)
        if step >= args.warmup:
            tot_sims += r['sims']
            tot_plies += r['plies']
            tot_secs += r['seconds']
            sample = r['sample']
        if args.evaluator == 'net' and step >= 1 and tot_secs > 240:
            break
    value = tot_sims / tot_secs
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * tot_secs / max(1, args.steps),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': shared_config(args),
        'moves_per_sec': tot_plies / tot_secs,
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads,
                         'kind': 'port', 'sample': sample, **reference_python_figures()},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
    }
    print_json(line)


# ------------------------------------------------------------------ ours ----

def select_bytes(d, n):
    """Algorithmic bytes of the select kernel from device counters, with the
    reference's field widths (SURVEY 8d): per level 12 B per child (N, W, P)
    + 8 B node link; virtual loss apply + undo 2 x (8 R + 8 W) per level;
    root masks 2 x ceil(n^2/32) x 4 B per descent; 4 B path entry per level."""
    nw = (n * n + 31) // 32
    return (12 * d['sum_children'] + 8 * d['sum_depth'] + 32 * d['sum_depth']
            + 8 * nw * d['simulations'] + 4 * d['sum_depth'])


def timed_steps(sp, steps, barrier, world, dev):
    """K lockstep moves bracketed by barrier + synchronize; device time by CUDA
    events on the launching stream, max over ranks.  Returns (ms, counter deltas)."""
    import torch
    import torch.distributed as dist
    c0 = sp.counters()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        sp.step_move()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    c1 = sp.counters()
    return ms, {k: c1[k] - c0[k] for k in c1}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from azalea_b200 import LockstepSelfPlay, StubEvaluator
    from azalea_b200.network import HexNetwork

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a GPU (no CPU fallback); '
                           'use --impl reference for the CPU baseline')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured' if 'hbm_gbs' in peaks else 'fallback'
    # kernels timed inside a long step: the sustained (power-capped) tensor figure
    bf16_peak = float(peaks.get('bf16_tflops_sustained', 1400.0))

    if args.evaluator == 'net':
        torch.manual_seed(0)
        evaluator = HexNetwork(args.board, 6, 64).eval().to(dev)
        evaluator.prepare_inference(torch.bfloat16)
    else:
        evaluator = StubEvaluator(args.stub_mode)
    sp = LockstepSelfPlay(evaluator, num_games=args.games, board_size=args.board,
                          seed=0xBAD5EED5, rank=rank, world_size=world,
                          device=dev, cuda_graph=not args.no_graph,
                          collect_replay=True,
                          streams=args.streams if args.evaluator == 'net' else 1,
                          nodes_per_game=args.nodes_per_game or None,
                          pack_leaves=bool(args.pack_leaves) and args.evaluator == 'net', **SEARCH)
    G, per_move = args.games, sp.sims_per_move
    n_streams = sp.streams
    steps = args.steps

    # ---- warm-up (also captures the CUDA graph) ----
    for _ in range(max(3, args.warmup)):
        sp.step_move()
    barrier()

    # ---- timed region 0: the opening (every game at the same early ply) ----
    opening = None
    with ClockSampler(local) as clk:
        if args.preroll > 0:
            ms0, d0 = timed_steps(sp, steps, barrier, world, dev)
            opening = {'value': world * G * per_move * steps / (ms0 * 1e-3), 'unit': UNIT,
                       'ms_per_step': ms0 / steps,
                       'mean_depth': d0['sum_depth'] / max(1, d0['simulations']),
                       'note': 'plies %d..%d of games started together from empty boards'
                               % (max(3, args.warmup), max(3, args.warmup) + steps)}
            # ---- stagger the games, then let the trees fill again ----
            sp.preroll(args.preroll)
            for _ in range(2):
                sp.step_move()
            barrier()
        # ---- timed region 1: device-resident steady state, K steps ----
        ms, d_run = timed_steps(sp, steps, barrier, world, dev)
    total_sims = world * G * per_move * steps
    value = total_sims / (ms * 1e-3)
    moves_per_sec = world * G * steps / (ms * 1e-3)

    # ---- timed region 2: end to end through the host-facing call ----
    # per step: new evaluator weights arrive from pinned host memory (the
    # trainer's hand-off; the reference pickles the whole agent per game,
    # parallel_player.py:36-38), the move runs, and the step's results --
    # every game's (move, move_id, result, ply) and the replay rows of the
    # games that finished -- are read back to the host (gathered to rank 0).
    h2d = d2h = 0
    if args.evaluator == 'net':
        host_w = [p.detach().float().cpu().pin_memory() for p in evaluator.parameters()]
        h2d_step = sum(w.numel() * 4 for w in host_w)
    else:
        host_w, h2d_step = [], 0
    chosen_host = torch.zeros(G, 4, dtype=torch.int32).pin_memory()
    # untimed: first use sets up the exchange (NCCL communicator / the pinned row buffer)
    sp.harvest_end(sp.harvest_begin(gather=world > 1))
    barrier()
    def upload():
        # the trainer's hand-off: weights from pinned host memory, inference tensors rebuilt
        if host_w:
            with torch.no_grad():
                for p, w in zip(evaluator.parameters(), host_w):
                    p.copy_(w, non_blocking=True)
            evaluator.prepare_inference(torch.bfloat16)
        return h2d_step

    # The host loop is software-pipelined (every step still has its own upload and its own
    # read-back inside the timed region): step k+1's weights are enqueued behind step k, so the
    # host's launches run while the GPU plays step k; after the one sync on step k's row count the
    # rows' copy, the clear and step k+1 are enqueued, and the rows are sorted under step k+1.
    dbg = os.environ.get('AZ_BENCH_E2E_DEBUG')

    def e2e_loop(nsteps):
        rows_out = up = down = 0
        up += upload()
        # (events around every move: how much of an end-to-end step is the move itself)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(nsteps)]

        def move(i):
            ev[i][0].record()
            sp.step_move()
            ev[i][1].record()
        move(0)
        for k in range(nsteps):
            c0 = time.perf_counter()
            chosen_host.copy_(sp.chosen, non_blocking=True)
            if k + 1 < nsteps:
                up += upload()
            c1 = time.perf_counter()
            # syncs on the row count(s) only; world > 1: rows of all ranks to rank 0 over NCCL
            handle = sp.harvest_begin(gather=world > 1)
            c2 = time.perf_counter()
            if k + 1 < nsteps:
                move(k + 1)
            c3 = time.perf_counter()
            rows = sp.harvest_end(handle)
            if dbg:
                print('e2e step %d: upload %.2f ms, harvest_begin %.2f, launch %.2f, harvest_end %.2f (host)'
                      % (k, (c1 - c0) * 1e3, (c2 - c1) * 1e3, (c3 - c2) * 1e3,
                         (time.perf_counter() - c3) * 1e3), file=sys.stderr)
            rows_out += len(rows)
            down += chosen_host.numel() * 4 + rows.nbytes + 8
        return rows_out, up, down, ev, rows

    # one untimed pass of the same loop: the first pipelined iteration pays one-off set-up
    # (30 ms of stream time between its two moves, measured) that a long run never sees again
    e2e_loop(2)
    barrier()
    t0 = time.perf_counter()
    rows_out, h2d, d2h, move_ev, last_rows = e2e_loop(steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:
        # chosen_host holds the last step's (move, move_id, result, ply): harvest_end waited for it
        dump_outputs(args.dump_outputs, chosen_host.numpy(), last_rows, args.board)
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = total_sims / e2e_s
    e2e_move_ms = sum(a.elapsed_time(b) for a, b in move_ev) / steps
    # stream time between two moves: the next weights' copies and prepare_inference kernels, the
    # row-count sync, the rows' copy and the graph launch
    if dbg:
        print('e2e gaps between moves (stream ms):',
              [round(move_ev[i][1].elapsed_time(move_ev[i + 1][0]), 2) for i in range(steps - 1)], file=sys.stderr)
    e2e_gap_ms = sum(move_ev[i][1].elapsed_time(move_ev[i + 1][0]) for i in range(steps - 1)) / max(1, steps - 1)

    # ---- kernel leg: per-launch timing of our kernels with CUDA events ----
    eng = sp.eng
    stream = torch.cuda.current_stream()
    sel_ev, exp_ev = [], []
    cs0 = sp.counters()
    sel_ms = exp_ms = 0.0
    conv_ev = None
    if args.evaluator == 'net' and getattr(evaluator, 'tower', None) == 'tcgen05':
        conv_ev = evaluator.conv_events = []
    eng.select_root()
    sp._evaluate(True)
    eng.expand_root(None, 1 if args.evaluator == 'net' else 0)
    for _ in range(sp.num_batches):
        a, b, c, d = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        a.record(stream)
        eng.select(sp.batch, sp.coef, sp.noise_scale, sp.noise_alpha)
        b.record(stream)
        v, p, kind = sp._evaluate(False)
        c.record(stream)
        eng.expand_backup(v, p, kind)
        d.record(stream)
        sel_ev.append((a, b))
        exp_ev.append((c, d))
    eng.play_commit(sp.temperature, sp.depth, sp.move_sampling, True, True, sp.chosen)
    torch.cuda.synchronize()
    if conv_ev is not None:
        evaluator.conv_events = None
    sel_ms = sum(a.elapsed_time(b) for a, b in sel_ev)
    exp_ms = sum(a.elapsed_time(b) for a, b in exp_ev)
    cs1 = sp.counters()
    dk = {k: cs1[k] - cs0[k] for k in cs1}
    sel_bytes = select_bytes(dk, args.board)
    launches = sp.num_batches
    sel_avg_ms = sel_ms / launches
    achieved = sel_bytes / launches / (sel_avg_ms * 1e-3) / 1e9
    tj = {}
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
    except Exception:
        pass
    traffic = None
    try:
        key = f'{args.board}x{args.board}/{G}/' + ('noise' if sp.noise_scale else 'nonoise')
        traffic = tj['k_select'][key]['traffic_bytes']
    except Exception:
        pass
    roofline = {
        'kernel': 'k_select', 'bound': 'hbm', 'achieved': achieved,
        'peak': hbm_peak, 'unit': 'GB/s', 'frac': achieved / hbm_peak,
        'traffic': traffic, 'peak_source': peak_src,
        'avg_launch_ms': sel_avg_ms,
        'alg_bytes_per_launch': sel_bytes / launches,
        'alg_bytes_per_sim': sel_bytes / max(1, dk['simulations']),
        'mean_depth': dk['sum_depth'] / max(1, dk['simulations']),
        'mean_children': dk['sum_children'] / max(1, dk['sum_depth']),
        'select_share_of_step': sel_ms / (ms / steps),
        'expand_backup_avg_launch_ms': exp_ms / launches,
        'note': 'latency/occupancy-bound pointer chasing; see DESIGN.md',
    }
    roofline_tree = None
    if conv_ev:
        roofline_tree = roofline
        live_frac = dk['nn_rows'] / (launches * G * sp.batch) if sp.pack_leaves else 1.0
        roofline = tower_roofline(conv_ev, args.board, G * sp.batch, ms / steps, hbm_peak,
                                  bf16_peak, peak_src, 'bf16_tflops_sustained' in peaks, tj, live_frac)
        roofline['rows_per_launch'] = live_frac * G * sp.batch
        roofline['packed_leaves'] = bool(sp.pack_leaves)
    nn_info = None
    if args.evaluator == 'net':
        step_ms = ms / steps
        rows = d_run['nn_rows'] / steps
        # rows the evaluator runs over: every leaf slot, or the packed live rows (+ the roots)
        padded = G * (per_move + 1) if not sp.pack_leaves else rows + G
        flop = NN_FLOP_PER_LEAF.get(args.board)
        if flop:
            nn_ms = step_ms - (sel_ms + exp_ms)
            nn_info = {'useful_rows_per_step': rows, 'padded_rows_per_step': padded,
                       'tflops_padded': padded * flop / (nn_ms * 1e-3) / 1e12,
                       'tflops_useful': rows * flop / (nn_ms * 1e-3) / 1e12,
                       'peak_bf16_tflops_sustained': bf16_peak,
                       'approx_nn_ms_per_step': nn_ms}
    counters_total = sp.counters()
    launches_per_step = sp_launches(args, per_move, evaluator)

    # ---- tree-only figure (stub evaluator) next to the headline ----
    del sp, eng
    torch.cuda.empty_cache()
    tree_only = None
    if args.evaluator == 'net' and not args.skip_tree_only:
        sp2 = LockstepSelfPlay(StubEvaluator(2), num_games=args.games,
                               board_size=args.board, seed=1, rank=rank,
                               world_size=world, device=dev, cuda_graph=True,
                               collect_replay=True,
                               nodes_per_game=args.nodes_per_game or None, **SEARCH)
        for _ in range(3):
            sp2.step_move()
        if args.preroll > 0:
            sp2.preroll(args.preroll)
            for _ in range(2):
                sp2.step_move()
        ms2, d2 = timed_steps(sp2, steps, barrier, world, dev)
        tree_only = {'value': world * G * per_move * steps / (ms2 * 1e-3), 'unit': UNIT,
                     'evaluator': 'device stub (mode 2)', 'ms_per_step': ms2 / steps,
                     'moves_per_sec': world * G * steps / (ms2 * 1e-3),
                     'mean_depth': d2['sum_depth'] / max(1, d2['simulations']),
                     'games_finished_per_step': d2['games'] / steps}
        del sp2
        torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations, same JSON line ----
    config5 = config4 = config1 = None
    if not args.skip_configs:
        config5 = guarded(lambda: bench_config5(args, rank, world, dev, barrier, hbm_peak, bf16_peak))
        torch.cuda.empty_cache()
        config4 = guarded(lambda: bench_config4(args, rank, world, dev, barrier))
        torch.cuda.empty_cache()
        if rank == 0:
            config1 = guarded(lambda: bench_config1(dev))
        barrier()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        # bounded sample, ~10-30 s of CPU work: one ply of 4 games per core with
        # the network, 16 whole games per core with the stub evaluator
        games = args.cpu_games or (4 * cores if args.evaluator == 'net' else 16 * cores)
        r = cpu_selfplay_sample(args.board, args.evaluator, args.stub_mode, games,
                                1, cores)
        cpu_baseline = {'value': r['sims'] / r['seconds'], 'unit': UNIT,
                        'cores': cores, 'kind': 'port', 'sample': r['sample'],
                        'seconds': r['seconds']}
        cpu_baseline.update(reference_python_figures())

    if rank == 0:
        failed = counters_total['games_failed']
        skipped = counters_total['pool_skipped_expansions']
        if failed or skipped:
            print(f'WARNING: {failed} games dropped (tree/pool full), {skipped} expansions '
                  f'skipped on a full pool -- raise --nodes-per-game', file=sys.stderr)
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world,
            'steps': steps, 'warmup': max(3, args.warmup),
            'ms_per_step': ms / steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 tree statistics (bit-exact PUCT); bf16 network'
            if args.evaluator == 'net' else 'f32',
            'data': 'synthetic',
            'config': shared_config(args),
            'run': {'window': ('steady state: game slot g pre-rolled by g*%d/G random plies, so '
                               'games end, restart and reuse subtrees inside the timed steps'
                               % args.preroll) if args.preroll > 0 else 'opening',
                    'l2_policy': 'working set (node pools, > 1 GB) exceeds the 126 MB L2',
                    'cuda_graph': not args.no_graph, 'streams': n_streams,
                    'tower': (('all residual blocks chained in one launch' if evaluator.tower_fused >= 2
                               else 'one fused launch per residual block')
                              if getattr(evaluator, 'tower_fused', 0)
                              and getattr(evaluator, '_fast', {}).get('tower_fused') else 'two launches per block')
                    if args.evaluator == 'net' else None},
            'moves_per_sec': moves_per_sec,
            'clocks': clk.summary(),
            'e2e': {'value': e2e_value, 'unit': UNIT,
                    'h2d_bytes_per_step': h2d // max(1, steps),
                    'd2h_bytes_per_step': d2h // max(1, steps),
                    'ms_per_step': 1e3 * e2e_s / steps,
                    'replay_rows_per_step': rows_out / steps,
                    'move_gpu_ms_per_step': e2e_move_ms, 'between_moves_gpu_ms': e2e_gap_ms,
                    'pipeline': 'weights of step k+1 enqueued behind step k; one sync per step on the row '
                                'count, rows copied to pinned memory and sorted under step k+1'},
            'gpu_launches': steps * launches_per_step,
            'roofline': roofline,
            'roofline_tree': roofline_tree,
            'cpu_baseline': cpu_baseline,
            'tree_only': tree_only,
            'opening': opening,
            'network': nn_info,
            'counters_per_step': {k: v / steps for k, v in d_run.items()},
            'mean_depth': d_run['sum_depth'] / max(1, d_run['simulations']),
            'games_failed_total': failed, 'pool_skipped_expansions_total': skipped,
            'config1': config1, 'config4': config4, 'config5': config5,
        }
        print_json(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, chosen, rows, board):
    """What one end-to-end step hands its caller, as float64 / float32 .npy
    files: per game slot the chosen move, its ordinal among the legal moves,
    the result after it and the new ply (chosen_*.npy); per replay row of the
    games that finished in the step, the header fields (replay_<field>.npy),
    the board before the move (replay_board.npy) and the root's visit counts
    (replay_visits.npy).  Rows are sorted by (game id, ply); if they exceed
    the size limit a fixed seeded sample of them is written."""
    from azalea_b200.engine import decode_replay_rows
    os.makedirs(out_dir, exist_ok=True)
    out = {f'chosen_{f}': chosen[:, i].astype(np.float64)
           for i, f in enumerate(('move', 'move_id', 'result', 'ply'))}
    head, boards, visits = decode_replay_rows(rows, board)
    fields = [f for f in head.dtype.names if f != 'reserved']
    row_bytes = 8 * len(fields) + 4 * boards[0].size + 4 * visits.shape[1] if len(rows) else 1
    cap = (DUMP_BYTES - sum(a.nbytes for a in out.values())) // row_bytes
    keep = np.arange(len(rows))
    if len(rows) > cap:
        keep = np.sort(np.random.RandomState(0).choice(len(rows), cap, replace=False))
    for f in fields:
        out[f'replay_{f}'] = head[f][keep].astype(np.float64)
    out['replay_board'] = boards[keep].astype(np.float32)
    out['replay_visits'] = visits[keep].astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def guarded(fn):
    """A side leg must never cost the headline line."""
    try:
        return fn()
    except Exception as exc:        # noqa: BLE001
        import traceback
        traceback.print_exc()
        return {'error': f'{type(exc).__name__}: {exc}'}


def tower_roofline(conv_ev, board, boards, step_ms, hbm_peak, bf16_peak, peak_src,
                   tensor_measured, tj, live_frac=1.0):
    """Roofline of the step's dominant kernel, the evaluator's tower
    convolutions, from per-launch CUDA events (DESIGN.md 3.5).

    Fused block (k_resblock, one launch per residual block): both
    convolutions from one read and one write of the activations, so the
    kernel is bound by the tensor pipe: useful FLOPs = 2 x 2*64*576 per cell.
    Two-launch path (k_conv3x3): plain launch 2 units of HBM traffic,
    residual launch 3."""
    cell_bytes = board * board * 128
    conv_flop = board * board * 2 * 64 * 576
    # packed leaves: a search batch's launch runs over its live rows only (device-side count);
    # live_frac = rows the network had to evaluate / leaf slots, from the device counters
    kinds = {}
    for e0, e1, kind, nb in conv_ev:
        kinds.setdefault(kind, []).append((e0.elapsed_time(e1), nb * live_frac if nb == boards else nb))
    tot_ms = sum(t for v in kinds.values() for t, _ in v)
    n_launch = sum(len(v) for v in kinds.values())
    units = {'plain': 2, 'residual': 3, 'block': 2}
    convs = {'plain': 1, 'residual': 1, 'block': 2}
    chain = 0
    for k in kinds:
        if k.startswith('chain'):       # 'chainK': K residual blocks chained in one launch
            chain = int(k[5:])
            units[k], convs[k] = 2 * chain, 2 * chain
    cbytes = sum(nb * cell_bytes * units[k] for k, v in kinds.items() for _, nb in v)
    cflop = sum(nb * conv_flop * convs[k] for k, v in kinds.items() for _, nb in v)
    tflops = cflop / (tot_ms * 1e-3) / 1e12
    gbs = cbytes / (tot_ms * 1e-3) / 1e9
    fused = 'block' in kinds or chain > 0
    out = {
        'kernel': 'k_resblock' if fused else 'k_conv3x3',
        'launches_timed': n_launch, 'avg_launch_ms': tot_ms / n_launch,
        'share_of_step': tot_ms / step_ms,
        'useful_tflops': tflops, 'alg_gbs': gbs,
        'alg_bytes_per_launch': cbytes / n_launch, 'alg_flop_per_launch': cflop / n_launch,
        'per_kind_avg_ms': {k: sum(t for t, _ in v) / len(v) for k, v in kinds.items()},
        'hbm_frac': gbs / hbm_peak, 'tensor_frac': tflops / bf16_peak,
        'hbm_peak_gbs': hbm_peak, 'tensor_peak_tflops_sustained': bf16_peak,
        'peak_source': peak_src if tensor_measured else 'fallback',
    }
    key = ('k_resblock' if fused else 'k_conv3x3')
    try:
        ent = tj[key][f'{board}x{board}/{boards}' + (f'/chain{chain}' if chain else '')]
        # the capture is a launch over all `boards` rows; a packed-leaves launch moves live_frac of it
        out['traffic'] = ent['traffic_bytes'] * live_frac
        out['traffic_source'] = ent.get('profile')
    except Exception:
        out['traffic'] = None
    if chain:
        out['blocks_per_launch'] = chain
    if fused:
        out.update(bound='tensor', achieved=tflops, peak=bf16_peak, unit='TFLOP/s',
                   frac=tflops / bf16_peak,
                   note=('the residual tower chained in one launch: ' if chain else 'one launch per residual block: ')
                        + '2 convolutions per block from one read + one write of '
                        'the activations; useful FLOPs exclude the pad cells of the slab layout '
                        '(110 of 128 MMA rows are real cells at 11x11); peak = sustained cuBLAS bf16')
    else:
        out.update(bound='hbm', achieved=gbs, peak=hbm_peak, unit='GB/s', frac=gbs / hbm_peak,
                   note='two launches per residual block: x->y (2 units of traffic, close to the '
                        'tensor ridge) and y,x->x (3 units, on the HBM roofline)')
    return out


def reference_python_figures():
    """The UNMODIFIED Python/Numba reference, timed on the build box by
    tools/measure_reference.py (it cannot travel to the GPU box)."""
    try:
        r = json.load(open(os.path.join(ROOT, 'profiles', 'r02_reference_python.json')))
    except Exception:
        return {}
    out = {'reference_python_sims_per_s': r['one_process']['sims_per_s'],
           'reference_python_s_per_move': r['one_process']['s_per_move'],
           'reference_python_cores': 1,
           'reference_python_box': f"{r['box']} ({r['cores']} cores), stub evaluator, "
                                   'profiles/r02_reference_python.json'}
    if 'process_pool' in r:
        out['reference_python_pool_sims_per_s'] = r['process_pool']['sims_per_s']
        out['reference_python_pool_workers'] = r['process_pool']['workers']
    return out


# ------------------------------------------------- BASELINE.json configs[4] --

def bench_config5(args, rank, world, dev, barrier, hbm_peak, bf16_peak):
    """Hex 19x19 deep-search stress test: many simulations per move, a node
    pool sized for them, 6x64 network.  Every rank runs its own games (weak
    scaling, like the headline)."""
    import torch
    from azalea_b200 import LockstepSelfPlay
    from azalea_b200.network import HexNetwork
    n, G, sims = 19, args.c5_games, args.c5_sims
    torch.manual_seed(0)
    net = HexNetwork(n, 6, 64).eval().to(dev)
    net.prepare_inference(torch.bfloat16)
    search = dict(SEARCH, simulations=sims)
    sp = LockstepSelfPlay(net, num_games=G, board_size=n, seed=0xC0F165, rank=rank,
                          world_size=world, device=dev, cuda_graph=True, collect_replay=True,
                          **search)
    per_move = sp.sims_per_move
    for _ in range(3):
        sp.step_move()
    steps = args.steps
    ms, d = timed_steps(sp, steps, barrier, world, dev)
    # per-launch shares from one eager move
    eng, stream = sp.eng, torch.cuda.current_stream()
    conv_ev = net.conv_events = []
    sel = []
    eng.select_root()
    sp._evaluate(True)
    eng.expand_root(None, 1)
    c0 = sp.counters()
    for _ in range(sp.num_batches):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng.select(sp.batch, sp.coef, sp.noise_scale, sp.noise_alpha)
        b.record(stream)
        sp._evaluate(False)
        eng.expand_backup(None, None, 1)
        sel.append((a, b))
    eng.play_commit(sp.temperature, sp.depth, sp.move_sampling, True, True, sp.chosen)
    torch.cuda.synchronize()
    net.conv_events = None
    c1 = sp.counters()
    dk = {k: c1[k] - c0[k] for k in c1}
    sel_ms = sum(a.elapsed_time(b) for a, b in sel)
    sel_b = select_bytes(dk, n)
    tower = tower_roofline(conv_ev, n, G * sp.batch, ms / steps, hbm_peak, bf16_peak,
                           'measured', True, {})
    tot = sp.counters()
    out = {'workload': f'Hex 19x19 deep search, {G} games/GPU, 6x64 resnet bf16, {sims} sims batch 10',
           'value': world * G * per_move * steps / (ms * 1e-3), 'unit': UNIT,
           'moves_per_sec': world * G * steps / (ms * 1e-3), 'ms_per_step': ms / steps,
           'steps': steps, 'n_gpus': world, 'sims_per_move': per_move,
           'nodes_per_game_half': eng.nodes_per_game,
           'node_pool_gb_per_gpu': G * 2 * eng.nodes_per_game * 16 / 1e9,
           'mean_depth': d['sum_depth'] / max(1, d['simulations']),
           'mean_children': d['sum_children'] / max(1, d['sum_depth']),
           'k_select12': {'avg_launch_ms': sel_ms / sp.num_batches,
                          'alg_gbs': sel_b / (sel_ms * 1e-3) / 1e9,
                          'hbm_frac': sel_b / (sel_ms * 1e-3) / 1e9 / hbm_peak,
                          'share_of_step': sel_ms / (ms / steps)},
           'tower': {k: tower[k] for k in ('kernel', 'avg_launch_ms', 'useful_tflops', 'alg_gbs',
                                           'hbm_frac', 'tensor_frac', 'share_of_step')},
           'games_failed': tot['games_failed'],
           'pool_skipped_expansions': tot['pool_skipped_expansions']}
    del sp, eng
    return out


# ------------------------------------------------- BASELINE.json configs[3] --

def bench_config4(args, rank, world, dev, barrier):
    """Round-robin tournament with compare() semantics (compare_cli.py:57-82,
    evaluation.py:17-80): 4 random-init 6x64 policies + the <random> anchor = 5
    agents, 10 pairs per round, move_sampling on, noise off, two trees per
    game; (round, pair) games dealt round-robin to the ranks, tallies reduced
    to rank 0.  Rounds scale with the world size (weak scaling)."""
    import torch
    import torch.distributed as dist
    import azalea_b200 as az
    from azalea_b200.evaluation import evaluate, reduce_tallies, gen_pairs
    n = args.board
    agents = [az.AzaleaAgent(lambda: az.HexGame(n))]            # <random>, Elo anchor
    for i in range(4):
        torch.manual_seed(i)
        p = az.Policy()
        p.initialize(dict(device=str(dev), network='HexNetwork', board_size=n, num_blocks=6,
                          base_chans=64, simulations=SEARCH['simulations'],
                          search_batch_size=SEARCH['search_batch_size'],
                          exploration_coef=SEARCH['exploration_coef'],
                          exploration_depth=SEARCH['exploration_depth'],
                          exploration_noise_alpha=SEARCH['exploration_noise_alpha'],
                          exploration_noise_scale=SEARCH['exploration_noise_scale'],
                          exploration_temperature=SEARCH['exploration_temperature']))
        a = az.AzaleaAgent(lambda: az.HexGame(n), policy=p)
        a.settings['move_sampling'] = True                      # compare_cli.py:70-71
        agents.append(a)
    rounds = args.c4_rounds * world
    stats = {}
    barrier()
    t0 = time.perf_counter()
    ok, share = 1, None
    try:
        share = evaluate(agents, rounds, rank=rank, world_size=world, reduce=False,
                         device=dev, stats=stats)
    except Exception:       # noqa: BLE001  keep the ranks in step: agree before the collective
        import traceback
        traceback.print_exc()
        ok = 0
    pairs = gen_pairs(len(agents))
    if world > 1:
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = int(flag.item())
    if not ok:
        return {'error': 'a rank failed during the tournament'}
    tally = np.array([share[pr] for pr in pairs], dtype=np.int64)
    work = np.array([stats['plies'], stats['simulations'], len(share) and int(tally.sum())],
                    dtype=np.int64)
    if world > 1:
        tally = reduce_tallies(tally, device=dev)
        t = torch.from_numpy(work).to(dev)
        dist.all_reduce(t)
        work = t.cpu().numpy()
    barrier()
    secs = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([secs], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t.item())
    games = int(work[2])
    return {'workload': f'Hex {n}x{n} round-robin tournament, 4 random-init 6x64 policies + <random>, '
                        f'{rounds} rounds x 10 pairs, 800 sims batch 10, two trees per game',
            'n_gpus': world, 'rounds': rounds, 'games': games, 'seconds': secs,
            'games_per_sec': games / secs, 'moves_per_sec': int(work[0]) / secs,
            'value': int(work[1]) / secs, 'unit': UNIT,
            'sharding': 'task t = round * 10 + pair on rank t % world; [10, 3] tallies reduced to rank 0',
            'timing': 'host wall clock around the whole tournament (eager launches, engines and '
                      'evaluators set up inside), max over ranks',
            'tallies': {f'{a}-{b}': [int(x) for x in tally[s]] for s, (a, b) in enumerate(pairs)}
            if rank == 0 else None,
            'pool_skipped_expansions': stats.get('pool_skipped_expansions')}


# ------------------------------------------------- BASELINE.json configs[0] --

class UniformStubNet:
    """The evaluator plug-in of BASELINE.md section 3: value 0, uniform
    moves_logprob over the legal moves (padding -99, network.py:150), with the
    interface the search calls (mcts.py:203-210)."""

    def __init__(self):
        import torch
        self.device = torch.device('cpu')

    def eval(self):
        return self

    def run(self, batch):
        import torch
        legal = batch['legal_moves']
        logit = torch.where(legal > 0, torch.zeros(legal.shape), torch.full(legal.shape, -99.0))
        return {'value': torch.zeros(len(legal)), 'moves_logprob': torch.log_softmax(logit, dim=1)}


def bench_config1(dev):
    """The single-game drop-in (AzaleaAgent.choose_action / execute_action on a
    1-game engine, evaluator called on the host exactly as the reference calls
    it): latency per move of BASELINE.json config 1, to put beside the
    reference's 0.16-0.25 s/move."""
    import azalea_b200 as az
    p = az.Policy()
    p.net = UniformStubNet()
    p.simulations, p.search_batch_size = SEARCH['simulations'], SEARCH['search_batch_size']
    p.exploration_coef, p.exploration_depth = SEARCH['exploration_coef'], SEARCH['exploration_depth']
    p.exploration_noise_alpha = SEARCH['exploration_noise_alpha']
    p.exploration_noise_scale = SEARCH['exploration_noise_scale']
    p.exploration_temperature = SEARCH['exploration_temperature']
    agent = az.AzaleaAgent(lambda: az.HexGame(11), policy=p)
    agent.settings['move_sampling'] = True
    agent.settings['move_exploration'] = True
    agent.reset()
    agent.seed(1)
    for _ in range(2):
        agent.execute_action(agent.choose_action())
    t0 = time.perf_counter()
    moves = 0
    while moves < 20 and not agent.game.state.result:
        agent.execute_action(agent.choose_action())
        moves += 1
    secs = time.perf_counter() - t0
    per_move = (SEARCH['simulations'] // SEARCH['search_batch_size'] + 1) * SEARCH['search_batch_size']
    out = {'workload': 'Hex 11x11 single game through AzaleaAgent/Policy (drop-in API), uniform stub '
                       'evaluator on the host, 800 sims batch 10, self-play settings',
           'moves': moves, 's_per_move': secs / moves, 'moves_per_sec': moves / secs,
           'value': per_move * moves / secs, 'unit': UNIT,
           'host_copies_per_search_batch': {'d2h': 1, 'h2d': 1, 'syncs': 1}}
    out.update(reference_python_figures())
    return out


def sp_launches(args, per_move, evaluator=None):
    """Kernels of ours per step: select_root, expand_root, commit, and per
    search batch select + expand_backup, plus per evaluation (root + every
    search batch) the stub kernel, or the network's stem + heads kernels and,
    with the tcgen05 tower, two k_conv3x3 per residual block."""
    nb = per_move // SEARCH['search_batch_size']
    per = 3 + 2 * nb
    if args.evaluator == 'stub':
        per += nb + 1
    else:
        own = 2                 # stem, heads
        if getattr(evaluator, 'tower', None) == 'tcgen05':
            own += 1            # tail
            level = int(getattr(evaluator, 'tower_fused', 0)) if evaluator._fast.get('tower_fused') else 0
            nblk = len(evaluator.resblocks)
            own += 2 * nblk if level == 0 else nblk if level == 1 else -(-nblk // 8)
        per += (nb + 1) * own
    return per


def main():
    args = parse_args()
    # libraries (NCCL's version banner) may write to stdout: keep fd 1 for
    # the ONE JSON line and send everything else to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    global print_json

    def print_json(line):
        os.write(json_fd, (json.dumps(line) + '\n').encode())

    if args.impl == 'reference':
        rank = int(os.environ.get('RANK', 0))
        if rank != 0:
            return
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
