"""The noised root search (k_select<., true>) against the oracle, bit for bit.

The engine draws descent b's Dirichlet vector from a counter: (seed, global
game id, meta[M_PLY], meta[M_SIM] + b).  Engine.noise_sample returns the same
vector for any counter through the same az_dirichlet_noise, so an oracle tree
fed those vectors (oracle/forced.c) must reach the engine's root statistics
exactly: this pins which vector each descent draws, which child each
component lands on, the float64 mix, where noise is mixed (the root of a full
ply only) and which prior forcing reads.  The sampler's law against NumPy's is
test_dirichlet_noise_distribution (test_mcts_gpu.py)."""
import numpy as np
import pytest
import torch

import oracle
from oracle import forced, stubs
from oracle.lockstep import assert_root_matches, bits
from oracle.philox import full_ply, game_ids

gpu = pytest.mark.gpu
M_SIM = 8


# n, G, sims, batch, c, eps, alpha, plies (None: to the end), extra settings
CONFIGS = {
    # k_select<4,true> at production settings; packed leaves, launches alternating over two
    # windows: the counters do not depend on the window
    'n11_production': (11, 64, 200, 10, 0.5, 0.25, 0.03, 8, dict(pack=True, windows=True)),
    # eps = 1: the prior is replaced by the noise outright
    'n11_eps1': (11, 32, 120, 8, 1.25, 1.0, 0.3, 4, {}),
    # alpha = 1: GS rejects about 27 % of its candidates, the retry loop runs constantly; k down to 1
    'n7_alpha1': (7, 128, 60, 6, 0.5, 0.25, 1.0, None, {}),
    # alpha > 1 with a fraction: exponentials added; k < 32 (idle lanes); forcing with noise
    'n5_alpha2.5_forced': (5, 64, 30, 4, 0.5, 0.25, 2.5, None, dict(forced_k=2.0)),
    # integer alpha (no GS draw at all); batch > k, so duplicate leaves
    'n3_alpha2_dup': (3, 64, 20, 16, 2.0, 0.25, 2.0, None, {}),
    # k_select<12,true> with k = 361: all twelve slots
    'n19_k361': (19, 8, 400, 10, 0.5, 0.25, 0.03, 3, {}),
    # k_select<12,true> under the playout cap: fast plies draw nothing, forcing on full plies
    'n13_cap_forced': (13, 16, 100, 8, 0.5, 0.25, 0.03, 8, dict(cap=(0.5, 20), forced_k=2.0)),
}


def _repack(eng, g0, cnt):
    """Packed leaves: move the stub evaluator's slot-indexed rows of the
    window to the packed rows k_select assigned (leaf_info[..][3] >> 10)."""
    info = eng.leaf_info[g0:g0 + cnt].reshape(-1, 4)
    need = (info[:, 0] >= 0) & ((info[:, 1] & 0xff) == 0)
    rows = (info[:, 3] >> 10)[need].long()
    value = eng.value[g0:g0 + cnt].reshape(-1)
    prior = eng.prior[g0:g0 + cnt].reshape(value.shape[0], -1)
    v, p = value[need].clone(), prior[need].clone()
    value[rows] = v
    prior[rows] = p


def _noise(eng, alpha, k, sim0, rows, games):
    """noise[g] = [rows][k]: the vectors of descents sim0[g] .. sim0[g] +
    rows - 1 of each game g in ``games``, grouped by sim0."""
    out = {}
    for s in sorted({int(sim0[g]) for g in games}):
        block = torch.stack([eng.noise_sample(alpha, k, s + i) for i in range(rows)], 1).cpu().numpy()
        for g in games:
            if sim0[g] == s:
                out[g] = block[g]
    return out


def _oracle_search(tree, game, sims, batch, coef, mode, fk, eps, noise, mix=forced.MIX_F64):
    forced.sample_paths_stub_noise(tree, game, sims, batch, coef, mode, fk, eps, noise, mix)
    v, w, p = tree.root_stats()
    return bits(v), bits(w), bits(p), tree.root_node(), tree.num_nodes


def _mutations(noise):
    """Deliberately wrong noise for each game: the self-check of the exact
    comparison."""
    keys = sorted(noise)
    return {
        'descent i + 1': {g: np.roll(noise[g], -1, axis=0) for g in keys},
        'children rolled by one': {g: np.roll(noise[g], 1, axis=1) for g in keys},
        'row 0 for the whole search': {g: np.repeat(noise[g][:1], len(noise[g]), 0) for g in keys},
        'game g + 1': {g: noise[keys[(i + 1) % len(keys)]] for i, g in enumerate(keys)},
    }


@gpu
@pytest.mark.parametrize('name', list(CONFIGS))
def test_noised_search_matches_the_oracle(name):
    """Engine driven like LockstepSelfPlay with tree reuse (select_root,
    num_batches x (select with noise, stub_eval, expand_backup), root_stats,
    play_commit at temperature 0): after every ply each live game's root
    (visits, W, priors, root N/W, node count) equals an oracle tree fed the
    device's own noise vectors, bit for bit.  Oracle trees searched without
    noise along the same moves differ on most noised plies, and at ply 0
    wrong noise (another descent's, another child's, another game's, one
    vector for the whole search) changes the search of most games."""
    from azalea_b200 import Engine
    n, G, sims, batch, coef, eps, alpha, plies, extra = CONFIGS[name]
    mode, seed = stubs.ROUGH, 13
    fk = extra.get('forced_k', 0.0)
    cap = extra.get('cap')
    num_batches = sims // batch + 1
    rows = num_batches * batch
    eng = Engine(G, n, max_batch=batch, seed=seed, nodes_per_game=200_000,
                 pack_leaves=extra.get('pack', False))
    if fk:
        eng.set_forced_playouts(fk, coef)
    if cap:
        fast_sims = cap[1]
        eng.set_playout_cap(cap[0], (fast_sims // batch + 1) * batch)
    halves = [(0, G // 2), (G // 2, G - G // 2)]
    trees = [oracle.Tree(max_nodes=2_000_000) for _ in range(G)]
    plain = [oracle.Tree(max_nodes=2_000_000) for _ in range(G)]
    games = [oracle.Hex(n) for _ in range(G)]
    chosen = torch.zeros(G, 4, dtype=torch.int32, device='cuda')
    done = np.zeros(G, bool)
    compared = noised = differ = fast = 0
    report = {}
    for it in range(plies or n * n):
        if done.all():
            break
        eng.set_window(0, 0)
        gid, ply = game_ids(eng)
        sim0 = eng.meta[:, M_SIM].cpu().numpy().astype(np.int64)
        live = np.flatnonzero(~done)
        k = n * n - int(ply[live[0]])
        full = {g: not cap or bool(full_ply(seed, int(gid[g]), int(ply[g]), cap[0])) for g in live}
        noise = _noise(eng, alpha, k, sim0, rows, [g for g in live if full[g]])
        eng.select_root()
        eng.stub_eval(mode)
        eng.expand_root()
        for b in range(num_batches):
            for g0, cnt in (halves if b % 2 == 0 else halves[::-1]) if extra.get('windows') else [(0, G)]:
                eng.set_window(g0, cnt if extra.get('windows') else 0)
                eng.select(batch, coef, eps, alpha)
                eng.stub_eval(mode)
                if eng.pack_leaves:
                    _repack(eng, g0, cnt)
                eng.expand_backup()
        eng.set_window(0, 0)
        stats = [x.cpu().numpy() for x in eng.root_stats()]
        v, w, p, kk, _, _ = stats
        eng.play_commit(0.0, 0, False, False, False, chosen)
        ch = chosen.cpu().numpy()
        if it == 0:
            # the self-check, on fresh trees: how many searches each kind of wrong noise changes
            def changed(g, bad, mix=forced.MIX_F64):
                out = _oracle_search(oracle.Tree(max_nodes=2_000_000), oracle.Hex(n), sims, batch, coef,
                                     mode, fk, eps, bad, mix)
                return out[:3] != (bits(v[g, :k]), bits(w[g, :k]), bits(p[g, :k]))
            for what, bad in _mutations(noise).items():
                report[what] = sum(changed(g, bad[g]) for g in noise)
            report['fp32 mix'] = sum(changed(g, noise[g], forced.MIX_F32) for g in noise)
            report['fp32 mix with FMA'] = sum(changed(g, noise[g], forced.MIX_F32_FMA) for g in noise)
            report['games'] = len(noise)
        for g in live:
            assert int(kk[g]) == k, (g, int(kk[g]), k)
            g_sims = sims if full[g] else cap[1]
            forced.sample_paths_stub_noise(trees[g], games[g], g_sims, batch, coef, mode, fk if full[g] else 0.0,
                                           eps if full[g] else 0.0, noise.get(g))
            ov = assert_root_matches(stats, g, trees[g], (name, g, int(ply[g]), full[g]))
            ref = _oracle_search(plain[g], games[g], g_sims, batch, coef, mode, fk if full[g] else 0.0, 0.0, None)
            compared += 1
            if full[g]:
                noised += 1
                differ += ref[0] != bits(ov)
            else:
                fast += 1           # (compared above with an oracle search without noise)
            mid = int(ch[g, 1])
            trees[g].move(mid)
            plain[g].move(mid)
            games[g].step(int(ch[g, 0]))
            if ch[g, 2] != 0:
                assert games[g].result() == ch[g, 2]
                done[g] = True
    print('\n%s: %d plies compared, %d noised, %d of them differ from eps = 0, %d fast; '
          'searches changed by wrong noise at ply 0: %s' % (name, compared, noised, differ, fast, report))
    assert (eng.status().cpu().numpy() == 0).all()
    assert noised > 0 and differ > noised // 2, (differ, noised)
    assert fast > 0 if cap else fast == 0
    if name == 'n11_production':
        for what in ('descent i + 1', 'children rolled by one', 'row 0 for the whole search', 'game g + 1'):
            assert report[what] > report['games'] // 2, (what, report)
