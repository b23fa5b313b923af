"""The bf16 evaluator (stem -> residual tower -> heads -> FC GEMM -> tail)
against fp64 references tight enough to see a dropped bias.

Two references, both plain torch in fp64 on the GPU:

* ``emulate``: the tcgen05 arm's arithmetic, rounding to bf16 at exactly
  the points where its kernels round (stem table, slab-stem row sums and
  output, every convolution's output with bf16 weights and fp32 bias, the
  heads, the GEMM output); fp64 everywhere else.  The three tcgen05 tower
  variants are held to it.
* ``reference``: the plain fp64 ``HexNetwork`` (``_trunk`` + ``move_fc``).
  The cuDNN tower, the glue path at 32 and 128 channels and the fp32 path,
  which round at other points, are held to it.

Every bound is about twice the largest error measured on a B200.  For every
board size the test checks that the bugs the bounds are meant to see -- a
dropped or shifted bias, a zeroed block, a transposed board -- move the fp64
outputs by at least MARGIN times the bound in one of the two weight sets, so a
bound cannot be widened until such a bug fits under it.  The glue arms are
exempt: their stem sums nine bf16 taps, and their FC bias and value are bf16,
so their bounds sit too close to the smallest of these bugs.  Stage checks
feed each kernel its predecessor's own output and hold it to one bf16
rounding.
"""
import copy
import ctypes

import pytest
import torch
import torch.nn.functional as F

from azalea_b200 import _cabi, tower_layout as tl
from azalea_b200.network import HexNetwork, _fold

pytestmark = pytest.mark.gpu

BLOCKS = 6
# (max |value - ref|, max |logit - ref|) per arm and weight set; logits are
# compared raw, not up to a per-row constant.  About twice the largest error
# measured on a B200 (1000 W), rounded up; the measured values are in DESIGN 4.
BOUNDS = {
    'chain': {'default': (2e-3, 8e-3), 'loud': (5e-2, 7e-2)},
    'block': {'default': (2e-3, 8e-3), 'loud': (5e-2, 7e-2)},
    'plain': {'default': (2e-3, 8e-3), 'loud': (5e-2, 7e-2)},
    'cudnn': {'default': (4e-3, 2e-2), 'loud': (5e-2, 9e-2)},
    'fp32': {'default': (2e-4, 9e-4), 'loud': (4e-3, 6e-3)},
    'glue32': {'default': (3e-3, 3e-2), 'loud': (5e-2, 2e-1)},
    'glue128': {'default': (4e-3, 2e-2), 'loud': (1e-1, 2e-1)},
}
MARGIN = 4
# largest error seen per (arm, weight set), printed by the end-to-end test
# (pytest -s): what the bounds are calibrated on
OBSERVED = {}


def bf(t):
    """Round to bf16, keep the dtype."""
    return t.to(torch.bfloat16).to(t.dtype)


def bf16_ulp(t):
    """One bf16 ulp of each element of t (fp64), for normal numbers."""
    return torch.exp2(torch.floor(torch.log2(t.abs().clamp_min(2.0 ** -126))) - 7)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def make_net(n, loud, chans=64, blocks=BLOCKS):
    """Random-init HexNetwork on cuda with randomised BatchNorm statistics.
    ``loud``: BN beta ~ N(0, 0.3), move_fc / value_fc2 / value_fc3 weights x 4
    and biases ~ N(0, 0.5), so every bias matters on the scale of the signal."""
    torch.manual_seed(1000 * n + chans + loud)
    net = HexNetwork(n, blocks, chans).eval()
    gen = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen) + 0.5)
                m.weight.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=gen) * (0.3 if loud else 0.1))
        if loud:
            for lin in (net.move_fc, net.value_fc2, net.value_fc3):
                lin.weight.mul_(4)
                lin.bias.normal_(0, 0.5, generator=gen)
    return net.cuda()


def make_cells(n, N, seed):
    """int8 network-view boards [N, stride]; the row padding past n*n holds
    2s, which no kernel may read."""
    nn = n * n
    cells = torch.full((N, (nn + 15) & ~15), 2, dtype=torch.int8, device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(seed)
    cells[:, :nn] = torch.randint(0, 3, (N, nn), generator=gen, device='cuda', dtype=torch.int8)
    return cells


def batch_sizes(n):
    bpg = 128 // (n + 1)
    return sorted({1, bpg - 1, bpg, bpg + 1, 1000})


# ------------------------------------------------------------- references --
def stem_rows(net, cells, acc_dtype):
    """The slab stem's three bf16 row sums per cell, [3][N, n, n, C] in fp64:
    T3[dy][code] = bf16((bias if dy == 1) + T[dy,0][v0] + T[dy,1][v1] + T[dy,2][v2])
    with the table T = bf16(fp32 W_fold x embedding) as prepare_inference
    builds it, summed in ``acc_dtype`` (fp32 in the kernel's order, or fp64)."""
    n, N = net.board_size, len(cells)
    ws, bs = _fold(net.conv1, net.bn1)
    tab = bf(torch.einsum('ocyx,vc->yxvo', ws.float(), net.encoder.weight.float()))
    tab = F.pad(tab, (0, 0, 0, 1)).to(acc_dtype)                # cell value 3: off board
    pc = F.pad(cells[:, :n * n].long().view(N, n, n), (1, 1, 1, 1), value=3)
    rows = []
    for dy in range(3):
        acc = bs.to(acc_dtype) if dy == 1 else torch.zeros((), dtype=acc_dtype, device=cells.device)
        for dx in range(3):
            acc = acc + tab[dy, dx][pc[:, dy:dy + n, dx:dx + n]]
        rows.append(bf(acc).double())
    return rows


@torch.no_grad()
def emulate(net, cells):
    """The tcgen05 arm in fp64 with its bf16 rounding points -> value [N],
    logits [N, n*n]."""
    d = torch.float64
    T3 = stem_rows(net, cells, d)
    x = bf(F.relu(T3[0] + T3[1] + T3[2])).permute(0, 3, 1, 2)
    for b in net.resblocks:
        (w1, b1), (w2, b2) = _fold(b.conv1, b.bn1), _fold(b.conv2, b.bn2)
        y = bf(F.relu(F.conv2d(x, bf(w1).to(d), b1.to(d), padding=1)))
        x = bf(F.relu(F.conv2d(y, bf(w2).to(d), b2.to(d), padding=1) + x))
    (wv, bv), (wp, bp) = _fold(net.value_conv1, net.value_bn1), _fold(net.move_conv1, net.move_bn1)
    h = bf(F.relu(F.conv2d(x, torch.cat([wv, wp]).to(d), torch.cat([bv, bp]).to(d))))
    yv = bf(h[:, :2].flatten(1) @ bf(net.value_fc2.weight).to(d).t())
    yp = bf(h[:, 2:].flatten(1) @ bf(net.move_fc.weight).to(d).t())
    logits = yp + net.move_fc.bias.to(d)
    v = F.relu(yv + net.value_fc2.bias.to(d)) @ net.value_fc3.weight.to(d).t()
    return torch.tanh(v + net.value_fc3.bias.to(d)).squeeze(1), logits


@torch.no_grad()
def reference(net, cells, mutate=None):
    """The plain fp64 HexNetwork on the same parameters (optionally mutated
    first) -> value [N], logits [N, n*n]."""
    n, N = net.board_size, len(cells)
    d = HexNetwork(n, len(net.resblocks), net.conv1.out_channels).eval()
    d.load_state_dict(net.state_dict())
    d = d.to(cells.device, torch.float64)
    if mutate is not None:
        mutate(d)
    v, p = d._trunk(d.encoder(cells[:, :n * n].long().view(N, n, n)).permute(0, 3, 1, 2))
    return v, d.move_fc(p)


def _drop_stem_bias(m):
    # the folded stem bias beta - mean * scale becomes zero
    bn = m.bn1
    bn.bias.copy_(bn.running_mean * bn.weight / torch.sqrt(bn.running_var + bn.eps))


MUTATIONS = {
    'move_fc bias dropped': lambda m: m.move_fc.bias.zero_(),
    'move_fc bias shifted by one tile': lambda m: m.move_fc.bias.copy_(m.move_fc.bias.roll(1)),
    'value_fc2 bias dropped': lambda m: m.value_fc2.bias.zero_(),
    'value_fc3 bias dropped': lambda m: m.value_fc3.bias.zero_(),
    'stem bias dropped': _drop_stem_bias,
    "last block's conv2 zeroed": lambda m: m.resblocks[-1].conv2.weight.zero_(),
    'board transposed': None,
}


def mutation_effects(net, cells, ref):
    """{bug: (max |value change|, max |logit change|)} of each bug of
    MUTATIONS on the fp64 network."""
    n = net.board_size
    out = {}
    for name, mutate in MUTATIONS.items():
        if mutate is None:
            t = cells[:, :n * n].view(-1, n, n).transpose(1, 2).reshape(-1, n * n)
            v, l = reference(net, t)
        else:
            v, l = reference(net, cells, mutate)
        out[name] = float((v - ref[0]).abs().max()), float((l - ref[1]).abs().max())
    return out


def check_mutations(effects, arms, what):
    """Each bug moves the fp64 outputs by at least MARGIN x the bound of every
    arm in ``arms``, in at least one of the two weight sets (``effects``:
    {weight set: mutation_effects}): a kernel with that bug fails the
    comparison of that set."""
    for arm in arms:
        for name in MUTATIONS:
            seen = {w: max(e[name][0] / BOUNDS[arm][w][0], e[name][1] / BOUNDS[arm][w][1])
                    for w, e in effects.items()}
            assert max(seen.values()) >= MARGIN, \
                f'{what}: {name} moves the outputs by only {seen} x the bounds of {arm}'


def check_arm(arm, weights, got, want, what):
    dv = float((got[0].double() - want[0]).abs().max())
    dl = float((got[1].double() - want[1]).abs().max())
    o = OBSERVED.setdefault((arm, weights), [0.0, 0.0])
    o[0], o[1] = max(o[0], dv), max(o[1], dl)
    bv, bl = BOUNDS[arm][weights]
    assert dv <= bv and dl <= bl, f'{arm} {what}: value off by {dv:.2e} (bound {bv:.0e}), logits by {dl:.2e} (bound {bl:.0e})'


def run_tcgen05(net, cells, fused):
    net.tower, net.tower_fused = 'tcgen05', fused
    return net.evaluate_cells(cells)


# ------------------------------------------------------------- end to end --
@pytest.mark.parametrize('n', (2, 3, 5, 7, 11, 13, 19))
def test_evaluator_matches_fp64_references(n):
    """evaluate_cells on every arm against emulate / reference at its bound,
    both weight sets, at batch sizes around a tower group (1, bpg - 1, bpg,
    bpg + 1, 1000), 40960 boards of 11x11 once on the 64-channel arms.  Then
    the mutation self-check on the 1000 boards."""
    effects = {}
    for loud in (False, True):
        w = 'loud' if loud else 'default'
        net = make_net(n, loud)
        net.prepare_inference(torch.bfloat16)
        assert net._fast['tower'] is not None
        net32 = copy.deepcopy(net).prepare_inference(torch.float32)
        glue = {c: make_net(n, loud, chans=c).prepare_inference(torch.bfloat16) for c in (32, 128)}
        for N in batch_sizes(n) + ([40960] if n == 11 else []):
            cells = make_cells(n, N, seed=N)
            what = f'n={n} {w} N={N}'
            emu, ref = emulate(net, cells), reference(net, cells)
            for arm, fused in (('chain', 2), ('block', 1), ('plain', 0)):
                check_arm(arm, w, run_tcgen05(net, cells, fused), emu, what)
            net.tower = 'cudnn'
            check_arm('cudnn', w, net.evaluate_cells(cells), ref, what)
            net.tower = 'tcgen05'
            check_arm('fp32', w, net32.evaluate_cells(cells), ref, what)
            if N == 1000:
                effects[w] = mutation_effects(net, cells, ref)
            for c, g in (glue.items() if N <= 1000 else ()):
                check_arm(f'glue{c}', w, g.evaluate_cells(cells), reference(g, cells), what)
    check_mutations(effects, ('chain', 'block', 'plain', 'cudnn', 'fp32'), f'n={n}')
    for (arm, w), (dv, dl) in sorted(OBSERVED.items()):
        print(f'{arm} {w}: value {dv:.2e} logits {dl:.2e} (largest so far)')


# ---------------------------------------------------------- stage by stage --
@pytest.mark.parametrize('n,N', ((2, 43), (3, 1), (5, 22), (7, 1000), (11, 1000), (13, 10), (19, 7)))
@torch.no_grad()
def test_evaluator_stages_on_their_own_inputs(n, N):
    """Each stage of the tcgen05 arm, fed the kernels' own previous output, is
    within one bf16 ulp of fp64 (plus the fp32 accumulation's share): the
    slab stem on its own buffer, the heads on the tower output, the GEMM on
    the heads output; the tail's logits are the one fp32 add bit for bit and
    its value is within a few fp32 ulps.  Nothing that is not a board cell or
    a real column is written."""
    net = make_net(n, True)
    net.prepare_inference(torch.bfloat16)
    f = net._fast
    L = _cabi.lib()
    nn = n * n
    cells = make_cells(n, N, seed=7)
    value, logits = run_tcgen05(net, cells, 2)
    x, _, flat, yfc, _ = f['tower_buf'][(N, cells.device, torch.cuda.current_stream().cuda_stream)]
    torch.cuda.synchronize()
    # stem: emulated in fp32 in the kernel's order up to the bf16 row sums
    xs = torch.zeros(L.az_nn_tower_rows(n, N), 64, dtype=torch.bfloat16, device='cuda')
    _cabi.check(L.az_nn_stem_live(ptr(cells), cells.stride(0), n, N, ptr(f['stem_table']),
                                  ptr(f['stem_bias']), ptr(xs), 64, 1, None, stream_ptr()))
    got, rest = tl.from_slabs(xs, n, N)
    assert rest == 0.0
    bpg = tl.boards_per_group(n)
    assert float(tl.from_slabs(xs, n, -(-N // bpg) * bpg)[0][N:].float().abs().sum()) == 0.0
    T3 = stem_rows(net, cells, torch.float32)
    want = F.relu(T3[0] + T3[1] + T3[2])
    slack = 2.0 ** -22 * (T3[0].abs() + T3[1].abs() + T3[2].abs())
    err = (got.double() - want).abs() - bf16_ulp(want) - slack
    assert float(err.max()) <= 0, float(err.max())
    # heads on the kernel's tower output; K padding of flat stays zero
    xt = tl.from_slabs(x, n, N)[0].double().reshape(N, nn, 64)
    (wv, bv), (wp, bp) = _fold(net.value_conv1, net.value_bn1), _fold(net.move_conv1, net.move_bn1)
    w, b = torch.cat([wv, wp]).flatten(1).double(), torch.cat([bv, bp]).double()
    want = F.relu(xt @ w.t() + b)
    slack = 2.0 ** -15 * (xt.abs() @ w.abs().t())
    got = flat[:, :nn * 6].double().view(N, nn, 6)
    err = (got - want).abs() - bf16_ulp(want) - slack
    assert float(err.max()) <= 0, float(err.max())
    assert float(flat[:, nn * 6:].float().abs().sum()) == 0.0
    # GEMM
    a, wfc = flat.double(), f['fc_pad'][0].double()
    want = a @ wfc.t()
    slack = 2.0 ** -16 * (a.abs() @ wfc.abs().t())
    err = (yfc.double() - want).abs() - bf16_ulp(want) - slack
    assert float(err.max()) <= 0, float(err.max())
    # tail on the kernel's yfc, with the module's own fp32 parameters
    k2 = net.value_fc2.out_features
    assert torch.equal(logits, yfc[:, k2:k2 + nn].float() + net.move_fc.bias)
    want_v, tol = tail_value(yfc[:, :k2], net.value_fc2.bias, net.value_fc3.weight.reshape(-1),
                             net.value_fc3.bias)
    assert float(((value.double() - want_v).abs() - tol).max()) <= 0


def tail_value(y, b, w3, b3):
    """fp64 value head tail and a tolerance of a few fp32 ulps of the terms."""
    t = F.relu(y.double() + b.double()) * w3.double()
    s = t.sum(1) + b3.double()
    return torch.tanh(s), 2.0 ** -20 * (t.abs().sum(1) + b3.double().abs() + 1)


@pytest.mark.parametrize('n', range(2, 20))
def test_tail_kernel_strides_nulls_and_live_rows(n):
    """az_nn_tail / az_nn_tail_live on random bf16 pre-activations, odd and
    even nfc2 + n*n, with a bias of exactly nfc2 + n*n elements: logits are
    y + bias bit for bit, value within a few fp32 ulps of fp64; strided
    outputs leave the gaps alone, a NULL output is not written, N = 0 and
    device-side live counts of 0, 1, N - 1 and N write exactly those rows."""
    L = _cabi.lib()
    nn, k2, N = n * n, 64, 37
    ld = (k2 + nn + 7) // 8 * 8
    gen = torch.Generator(device='cuda').manual_seed(n)
    y = (torch.randn(N, ld, generator=gen, device='cuda') * 2).to(torch.bfloat16)
    bias = torch.randn(k2 + nn, generator=gen, device='cuda')
    w3 = torch.randn(k2, generator=gen, device='cuda') * 0.3
    b3 = torch.randn(1, generator=gen, device='cuda')
    want_l = y[:, k2:k2 + nn].float() + bias[k2:]
    want_v, tol = tail_value(y[:, :k2], bias[:k2], w3, b3)
    vs, ls = 3, nn + 5
    sentinel = -77.0

    def call(rows, value, logits, live=None):
        args = (ptr(y), rows, ld, k2, n, ptr(bias), ptr(w3), ptr(b3), ptr(value), vs, ptr(logits), ls)
        if live is None:
            _cabi.check(L.az_nn_tail(*args, stream_ptr()))
        else:
            _cabi.check(L.az_nn_tail_live(*args, ptr(live), stream_ptr()))

    for live in (None, 0, 1, N - 1, N):
        for which in ('both', 'value', 'logits'):
            value = torch.full((N * vs + 1,), sentinel, device='cuda')
            logits = torch.full((N * ls + 1,), sentinel, device='cuda')
            call(N, value if which != 'logits' else None, logits if which != 'value' else None,
                 None if live is None else torch.tensor([live], dtype=torch.int32, device='cuda'))
            torch.cuda.synchronize()
            k = N if live is None else live
            v2, l2 = value[:N * vs].view(N, vs), logits[:N * ls].view(N, ls)
            if which != 'logits':
                assert ((v2[:k, 0].double() - want_v[:k]).abs() <= tol[:k]).all()
                assert (v2[k:, 0] == sentinel).all()
            else:
                assert (value == sentinel).all()
            if which != 'value':
                assert torch.equal(l2[:k, :nn], want_l[:k])
                assert (l2[k:, :nn] == sentinel).all()
            else:
                assert (logits == sentinel).all()
            assert (v2[:, 1:] == sentinel).all() and value[-1].item() == sentinel
            assert (l2[:, nn:] == sentinel).all() and logits[-1].item() == sentinel
    value = torch.full((4,), sentinel, device='cuda')
    call(0, value, None)
    torch.cuda.synchronize()
    assert (value == sentinel).all()


# ------------------------------------------------- the engine's own buffers --
def test_evaluator_writes_into_engine_buffers():
    """The two calls selfplay._evaluate makes: root mode writes the slot-0
    prior rows (logits_stride = max_batch * n*n, no value) and nothing else;
    leaf mode writes value / prior rows of the live count and nothing past
    it.  The rows written equal the dense evaluation."""
    from azalea_b200 import Engine
    n, G, B = 7, 40, 6
    nn = n * n
    net = make_net(n, True)
    net.prepare_inference(torch.bfloat16)
    eng = Engine(G, n, max_batch=B, device='cuda')
    cs = eng.cell_stride
    gen = torch.Generator(device='cuda').manual_seed(3)
    eng.leaf_board[:, :, :nn] = torch.randint(0, 3, (G, B, nn), generator=gen, device='cuda',
                                              dtype=torch.int8)
    sentinel = -55.0
    eng.value.fill_(sentinel)
    eng.prior.fill_(sentinel)
    net.evaluate_cells(eng.leaf_board[:, 0], logits_out=eng.prior[:, 0],
                       logits_stride=B * nn, want_value=False)
    _, want = net.evaluate_cells(eng.leaf_board[:, 0].contiguous())
    torch.cuda.synchronize()
    assert torch.equal(eng.prior[:, 0], want)
    assert (eng.prior[:, 1:] == sentinel).all() and (eng.value == sentinel).all()
    cells = eng.leaf_board.view(G * B, cs)
    want_v, want_l = (t.clone() for t in net.evaluate_cells(cells.clone()))
    for live in (G * B, G * B - 1, 100, 1, 0):
        eng.value.fill_(sentinel)
        eng.prior.fill_(sentinel)
        cnt = torch.tensor([live], dtype=torch.int32, device='cuda')
        net.evaluate_cells(cells, value_out=eng.value.view(-1), logits_out=eng.prior.view(-1, nn),
                           logits_stride=nn, live_rows=cnt)
        torch.cuda.synchronize()
        v, p = eng.value.view(-1), eng.prior.view(-1, nn)
        assert torch.equal(v[:live], want_v[:live]) and torch.equal(p[:live], want_l[:live]), live
        assert (v[live:] == sentinel).all() and (p[live:] == sentinel).all(), live


# ---------------------------------------------------- in-place weight refresh --
def _pointers(obj, out):
    if isinstance(obj, torch.Tensor):
        out.append(obj.data_ptr())
    elif isinstance(obj, dict):
        for k in sorted(obj, key=repr):
            _pointers(obj[k], out)
    elif isinstance(obj, (list, tuple)):
        for o in obj:
            _pointers(o, out)
    return out


def test_prepare_inference_refreshes_in_place_for_graphs():
    """prepare_inference() after load_state_dict refreshes every folded tensor
    at its old address: eager outputs and the replay of a graph captured
    before the refresh equal a freshly prepared network bit for bit, and
    graphed self-play refreshed from A to B plays the moves of self-play built
    on B."""
    from azalea_b200 import LockstepSelfPlay
    n, N = 7, 300
    a, b = make_net(n, False), make_net(n, True)
    cells = make_cells(n, N, seed=5)
    a.prepare_inference(torch.bfloat16)
    a.evaluate_cells(cells)                 # buffers and library handles before capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        a.evaluate_cells(cells)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gv, gl = a.evaluate_cells(cells)
    ptrs = _pointers(a._fast, [])
    a.load_state_dict(b.state_dict())
    a.prepare_inference(torch.bfloat16)
    assert _pointers(a._fast, []) == ptrs
    b.prepare_inference(torch.bfloat16)
    wv, wl = (t.clone() for t in b.evaluate_cells(cells))
    ev, el = a.evaluate_cells(cells)
    assert torch.equal(ev, wv) and torch.equal(el, wl)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gv, wv) and torch.equal(gl, wl)
    del graph

    def play(net, refresh=None):
        sp = LockstepSelfPlay(net, num_games=32, board_size=n, simulations=24,
                              search_batch_size=6, seed=11, cuda_graph=True)
        sp.capture()
        if refresh is not None:
            net.load_state_dict(refresh.state_dict())
            net.prepare_inference(torch.bfloat16)
        chosen = []
        for _ in range(4):
            sp.step_move()
            chosen.append(sp.chosen.clone())
        return torch.stack(chosen).cpu()
    a2 = make_net(n, False).prepare_inference(torch.bfloat16)
    refreshed = play(a2, refresh=make_net(n, True))
    b2 = make_net(n, True).prepare_inference(torch.bfloat16)
    assert torch.equal(refreshed, play(b2))
    # and the refresh is not a no-op: A's own games differ
    assert not torch.equal(refreshed, play(make_net(n, False).prepare_inference(torch.bfloat16)))

