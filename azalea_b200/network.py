"""The evaluator: 6x64 residual tower with value and policy heads.

Same architecture, parameter names and ``run`` contract as the reference's
``HexNetwork`` (azalea/network.py:17-152), so reference checkpoints load and
this module can be dropped into the reference's ``Policy``.  Two ways in:

* ``forward`` / ``run``: the reference's interface (int32 boards + padded
  legal-move lists -> value, moves_logprob), in the module's own dtype.
* ``evaluate_cells``: the lockstep path.  Takes the int8 network-view boards
  the select kernel wrote ([N, cell_stride]) and returns fp32 value [N] and
  fp32 logits over all n*n tiles [N, n*n]; BatchNorm is folded into the
  convolutions, activations are bf16 channels-last, and on CUDA every
  convolution is one cuDNN call with bias, ReLU and the residual add in its
  epilogue (2.8x over separate conv / bias / add / relu kernels on B200,
  profiles/r01_nn_variants.txt).  Gathering the legal tiles and the masked
  softmax happen in the expand kernel (AZ_PRIOR_LOGITS), not here.

The network is the only dense contraction on the path and stays a PyTorch
(cuDNN / cuBLAS) call by design; the tree kernels around it are ours.
"""
import logging

import torch
from torch import nn
from torch.nn import functional as F


def conv3x3(cin, cout):
    return nn.Conv2d(cin, cout, kernel_size=3, padding=1, bias=False)


def conv1x1(cin, cout):
    return nn.Conv2d(cin, cout, kernel_size=1, bias=False)


class Resblock(nn.Module):
    """network.py:17-39 (in_dim == dim on this path: no projection)."""

    def __init__(self, in_dim, dim):
        super().__init__()
        self.conv1 = conv3x3(in_dim, dim)
        self.bn1 = nn.BatchNorm2d(dim)
        self.conv2 = conv3x3(dim, dim)
        self.bn2 = nn.BatchNorm2d(dim)
        if dim != in_dim:
            self.res_conv = conv1x1(in_dim, dim)
            self.res_bn = nn.BatchNorm2d(dim)
        else:
            self.res_conv = self.res_bn = None

    def forward(self, x):
        y = F.relu(self.bn1(self.conv1(x)))
        y = self.bn2(self.conv2(y))
        if self.res_conv is not None:
            x = self.res_bn(self.res_conv(x))
        return F.relu(y + x)


def _fold(conv, bn):
    """conv (no bias) followed by eval-mode BatchNorm -> weight, bias."""
    scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    return conv.weight * scale[:, None, None, None], \
        bn.bias - bn.running_mean * scale


class HexNetwork(nn.Module):
    def __init__(self, board_size=11, num_blocks=6, base_chans=64):
        super().__init__()
        self.board_size = board_size
        value_chans, policy_chans, input_dim = 2, 4, 4
        nn2 = board_size * board_size
        self.conv1 = conv3x3(input_dim, base_chans)
        self.bn1 = nn.BatchNorm2d(base_chans)
        self.resblocks = nn.Sequential(
            *[Resblock(base_chans, base_chans) for _ in range(num_blocks)])
        self.value_conv1 = conv1x1(base_chans, value_chans)
        self.value_bn1 = nn.BatchNorm2d(value_chans)
        self.value_fc2 = nn.Linear(value_chans * nn2, 64)
        self.value_fc3 = nn.Linear(64, 1)
        self.move_conv1 = conv1x1(base_chans, policy_chans)
        self.move_bn1 = nn.BatchNorm2d(policy_chans)
        self.encoder = nn.Embedding(3, 4)
        self.move_fc = nn.Linear(policy_chans * nn2, nn2)
        self._fast = None
        # 'tcgen05' (default): the tower runs on our implicit-GEMM kernel
        # (csrc/az_tower.cuh; 64 channels, bf16, board <= 19);
        # 'cudnn': twelve fused cuDNN calls (also used for other widths)
        import os
        self.tower = os.environ.get('AZALEA_B200_TOWER', 'tcgen05')
        # the residual tower on the fused kernel (csrc/az_block.cuh): AZALEA_B200_FUSED=2
        # (default) chains all blocks in one launch, 1 is one launch per block, 0 the
        # two az_nn_conv3x3 launches per block
        self.tower_fused = int(os.environ.get('AZALEA_B200_FUSED', '2'))
        nnet = sum(p.nelement() for p in self.parameters())
        nenc = sum(p.nelement() for p in self.encoder.parameters())
        logging.info('Net params: %d  Embedding params: %d', nnet - nenc, nenc)

    @property
    def device(self):
        return self.conv1.weight.device

    # ------------------------------------------------ reference interface --
    def _trunk(self, x):
        x = F.relu(self.bn1(self.conv1(x)))
        x = self.resblocks(x)
        v = F.relu(self.value_bn1(self.value_conv1(x)))
        v = F.relu(self.value_fc2(v.flatten(1)))
        value = torch.tanh(self.value_fc3(v)).squeeze(1)
        p = F.relu(self.move_bn1(self.move_conv1(x)))
        return value, p.flatten(1)

    def forward(self, x, legal_moves):
        """network.py:134-152.  x int32 [B, n, n] (first-player view),
        legal_moves int32 [B, K] zero padded."""
        x = self.encoder(x.long()).permute(0, 3, 1, 2).contiguous()
        value, p = self._trunk(x)
        logit = self.move_fc(p)
        tiles = (legal_moves - 1).clamp(min=0)
        logit = torch.gather(logit, 1, tiles.long())
        logit = logit.masked_fill(legal_moves == 0, -99)
        return dict(value=value, moves_logprob=F.log_softmax(logit, dim=1))

    def run(self, batch, *, compute_loss=False):
        """network.py:87-105."""
        output = self.forward(batch['board'], batch['legal_moves'])
        if not compute_loss:
            return {k: v.detach() for k, v in output.items()}
        moves_prob = batch['moves_prob']
        value_loss = F.mse_loss(output['value'], batch['reward'])
        moves_loss = -(moves_prob * output['moves_logprob']).sum() \
            / len(moves_prob)
        loss = value_loss.to(moves_loss.device) + moves_loss
        output = {k: v.detach() for k, v in output.items()}
        output.update(value_loss=value_loss.item(),
                      moves_loss=moves_loss.item())
        return output, loss

    # ------------------------------------------------------- lockstep path --
    @torch.no_grad()
    def prepare_inference(self, dtype=torch.bfloat16):
        """Fold BatchNorm into the convolutions and cast for inference.

        Calling it again after the parameters changed refreshes the folded
        tensors IN PLACE (same device addresses), so a captured CUDA graph
        keeps reading the current weights."""
        assert not self.training, 'call .eval() first'
        dev = self.device
        old = self._fast if (self._fast is not None
                             and self._fast['dtype'] == dtype
                             and self._fast['emb'].device == dev) else None
        slot = [0]

        def keep(t, channels_last=False, dtype_=None):
            t = t.to(dev, dtype_ or dtype)
            t = t.contiguous(memory_format=torch.channels_last) \
                if channels_last else t.contiguous()
            if old is not None:
                dst = old['_flat'][slot[0]]
                dst.copy_(t)
                t = dst
            slot[0] += 1
            flat.append(t)
            return t

        def keep32(t):
            return keep(t, dtype_=torch.float32)

        def pack(w, b):
            return keep(w, True), keep(b)

        flat = []
        fast = {'dtype': dtype, '_flat': flat}
        fast['emb'] = keep(self.encoder.weight)
        ws, bs = _fold(self.conv1, self.bn1)
        fast['stem'] = pack(ws, bs)
        # stem as a table for az_nn_stem: T[tap][cell value][c_out]
        tab = torch.einsum('ocyx,vc->yxvo', ws.float(), self.encoder.weight.float())
        tab = F.pad(tab, (0, 0, 0, 1)).reshape(9, 4, -1)
        fast['stem_table'] = keep(tab)
        fast['stem_bias'] = keep32(bs)
        fast['blocks'] = [(pack(*_fold(b.conv1, b.bn1)),
                           pack(*_fold(b.conv2, b.bn2)))
                          for b in self.resblocks]
        # the same layers packed for az_nn_conv3x3 (csrc/az_tower.cuh):
        # [kx][ky][c_out][c_in] bf16, 16-byte chunk j of row r stored at
        # chunk j ^ (r & 7); bias stays fp32
        fast['tower'] = None
        if ws.shape[0] == 64 and dtype == torch.bfloat16:
            from .tower_layout import pack_conv_weights

            def pack_tower(conv, bn):
                w, b = _fold(conv, bn)
                return keep(pack_conv_weights(w.to(dev, dtype))), keep32(b)
            fast['tower'] = [(pack_tower(b.conv1, b.bn1), pack_tower(b.conv2, b.bn2))
                             for b in self.resblocks]
            # the same, block by block, for the fused launch (csrc/az_block.cuh)
            fast['tower_fused'] = [
                (keep(torch.cat([w1, w2])), keep32(torch.cat([b1, b2])))
                for (w1, b1), (w2, b2) in fast['tower']]
            # and all blocks back to back for the chained launch
            fast['tower_chain'] = (keep(torch.cat([w for w, _ in fast['tower_fused']])),
                                   keep32(torch.cat([b for _, b in fast['tower_fused']])))
        fast['tower_buf'] = old['tower_buf'] if old is not None else {}
        # the two 1x1 head convolutions read the same activations: one conv;
        # the two first fully connected layers read its output: one GEMM over
        # the channels-last flattening (hw-major, channel-minor), so no
        # layout change is needed between the conv and the GEMM
        wv, bv = _fold(self.value_conv1, self.value_bn1)
        wp, bp = _fold(self.move_conv1, self.move_bn1)
        fast['heads'] = pack(torch.cat([wv, wp]), torch.cat([bv, bp]))
        fast['heads_w32'] = keep32(torch.cat([wv, wp]).flatten(1))
        fast['heads_b32'] = keep32(torch.cat([bv, bp]))
        nv, npc = wv.shape[0], wp.shape[0]
        hw = self.board_size ** 2
        hc = nv + npc
        w2, wm = self.value_fc2.weight, self.move_fc.weight
        merged = torch.zeros(w2.shape[0] + wm.shape[0], hw * hc,
                             dtype=w2.dtype, device=w2.device)
        # reference flattening is channel-major: column c * hw + p
        merged[:w2.shape[0]].view(-1, hw, hc)[:, :, :nv] = \
            w2.view(-1, nv, hw).permute(0, 2, 1)
        merged[w2.shape[0]:].view(-1, hw, hc)[:, :, nv:] = \
            wm.view(-1, npc, hw).permute(0, 2, 1)
        fast['fc'] = (keep(merged),
                      keep(torch.cat([self.value_fc2.bias, self.move_fc.bias])))
        # K and N padded to multiples of 8 with zeros for the tcgen05 path
        kp, npd = (merged.shape[1] + 7) // 8 * 8, (merged.shape[0] + 7) // 8 * 8
        wpad = torch.zeros(npd, kp, dtype=merged.dtype, device=merged.device)
        wpad[:merged.shape[0], :merged.shape[1]] = merged
        bpad = torch.zeros(npd, dtype=merged.dtype, device=merged.device)
        bpad[:merged.shape[0]] = torch.cat([self.value_fc2.bias, self.move_fc.bias])
        fast['fc_pad'] = (keep(wpad), keep(bpad))
        fast['nfc2'] = w2.shape[0]
        fast['value_fc3'] = (keep(self.value_fc3.weight), keep(self.value_fc3.bias))
        # operands of the tail kernel (csrc/az_nn_glue.cuh: k_nn_tail): the GEMM
        # runs without bias, the fp32 bias is added where the results are
        # converted to fp32
        fast['fc_pad_t'] = fast['fc_pad'][0].t()
        fast['fc_bias32'] = keep32(bpad)
        fast['value_fc3_32'] = (keep32(self.value_fc3.weight.reshape(-1)),
                                keep32(self.value_fc3.bias.reshape(-1)))
        self._fast = fast
        return self

    @torch.no_grad()
    def evaluate_cells(self, cells, value_out=None, logits_out=None,
                       logits_stride=None, want_value=True, live_rows=None):
        """int8 [N, >= n*n] network-view boards -> value f32 [N], logits
        f32 [N, n*n] over tiles (no legal-move gather, no softmax).  The
        optional outputs are written in place (see _evaluate_cells_tcgen05).
        ``live_rows``: int32 device tensor holding the number of leading rows
        that hold boards (packed leaves, AZ_CFG_PACK_LEAVES); our kernels then
        work on that many rows, the comparison arms ignore it and evaluate all N."""
        f = self._fast
        if f is None:
            raise RuntimeError('call prepare_inference() first')
        n = self.board_size
        N = cells.shape[0]
        C_ = f['stem_bias'].numel()
        glue = (cells.is_cuda and f['dtype'] == torch.bfloat16
                and C_ in (32, 64, 128) and cells.dtype == torch.int8
                and cells.stride(1) == 1)
        if glue and self.tower == 'tcgen05' and f['tower'] is not None:
            return self._evaluate_cells_tcgen05(cells, value_out, logits_out,
                                                logits_stride, want_value, live_rows)
        if glue:
            # our kernels at both ends of the tower (csrc/az_nn_glue.cuh)
            from . import _cabi
            import ctypes
            L = _cabi.lib()
            stream = ctypes.c_void_p(torch.cuda.current_stream(cells.device).cuda_stream)
            x = torch.empty(N, n, n, C_, dtype=torch.bfloat16, device=cells.device)
            _cabi.check(L.az_nn_stem(
                ctypes.c_void_p(cells.data_ptr()), cells.stride(0), n, N,
                ctypes.c_void_p(f['stem_table'].data_ptr()),
                ctypes.c_void_p(f['stem_bias'].data_ptr()),
                ctypes.c_void_p(x.data_ptr()), C_, 0, stream))
            x = x.permute(0, 3, 1, 2)       # NCHW view of NHWC memory
        else:
            idx = cells[:, :n * n].to(torch.int32)
            x = F.embedding(idx, f['emb']).view(N, n, n, 4).permute(0, 3, 1, 2)
        if x.is_cuda and f['dtype'] != torch.float32:
            one, pad, nopad = (1, 1), (1, 1), (0, 0)
            if not glue:
                x = torch.cudnn_convolution_relu(x, *f['stem'], one, pad, one, 1)
            for (w1, b1), (w2, b2) in f['blocks']:
                y = torch.cudnn_convolution_relu(x, w1, b1, one, pad, one, 1)
                x = torch.cudnn_convolution_add_relu(y, w2, x, 1.0, b2, one,
                                                     pad, one, 1)
            if glue:
                xh = x.permute(0, 2, 3, 1)
                if not xh.is_contiguous():
                    xh = xh.contiguous()
                flat = torch.empty(N, n * n * 6, dtype=torch.bfloat16,
                                   device=cells.device)
                _cabi.check(L.az_nn_heads(
                    ctypes.c_void_p(xh.data_ptr()), N * n * n,
                    ctypes.c_void_p(f['heads_w32'].data_ptr()),
                    ctypes.c_void_p(f['heads_b32'].data_ptr()),
                    ctypes.c_void_p(flat.data_ptr()), 0, C_, 6, 0, stream))
                h = None
            else:
                h = torch.cudnn_convolution_relu(x, *f['heads'], one, nopad, one, 1)
        else:
            x = F.relu_(F.conv2d(x, *f['stem'], padding=1))
            for (w1, b1), (w2, b2) in f['blocks']:
                y = F.relu_(F.conv2d(x, w1, b1, padding=1))
                y = F.conv2d(y, w2, b2, padding=1)
                x = F.relu_(y.add_(x))
            h = F.relu_(F.conv2d(x, *f['heads']))
        # [N, C, n, n] channels-last == [N, n*n*C] row-major: free view
        if h is not None:
            flat = h.permute(0, 2, 3, 1).reshape(N, -1)
        y = F.linear(flat, *f['fc'])
        k2 = f['nfc2']
        value = torch.tanh(F.linear(F.relu(y[:, :k2]), *f['value_fc3'])).squeeze(1)
        logits = y[:, k2:]
        value, logits = value.float(), logits.float()
        # comparison arms (cuDNN tower, fp32, CPU): honour the in-place outputs by copying
        if value_out is not None:
            value_out.copy_(value)
            value = value_out
        if logits_out is not None:
            stride = int(logits_stride or n * n)
            torch.as_strided(logits_out, (N, n * n), (stride, 1)).copy_(logits)
            logits = logits_out
        return value, logits

    @torch.no_grad()
    def _evaluate_cells_tcgen05(self, cells, value_out=None, logits_out=None,
                                logits_stride=None, want_value=True, live_rows=None):
        """evaluate_cells with the whole tower on our tcgen05 convolution
        (csrc/az_tower.cuh): stem kernel -> 12 x az_nn_conv3x3 over the slab
        activation layout (residual added in the epilogue, in place) -> heads
        kernel -> one GEMM -> tail kernel (bias, value head tail, fp32
        outputs).  ``value_out`` f32 [N] / ``logits_out`` f32 rows of
        ``logits_stride`` elements (default n*n, dense) receive the results in
        place -- the lockstep path passes views of the engine's value / prior
        buffers, so nothing is copied between the network and the tree."""
        import ctypes
        from . import _cabi
        f = self._fast
        L = _cabi.lib()
        n, N, dev = self.board_size, cells.shape[0], cells.device
        nn2 = n * n
        npad = N
        rows = L.az_nn_tower_rows(n, N)
        wfc, bfc = f['fc_pad']
        # one set of activation buffers per (batch size, stream): two halves of the games
        # may be evaluated concurrently on two streams (LockstepSelfPlay(streams=2))
        stream_id = torch.cuda.current_stream(dev).cuda_stream
        bufs = f['tower_buf'].get((npad, dev, stream_id))
        if bufs is None:
            # halos and pad cells must be zero; the kernels keep them zero
            bufs = (torch.zeros(rows, 64, dtype=torch.bfloat16, device=dev),
                    torch.zeros(rows, 64, dtype=torch.bfloat16, device=dev),
                    torch.zeros(N, wfc.shape[1], dtype=torch.bfloat16, device=dev),
                    torch.empty(N, wfc.shape[0], dtype=torch.bfloat16, device=dev),
                    # scratch argument of the fused residual block (unused: az_nn_resblock_scratch_bytes() is 0)
                    torch.zeros(max(16, L.az_nn_resblock_scratch_bytes()), dtype=torch.uint8, device=dev))
            f['tower_buf'][(npad, dev, stream_id)] = bufs
        x, y, flat, yfc, scratch = bufs
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        live = p(live_rows) if live_rows is not None else None
        _cabi.check(L.az_nn_stem_live(p(cells), cells.stride(0), n, N, p(f['stem_table']),
                                      p(f['stem_bias']), p(x), 64, 1, live, stream))
        ev = getattr(self, 'conv_events', None)     # bench.py: per-launch CUDA events
        cur = torch.cuda.current_stream(dev)

        def timed(fn, kind):
            if ev is None:
                return fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(cur)
            fn()
            e1.record(cur)
            ev.append((e0, e1, kind, N))

        fused = f.get('tower_fused') if self.tower_fused else None
        if fused is not None and self.tower_fused >= 2:
            # the whole tower chained in one launch (csrc/az_block.cuh), in place
            wall, ball = f['tower_chain']
            timed(lambda: _cabi.check(L.az_nn_resblocks_live(
                p(x), p(wall), p(ball), p(scratch), n, npad, len(fused), live, stream)), 'chain%d' % len(fused))
        elif fused is not None:
            # one launch per residual block, in place
            for w12, b12 in fused:
                timed(lambda: _cabi.check(L.az_nn_resblock(
                    p(x), p(w12), p(b12), p(scratch), n, npad, stream)), 'block')
        else:
            for (w1, b1), (w2, b2) in f['tower']:
                timed(lambda: _cabi.check(L.az_nn_conv3x3(
                    p(x), p(w1), p(b1), None, p(y), n, npad, stream)), 'plain')
                timed(lambda: _cabi.check(L.az_nn_conv3x3(
                    p(y), p(w2), p(b2), p(x), p(x), n, npad, stream)), 'residual')
        # head activations with the board row padded to a multiple of 8 (zeros):
        # the merged FC GEMM then runs a current cuBLAS kernel (K = 726 falls
        # back to a legacy one, 0.15 ms instead of 0.03)
        _cabi.check(L.az_nn_heads_live(p(x), N * nn2, p(f['heads_w32']), p(f['heads_b32']),
                                       p(flat), flat.shape[1], 64, 6, n, live, stream))
        torch.mm(flat, f['fc_pad_t'], out=yfc)
        k2 = f['nfc2']
        if value_out is None and want_value:
            value_out = torch.empty(N, dtype=torch.float32, device=dev)
        if logits_out is None:
            logits_out = torch.empty(N, nn2, dtype=torch.float32, device=dev)
            logits_stride = nn2
        w3, b3 = f['value_fc3_32']
        _cabi.check(L.az_nn_tail_live(
            p(yfc), N, yfc.shape[1], k2, n, p(f['fc_bias32']), p(w3), p(b3),
            p(value_out) if value_out is not None else None, 1,
            p(logits_out), int(logits_stride or nn2), live, stream))
        return value_out, logits_out
