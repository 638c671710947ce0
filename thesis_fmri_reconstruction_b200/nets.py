"""Layer- and network-level forward / backward of the VAE/GAN sub-networks on raw device buffers.

Everything here is orchestration: each arithmetic step is one call into libfmri_b200.so (hand-written sm_100a kernels,
see include/fmri_b200.h). There is no autograd and no torch compute in this file -- torch is used to own device
memory only. The same code serves both front ends:
  * the fused training engine (engine.py), which runs the minimal backward of SURVEY.md section 8d, and
  * the nn.Module drop-in surface (models/vae_gan.py), whose autograd Functions call forward()/backward() below.

Layouts: activations are channels-last [N,H,W,C] in ``adt`` (torch.bfloat16 -> tcgen05/TMA tensor path,
torch.float32 -> exact CUDA-core path used for tight parity checks); images at the network edges are NCHW fp32 as in
the reference; weights, gradients and statistics are fp32 in the reference layouts.
Parameter / buffer dictionaries are keyed by the reference's state_dict names relative to the sub-network
(/root/reference/models/vae_gan.py:63-232, 499-529).
"""
from __future__ import annotations

import torch

from . import lib as L

BN_EPS = 1e-5
BN_MOMENTUM = 0.9  # /root/reference/models/vae_gan.py:21,54,80,108,158,200
F32, BF16, F64 = torch.float32, torch.bfloat16, torch.float64


def E(*shape, dtype=F32):
    return torch.empty(shape, dtype=dtype, device="cuda")


def Z(*shape, dtype=F32):
    return torch.zeros(shape, dtype=dtype, device="cuda")


class Ctx(dict):
    """Saved forward state of one layer / network (attribute access)."""
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


def _pad8(n):
    return (n + 7) // 8 * 8


class _EdgeWs:
    """Grow-only workspace of the edge convolutions (sized by fmri_edge_workspace of the largest descriptor seen)."""

    def __init__(self):
        self.buf = None

    def get(self, d):
        need = L.edge_workspace(d)
        if self.buf is None or self.buf.numel() < need:
            self.buf = E(need, dtype=torch.uint8)
        return self.buf


# ====================================================================================================== BatchNorm
class BatchNorm:
    """nn.BatchNorm{1,2}d(momentum=0.9) + optional ReLU over a channels-last [rows, C] matrix."""

    def __init__(self, prefix, C):
        self.prefix, self.C = prefix, C
        self._ws = self._ws2 = None

    def names(self):
        return [self.prefix + "weight", self.prefix + "bias"]

    def forward(self, P, S, raw, rows, out_dtype, relu, train, n_updates, stats=None, nbt=None):
        C, pre = self.C, self.prefix
        mean, invstd = E(C), E(C)
        if train:
            if stats is None:
                stats = (E(C, dtype=F64), E(C, dtype=F64))
                L.colstats(raw, rows, C, stats[0], stats[1])
            L.bn_finalize(stats[0], stats[1], rows, C, BN_EPS, BN_MOMENTUM, mean, invstd,
                          S[pre + "running_mean"] if n_updates > 0 else None,
                          S[pre + "running_var"] if n_updates > 0 else None)
            for _ in range(n_updates - 1):  # the reference runs the discriminator twice per step (vae_gan.py:284-285)
                L.bn_finalize(stats[0], stats[1], rows, C, BN_EPS, BN_MOMENTUM, mean, invstd,
                              S[pre + "running_mean"], S[pre + "running_var"])
            if nbt is not None and n_updates:
                nbt[pre + "num_batches_tracked"] = nbt.get(pre + "num_batches_tracked", 0) + n_updates
        else:
            L.bn_eval_stats(S[pre + "running_mean"], S[pre + "running_var"], C, BN_EPS, mean, invstd)
        y = torch.empty(raw.shape, dtype=out_dtype, device=raw.device)
        L.bn_apply(raw, y, rows, C, mean, invstd, P[pre + "weight"], P[pre + "bias"], relu)
        return y, Ctx(raw=raw, mean=mean, invstd=invstd, rows=rows, relu=relu, train=train)

    def backward(self, P, c, dy, G, acc, need_dw):
        """dy has the gradient dtype; returns d(raw) in the same dtype."""
        C, pre = self.C, self.prefix
        if self._ws is None:
            self._ws = E(3 * C, dtype=F64)
        draw = torch.empty(c.raw.shape, dtype=dy.dtype, device=dy.device)
        L.bn_backward(c.raw, dy, draw, c.rows, C, c.mean, c.invstd, P[pre + "weight"], P[pre + "bias"], c.relu,
                      c.train, G[pre + "weight"] if need_dw else None, G[pre + "bias"] if need_dw else None, acc,
                      self._ws)
        return draw

    def backward_pair(self, P, c, dya, dyb, G, acc, need_dw, rows_b=None):
        """Two upstreams through this layer with the forward tensor read once for both (the layer is linear in its upstream).
        Parameter gradients come from upstream a. rows_b = (row0, nrows): upstream b's gradient for those rows only.
        Returns one buffer holding d(raw) of a, then of b, stacked along the leading (batch) dimension."""
        C, pre = self.C, self.prefix
        if self._ws2 is None:
            self._ws2 = E(6 * C, dtype=F64)
        lead, per = c.raw.shape[0], c.rows // c.raw.shape[0]
        row0, nb = rows_b if rows_b is not None else (0, c.rows)
        out = torch.empty((lead + nb // per,) + tuple(c.raw.shape[1:]), dtype=dya.dtype, device=dya.device)
        args = (C, c.mean, c.invstd, P[pre + "weight"], P[pre + "bias"], c.relu, c.train,
                G[pre + "weight"] if need_dw else None, G[pre + "bias"] if need_dw else None, acc, self._ws2)
        if rows_b is None:
            L.bn_backward_pair(c.raw, dya, dyb, out[:lead], out[lead:], c.rows, *args)
        else:
            L.bn_backward_pair_slice(c.raw, dya, dyb, out[:lead], out[lead:], c.rows, row0, nb, *args)
        return out


# ====================================================================================================== conv blocks
class ConvBlock:
    """EncoderBlock / DecoderBlock (vae_gan.py:11-60): 5x5 stride-2 Conv2d or ConvTranspose2d (no bias) -> BN -> ReLU,
    channels >= 32 on both sides: tcgen05 implicit GEMM (bf16) or direct conv (fp32)."""

    def __init__(self, prefix, Cin, Cout, transposed, output_pad, adt):
        self.prefix, self.Cin, self.Cout, self.transposed, self.output_pad, self.adt = (
            prefix, Cin, Cout, transposed, int(output_pad), adt)
        self.bn = BatchNorm(prefix + "bn.", Cout)
        self.pack_f = self.pack_d = None
        self._ws = None

    def names(self):
        return [self.prefix + "conv.weight"] + self.bn.names()

    def desc(self, N, H, W):
        return L.conv_desc(N, H, W, self.Cin, self.Cout, 2, self.transposed, self.output_pad, self.adt)

    def refresh(self, P, inplace=True):
        if self.adt != BF16:
            return
        n = L.conv_pack_elems(self.desc(1, 8, 8))
        if self.pack_f is None or not inplace:
            self.pack_f, self.pack_d = E(n, dtype=BF16), E(n, dtype=BF16)
        L.conv_pack_weights(self.desc(1, 8, 8), P[self.prefix + "conv.weight"], self.pack_f, self.pack_d)

    def forward(self, P, S, x, N, H, W, train, n_updates, nbt=None):
        d = self.desc(N, H, W)
        OH, OW = L.conv_out_hw(d)
        raw = E(N, OH, OW, self.Cout, dtype=self.adt)
        stats = (E(self.Cout, dtype=F64), E(self.Cout, dtype=F64)) if train else (None, None)
        L.conv_fprop(d, x, P[self.prefix + "conv.weight"], self.pack_f, None, L.ACT_NONE, raw, stats[0], stats[1])
        y, cb = self.bn.forward(P, S, raw, N * OH * OW, self.adt, True, train, n_updates,
                                stats if train else None, nbt)
        return y, Ctx(d=d, x=x, bn=cb, pack_f=self.pack_f, pack_d=self.pack_d, OH=OH, OW=OW)

    def backward(self, P, c, dy, G, acc, need_dw, need_dx, relu_mask=None):
        """relu_mask: (y, bits) of the bias+ReLU layer BELOW, whose ReLU backward this layer's data-gradient kernel applies."""
        draw = self.bn.backward(P, c.bn, dy, G, acc, need_dw)
        return self.backward_raw(P, c, draw, G, acc, need_dw, need_dx, relu_mask)

    def backward_pair(self, P, c, dya, dyb, G, acc, need_dw):
        """Two upstreams through this block's saved forward state: one BatchNorm backward for both, one data-gradient launch
        over the two stacked along the batch, the weight gradient from upstream a. Returns dx of a, then of b, stacked
        [2N, H, W, Cin]."""
        N = c.d.N
        draw = self.bn.backward_pair(P, c.bn, dya, dyb, G, acc, need_dw)
        dx = E(2 * N, c.d.H, c.d.W, self.Cin, dtype=self.adt)
        L.conv_dgrad(self.desc(2 * N, c.d.H, c.d.W), draw, P[self.prefix + "conv.weight"], c.pack_d, dx)
        self.backward_raw(P, c, draw[:N], G, acc, need_dw, False)
        return dx

    def backward_dx_slice(self, P, c, dy, n0, n1, relu_mask=None):
        """Data gradient only, for images [n0, n1) of the batch. Train-mode BatchNorm couples all samples through its two
        backward sums, so those run over the whole batch; the BN apply pass and the conv data gradient run on the slice only
        (the discriminator's feature-tap sweep needs the image gradient of ONE of its three sources). Returns dx of the slice."""
        C, pre, cb = self.Cout, self.prefix + "bn.", c.bn
        per = c.OH * c.OW
        N = c.d.N
        if self.bn._ws is None:
            self.bn._ws = E(3 * C, dtype=F64)
        draw = E(n1 - n0, c.OH, c.OW, C, dtype=dy.dtype)
        L.bn_backward_slice(cb.raw, dy, draw, N * per, n0 * per, (n1 - n0) * per, C, cb.mean, cb.invstd, P[pre + "weight"],
                            P[pre + "bias"], cb.relu, cb.train, self.bn._ws)
        dsub = self.desc(n1 - n0, c.d.H, c.d.W)
        dx = E(n1 - n0, c.d.H, c.d.W, self.Cin, dtype=self.adt)
        L.conv_dgrad(dsub, draw, P[self.prefix + "conv.weight"], c.pack_d, dx, relu_mask)
        return dx

    def backward_raw(self, P, c, draw, G, acc, need_dw, need_dx, relu_mask=None):
        """Backward from a gradient on the raw (pre-BN) conv output -- the discriminator's feature tap (vae_gan.py:169-173)."""
        w = P[self.prefix + "conv.weight"]
        dx = None
        if need_dx:
            dx = torch.empty(c.x.shape, dtype=self.adt, device=draw.device)
            L.conv_dgrad(c.d, draw, w, c.pack_d, dx, relu_mask)
        if need_dw:
            if self._ws is None:
                self._ws = E(max(1, L.conv_wgrad_workspace(c.d)), dtype=torch.uint8)
            if WGRAD_SIDE_STREAM and self.adt == BF16:
                # The weight gradient is a leaf of the backward graph: nothing downstream in this sweep reads it. It goes
                # to a side stream, ordered AFTER this layer's data-gradient kernel (both are tensor-pipe bound and would
                # only time-share the SMs), so that it runs beside the HBM-bound BatchNorm backward of the layer below.
                # All weight-gradient launches share the one side stream, so accumulation into G stays ordered;
                # consumers of G join it (join_side / side_into).
                side, cur = side_stream(), torch.cuda.current_stream()
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    L.conv_wgrad(c.d, c.x, draw, G[self.prefix + "conv.weight"], acc, self._ws)
                draw.record_stream(side)
                c.x.record_stream(side)
            else:
                L.conv_wgrad(c.d, c.x, draw, G[self.prefix + "conv.weight"], acc, self._ws)
        return dx


class BlockNet:
    """A standalone EncoderBlock / DecoderBlock (vae_gan.py:11-60) on NCHW fp32 tensors, as the reference's modules are
    callable on their own: forward(ten, out) -> relu(bn(conv(ten))) [, raw conv output]. Inside Encoder / Decoder /
    Discriminator the blocks run in their network's fused pipeline instead (no layout passes). Channel counts the tensor path
    does not tile (e.g. a 3-channel input) run on the exact fp32 CUDA-core path."""

    def __init__(self, Cin, Cout, transposed, output_pad, adt):
        ok = (Cin % 64 == 0 and Cout % 32 == 0) if transposed else (Cin % 32 == 0 and Cout % 64 == 0)
        self.adt = adt if ok else F32
        self.Cin, self.Cout = Cin, Cout
        self.block = ConvBlock("", Cin, Cout, transposed, output_pad, self.adt)

    def refresh(self, P, inplace=True):
        self.block.refresh(P, inplace)

    def forward(self, P, S, x, train, out, nbt):
        N, _, H, W = x.shape
        xs = E(N, H, W, self.Cin, dtype=self.adt)
        L.nchw_to_nhwc(x, xs, N, self.Cin, H, W)
        y, c = self.block.forward(P, S, xs, N, H, W, train, 1, nbt)
        yo = E(N, self.Cout, c.OH, c.OW)
        L.nhwc_to_nchw(y, yo, N, self.Cout, c.OH, c.OW)
        ro = None
        if out:
            ro = E(N, self.Cout, c.OH, c.OW)
            L.nhwc_to_nchw(c.bn.raw, ro, N, self.Cout, c.OH, c.OW)
        c.N, c.H, c.W = N, H, W
        return yo, ro, c

    def backward(self, P, c, dy, draw_extra, G, need_dw, need_dx):
        """dy / draw_extra: NCHW fp32 gradients on the block output / on the raw conv output (either may be None)."""
        N, OH, OW = c.N, c.OH, c.OW
        draw = None
        if dy is not None:
            g = E(N, OH, OW, self.Cout, dtype=self.adt)
            L.nchw_to_nhwc(dy, g, N, self.Cout, OH, OW)
            draw = self.block.bn.backward(P, c.bn, g, G, False, need_dw)
        elif need_dw:
            G["bn.weight"].zero_()
            G["bn.bias"].zero_()
        if draw_extra is not None:
            t = E(N, OH, OW, self.Cout, dtype=self.adt)
            L.nchw_to_nhwc(draw_extra, t, N, self.Cout, OH, OW)
            draw = t if draw is None else draw.add_(t)
        dx = self.block.backward_raw(P, c, draw, G, False, need_dw, need_dx)
        if dx is None:
            return None
        dxo = E(N, self.Cin, c.H, c.W)
        L.nhwc_to_nchw(dx, dxo, N, self.Cin, c.H, c.W)
        return dxo


import os as _os

# Tensor-core weight gradients on a side stream: OFF by default (FMRI_WGRAD_STREAM=1 enables). Measured on one B200: -0.7 % step
# time at batch 4096 (the GPU is power-capped, so overlapping tensor-pipe and HBM-bound kernels buys little), but 2x slower at
# batch 64, where the step is launch-bound and the stream switches / record_stream bookkeeping dominate.
WGRAD_SIDE_STREAM = _os.environ.get("FMRI_WGRAD_STREAM", "0") == "1"
_SIDE = None


def side_stream():
    global _SIDE
    if _SIDE is None:
        _SIDE = torch.cuda.Stream()
    return _SIDE


def join_side():
    """The current stream waits for every weight-gradient launch issued so far (before anything reads a gradient bucket)."""
    if _SIDE is not None:
        torch.cuda.current_stream().wait_stream(_SIDE)


def side_into(stream):
    """`stream` (the gradient all-reduce stream) waits for the weight-gradient side stream."""
    if _SIDE is not None:
        stream.wait_stream(_SIDE)


def _backward_chain(blocks, ctxs, P, dy, G, acc, need_dw, relu_mask=None):
    """Backward through a stack of ConvBlocks (last block first); returns dx of blocks[0]. relu_mask = (y, bits): the layer
    below blocks[0] is bias+ReLU without BatchNorm, and its ReLU backward rides in blocks[0]'s data-gradient epilogue."""
    for i in range(len(blocks) - 1, -1, -1):
        dy = blocks[i].backward(P, ctxs[i], dy, G, acc, need_dw, True, relu_mask if i == 0 else None)
    return dy


# ====================================================================================================== linear pieces
class LinearOp:
    """nn.Linear on [M, K] row-major activations. bf16 mode keeps two bf16 packs of the fp32 master weight: wp [N, Kp]
    (fprop) and wpt [K, Np] (dgrad), pitches padded to 8 elements (16-byte TMA pitch; K = 3620 voxels -> 3624).

    chw = (C, h, w): the layer consumes a flattened conv output. The reference flattens NCHW (vae_gan.py:89,180), the conv
    kernels here produce NHWC; instead of transposing the activations (and their gradients) every step, the PACKS carry the
    columns in (h, w, c) order -- the [M, K] activation matrix is then just a view of the NHWC tensor -- and the weight
    gradient is computed in that order and transposed back into the reference layout once (a pass over K*N weights instead
    of four passes over M*K activations)."""

    def __init__(self, wname, bname, N, K, adt, chw=None):
        self.wname, self.bname, self.N, self.K, self.adt = wname, bname, N, K, adt
        self.Kp, self.Np = _pad8(K), _pad8(N)
        self.wp = self.wpt = None
        self.chw = chw if adt == BF16 else None
        if self.chw is not None and (self.Kp != K or self.Np != N or chw[0] * chw[1] * chw[2] != K):
            raise L.FmriError("permuted linear packs need unpadded K and N")
        self._dw = None

    def names(self):
        return [self.wname] + ([self.bname] if self.bname else [])

    def refresh(self, P, inplace=True):
        if self.adt != BF16:
            return
        if self.wp is None or not inplace:
            self.wp, self.wpt = Z(self.N, self.Kp, dtype=BF16), Z(self.K, self.Np, dtype=BF16)
        if self.chw is not None:
            C_, h, w = self.chw
            L.nchw_to_nhwc(P[self.wname], self.wp, self.N, C_, h, w)      # every weight row: [C][hw] -> [hw][C], bf16
            L.nchw_to_nhwc(self.wp, self.wpt, 1, self.N, 1, self.K)       # [N][K] -> [K][N]
            return
        L.linear_pack_weights(L.linear_desc(1, self.N, self.K, BF16), P[self.wname], self.wp, self.Kp, self.wpt, self.Np)

    def packs(self):
        return (self.wp, self.wpt)

    def fprop(self, P, x, ldx, M, y, ldy, act=L.ACT_NONE, packs=None):
        wp = (packs or self.packs())[0]
        L.linear_fprop(L.linear_desc(M, self.N, self.K, self.adt), x, ldx, P[self.wname], wp, self.Kp,
                       P[self.bname] if self.bname else None, act, y, ldy)

    def dgrad(self, P, dy, lddy, M, dx, lddx, accumulate=False, packs=None):
        wpt = (packs or self.packs())[1]
        L.linear_dgrad(L.linear_desc(M, self.N, self.K, self.adt), dy, lddy, P[self.wname], wpt, self.Np, dx, lddx,
                       accumulate)

    def wgrad(self, x, ldx, dy, lddy, M, G, acc):
        if self.chw is not None:   # gradient in (h, w, c) column order, then back to the reference's (c, h, w)
            if self._dw is None:
                self._dw = E(self.N, self.K)
            C_, h, w = self.chw
            L.linear_wgrad(L.linear_desc(M, self.N, self.K, self.adt), x, ldx, dy, lddy, self._dw, False)
            L.nhwc_to_nchw(self._dw, G[self.wname], self.N, C_, h, w, acc)
        else:
            L.linear_wgrad(L.linear_desc(M, self.N, self.K, self.adt), x, ldx, dy, lddy, G[self.wname], acc)
        if self.bname:
            if not acc:
                G[self.bname].zero_()
            if lddy != self.N:
                raise L.FmriError("bias gradient needs a dense dy")
            L.colsum(dy, M, self.N, G[self.bname])


class LinearBlock:
    """nn.Linear(bias=False) -> BatchNorm1d -> ReLU (Encoder.fc, Decoder.fc, Discriminator.fc[0:3], CognitiveEncoder.fc1).
    The pre-BN output is kept in fp32 (split-K accumulates in fp32; BN statistics from unrounded values)."""

    def __init__(self, wname, bn_prefix, N, K, adt, chw=None):
        self.lin = LinearOp(wname, None, N, K, adt, chw)
        self.bn = BatchNorm(bn_prefix, N)
        self.N, self.K, self.adt = N, K, adt
        self.nhwc_in = self.lin.chw is not None   # the input matrix is the NHWC conv output itself

    def names(self):
        return self.lin.names() + self.bn.names()

    def refresh(self, P, inplace=True):
        self.lin.refresh(P, inplace)

    def forward(self, P, S, x, ldx, M, train, n_updates, nbt=None):
        raw = E(M, self.N)
        self.lin.fprop(P, x, ldx, M, raw, self.N)
        y, cb = self.bn.forward(P, S, raw, M, self.adt, True, train, n_updates, None, nbt)
        return y, Ctx(x=x, ldx=ldx, M=M, bn=cb, packs=self.lin.packs())

    def backward(self, P, c, dy, G, acc, need_dw, need_dx, dx_dtype=None):
        draw = self.bn.backward(P, c.bn, dy, G, acc, need_dw)  # dtype of dy
        if draw.dtype != self.adt:
            t = E(c.M, self.N, dtype=self.adt)
            L.cast2d(draw, self.N, t, self.N, c.M, self.N)
            draw = t
        if need_dw:
            self.lin.wgrad(c.x, c.ldx, draw, self.N, c.M, G, acc)
        dx = None
        if need_dx:
            dx = E(c.M, self.K, dtype=dx_dtype or self.adt)
            self.lin.dgrad(P, draw, self.N, c.M, dx, self.K, packs=c.packs)
        return dx

    def backward_pair(self, P, c, dya, dyb, G, acc, dx_dtype=None):
        """Upstream a -> the parameter gradients, upstream b -> the input gradient, with one BatchNorm backward for both."""
        M = c.M
        draw = self.bn.backward_pair(P, c.bn, dya, dyb, G, acc, True)
        if draw.dtype != self.adt:
            t = E(2 * M, self.N, dtype=self.adt)
            L.cast2d(draw, self.N, t, self.N, 2 * M, self.N)
            draw = t
        self.lin.wgrad(c.x, c.ldx, draw[:M], self.N, M, G, acc)
        dx = E(M, self.K, dtype=dx_dtype or self.adt)
        self.lin.dgrad(P, draw[M:], self.N, M, dx, self.K, packs=c.packs)
        return dx


class LatentHeads:
    """l_mu / l_var (vae_gan.py:84-85, 206-207): two Linear(1024, z) + bias writing the halves of one [B, 2z] fp32 matrix."""

    def __init__(self, z, K, adt):
        self.z, self.K, self.adt = z, K, adt
        self.mu = LinearOp("l_mu.weight", "l_mu.bias", z, K, adt)
        self.lv = LinearOp("l_var.weight", "l_var.bias", z, K, adt)

    def names(self):
        return self.mu.names() + self.lv.names()

    def refresh(self, P, inplace=True):
        self.mu.refresh(P, inplace)
        self.lv.refresh(P, inplace)

    def forward(self, P, h, M):
        z = self.z
        ycat = E(M, 2 * z)
        self.mu.fprop(P, h, self.K, M, ycat[:, :z], 2 * z)
        self.lv.fprop(P, h, self.K, M, ycat[:, z:], 2 * z)
        return ycat, Ctx(h=h, M=M, pm=self.mu.packs(), pl=self.lv.packs())

    def backward(self, P, c, dycat, G, acc, need_dw, need_lv=True):
        """dycat: [M, 2z] in adt (d mu | d logvar). Returns d h as fp32 [M, K]."""
        z, M = self.z, c.M
        dh = E(M, self.K)
        self.mu.dgrad(P, dycat[:, :z], 2 * z, M, dh, self.K, False, c.pm)
        if need_lv:
            self.lv.dgrad(P, dycat[:, z:], 2 * z, M, dh, self.K, True, c.pl)
        if need_dw:
            for op, sl in ((self.mu, dycat[:, :z]), (self.lv, dycat[:, z:])):
                if op is self.lv and not need_lv:
                    continue
                L.linear_wgrad(L.linear_desc(M, z, self.K, self.adt), c.h, self.K, sl, 2 * z, G[op.wname], acc)
            # bias gradients: column sums of the dense [M, 2z] matrix into a scratch, then split
            tmp = Z(2 * z)
            L.colsum(dycat, M, 2 * z, tmp)
            for op, sl in ((self.mu, tmp[:z]), (self.lv, tmp[z:])):
                if op is self.lv and not need_lv:
                    continue
                L.axpby_tanh_bwd(1.0, sl, 1.0, G[op.bname] if acc else None, None, G[op.bname])
        return dh


# ====================================================================================================== Encoder
class EncoderNet:
    """Encoder (vae_gan.py:63-96): 3 x EncoderBlock (3->64->128->256) -> flatten -> Linear -> BN1d -> ReLU -> l_mu | l_var."""

    def __init__(self, cfg, z, adt):
        ch = cfg["encoder_channels"]
        self.cfg, self.z, self.adt = cfg, z, adt
        self.C0 = ch[0]
        self.bn0 = BatchNorm("conv.0.bn.", ch[0])
        self.blocks = [ConvBlock(f"conv.{i}.", ch[i - 1], ch[i], False, 0, adt) for i in (1, 2)]
        self.fi = cfg["fc_input"]
        self.fc = LinearBlock("fc.0.weight", "fc.1.", cfg["fc_output"], self.fi ** 2 * ch[2], adt, (ch[2], self.fi, self.fi))
        self.heads = LatentHeads(z, cfg["fc_output"], adt)
        self.Clast = ch[2]
        self._ews = None
        self._ewsm = _EdgeWs()

    def param_names(self):
        n = ["conv.0.conv.weight"] + self.bn0.names()
        for b in self.blocks:
            n += b.names()
        return n + self.fc.names() + self.heads.names()

    def refresh(self, P, inplace=True):
        for m in self.blocks + [self.fc, self.heads]:
            m.refresh(P, inplace)

    def _edge(self, N, H, W):
        d = L.edge_desc(N, H, W, self.C0, 2, self.adt)
        self._ews = self._ewsm.get(d)
        return d

    def forward(self, P, S, x, train=True, n_updates=1, nbt=None):
        """x: [B,3,H,W] fp32 NCHW. Returns (ycat [B, 2z] fp32 = mu | logvar, ctx)."""
        B, _, H, W = x.shape
        d0 = self._edge(B, H, W)
        OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        raw0 = E(B, OH, OW, self.C0, dtype=self.adt)
        L.edge_in_fprop(d0, [x], B, P["conv.0.conv.weight"], None, L.ACT_NONE, raw0, self._ews)
        y, c0 = self.bn0.forward(P, S, raw0, B * OH * OW, self.adt, True, train, n_updates, None, nbt)
        cs = []
        h, w = OH, OW
        for b in self.blocks:
            y, c = b.forward(P, S, y, B, h, w, train, n_updates, nbt)
            cs.append(c)
            h, w = c.OH, c.OW
        if self.fc.nhwc_in:   # the fc packs carry their columns in (h, w, c) order: no activation transpose
            flat = y.view(B, -1)
        else:
            flat = E(B, self.Clast * h * w, dtype=self.adt)
            L.nhwc_to_nchw(y, flat, B, self.Clast, h, w)  # the reference flattens NCHW (vae_gan.py:89)
        hfc, cfc = self.fc.forward(P, S, flat, flat.shape[1], B, train, n_updates, nbt)
        ycat, ch = self.heads.forward(P, hfc, B)
        return ycat, Ctx(x=x, d0=d0, c0=c0, blocks=cs, fc=cfc, heads=ch, B=B, hw=(h, w))

    def backward(self, P, c, dycat, G, acc=False, need_dw=True, need_lv=True, after_fc=None):
        """dycat [B, 2z] in adt. Parameter gradients into G (no image gradient: the input is data). after_fc(): called once the
        gradients of fc / l_mu / l_var (93 % of the encoder's parameters) are issued -- the data-parallel engine starts their
        all-reduce there, so that only the small conv part is exchanged after the last backward kernel."""
        B = c.B
        dh = self.heads.backward(P, c.heads, dycat, G, acc, need_dw, need_lv)
        dflat = self.fc.backward(P, c.fc, dh, G, acc, need_dw, True)
        if after_fc is not None:
            after_fc()
        h, w = c.hw
        if self.fc.nhwc_in:
            dy = dflat.view(B, h, w, self.Clast)
        else:
            dy = E(B, h, w, self.Clast, dtype=self.adt)
            L.nchw_to_nhwc(dflat, dy, B, self.Clast, h, w)
        dy = _backward_chain(self.blocks, c.blocks, P, dy, G, acc, need_dw)
        draw0 = self.bn0.backward(P, c.c0, dy, G, acc, need_dw)
        if need_dw:
            L.edge_in_wgrad(c.d0, [c.x], B, draw0, G["conv.0.conv.weight"], acc, self._ews)


# ====================================================================================================== Decoder
class DecoderNet:
    """Decoder (vae_gan.py:99-132): Linear -> BN1d -> ReLU -> view [B,size,f,f] -> 3 x DecoderBlock -> Conv2d(C,3,5,s1)+bias -> tanh."""

    def __init__(self, cfg, z, adt, size=256):
        dc = cfg["decoder_channels"]
        self.cfg, self.z, self.adt, self.size = cfg, z, adt, size
        self.fi = cfg["fc_input"]
        self.fc = LinearBlock("fc.0.weight", "fc.1.", self.fi ** 2 * size, z, adt)
        chans = [(size, size), (size, dc[1]), (dc[1], dc[2])]
        self.blocks = [ConvBlock(f"conv.{i}.", ci, co, True, cfg["output_pad_dec"][i], adt)
                       for i, (ci, co) in enumerate(chans)]
        self.Cl = dc[2]
        self._ews = None
        self._ewsm = _EdgeWs()

    def param_names(self):
        n = self.fc.names()
        for b in self.blocks:
            n += b.names()
        return n + ["conv.3.0.weight", "conv.3.0.bias"]

    def refresh(self, P, inplace=True):
        for m in [self.fc] + self.blocks:
            m.refresh(P, inplace)

    def forward(self, P, S, zin, train=True, n_updates=1, nbt=None):
        """zin [B, z] fp32 (row pitch may exceed z). Returns (img [B,3,H,W] fp32 NCHW after tanh, ctx)."""
        B = zin.shape[0]
        ld = zin.stride(0)
        if self.adt == BF16:
            zb = E(B, self.z, dtype=BF16)
            L.cast2d(zin, ld, zb, self.z, B, self.z)
        elif ld != self.z:
            zb = E(B, self.z)
            L.cast2d(zin, ld, zb, self.z, B, self.z)
        else:
            zb = zin
        hfc, cfc = self.fc.forward(P, S, zb, self.z, B, train, n_updates, nbt)
        f = self.fi
        y = E(B, f, f, self.size, dtype=self.adt)
        L.nchw_to_nhwc(hfc, y, B, self.size, f, f)  # view(B, size, f, f) of the reference (vae_gan.py:127)
        cs = []
        h = w = f
        for b in self.blocks:
            y, c = b.forward(P, S, y, B, h, w, train, n_updates, nbt)
            cs.append(c)
            h, w = c.OH, c.OW
        d3 = L.edge_desc(B, h, w, self.Cl, 1, self.adt)
        self._ews = self._ewsm.get(d3)
        img = E(B, 3, h, w)
        L.edge_out_fprop(d3, y, P["conv.3.0.weight"], P["conv.3.0.bias"], L.ACT_TANH, img, self._ews)
        return img, Ctx(fc=cfc, blocks=cs, d3=d3, a3=y, img=img, B=B, hw=(h, w))

    def backward(self, P, c, a, gx, b, gy, G, acc=False, need_dw=True, need_dz=False):
        """Upstream image gradient (a*gx + b*gy) (gy may be None), NCHW fp32. Returns dz [B, z] fp32 or None."""
        B = c.B
        h, w = c.hw
        dpre = E(B, 3, h, w)
        L.axpby_tanh_bwd(a, gx, b, gy, c.img, dpre)
        if need_dw:
            L.chansum_nchw(dpre, B, 3, h * w, G["conv.3.0.bias"], acc)
            L.edge_out_wgrad(c.d3, c.a3, dpre, G["conv.3.0.weight"], acc, self._ews)
        dy = torch.empty(c.a3.shape, dtype=self.adt, device=dpre.device)
        L.edge_out_dgrad(c.d3, dpre, P["conv.3.0.weight"], dy, self._ews)
        dy = _backward_chain(self.blocks, c.blocks, P, dy, G, acc, need_dw)
        f = self.fi
        dflat = E(B, self.size * f * f, dtype=self.adt)
        L.nhwc_to_nchw(dy, dflat, B, self.size, f, f)
        return self.fc.backward(P, c.fc, dflat, G, acc, need_dw, need_dz, dx_dtype=F32)

    def backward_pair(self, P, c, a, gx, b, gy, a2, gx2, G, acc=False):
        """Two sweeps through one saved forward state: upstream (a*gx + b*gy) -> parameter gradients into G, upstream a2*gx2
        -> dz. The same as backward(P, c, a, gx, b, gy, G, acc, True, False) followed by backward(P, c, a2, gx2, 0, None, None,
        need_dw=False, need_dz=True), with every BatchNorm backward shared by the two and every data gradient run once over
        the two upstreams stacked along the batch (the 3-channel output conv's data gradient stays two launches: its kernel
        does not give the same bits for a doubled batch at every size). Returns dz [B, z] fp32."""
        B = c.B
        h, w = c.hw
        dpre = E(2 * B, 3, h, w)
        L.axpby_tanh_bwd(a, gx, b, gy, c.img, dpre[:B])
        L.axpby_tanh_bwd(a2, gx2, 0.0, None, c.img, dpre[B:])
        L.chansum_nchw(dpre[:B], B, 3, h * w, G["conv.3.0.bias"], acc)
        L.edge_out_wgrad(c.d3, c.a3, dpre[:B], G["conv.3.0.weight"], acc, self._ews)
        dy = E(2 * B, h, w, self.Cl, dtype=self.adt)
        L.edge_out_dgrad(c.d3, dpre[:B], P["conv.3.0.weight"], dy[:B], self._ews)
        L.edge_out_dgrad(c.d3, dpre[B:], P["conv.3.0.weight"], dy[B:], self._ews)
        for i in range(len(self.blocks) - 1, -1, -1):
            dy = self.blocks[i].backward_pair(P, c.blocks[i], dy[:B], dy[B:], G, acc, True)
        f = self.fi
        dflat = E(2 * B, self.size * f * f, dtype=self.adt)
        L.nhwc_to_nchw(dy, dflat, 2 * B, self.size, f, f)
        return self.fc.backward_pair(P, c.fc, dflat[:B], dflat[B:], G, acc, dx_dtype=F32)


# ====================================================================================================== Discriminator
class DiscriminatorNet:
    """Discriminator (vae_gan.py:135-187) on the batch-concatenation of up to three image sources (the torch.cat of
    :165 is never materialised): Conv2d(3,32,5,s)+bias+ReLU -> 3 x EncoderBlock -> [feature tap = raw output of block 3]
    -> flatten -> Linear -> BN1d -> ReLU -> Linear(.,1)+bias -> sigmoid."""

    def __init__(self, cfg, adt, recon_level=3):
        ch = cfg["discrim_channels"]
        if recon_level not in (1, 2, 3):   # vae_gan.py:169-173: conv[0] is a plain Sequential and cannot be the tap
            raise L.FmriError("recon_level must be 1, 2 or 3 (the EncoderBlock whose raw conv output is the feature tap)")
        self.cfg, self.adt, self.level = cfg, adt, int(recon_level)
        self.C0, self.stride0 = ch[0], cfg["stride_gan"]
        self.blocks = [ConvBlock(f"conv.{i}.", ch[i - 1], ch[i], False, 0, adt) for i in (1, 2, 3)]
        self.Cl = ch[3]
        self.fg = cfg["fc_input_gan"]
        self.fc = LinearBlock("fc.0.weight", "fc.1.", cfg["fc_output_gan"], self.fg ** 2 * ch[3], adt, (ch[3], self.fg, self.fg))
        self.F = cfg["fc_output_gan"]
        self._ews = None
        self._ewsm = _EdgeWs()

    def param_names(self):
        n = ["conv.0.0.weight", "conv.0.0.bias"]
        for b in self.blocks:
            n += b.names()
        return n + self.fc.names() + ["fc.3.weight", "fc.3.bias"]

    def refresh(self, P, inplace=True):
        for m in self.blocks + [self.fc]:
            m.refresh(P, inplace)

    def forward(self, P, S, imgs, train=True, n_updates=1, head=True, nbt=None, head_updates=1):
        """imgs: list of 1..3 NCHW fp32 tensors of equal shape [Bs,3,H,W]. Returns (NHWC feature tap = raw conv output of block
        `recon_level`, p [N] or None, ctx). head=False is the reference's "REC" pass, which stops after block `recon_level`
        (vae_gan.py:166-175: the later blocks neither run nor update their BatchNorm statistics).
        n_updates: BN running-stat updates of the conv blocks (2 when one pass stands for the reference's REC + GAN passes,
        vae_gan.py:284-285; only valid for recon_level 3, where both passes run every block); head_updates: of fc[1], which
        only the GAN pass reaches."""
        if n_updates > 1 and self.level != 3:
            raise L.FmriError("one pass standing for REC + GAN needs recon_level 3 (lower taps update fewer BatchNorm layers)")
        Bs, _, H, W = imgs[0].shape
        N = Bs * len(imgs)
        d0 = L.edge_desc(N, H, W, self.C0, self.stride0, self.adt)
        self._ews = self._ewsm.get(d0)
        OH, OW = (H - 1) // self.stride0 + 1, (W - 1) // self.stride0 + 1
        y0 = E(N, OH, OW, self.C0, dtype=self.adt)
        L.edge_in_fprop(d0, imgs, Bs, P["conv.0.0.weight"], P["conv.0.0.bias"], L.ACT_RELU, y0, self._ews)
        mask0 = None
        if train and self.adt == BF16 and self.C0 == 32:   # ReLU mask as 4 B per pixel for the fused backward (see _backward_chain)
            mask0 = torch.empty(N * OH * OW, dtype=torch.int32, device=y0.device)
            L.relu_bitmask(y0, N * OH * OW, self.C0, mask0)
        cs, y, h, w = [], y0, OH, OW
        for b in (self.blocks if head else self.blocks[:self.level]):
            y, c = b.forward(P, S, y, N, h, w, train, n_updates, nbt)
            cs.append(c)
            h, w = c.OH, c.OW
        ctx = Ctx(imgs=list(imgs), Bs=Bs, N=N, d0=d0, y0=y0, mask0=mask0, blocks=cs, hw=(h, w), H=H, W=W, hw0=(OH, OW))
        raw3 = cs[self.level - 1].bn.raw
        p = None
        if head:
            if self.fc.nhwc_in:
                flat = y.view(N, -1)
            else:
                flat = E(N, self.Cl * h * w, dtype=self.adt)
                L.nhwc_to_nchw(y, flat, N, self.Cl, h, w)  # ten.view(len(ten), -1) on NCHW (vae_gan.py:180)
            hfc, cfc = self.fc.forward(P, S, flat, flat.shape[1], N, train, head_updates, nbt)
            p = E(N)
            L.head_sigmoid_fwd(hfc, P["fc.3.weight"], P["fc.3.bias"], p, N, self.F)
            ctx.fc, ctx.hfc, ctx.p = cfc, hfc, p
        return raw3, p, ctx

    def _conv0_backward(self, P, c, dy0, G, acc, need_dw, img_slices):
        """ReLU backward of conv[0], its weight/bias gradient, and image gradients for the requested source slices
        (a contiguous range [s0, s1) of sources -> one [ (s1-s0)*Bs, 3, H, W ] fp32 tensor)."""
        dpre = dy0   # conv[0]'s ReLU backward was applied by the data-gradient kernel of block 1 (_backward_chain relu_mask)
        OH, OW = c.hw0
        if need_dw:
            L.edge_in_wgrad(c.d0, c.imgs, c.Bs, dpre, G["conv.0.0.weight"], acc, self._ews, G["conv.0.0.bias"])
        if img_slices is None:
            return None
        s0, s1 = img_slices
        n = (s1 - s0) * c.Bs
        dimg = E(n, 3, c.H, c.W)
        dsl = L.edge_desc(n, c.H, c.W, self.C0, self.stride0, self.adt)
        L.edge_in_dgrad(dsl, dpre[s0 * c.Bs:s1 * c.Bs], P["conv.0.0.weight"], dimg, self._ews)
        return dimg

    def backward_gan(self, P, c, gp, G, acc=False, need_dw=True, img_slices=None):
        """Backward of the class-score path from gp = dL/dp [N] fp32. Returns image gradients for `img_slices`."""
        N = c.N
        dh = E(N, self.F, dtype=self.adt)
        if need_dw and not acc:
            G["fc.3.weight"].zero_()
            G["fc.3.bias"].zero_()
        L.head_sigmoid_bwd(c.hfc, P["fc.3.weight"], c.p, gp, dh, G["fc.3.weight"] if need_dw else None,
                           G["fc.3.bias"] if need_dw else None, N, self.F)
        dflat = self.fc.backward(P, c.fc, dh, G, acc, need_dw, True)
        h, w = c.hw
        if self.fc.nhwc_in:
            dy = dflat.view(N, h, w, self.Cl)
        else:
            dy = E(N, h, w, self.Cl, dtype=self.adt)
            L.nchw_to_nhwc(dflat, dy, N, self.Cl, h, w)
        dy = _backward_chain(self.blocks, c.blocks, P, dy, G, acc, need_dw, (c.y0, c.mask0))
        return self._conv0_backward(P, c, dy, G, acc, need_dw, img_slices)

    def backward_pair(self, P, c, gp, draw3, G, acc=False, live=(0, 2), after_dw=None):
        """The class path (backward_gan with img_slices=(1, 3)) and the feature tap of recon_level 3 (backward_rec with
        need_dw=False, img_slices=(1, 2)) in one sweep over the saved forward state of three sources: below the tap both
        upstreams share every BatchNorm backward, and block 2's data gradient runs once over the two. after_dw(): called once the last weight gradient is issued. Returns (image gradient of the class path for
        sources 1 and 2 [2Bs, 3, H, W], image gradient of the feature tap for source 1 [Bs, 3, H, W])."""
        if self.level != 3 or len(c.imgs) != 3:
            raise L.FmriError("the paired discriminator sweep needs recon_level 3 and three image sources")
        Bs, N = c.Bs, c.N
        (b1, b2, b3), (c1, c2, c3) = self.blocks, c.blocks
        dh = E(N, self.F, dtype=self.adt)
        if not acc:
            G["fc.3.weight"].zero_()
            G["fc.3.bias"].zero_()
        L.head_sigmoid_bwd(c.hfc, P["fc.3.weight"], c.p, gp, dh, G["fc.3.weight"], G["fc.3.bias"], N, self.F)
        dflat = self.fc.backward(P, c.fc, dh, G, acc, True, True)
        h, w = c.hw
        if self.fc.nhwc_in:
            dy = dflat.view(N, h, w, self.Cl)
        else:
            dy = E(N, h, w, self.Cl, dtype=self.adt)
            L.nchw_to_nhwc(dflat, dy, N, self.Cl, h, w)
        # block 3: the class path through its BatchNorm; the feature tap enters at its raw conv output, live sources only
        dy2 = E(2 * N, c3.d.H, c3.d.W, b3.Cin, dtype=self.adt)
        dy2b = dy2[N:]
        draw =b3.bn.backward(P, c3.bn, dy, G, acc, True)
        w3 = P[b3.prefix + "conv.weight"]
        L.conv_dgrad(c3.d, draw, w3, c3.pack_d, dy2[:N])
        b3.backward_raw(P, c3, draw, G, acc, True, False)
        l0, l1 = live
        if l0 > 0:
            dy2b[:l0 * Bs].zero_()
        if l1 < 3:
            dy2b[l1 * Bs:].zero_()
        L.conv_dgrad(b3.desc((l1 - l0) * Bs, c3.d.H, c3.d.W), draw3[l0 * Bs:l1 * Bs], w3, c3.pack_d, dy2b[l0 * Bs:l1 * Bs])
        # block 2: both upstreams
        dy1 = b2.backward_pair(P, c2, dy2[:N], dy2b, G, acc, True)
        # block 1: the class path over all N images, the feature tap on source 1 only (the BatchNorm sums of both run over N)
        per = c1.OH * c1.OW
        draw = b1.bn.backward_pair(P, c1.bn, dy1[:N], dy1[N:], G, acc, True, rows_b=(Bs * per, Bs * per))
        OH, OW = c.hw0
        dy0 = E(N + Bs, OH, OW, self.C0, dtype=self.adt)
        w1 = P[b1.prefix + "conv.weight"]
        L.conv_dgrad(c1.d, draw[:N], w1, c1.pack_d, dy0[:N], (c.y0, c.mask0))
        bits = c.mask0[Bs * OH * OW:2 * Bs * OH * OW] if c.mask0 is not None else None
        L.conv_dgrad(b1.desc(Bs, c1.d.H, c1.d.W), draw[N:], w1, c1.pack_d, dy0[N:], (c.y0[Bs:2 * Bs], bits))
        b1.backward_raw(P, c1, draw[:N], G, acc, True, False)
        # conv[0]: weight gradient of the class path, image gradients of its sources 1, 2 and of the feature tap's source 1
        # (two launches: the edge kernel does not give the same bits for the merged 3Bs rows at every batch size)
        L.edge_in_wgrad(c.d0, c.imgs, Bs, dy0[:N], G["conv.0.0.weight"], acc, self._ews, G["conv.0.0.bias"])
        if after_dw is not None:
            after_dw()
        dimg = E(N, 3, c.H, c.W)
        w0 = P["conv.0.0.weight"]
        for n, src, dst in ((2 * Bs, dy0[Bs:N], dimg[:2 * Bs]), (Bs, dy0[N:], dimg[2 * Bs:])):
            L.edge_in_dgrad(L.edge_desc(n, c.H, c.W, self.C0, self.stride0, self.adt), src, w0, dst, self._ews)
        return dimg[:2 * Bs], dimg[2 * Bs:]

    def backward_rec(self, P, c, draw3, G=None, acc=False, need_dw=False, img_slices=None, live=None):
        """Backward of the feature-tap path from a gradient on the raw conv output of block 3 [N,h,w,C] (adt).
        live = (s0, s1): only sources [s0, s1) of draw3 are non-zero (the feature-matching loss compares x and x_tilde; the
        x_p third gets no gradient at the tap, train_vgan_stage1.py:369 / vae_gan.py:313).
        Data-gradient-only fast path (need_dw False): block 3's data gradient runs on the live sources only
        (the rest of its output is exactly zero), and block 1's BN apply + data gradient + conv[0] run on the requested image
        slice only -- BatchNorm's coupling of the whole 3B batch is kept by running every BN's backward SUMS over all of it."""
        top = self.level - 1
        mask0 = (c.y0, c.mask0)
        if top != 2:   # feature tap below block 3: plain chain from the tap's block down
            dy = self.blocks[top].backward_raw(P, c.blocks[top], draw3, G, acc, need_dw, True, mask0 if top == 0 else None)
            if top > 0:
                dy = _backward_chain(self.blocks[:top], c.blocks[:top], P, dy, G, acc, need_dw, mask0)
            return self._conv0_backward(P, c, dy, G, acc, need_dw, img_slices)
        if not need_dw and img_slices is not None and len(c.imgs) > 1:
            Bs = c.Bs
            l0, l1 = live if live is not None else (0, len(c.imgs))
            b3, c3 = self.blocks[2], c.blocks[2]
            dy = torch.empty(c3.x.shape, dtype=self.adt, device=draw3.device)
            if l0 > 0:
                dy[:l0 * Bs].zero_()
            if l1 < len(c.imgs):
                dy[l1 * Bs:].zero_()
            L.conv_dgrad(b3.desc((l1 - l0) * Bs, c3.d.H, c3.d.W), draw3[l0 * Bs:l1 * Bs], P[b3.prefix + "conv.weight"],
                         c3.pack_d, dy[l0 * Bs:l1 * Bs])
            dy = self.blocks[1].backward(P, c.blocks[1], dy, None, False, False, True)
            s0, s1 = img_slices
            OH, OW = c.hw0
            bits = c.mask0[s0 * Bs * OH * OW:s1 * Bs * OH * OW] if c.mask0 is not None else None
            dy0 = self.blocks[0].backward_dx_slice(P, c.blocks[0], dy, s0 * Bs, s1 * Bs, (c.y0[s0 * Bs:s1 * Bs], bits))
            n = (s1 - s0) * Bs
            dimg = E(n, 3, c.H, c.W)
            L.edge_in_dgrad(L.edge_desc(n, c.H, c.W, self.C0, self.stride0, self.adt), dy0, P["conv.0.0.weight"], dimg,
                            self._ews)
            return dimg
        dy = self.blocks[2].backward_raw(P, c.blocks[2], draw3, G, acc, need_dw, True)
        dy = _backward_chain(self.blocks[:2], c.blocks[:2], P, dy, G, acc, need_dw, mask0)
        return self._conv0_backward(P, c, dy, G, acc, need_dw, img_slices)


# ====================================================================================================== Cognitive encoder
class CognitiveEncoderNet:
    """CognitiveEncoder (vae_gan.py:190-232): Linear(V,1024, no bias) -> BN1d -> ReLU -> l_mu | l_var."""

    def __init__(self, input_size, z, adt):
        self.V, self.z, self.adt = input_size, z, adt
        self.Vp = _pad8(input_size)
        self.fc = LinearBlock("fc1.0.weight", "fc1.1.", 1024, input_size, adt)
        self.heads = LatentHeads(z, 1024, adt)

    def param_names(self):
        return self.fc.names() + self.heads.names()

    def refresh(self, P, inplace=True):
        self.fc.refresh(P, inplace)
        self.heads.refresh(P, inplace)

    def forward(self, P, S, v, train=True, n_updates=1, nbt=None):
        """v [B, V] fp32. bf16 mode stages it as bf16 with the row pitch padded to 8 elements (V = 3620 -> 3624)."""
        B = v.shape[0]
        if self.adt == BF16:
            vb = Z(B, self.Vp, dtype=BF16)
            L.cast2d(v, v.stride(0), vb, self.Vp, B, self.V)
            ld = self.Vp
        else:
            vb, ld = v, v.stride(0)
        hfc, cfc = self.fc.forward(P, S, vb, ld, B, train, n_updates, nbt)
        ycat, ch = self.heads.forward(P, hfc, B)
        return ycat, Ctx(fc=cfc, heads=ch, B=B)

    def backward(self, P, c, dycat, G, acc=False, need_dw=True, need_lv=True):
        dh = self.heads.backward(P, c.heads, dycat, G, acc, need_dw, need_lv)
        self.fc.backward(P, c.fc, dh, G, acc, need_dw, False)


# ====================================================================================================== WAE discriminator
class WaeDiscriminatorNet:
    """WaeDiscriminator (vae_gan.py:499-529): 4 x [Linear + bias + ReLU] -> Linear(512,1) + bias -> sigmoid on latents."""

    def __init__(self, z, adt, dim_h=512):
        self.z, self.adt, self.H = z, adt, dim_h
        dims = [(dim_h, z), (dim_h, dim_h), (dim_h, dim_h), (dim_h, dim_h)]
        self.lins = [LinearOp(f"main.{i}.weight", f"main.{i}.bias", n, k, adt) for i, (n, k) in zip((0, 2, 4, 6), dims)]

    def param_names(self):
        n = []
        for l in self.lins:
            n += l.names()
        return n + ["main.8.weight", "main.8.bias"]

    def refresh(self, P, inplace=True):
        for l in self.lins:
            l.refresh(P, inplace)

    def forward(self, P, zin):
        """zin [M, z] fp32 (row pitch may exceed z). Returns (p [M] fp32, ctx)."""
        M, ld = zin.shape[0], zin.stride(0)
        x = E(M, self.z, dtype=self.adt)
        L.cast2d(zin, ld, x, self.z, M, self.z)
        acts = [x]
        for l in self.lins:
            y = E(M, l.N, dtype=self.adt)
            l.fprop(P, acts[-1], l.K, M, y, l.N, L.ACT_RELU)
            acts.append(y)
        p = E(M)
        L.head_sigmoid_fwd(acts[-1], P["main.8.weight"], P["main.8.bias"], p, M, self.H)
        return p, Ctx(acts=acts, p=p, M=M, packs=[l.packs() for l in self.lins])

    def backward(self, P, c, gp, G, acc=False, need_dw=True, need_dz=False):
        """gp = dL/dp [M] fp32. Returns dz [M, z] fp32 or None."""
        M = c.M
        dy = E(M, self.H, dtype=self.adt)
        if need_dw and not acc:
            G["main.8.weight"].zero_()
            G["main.8.bias"].zero_()
        L.head_sigmoid_bwd(c.acts[-1], P["main.8.weight"], c.p, gp, dy, G["main.8.weight"] if need_dw else None,
                           G["main.8.bias"] if need_dw else None, M, self.H)
        for i in range(len(self.lins) - 1, -1, -1):
            l = self.lins[i]
            dpre = torch.empty_like(dy)
            L.relu_backward(c.acts[i + 1], dy, dpre)
            if need_dw:
                l.wgrad(c.acts[i], l.K, dpre, l.N, M, G, acc)
            if i == 0 and not need_dz:
                return None
            dy = E(M, l.K, dtype=F32 if i == 0 else self.adt)
            l.dgrad(P, dpre, l.N, M, dy, l.K, packs=c.packs[i])
        return dy
