"""Inference fast path (SURVEY.md 8f-2): the eval-mode forward of the reference's composites with BatchNorm FOLDED into
the preceding layer, and the image-quality metrics it is evaluated with, all as launches of libfmri_b200.so.

Reference behaviour reproduced (all paths relative to /root/reference):
  * VaeGan.forward eval branch (models/vae_gan.py:288-297): encoder -> reparameterize (it STILL samples in eval mode) ->
    decoder; x is None -> decoder(randn(gen_size, z)). VaeGanCognitive eval (:397-402) is the same with the CognitiveEncoder.
    WaeGan / WaeGanCognitive eval (:484-496, :575-578) decode the mean (no sampling).
  * BatchNorm in eval mode uses the running statistics (:21,54,80,108,158,200): y = gamma * (x - rm) / sqrt(rv + eps) + beta.
    Every BatchNorm here follows a bias-free conv / linear layer, so it folds exactly: conv(x, w * s) + (beta - rm * s),
    s = gamma / sqrt(rv + eps) per output channel (fmri_bn_fold). The folded layer runs as ONE kernel: implicit GEMM with a
    bias + ReLU epilogue. An eval forward is 9 (encoder) + 5 (decoder) launches instead of 27 + 17, and no activation is
    written twice.
  * metrics: PearsonCorrelation, StructuralSimilarity (train/train_utils.py:267-425), nn.MSELoss -- as the train scripts'
    per-epoch evaluation computes them (train/train_vgan_stage1.py:489-560).
  * identification (the question objective_assessment, train_utils.py:752, answers by sampling distractors on the host):
    is reconstruction i more similar to its own stimulus than to the others? similarity_matrix() gives every PCC or SSIM
    value of reconstructions against stimuli, identification() the wins per reconstruction and the exact expected n-way
    accuracy over all distractor draws. Over a test set:

        r = Reconstructor(checkpoint, hp.CFG64, z=128, kind="cognitive")
        recon = torch.cat([r(fmri_batch, sample=False) for fmri_batch in test_fmri])       # [N, 3, 64, 64]
        S = similarity_matrix(recon, stimuli, metric="ssim")                               # [N, N], row i vs stimulus j
        wins, acc = identification(S, ns=(2, 5, 10))                                       # acc[0]: pairwise accuracy
"""
from __future__ import annotations

from collections import OrderedDict

import torch

from . import lib as L
from . import nets as NN
from .nets import BF16, F32, F64, E, Z


def _fold(w, inner, Cc, S, P, pre):
    wf, bf = torch.empty_like(w), E(Cc)
    L.bn_fold(w, inner, Cc, S[pre + "running_mean"], S[pre + "running_var"], P[pre + "weight"], P[pre + "bias"], NN.BN_EPS,
              wf, bf)
    return wf, bf


class _FoldedConv:
    """ConvBlock (EncoderBlock / DecoderBlock) in eval mode: conv + folded-BN bias + ReLU in one launch."""

    def __init__(self, blk, P, S):
        self.blk = blk
        w = P[blk.prefix + "conv.weight"]
        inner = 25 if blk.transposed else blk.Cin * 25
        self.w, self.b = _fold(w, inner, blk.Cout, S, P, blk.prefix + "bn.")
        self.pack = None
        if blk.adt == BF16:
            d = blk.desc(1, 8, 8)
            self.pack = E(L.conv_pack_elems(d), dtype=BF16)
            L.conv_pack_weights(d, self.w, self.pack, None)

    def __call__(self, x, N, H, W):
        d = self.blk.desc(N, H, W)
        OH, OW = L.conv_out_hw(d)
        y = E(N, OH, OW, self.blk.Cout, dtype=self.blk.adt)
        L.conv_fprop(d, x, self.w, self.pack, self.b, L.ACT_RELU, y)
        return y, OH, OW


class _FoldedLinear:
    """LinearBlock (Linear, no bias -> BatchNorm1d -> ReLU) in eval mode: GEMM + bias + ReLU epilogue."""

    def __init__(self, lb, P, S):
        self.lb = lb
        w = P[lb.lin.wname]
        self.w, self.b = _fold(w, lb.K, lb.N, S, P, lb.bn.prefix)
        self.Kp = lb.lin.Kp
        self.wp = None
        if lb.adt == BF16:
            self.wp = Z(lb.N, self.Kp, dtype=BF16)
            L.linear_pack_weights(L.linear_desc(1, lb.N, lb.K, BF16), self.w, self.wp, self.Kp, None, 0)

    def __call__(self, x, ldx, M):
        y = E(M, self.lb.N, dtype=self.lb.adt)
        L.linear_fprop(L.linear_desc(M, self.lb.N, self.lb.K, self.lb.adt), x, ldx, self.w, self.wp, self.Kp, self.b,
                       L.ACT_RELU, y, self.lb.N)
        return y


class FoldedEncoder:
    """Encoder (models/vae_gan.py:63-96) in eval mode, BatchNorm folded."""

    def __init__(self, P, S, cfg, z, adt=BF16):
        self.net = NN.EncoderNet(cfg, z, adt)
        self.net.heads.refresh(P)
        self.P = P
        n = self.net
        self.w0, self.b0 = _fold(P["conv.0.conv.weight"], 75, n.C0, S, P, "conv.0.bn.")
        self.blocks = [_FoldedConv(b, P, S) for b in n.blocks]
        self.fc = _FoldedLinear(n.fc, P, S)

    def __call__(self, x):
        n = self.net
        B, _, H, W = x.shape
        d0 = n._edge(B, H, W)
        h, w = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        y = E(B, h, w, n.C0, dtype=n.adt)
        L.edge_in_fprop(d0, [x], B, self.w0, self.b0, L.ACT_RELU, y, n._ews)
        for f in self.blocks:
            y, h, w = f(y, B, h, w)
        flat = E(B, n.Clast * h * w, dtype=n.adt)
        L.nhwc_to_nchw(y, flat, B, n.Clast, h, w)
        hfc = self.fc(flat, flat.shape[1], B)
        ycat, _ = n.heads.forward(self.P, hfc, B)
        return ycat


class FoldedCognitiveEncoder:
    """CognitiveEncoder (models/vae_gan.py:190-232) in eval mode, BatchNorm folded."""

    def __init__(self, P, S, z, voxels, adt=BF16):
        self.net = NN.CognitiveEncoderNet(voxels, z, adt)
        self.net.heads.refresh(P)
        self.P = P
        self.fc = _FoldedLinear(self.net.fc, P, S)

    def __call__(self, v):
        n = self.net
        B = v.shape[0]
        if n.adt == BF16:
            vb = Z(B, n.Vp, dtype=BF16)
            L.cast2d(v, v.stride(0), vb, n.Vp, B, n.V)
            ld = n.Vp
        else:
            vb, ld = v, v.stride(0)
        hfc = self.fc(vb, ld, B)
        ycat, _ = n.heads.forward(self.P, hfc, B)
        return ycat


class FoldedDecoder:
    """Decoder (models/vae_gan.py:99-132) in eval mode, BatchNorm folded; conv[3] + bias + tanh unchanged."""

    def __init__(self, P, S, cfg, z, adt=BF16, size=256):
        self.net = NN.DecoderNet(cfg, z, adt, size)
        self.P = P
        self.fc = _FoldedLinear(self.net.fc, P, S)
        self.blocks = [_FoldedConv(b, P, S) for b in self.net.blocks]

    def __call__(self, zin):
        n = self.net
        B, ld = zin.shape[0], zin.stride(0)
        zb = E(B, n.z, dtype=n.adt)
        L.cast2d(zin, ld, zb, n.z, B, n.z)
        hfc = self.fc(zb, n.z, B)
        f = n.fi
        y = E(B, f, f, n.size, dtype=n.adt)
        L.nchw_to_nhwc(hfc, y, B, n.size, f, f)
        h = w = f
        for blk in self.blocks:
            y, h, w = blk(y, B, h, w)
        d3 = L.edge_desc(B, h, w, n.Cl, 1, n.adt)
        ws = n._ewsm.get(d3)
        img = E(B, 3, h, w)
        L.edge_out_fprop(d3, y, self.P["conv.3.0.weight"], self.P["conv.3.0.bias"], L.ACT_TANH, img, ws)
        return img


def _split(full, prefix):
    return OrderedDict((k[len(prefix):], v) for k, v in full.items() if k.startswith(prefix))


class Reconstructor:
    """Eval-mode reconstruction of a trained model from its state_dict (the keys the reference's checkpoints use).

        r = Reconstructor(model.state_dict(), hp.CFG64, z=128, kind="vaegan")        # or a checkpoint loaded with torch.load
        x_hat = r(images)                     # VaeGan.forward(x) in eval mode (samples z like the reference)
        x_hat = r(images, sample=False)       # decode the mean (what WaeGan / WaeGanCognitive eval do)
        imgs  = r.generate(100)               # VaeGan.forward(None, 100)
        pcc, ssim, mse = r.metrics(x_hat, images)

    kind: "vaegan" | "waegan" (visual encoder) or "cognitive" | "wae_cognitive" (fMRI CognitiveEncoder, encoder.fc1.*).
    """

    def __init__(self, state_dict, cfg, z=128, kind="vaegan", adt=BF16, voxels=None):
        if kind not in ("vaegan", "waegan", "cognitive", "wae_cognitive"):
            raise L.FmriError("kind must be vaegan | waegan | cognitive | wae_cognitive")
        dev = torch.device("cuda")
        sd = OrderedDict((k, v.detach().to(dev, F32) if v.dtype.is_floating_point else v.detach().to(dev))
                         for k, v in state_dict.items())
        self.kind, self.z = kind, z
        self.sample_default = kind in ("vaegan", "cognitive")
        enc, dec = _split(sd, "encoder."), _split(sd, "decoder.")
        if kind in ("cognitive", "wae_cognitive"):
            V = voxels or enc["fc1.0.weight"].shape[1]
            self.enc = FoldedCognitiveEncoder(enc, enc, z, V, adt)
        else:
            self.enc = FoldedEncoder(enc, enc, cfg, z, adt)
        self.dec = FoldedDecoder(dec, dec, cfg, z, adt)
        self._ws = torch.empty(8, dtype=F64, device=dev)

    def encode(self, x):
        """(mu, logvar) fp32 [B, z] views of the encoder's head output."""
        ycat = self.enc(x.to("cuda", F32).contiguous())
        return ycat[:, :self.z], ycat[:, self.z:]

    def __call__(self, x, sample=None, eps=None):
        mu, lv = self.encode(x)
        if self.sample_default if sample is None else sample:
            B = mu.shape[0]
            if eps is None:
                eps = lv.data.new(B, self.z).normal_()      # same RNG call as VaeGan.reparameterize (vae_gan.py:266-269)
            zz = E(B, self.z)
            L.reparam_kl_fwd(mu, lv, eps, zz, None, B, self.z, ld=2 * self.z)
            return self.dec(zz)
        return self.dec(mu)

    def generate(self, gen_size=10, z_p=None):
        if z_p is None:
            z_p = torch.randn(gen_size, self.z).to("cuda")      # CPU RNG then moved, as vae_gan.py:290-291
        return self.dec(z_p.to("cuda", F32).contiguous())

    # ---- metrics (train/train_utils.py:267-425), device scalars
    def pcc(self, pred, target):
        out = E(1)
        L.pearson(pred.contiguous(), target.contiguous(), out, self._ws)
        return out[0]

    def ssim(self, pred, target):
        out = E(1)
        L.ssim(pred.contiguous(), target.contiguous(), out, self._ws)
        return out[0]

    def mse(self, pred, target):
        B = pred.shape[0]
        Fd = pred[0].numel()
        rows, out = E(B), Z(1)
        L.rowsqdiff_fwd(pred.contiguous(), target.contiguous(), rows, B, Fd, 1.0 / (B * Fd))
        L.vecsum(rows, B, 1.0, out)
        return out[0]

    def metrics(self, pred, target):
        return self.pcc(pred, target), self.ssim(pred, target), self.mse(pred, target)


def pcc(pred, target):
    """PearsonCorrelation()(pred, target) of train/train_utils.py:267-293 on the device (fp32 tensors of equal shape)."""
    out, ws = E(1), torch.empty(5, dtype=F64, device="cuda")
    L.pearson(pred.to("cuda", F32).contiguous(), target.to("cuda", F32).contiguous(), out, ws)
    return out[0]


def ssim(pred, target):
    """StructuralSimilarity()(pred, target) of train/train_utils.py:295-425 on the device ([N, C, H, W] fp32)."""
    out, ws = E(1), torch.empty(1, dtype=F64, device="cuda")
    L.ssim(pred.to("cuda", F32).contiguous(), target.to("cuda", F32).contiguous(), out, ws)
    return out[0]


# ---- all-pairs similarity and n-way identification
_METRICS = {"pcc": L.METRIC_PCC, "ssim": L.METRIC_SSIM}


def similarity_matrix(pred, target, metric="ssim"):
    """fp32 [N, M] device tensor of metric(pred[i:i+1], target[j:j+1]) (PearsonCorrelation or StructuralSimilarity of
    train/train_utils.py:267-425) for pred [N, C, H, W] and target [M, C, H, W]."""
    if metric not in _METRICS:
        raise L.FmriError(f"metric must be 'ssim' or 'pcc', not {metric!r}")
    if pred.dim() != 4 or target.dim() != 4 or tuple(pred.shape[1:]) != tuple(target.shape[1:]):
        raise L.FmriError(f"pred {tuple(pred.shape)} and target {tuple(target.shape)} must be [N, C, H, W] and [M, C, H, W]")
    N, Cc, H, W = pred.shape
    M = target.shape[0]
    if min(N, M, Cc, H, W) <= 0:
        raise L.FmriError("similarity_matrix needs non-empty image sets")
    if metric == "ssim" and (H < 11 or W < 11):
        raise L.FmriError(f"ssim: images smaller than the 11 x 11 window ({H} x {W})")
    p, t = pred.to("cuda", F32).contiguous(), target.to("cuda", F32).contiguous()
    ws = torch.empty(L.pairwise_workspace(N, M, Cc, H, W, _METRICS[metric]), dtype=torch.uint8, device="cuda")
    out = E(N, M)
    L.pairwise_similarity(p, t, _METRICS[metric], out, ws)
    return out


def identification(sim, ns=(2, 5, 10)):
    """(wins int32 [N], acc float64 [len(ns)]) on the device, no host sync, from a square similarity matrix sim [N, N]
    whose row i is reconstruction i and column i its own target: wins[i] = #{j != i : sim[i, i] > sim[i, j]} (strict, a
    NaN never wins) and acc[q] = mean_i C(wins[i], n-1) / C(N-1, n-1) for n = ns[q] in [2, N], the probability that the
    true target beats n-1 distractors drawn without replacement (n = 2: pairwise identification, n = N: top-1)."""
    if sim.dim() != 2 or sim.shape[0] != sim.shape[1]:
        raise L.FmriError(f"identification needs a square [N, N] matrix, got {tuple(sim.shape)}")
    N = sim.shape[0]
    ns = [int(n) for n in ns]
    if N < 2 or not ns or any(n < 2 or n > N for n in ns):
        raise L.FmriError(f"identification needs N >= 2 and every n in [2, N = {N}] (ns = {ns})")
    s = sim.to("cuda", F32).contiguous()
    wins, acc = E(N, dtype=torch.int32), E(len(ns), dtype=F64)
    L.identification(s, ns, wins, acc)
    return wins, acc
