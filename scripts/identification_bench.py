#!/usr/bin/env python
"""All-pairs similarity matrices (inference.similarity_matrix) against a stock-PyTorch formulation of the same matrix.

  python scripts/identification_bench.py [--sizes 1024,4096] [--res 64,100] [--metrics pcc,ssim] [--reps 3] [--no-torch]

For each size (N = M images of 3 x res x res, seeded) and metric, our call and the stock formulation run alternately,
each warmed up first and then timed with CUDA events over --reps calls, twice. One JSON line per size and metric: ms per
matrix (mean of the two windows) for both, the algorithmic FLOP per pair (alg_flop_per_pair below), our achieved fp32
rate and its share of the FMA peak at the SM clock sampled during our window (148 SMs x 128 lanes x 2 FLOP x clock), the
max |difference| between the two matrices, and the GPU's name, power limit and clock (read-only nvidia-smi queries).
The stock formulation:
  pcc  fp32 matmul (TF32 off) of the mean-centred images, divided by the outer product of their norms;
  ssim cuDNN depthwise F.conv2d for mu / sigma^2 of each set, then, over chunks of pred rows, G * (x_i y_j) of every pair
       product of the chunk as one depthwise F.conv2d, and the SSIM map and its mean in elementwise ops.
Each call of either side includes its per-image terms. Inputs are 50-490 MB per set, so the smaller ones stay in L2
between calls; both sides see the same.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402  (clock sampler)
from loss_mix_bench import gpu_info  # noqa: E402  (read-only nvidia-smi query of name, power limit, clocks)

SMS, LANES = 148, 128


def alg_flop_per_pair(metric, C, H, W):
    """pcc: one FMA per element of the centred images (2 CHW). ssim per output pixel: the product x_i y_j (1), the
    horizontal and the vertical 11-tap sums (2 x 11 FMAs = 44), and the SSIM expression of the epilogue (12): 57 CHW."""
    return 2 * C * H * W if metric == "pcc" else 57 * C * H * W


def torch_pcc(pred, target):
    import torch

    xa = pred.flatten(1)
    xb = target.flatten(1)
    xa = xa - xa.mean(1, keepdim=True)
    xb = xb - xb.mean(1, keepdim=True)
    return (xa @ xb.t()) / (xa.norm(dim=1)[:, None] * xb.norm(dim=1)[None, :]).to(torch.float32)


def torch_ssim(pred, target, chunk_bytes=8 << 30):
    import torch
    import torch.nn.functional as F

    from oracle.metrics import _window

    N, C, H, W = pred.shape
    M = target.shape[0]
    win = _window(11, C, torch.float32).to(pred.device)
    conv = lambda x: F.conv2d(x, win, padding=5, groups=C)
    mu_a, mu_b = conv(pred), conv(target)
    sg_a, sg_b = conv(pred * pred) - mu_a * mu_a, conv(target * target) - mu_b * mu_b
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    out = torch.empty(N, M, device=pred.device)
    rows = max(1, chunk_bytes // (M * C * H * W * 4 * 6))
    for i0 in range(0, N, rows):
        i1 = min(N, i0 + rows)
        prod = (pred[i0:i1, None] * target[None]).reshape(-1, C, H, W)
        s12 = conv(prod).view(i1 - i0, M, C, H, W)
        m12 = mu_a[i0:i1, None] * mu_b[None]
        num = (2 * m12 + C1) * (2 * (s12 - m12) + C2)
        den = (mu_a[i0:i1, None] ** 2 + mu_b[None] ** 2 + C1) * (sg_a[i0:i1, None] + sg_b[None] + C2)
        out[i0:i1] = (num / den).mean(dim=(2, 3, 4))
    return out


def timed(fn, reps):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--sizes", default="1024,4096")
    ap.add_argument("--res", default="64,100")
    ap.add_argument("--metrics", default="pcc,ssim")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-torch", action="store_true", help="skip the stock-PyTorch formulation")
    a = ap.parse_args()
    sys.dont_write_bytecode = True
    import torch

    from thesis_fmri_reconstruction_b200 import inference

    if not torch.cuda.is_available():
        raise SystemExit("identification_bench.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    info = gpu_info(0)
    for res in [int(v) for v in a.res.split(",")]:
        for n in [int(v) for v in a.sizes.split(",")]:
            g = torch.Generator().manual_seed(1000 + n + res)
            pred = (torch.rand(n, 3, res, res, generator=g) * 2 - 1).cuda()
            target = (pred.cpu() + 0.5 * torch.randn(n, 3, res, res, generator=g)).clamp(-1, 1).cuda()
            for metric in a.metrics.split(","):
                ours = lambda: inference.similarity_matrix(pred, target, metric=metric)
                stock = (lambda: torch_pcc(pred, target)) if metric == "pcc" else (lambda: torch_ssim(pred, target))
                X = ours()
                Y = None if a.no_torch else stock()
                torch.cuda.synchronize()
                t_ours, t_stock, clocks = [], [], []
                for _ in range(2):
                    ck = bench.ClockSampler(0)
                    ck.start()
                    ms, X = timed(ours, a.reps)
                    clocks.append(ck.stop())
                    t_ours.append(ms)
                    if Y is not None:
                        ms, Y = timed(stock, a.reps)
                        t_stock.append(ms)
                ms = sum(t_ours) / 2
                flop = alg_flop_per_pair(metric, 3, res, res) * n * n
                mhz = [c["sm_mhz"] for c in clocks if c.get("sm_mhz")]
                mhz = sum(mhz) / len(mhz) if mhz else None
                tflops = flop / (ms * 1e-3) / 1e12
                peak = SMS * LANES * 2 * mhz * 1e6 / 1e12 if mhz else None
                line = dict(metric=metric, n=n, res=res, reps=a.reps, ms=round(ms, 3), ms_runs=[round(v, 3) for v in t_ours],
                            alg_flop_per_pair=alg_flop_per_pair(metric, 3, res, res), tflops_fp32=round(tflops, 2),
                            sm_mhz=mhz, fma_peak_tflops=round(peak, 1) if peak else None,
                            frac_fma_peak=round(tflops / peak, 3) if peak else None,
                            throttle=sorted({r for c in clocks for r in c.get("reasons", [])}))
                if Y is not None:
                    ts = sum(t_stock) / 2
                    line.update(stock_ms=round(ts, 3), stock_ms_runs=[round(v, 3) for v in t_stock],
                                speedup=round(ts / ms, 2), max_abs_diff=float((X - Y).abs().max()))
                print(json.dumps(dict(line, **info)), flush=True)
                del X, Y
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
