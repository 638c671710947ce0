#!/usr/bin/env python
"""Step time of the fused Stage-I trainer (engine.VaeGanStage1) for the loss mixes of train_vgan_stage1.py:359-388.

  python scripts/loss_mix_bench.py [--batch 4096] [--resolution 64|100] [--graph] [--steps 20] [--warmup 3]

The modes run alternately, twice each, in one process (the power-capped B200 drifts by a few percent over a run, so one
mode timed after another would carry that drift into the comparison). Inputs and weights are seeded as in bench.py; every
mode is warmed up before the first timed window. One JSON line per timed run: ms/step, samples/s, the algorithmic
MFLOP/sample of that mode (alg_mflop below), whole-step TFLOP/s and its fraction of the sustained bf16 peak, and the GPU's
name, power limit and SM clock (read-only nvidia-smi queries). Then one line per mode for the module path
(models/vae_gan.py driven as the unchanged script drives it: two discriminator forwards, three autograd sweeps, the host-side
gate) at the same batch or, when that does not fit, the largest power-of-two fraction of it that does; and a summary line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (seeded inputs, peaks, clock sampler and the 'vae-gan' FLOP count of the benchmark)

MODES = ("vae-gan", "vae", "dcgan")


def alg_mflop(cfg, z, mode):
    """Algorithmic MFLOP per sample of one fused Stage-I step in `mode` (SURVEY.md 8d conventions, as bench.stage1_alg_mflop:
    2 x MACs of the necessary contractions; a transposed conv counts its input grid). E, D, S: forward of the encoder, the
    decoder and the discriminator; c0..c3 the discriminator's convs, fc the decoder's first Linear, e0 the encoder's first conv.
      vae-gan / beta-vae: E + 2D + 3S | class path 3S + 3(S - c0) + 2c0 | feature-tap path 2c3 + 3(c2 + c1) + c0 |
                          decoder 2(2D - fc) | decoder data gradient D | encoder 2E - e0
      dcgan:              E + 2D + 3S | class path 3S + 3(S - c0) + 2c0 | decoder 2(2D - fc)
      vae:                E + 2D + 3S | class path 3S + 3(S - c0) (g_dis only) | one decoder sweep 2D | encoder 2E - e0"""
    def conv(cin, cout, oh, ow):
        return 2.0 * oh * ow * cin * cout * 25

    half = lambda v: (v - 1) // 2 + 1
    s = cfg["image_size"]
    e, d, c = cfg["encoder_channels"], cfg["decoder_channels"], cfg["discrim_channels"]
    h1, h2, h3 = half(s), half(half(s)), half(half(half(s)))
    e0 = conv(3, e[0], h1, h1)
    E = e0 + conv(e[0], e[1], h2, h2) + conv(e[1], e[2], h3, h3) + 2.0 * h3 * h3 * e[2] * cfg["fc_output"] + \
        2 * 2.0 * cfg["fc_output"] * z
    f = cfg["fc_input"]
    g1 = 2 * f - 1 + int(cfg["output_pad_dec"][0])
    g2 = 2 * g1 - 1 + int(cfg["output_pad_dec"][1])
    g3 = 2 * g2 - 1 + int(cfg["output_pad_dec"][2])
    fc = 2.0 * z * f * f * 256
    D = fc + conv(256, 256, f, f) + conv(256, d[1], g1, g1) + conv(d[1], d[2], g2, g2) + conv(d[2], 3, g3, g3)
    d0 = (s - 1) // cfg["stride_gan"] + 1
    d1, d2, d3 = half(d0), half(half(d0)), half(half(half(d0)))
    c0, c1, c2, c3 = conv(3, c[0], d0, d0), conv(c[0], c[1], d1, d1), conv(c[1], c[2], d2, d2), conv(c[2], c[3], d3, d3)
    S = c0 + c1 + c2 + c3 + 2.0 * d3 * d3 * c[3] * cfg["fc_output_gan"] + 2.0 * cfg["fc_output_gan"]
    fwd = E + 2 * D + 3 * S
    if mode in ("vae-gan", "beta-vae"):
        bwd = (3 * S + 3 * (S - c0) + 2 * c0) + (2 * c3 + 3 * (c2 + c1) + c0) + 2 * (2 * D - fc) + D + (2 * E - e0)
    elif mode == "dcgan":
        bwd = (3 * S + 3 * (S - c0) + 2 * c0) + 2 * (2 * D - fc)
    elif mode == "vae":
        bwd = (3 * S + 3 * (S - c0)) + 2 * D + (2 * E - e0)
    else:
        raise ValueError(f"unknown loss mix {mode!r}")
    return (fwd + bwd) / 1e6


def gpu_info(index):
    """Read-only query of the card: name, power limit (W), max and current SM clock (MHz)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                              "--format=csv,noheader,nounits", "-i", str(index)], capture_output=True, text=True, timeout=30)
        name, plim, smax, sm = [v.strip() for v in out.stdout.strip().splitlines()[0].split(",")]
        return dict(gpu=name, power_limit_w=float(plim), sm_max_mhz=float(smax), sm_mhz_idle=float(sm))
    except Exception as ex:   # the numbers below are then reported without the card they were measured on
        return dict(gpu=None, nvidia_smi_error=str(ex))


def parse():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--resolution", type=int, default=64, choices=[64, 100])
    ap.add_argument("--graph", action="store_true", help="replay each mode's step from a CUDA graph (engine.GraphedStep)")
    ap.add_argument("--steps", type=int, default=20, help="timed steps per run (at least 20)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-module", action="store_true", help="skip the module-path leg")
    a = ap.parse_args()
    if a.steps < 20:
        ap.error("--steps must be at least 20")
    if a.batch < 2:
        ap.error("--batch must be at least 2")
    return a


def module_leg(P, S, cfg, z, res, mode, hp, batch, x_all, steps, warmup):
    """The module path's step at `batch` (halved until it fits). Returns (batch used, ms/step, error of the first failure)."""
    import torch

    import configs.models_config as mc
    from models.vae_gan import VaeGan
    from thesis_fmri_reconstruction_b200 import dp, lib

    mc.use_resolution(res)
    model = VaeGan(device="cuda", z_size=z)
    model.load_state_dict({**P, **S}, strict=True)
    model.train()
    opt = {b: torch.optim.RMSprop(getattr(model, b).parameters(), lr=hp["lr"], alpha=hp["alpha"], eps=hp["eps"])
           for b in ("encoder", "decoder", "discriminator")}
    lam, first_err = hp["lambda_mse"], None

    def step(x):
        B = x.shape[0]
        x_tilde, dc, dl, mus, lv = model(x)
        nle, kl, mse, bo, bp, bs = VaeGan.loss(x, x_tilde, dl[:B], dl[B:-B], dl[-B:], dc[:B], dc[B:-B], dc[-B:], mus, lv)
        if mode == "vae-gan":
            le, ld_ = torch.sum(kl) + torch.sum(mse), torch.sum(bo) + torch.sum(bp) + torch.sum(bs)
            lde, train_enc, dis_in = torch.sum(lam * mse) - (1.0 - lam) * ld_, True, True
        elif mode == "dcgan":
            le, ld_ = torch.sum(kl) + torch.sum(nle), torch.sum(bo) + torch.sum(bs)
            lde, train_enc, dis_in = torch.sum(lam * nle) - (1.0 - lam) * ld_, False, True
        else:
            le, ld_ = torch.sum(kl) + torch.sum(nle), torch.sum(bo) + torch.sum(bs)
            lde, train_enc, dis_in = torch.sum(lam * nle), True, False
        train_dis, train_dec = dp.gate_from_sums(torch.sum(bo).item(), torch.sum(bp).item(), B, hp["margin"],
                                                 hp["equilibrium"], dis_in)
        model.zero_grad()
        le.backward(retain_graph=True)
        if train_enc:
            opt["encoder"].step()
        model.zero_grad()
        lde.backward(retain_graph=True)
        if train_dec:
            opt["decoder"].step()
        model.discriminator.zero_grad()
        ld_.backward()
        if train_dis:
            opt["discriminator"].step()

    while batch >= 1:
        try:
            x = x_all[:batch]
            for _ in range(warmup):
                step(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(x)
            e1.record()
            torch.cuda.synchronize()
            return batch, e0.elapsed_time(e1) / steps, first_err
        except (torch.cuda.OutOfMemoryError, lib.FmriError) as ex:
            if "out of memory" not in str(ex).lower():
                raise
            first_err = first_err or str(ex).splitlines()[0][:200]
            model.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            batch //= 2
    return None, None, first_err


def main():
    args = parse()
    sys.dont_write_bytecode = True   # like bench.py: no __pycache__ of its imports in the tree
    import torch

    from thesis_fmri_reconstruction_b200 import engine, hp, init

    if not torch.cuda.is_available():
        raise SystemExit("loss_mix_bench.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    cfg, z = (hp.CFG64, 128) if args.resolution == 64 else (hp.CFG100, 512)
    B, IMG = args.batch, cfg["image_size"]
    gen = torch.Generator().manual_seed(1234)
    x = ((torch.rand(B, 3, IMG, IMG, generator=gen) * 2 - 1)).cuda()
    eps = torch.randn(B, z, generator=gen).cuda()
    z_p = torch.randn(B, z, generator=gen).cuda()
    P, S = init.init_vaegan(cfg, z, seed=12345)
    info = gpu_info(0)
    pk = bench.peaks()

    steps = {}
    for mode in MODES:
        tr = engine.VaeGanStage1(P, S, cfg, z, torch.bfloat16, mode=mode)
        if args.graph:
            g = engine.GraphedStep(tr, x, eps, z_p, warmup=args.warmup)
            steps[mode] = (tr, lambda g=g: g(x, eps, z_p))
        else:
            steps[mode] = (tr, lambda tr=tr: tr.step(x, eps, z_p))
            for _ in range(args.warmup):
                tr.step(x, eps, z_p)
    torch.cuda.synchronize()

    results = {m: [] for m in MODES}
    for rnd in range(2):
        for mode in MODES:
            tr, fn = steps[mode]
            clocks = bench.ClockSampler(0)
            clocks.start()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ck = clocks.stop()
            ms = e0.elapsed_time(e1) / args.steps
            mf = alg_mflop(cfg, z, mode)
            tflops = B * mf * 1e6 / (ms * 1e-3) / 1e12
            lo = tr.losses()
            finite = all(v == v and abs(v) != float("inf") for v in lo.values() if isinstance(v, float))
            results[mode].append(ms)
            print(json.dumps(dict(kind="fused", mode=mode, run=rnd, batch=B, resolution=args.resolution, graph=args.graph,
                                  steps=args.steps, ms_per_step=round(ms, 3), samples_per_s=round(B / (ms * 1e-3), 1),
                                  alg_mflop_per_sample=round(mf, 1), tflops=round(tflops, 1),
                                  frac_sustained_bf16=round(tflops / pk["tflops"], 3), peak_src=pk["src"],
                                  sm_mhz_median=ck.get("sm_mhz"), throttle=ck.get("reasons"), losses_finite=finite, **info)),
                  flush=True)

    module = {}
    if not args.no_module:
        steps.clear()   # frees the fused trainers before the module path allocates
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        from thesis_fmri_reconstruction_b200 import autograd as ag

        ag.set_compute_dtype(torch.bfloat16)
        for mode in MODES:
            bm, ms, err = module_leg(P, S, cfg, z, args.resolution, mode, hp.HP_VGAN, B, x, args.steps, args.warmup)
            module[mode] = (bm, ms)
            print(json.dumps(dict(kind="module", mode=mode, batch=bm, resolution=args.resolution, steps=args.steps,
                                  ms_per_step=round(ms, 3) if ms else None,
                                  samples_per_s=round(bm / (ms * 1e-3), 1) if ms else None, larger_batch_error=err,
                                  **info)), flush=True)
            torch.cuda.empty_cache()

    med = {m: sorted(v)[len(v) // 2] if len(v) % 2 else sum(v) / len(v) for m, v in results.items()}
    summ = dict(kind="summary", batch=B, resolution=args.resolution, graph=args.graph,
                fused_ms_per_step={m: round(v, 3) for m, v in med.items()},
                ratio_to_vae_gan={m: round(v / med["vae-gan"], 3) for m, v in med.items()},
                alg_flop_ratio_to_vae_gan={m: round(alg_mflop(cfg, z, m) / alg_mflop(cfg, z, "vae-gan"), 3) for m in MODES},
                **info)
    if module:
        summ["module_speedup"] = {m: round((module[m][1] / module[m][0]) / (med[m] / B), 2) if module[m][1] else None
                                  for m in MODES}
    print(json.dumps(summ), flush=True)


if __name__ == "__main__":
    main()
