#!/usr/bin/env python
"""Benchmark of the training hot path (BASELINE.json: "Stage-I VAE/GAN train samples/sec @64x64").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload stage1_vaegan] [--batch GLOBAL_B]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
  python bench.py --impl reference ...     # the CPU arm: the oracle port of the reference step on the host cores
  python bench.py ... --dump-outputs DIR   # also write the last timed step's outputs as DIR/<name>.npy (seeded inputs)

One step = one full training iteration (forward, minimal backward, gradient all-reduce for N > 1, three RMSprop updates,
bf16 operand repack) on one synthetic batch. `value` times K steps with inputs resident in HBM; `e2e` times K steps fed
from pinned host memory (H2D of the batch + noise, D2H of the loss sums, every step). Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic MFLOP per sample per optimisation step (SURVEY.md section 8d; 2 x MACs of the necessary GEMMs only)
ALG_MFLOP = {"stage1_vaegan": 16966.2, "stage1_waegan": 3352.8, "stage2_cognitive": 13866.1,
             # Stage III proper (train_vgan_stage3.py): fwd C+2D+3S = 4359.3, bwd [3S+3(S-c0)+2c0] + [2c3+3(c2+c1)+c0] + 2(2D-fc) = 11001.2
             "stage3_cognitive": 15360.4,
             # configs[3] composite (SURVEY.md 8d, C4): Stage III + teacher-encoder forward + latent-discriminator D-phase
             "stage3_dual": 15624.3,
             # WAE-MMD extension: E + D forward, 2D + (2E - c0) backward; the pairwise kernel adds 9 * B * Z flop / sample
             "stage1_wae_mmd": 3339.2,
             # WAE Stage II: fwd E + 2D (one unused teacher reconstruction) + C + 3W, bwd 5W + D (dgrad) + C; Stage III: fwd
             # E + C + D + 3W, bwd 4W + (2D - fc)   (same conventions as SURVEY.md 8d; W, C terms are < 1 %)
             "stage2_wae_cognitive": 2871.2, "stage3_wae_cognitive": 2857.4}
CONFIG_OF = {"stage1_vaegan": "configs[4] (configs[0] at --batch 64)", "stage1_waegan": "configs[1] (reference WAE/GAN step; "
             "the reference has no MMD)", "stage2_cognitive": "configs[2]", "stage3_cognitive": "train_vgan_stage3.py proper",
             "stage3_dual": "configs[3] (composite, SURVEY.md 8d C4)",
             "stage1_wae_mmd": "configs[1] with the MMD latent loss (extension: no reference code, parity unpinned)",
             "stage2_wae_cognitive": "train_wae_stage2.py step (SURVEY.md 8a row a15)",
             "stage3_wae_cognitive": "train_wae_stage3.py step (SURVEY.md 8a row a15)"}
METRIC = "stage1_vaegan_train_samples_per_sec_64x64"  # BASELINE.json metric; other workloads rename it below


def stage1_alg_mflop(cfg, z):
    """Algorithmic MFLOP per sample of the Stage-I VAE/GAN step for an architecture dict (same accounting as ALG_MFLOP /
    tests/test_flops_cpu.py: 2 x MACs of the necessary contractions; a transposed conv counts its input grid)."""
    def conv(cin, cout, oh, ow):
        return 2.0 * oh * ow * cin * cout * 25

    half = lambda v: (v - 1) // 2 + 1
    s = cfg["image_size"]
    e, d, c = cfg["encoder_channels"], cfg["decoder_channels"], cfg["discrim_channels"]
    h1, h2, h3 = half(s), half(half(s)), half(half(half(s)))
    enc_c = [conv(3, e[0], h1, h1), conv(e[0], e[1], h2, h2), conv(e[1], e[2], h3, h3)]
    E = sum(enc_c) + 2.0 * h3 * h3 * e[2] * cfg["fc_output"] + 2 * 2.0 * cfg["fc_output"] * z
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
    total = (E + 2 * D + 3 * S) + (3 * S + 3 * (S - c0) + 2 * c0) + (2 * c3 + 3 * (c2 + c1) + c0) + 2 * (2 * D - fc) + D + \
            (2 * E - enc_c[0])
    return total / 1e6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="stage1_vaegan", choices=["stage1_vaegan", "stage1_waegan", "stage2_cognitive", "stage3_cognitive", "stage3_dual", "stage1_wae_mmd",
                                                                    "stage2_wae_cognitive", "stage3_wae_cognitive"])
    ap.add_argument("--batch", type=int, default=4096, help="GLOBAL batch (BASELINE.json configs[4]: 4096, strong scaling)")
    ap.add_argument("--resolution", type=int, default=64, choices=[64, 100], help="architecture block of the reference's "
                    "configs/models_config.py: 64 (the BASELINE.json configs) or 100 (its ACTIVE 100x100 / latent-512 block; "
                    "stage1_vaegan only)")
    ap.add_argument("--cpu-batch", type=int, default=64, help="batch of the bounded CPU sample (BASELINE.json configs[0])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-stock-torch", action="store_true", help="skip the stock-PyTorch-on-this-GPU leg (child process)")
    ap.add_argument("--graph", action="store_true", help="replay the step from a CUDA graph (engine.GraphedStep; RMSprop "
                    "engines on one GPU): for launch-bound batch sizes such as configs[0]'s 64")
    ap.add_argument("--quick", action="store_true", help="device-resident timing only (for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (forward "
                    "outputs, loss sums, updated parameters and BatchNorm buffers; rank 0) as DIR/<name>.npy, at most 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.warmup < 0:
        ap.error("--warmup must not be negative")
    return a


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(tflops=float(p["bf16_tflops_sustained"]), hbm=float(p["hbm_gbs"]), src="measured (MEASURED_PEAKS.json, sustained bf16)")
    except Exception:
        return dict(tflops=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


def build_hash():
    """sha256 over the kernel sources + public header: ties a committed ncu capture to the build it was taken from."""
    import hashlib

    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "thesis_fmri_reconstruction_b200", "csrc")
    for f in sorted(os.listdir(csrc)) + [os.path.join(ROOT, "include", "fmri_b200.h")]:
        with open(f if os.path.isabs(f) else os.path.join(csrc, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def committed_traffic(workload, per_gpu_batch, family):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel family from the committed ncu capture
    (profiles/r2_traffic.json, written by scripts/ncu_traffic.py). None unless the capture is of THIS build, workload and
    per-GPU batch. Returns (bytes per launch or None, source string)."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
    except Exception:
        return None, "no committed capture (profiles/r2_traffic.json)"
    if t.get("build_hash") != build_hash():
        return None, "profiles/r2_traffic.json is of build %s, this build is %s: traffic withheld" % (t.get("build_hash"), build_hash())
    if t.get("workload") != workload or int(t.get("per_gpu_batch", -1)) != int(per_gpu_batch):
        return None, "profiles/r2_traffic.json is of %s at batch %s" % (t.get("workload"), t.get("per_gpu_batch"))
    fam = t.get("families", {}).get(family)
    if not fam:
        return None, "family %s not in profiles/r2_traffic.json" % family
    return fam["dram_bytes_per_launch"], "profiles/r2_traffic.json (%s; ncu, cold cache, %d launches)" % (t.get("source", "?"), fam["launches"])


def stock_torch_leg(workload, B):
    """Stock PyTorch on the same GPU (cuDNN / cuBLAS, bf16 autocast + channels_last: its best mode, BASELINE.md section 3), in a
    child process; the practical bar next to the hand-written path. Returns a dict or None."""
    if workload not in ("stage1_vaegan", "stage1_waegan", "stage2_cognitive", "stage3_cognitive"):
        return None
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "stock_torch_gpu_baseline.py"), "--workload", workload,
                            "--batch", str(B), "--steps", "3", "--warmup", "2", "--modes", "bf16_cl"],
                           capture_output=True, text=True, timeout=600, env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
        line = json.loads([x for x in r.stdout.splitlines() if x.startswith("{")][-1])
        if "samples_per_s" not in line:
            return dict(error=line.get("error", "failed"))
        return dict(value=line["samples_per_s"], unit="samples/s", ms_per_step=line["ms_per_step"], impl=line["impl"],
                    mode="bf16 autocast + channels_last", batch=B, steps=3, warmup=2)
    except Exception as ex:
        return dict(error=repr(ex)[:200])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(pw) if pw else None, samples=len(sm), reasons=sorted(reasons))


# ------------------------------------------------------------------------------------------------ CPU reference arm
def cpu_reference_steps(workload, B, steps, warmup, threads=None):
    """The oracle port of the reference step (oracle/vaegan.py: reference modules' arithmetic restated functionally, the
    reference's two discriminator passes and three autograd sweeps) on the host cores. Returns (samples/s, ms/step, cores)."""
    import torch

    from oracle import vaegan as O

    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    if workload == "stage1_vaegan":
        P, S = O.make_vaegan(O.CFG64, seed=12345, jitter=False)
        x = O.synthetic_images(B)
        eps, z_p = O.synthetic_noise(B, 128)
        sq = None

        def one():
            nonlocal P, sq
            out = O.stage1_vaegan_step(P, S, x, eps, z_p, sq=sq)
            P, sq = out["params"], out["square_avg"]
    elif workload == "stage1_waegan":
        P, S = O.make_waegan(O.CFG64, seed=12345, jitter=False)
        x = O.synthetic_images(B)
        z_fake = O.synthetic_noise(B, 128)[0] * 0.5
        st = dict(opt=None, t=1)

        def one():
            nonlocal P
            out = O.stage1_waegan_step(P, S, x, z_fake, opt=st["opt"], step=st["t"])
            P, st["opt"], st["t"] = out["params"], out["adam"], st["t"] + 1
    elif workload == "stage1_wae_mmd":
        P, S = O.make_waegan(O.CFG64, seed=12345, jitter=False)
        x = O.synthetic_images(B)
        z_fake = O.synthetic_noise(B, 128)[0] * 0.5
        st = dict(opt=None, t=1)

        def one():
            nonlocal P
            out = O.stage1_wae_mmd_step(P, S, x, z_fake, opt=st["opt"], step=st["t"])
            P, st["opt"], st["t"] = out["params"], out["adam"], st["t"] + 1
    elif workload in ("stage2_wae_cognitive", "stage3_wae_cognitive"):
        stage = 2 if workload == "stage2_wae_cognitive" else 3
        P, S = O.make_cognitive_wae(O.CFG64, seed=12345, jitter=False)
        fmri, x = O.synthetic_fmri(B), O.synthetic_images(B)
        st = dict(opt=None, t=1)

        def one():
            nonlocal P
            out = O.cognitive_wae_step(P, S, fmri, x, stage, opt=st["opt"], step=st["t"])
            P, st["opt"], st["t"] = out["params"], out["adam"], st["t"] + 1
    elif workload == "stage3_dual":
        P, S = O.make_dual_stage3(O.CFG64, seed=12345, jitter=False)
        fmri, x = O.synthetic_fmri(B), O.synthetic_images(B)
        eps, z_p = O.synthetic_noise(B, 128)
        st = dict(sq=None, opt=None, t=1)

        def one():
            nonlocal P
            out = O.dual_stage3_step(P, S, fmri, x, eps, z_p, sq=st["sq"], opt=st["opt"], step=st["t"],
                                     force_gate=(True, True))
            P, st["sq"], st["opt"], st["t"] = out["params"], out["square_avg"], out["adam"], st["t"] + 1
    else:
        stage = 2 if workload == "stage2_cognitive" else 3
        P, S = O.make_cognitive(O.CFG64, seed=12345, jitter=False)
        fmri, x = O.synthetic_fmri(B), O.synthetic_images(B)
        eps, z_p = O.synthetic_noise(B, 128)
        eps_t = O.synthetic_noise(B, 128, seed=99)[0]
        sq = None

        def one():
            nonlocal P, sq
            out = O.cognitive_vaegan_step(P, S, fmri, x, eps, eps_t, z_p, stage, sq=sq, force_gate=(True, True))
            P, sq = out["params"], out["square_avg"]
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return B / dt, dt * 1e3, threads


def find_reference_models():
    """Root of a checkout of the original project (named by $FMRI_REFERENCE_ROOT) that holds models/vae_gan.py, or None."""
    root = os.environ.get("FMRI_REFERENCE_ROOT")
    if root and os.path.exists(os.path.join(root, "models", "vae_gan.py")) and \
            os.path.exists(os.path.join(root, "configs", "models_config.py")):
        return root
    return None


def reference_modules_steps(ref_root, B, steps, warmup, threads=None):
    """Stage-I VAE/GAN on the UNMODIFIED reference modules (models/vae_gan.py imported from `ref_root` with its own
    configs.models_config switched to the 64x64 block, :23-31): VaeGan.forward (two discriminator passes), VaeGan.loss, the
    loss mix of train_vgan_stage1.py:368-372, and the script's three FULL backward sweeps loss_x.backward(retain_graph=True)
    (:408-432, discarded gradients included). The three RMSprop steps run after the third sweep: torch >= 1.5 rejects the
    script's interleaved step order on these modules (SURVEY.md 0-6), and under the torch-1.4 semantics the script was
    written for the result is the same (0-7). Returns (samples/s, ms/step, cores)."""
    import importlib

    import torch

    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    saved = list(sys.path)
    sys.path[:] = [ref_root] + [q for q in sys.path if os.path.abspath(q or ".") != ROOT]
    for m in [k for k in sys.modules if k.split(".")[0] in ("configs", "models")]:
        del sys.modules[m]
    try:
        mc = importlib.import_module("configs.models_config")
        assert os.path.abspath(mc.__file__).startswith(os.path.abspath(ref_root)), mc.__file__
        mc.image_size, mc.fc_input, mc.fc_input_gan, mc.fc_output_gan, mc.stride_gan, mc.latent_dim = 64, 8, 8, 512, 1, 128
        mc.output_pad_dec, mc.decoder_channels = [True, True, True], [256, 128, 32, 3]
        ref = importlib.import_module("models.vae_gan")
        assert os.path.abspath(ref.__file__).startswith(os.path.abspath(ref_root)), ref.__file__
    finally:
        sys.path[:] = saved
    torch.manual_seed(12345)
    model = ref.VaeGan(device=torch.device("cpu"), z_size=128)
    model.train()
    opts = [torch.optim.RMSprop(params=m.parameters(), lr=1e-4, alpha=0.9, eps=1e-8, weight_decay=0, momentum=0, centered=False)
            for m in (model.encoder, model.decoder, model.discriminator)]
    g = torch.Generator().manual_seed(1234)
    x = torch.rand(B, 3, 64, 64, generator=g) * 2 - 1
    lam = 1e-6

    def one():
        x_tilde, disc_class, disc_layer, mus, lv = model(x)
        nle, kld, mse, bo, bp, bs = ref.VaeGan.loss(x, x_tilde, disc_layer[:B], disc_layer[B:-B], disc_layer[-B:],
                                                    disc_class[:B], disc_class[B:-B], disc_class[-B:], mus, lv)
        loss_encoder = torch.sum(kld) + torch.sum(mse)
        loss_discriminator = torch.sum(bo) + torch.sum(bp) + torch.sum(bs)
        loss_decoder = torch.sum(lam * mse) - (1.0 - lam) * loss_discriminator
        grads = []
        for loss, mod in ((loss_encoder, model.encoder), (loss_decoder, model.decoder), (loss_discriminator, model.discriminator)):
            model.zero_grad()
            loss.backward(retain_graph=True)       # a full sweep through discriminator -> decoder -> encoder, as the script does
            grads.append([p.grad.clone() if p.grad is not None else None for p in mod.parameters()])
        for gl, mod, opt in zip(grads, (model.encoder, model.decoder, model.discriminator), opts):
            for p, gr in zip(mod.parameters(), gl):
                p.grad = gr
            opt.step()

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return B / dt, dt * 1e3, threads


def cpu_arm(workload, B, steps, warmup):
    """(samples/s, ms/step, cores, kind, how): the unmodified reference modules when a reference tree is present and the
    workload is the headline one, else the oracle port."""
    ref_root = find_reference_models() if workload == "stage1_vaegan" else None
    if ref_root is not None:
        v, ms, cores = reference_modules_steps(ref_root, B, steps, warmup)
        return v, ms, cores, "reference", ("unmodified reference modules (%s/models/vae_gan.py): VaeGan.forward + VaeGan.loss + the "
                                          "script's three full backward sweeps + 3 x torch.optim.RMSprop" % ref_root)
    v, ms, cores = cpu_reference_steps(workload, B, steps, warmup)
    return v, ms, cores, "port", "oracle port of the reference step (needed gradients only: cheaper than the script's three full sweeps)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    B = args.cpu_batch
    v, ms, cores, kind, how = cpu_arm(args.workload, B, steps, warm)
    sample = f"{steps} timed + {warm} warm-up steps of batch {B} (bounded sample of the workload), fp32, torch CPU; {how}"
    line = dict(metric=METRIC, value=v, unit="samples/s", n_gpus=args.gpus, steps=steps, warmup=warm, ms_per_step=ms,
                higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=f"{args.workload} 64x64 z=128 (BASELINE.json {CONFIG_OF[args.workload]}: global batch {args.batch})",
                            global_batch=args.batch, cpu_sample_batch=B,
                            note="reference arm on the host cores; each timed step is a batch-%d sample of the workload. %s" % (B, how)),
                cpu_baseline=dict(value=v, unit="samples/s", cores=cores, kind=kind, sample=sample),
                e2e=dict(value=v, unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write each tensor of `arrays` as <path>/<name>.npy: float64 and integer tensors as float64, all others as float32.
    Every array gets an equal share of DUMP_BYTES; a larger one is replaced by a fixed sample of its flattened elements (the
    positions depend only on the seed and the element count), so two builds run with the same arguments compare output for
    output."""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096          # room for the .npy header
    for name, t in arrays.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()
        cap = share // t.element_size()
        if t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def run_ours(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    group = None
    if world > 1:
        import torch.distributed as td

        td.init_process_group("nccl", device_id=torch.device("cuda", local))
        group = td.group.WORLD
    from thesis_fmri_reconstruction_b200 import engine, hp, init, lib

    if args.batch % world:
        raise SystemExit(f"global batch {args.batch} not divisible by {world} ranks")
    B = args.batch // world
    cfg, z = hp.CFG64, 128
    if args.resolution == 100:
        if args.workload != "stage1_vaegan":
            raise SystemExit("--resolution 100: workload stage1_vaegan only")
        cfg, z = hp.CFG100, 512
        ALG_MFLOP["stage1_vaegan"] = stage1_alg_mflop(cfg, z)
        args.no_cpu_baseline = True      # the CPU / stock-torch legs are the 64x64 restatements
    IMG = cfg["image_size"]
    gen = torch.Generator().manual_seed(1234 + rank)
    x_host = (torch.rand(B, 3, IMG, IMG, generator=gen) * 2 - 1).pin_memory()
    if args.workload == "stage1_vaegan":
        P, S = init.init_vaegan(cfg, z, seed=12345)
        tr = engine.VaeGanStage1(P, S, cfg, z, torch.bfloat16, dist_group=group, gate=True)
        n1_host = torch.randn(B, z, generator=gen).pin_memory()
        n2_host = torch.randn(B, z, generator=gen).pin_memory()
    elif args.workload in ("stage1_waegan", "stage1_wae_mmd"):
        P, S = init.init_waegan(cfg, z, seed=12345)
        tr = engine.WaeGanStage1(P, S, cfg, z, torch.bfloat16, dist_group=group,
                                 penalty="mmd" if args.workload == "stage1_wae_mmd" else "gan")
        n1_host = (torch.randn(B, z, generator=gen) * 0.5).pin_memory()
        n2_host = None
    else:
        if args.workload in ("stage2_wae_cognitive", "stage3_wae_cognitive"):
            P, S = init.init_cognitive_wae(cfg, z, seed=12345)
            tr = engine.WaeCognitiveStage(P, S, cfg, 2 if args.workload == "stage2_wae_cognitive" else 3, z,
                                          torch.bfloat16, dist_group=group)
        elif args.workload == "stage3_dual":
            P, S = init.init_dual_stage3(cfg, z, seed=12345)
            tr = engine.DualCognitiveStage3(P, S, cfg, z, torch.bfloat16, dist_group=group)
        else:
            stage = 2 if args.workload == "stage2_cognitive" else 3
            P, S = init.init_cognitive(cfg, z, seed=12345, with_teacher=stage == 2)
            tr = engine.VaeGanCognitiveStage(P, S, cfg, stage, z, torch.bfloat16, dist_group=group)
        n1_host = torch.randn(B, z, generator=gen).pin_memory()
        n2_host = torch.randn(B, z, generator=gen).pin_memory()
        fmri_host = torch.randn(B, hp.NUM_VOXELS, generator=gen).pin_memory()
        eps_t = torch.randn(B, z, generator=gen).cuda()
    x = x_host.cuda(non_blocking=True)
    n1 = n1_host.cuda(non_blocking=True)
    n2 = n2_host.cuda(non_blocking=True) if n2_host is not None else None
    cog = args.workload in ("stage2_cognitive", "stage3_cognitive", "stage3_dual", "stage2_wae_cognitive",
                            "stage3_wae_cognitive")
    dual = args.workload == "stage3_dual"
    waecog = args.workload in ("stage2_wae_cognitive", "stage3_wae_cognitive")
    fmri = fmri_host.cuda(non_blocking=True) if cog else None

    def step_inputs(xb, a, b2, fb=None):
        """Positional inputs of this workload's trainer.step()."""
        fb = fb if fb is not None else fmri
        if waecog:
            return (fb, xb)
        if dual:
            return (fb, xb, a, b2)
        if cog:
            return (fb, xb, a, eps_t, b2)
        if b2 is not None:
            return (xb, a, b2)
        return (xb, a)

    def run_step(xb, a, b2, fb=None):
        return tr.step(*step_inputs(xb, a, b2, fb))

    graphed = None
    if args.graph:
        if world > 1:
            raise SystemExit("--graph: one GPU")
        graphed = engine.GraphedStep(tr, *step_inputs(x, n1, n2, fmri))
    last = {}

    def step_dev():
        if graphed is not None:
            out = graphed(*step_inputs(x, n1, n2, fmri))
        else:
            out = run_step(x, n1, n2)
        if args.dump_outputs:
            last["out"] = out   # held only when dumping: the step's outputs are otherwise freed before the next step

    def sync_all():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            td.all_reduce(ms, op=td.ReduceOp.MAX)
        return ms.item()

    # ---------------------------------------------------------------- device-resident throughput (`value`)
    for _ in range(args.warmup):
        step_dev()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    lib.launch_count(reset=True)
    ms_total = timed(step_dev, args.steps)
    launches = lib.launch_count() if graphed is None else graphed.launches * args.steps  # replays bypass the host counter
    ck = clocks.stop() if rank == 0 else None
    losses = tr.losses()
    ms_step = ms_total / args.steps
    value = args.batch / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:   # before the e2e and profiling passes below step the trainer further
        arrays = {k: v for k, v in last["out"].items() if isinstance(v, torch.Tensor)}
        arrays["loss_sums"] = tr.sc
        arrays.update(("param." + k, v) for k, v in tr.named_parameters().items())
        arrays.update(("buffer." + k, v) for k, v in tr.named_buffers().items())
        dump_outputs(args.dump_outputs, arrays)

    if args.quick:
        if rank == 0:
            print(json.dumps(dict(metric=METRIC, value=value, unit="samples/s", ms_per_step=ms_step, gpu_launches=launches,
                                  quick=True, global_batch=args.batch)), flush=True)
        if world > 1:
            td.destroy_process_group()
        return
    # ---------------------------------------------------------------- end to end from pinned host memory (`e2e`)
    copy_stream = torch.cuda.Stream()
    bufs = [[torch.empty_like(x), torch.empty_like(n1), torch.empty_like(n2) if n2 is not None else None,
             torch.empty_like(fmri) if cog else None] for _ in range(2)]
    evs = [torch.cuda.Event(), torch.cuda.Event()]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    sc_host = torch.empty(16).pin_memory()
    state = dict(i=0)

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[slot])  # the step that last read this slot has finished
            bufs[slot][0].copy_(x_host, non_blocking=True)
            bufs[slot][1].copy_(n1_host, non_blocking=True)
            if n2 is not None:
                bufs[slot][2].copy_(n2_host, non_blocking=True)
            if cog:
                bufs[slot][3].copy_(fmri_host, non_blocking=True)
            evs[slot].record(copy_stream)

    def step_e2e():
        i = state["i"]
        slot = i & 1
        torch.cuda.current_stream().wait_event(evs[slot])
        upload(slot ^ 1)  # prefetch the next batch while this step computes (the DataLoader's role in the reference)
        b = bufs[slot]
        if graphed is not None:   # the replay copies the slot into the graph's static input buffers (device to device)
            graphed(*step_inputs(b[0], b[1], b[2], b[3]))
        else:
            run_step(b[0], b[1], b[2], b[3])
        done[slot].record()
        sc_host.copy_(tr.sc, non_blocking=True)  # D2H of the step's loss sums (what train_vgan_stage1.py:391-401 reads)
        state["i"] = i + 1

    done[0].record(); done[1].record()
    upload(0)
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps) / args.steps
    e2e_value = args.batch / (ms_e2e * 1e-3)
    h2d = world * (x_host.numel() + n1_host.numel() + (n2_host.numel() if n2_host is not None else 0) +
                   (fmri_host.numel() if cog else 0)) * 4
    d2h = world * 16 * 4

    # ---------------------------------------------------------------- per-kernel-family device times (CUDA events)
    pk = peaks()
    roof = None
    if not args.no_profile:
        from thesis_fmri_reconstruction_b200 import nets as _nets

        torch.cuda.synchronize()
        side = _nets.WGRAD_SIDE_STREAM
        _nets.WGRAD_SIDE_STREAM = False   # attribution pass: every kernel alone on the compute stream (no overlap)
        lib.profile_begin()
        psteps = max(1, min(3, args.steps))
        for _ in range(psteps):
            run_step(x, n1, n2)   # eager even under --graph: the per-entry-point events need real launches
        agg = lib.profile_end()
        _nets.WGRAD_SIDE_STREAM = side
        tot_ms = sum(a["ms"] for a in agg.values())
        fam = {}
        for name, a in agg.items():
            k = "igemm" if name in ("fmri_conv_fprop", "fmri_conv_dgrad", "fmri_linear_fprop", "fmri_linear_dgrad") else (
                "wgrad" if name in ("fmri_conv_wgrad", "fmri_linear_wgrad") else name)
            f = fam.setdefault(k, dict(ms=0.0, calls=0, flops=0.0))
            for q in ("ms", "calls", "flops"):
                f[q] += a[q]
        dom = max(("igemm", "wgrad"), key=lambda k: fam.get(k, dict(ms=0))["ms"])
        d = fam[dom]
        ach = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
        top = sorted(((k, round(v["ms"] / psteps, 3)) for k, v in fam.items()), key=lambda t: -t[1])[:16]
        roof = dict(bound="tensor", kernel=("igemm_kernel (conv/convT fprop+dgrad, linear fprop+dgrad)" if dom == "igemm"
                                            else "wgrad_kernel (conv/convT/linear weight gradients)"),
                    achieved=ach, peak=pk["tflops"], unit="TFLOP/s", frac=ach / pk["tflops"],
                    # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel family (mean over its launches of
                    # one step) from the committed ncu capture of THIS build and configuration; null otherwise
                    traffic=committed_traffic(args.workload, B, dom)[0],
                    traffic_source=committed_traffic(args.workload, B, dom)[1],
                    peak_source=pk["src"], kernel_ms_per_step=d["ms"] / psteps, kernel_launches_per_step=d["calls"] / psteps,
                    kernel_share_of_step=d["ms"] / tot_ms if tot_ms else None,
                    # whole job: algorithmic FLOPs of the step x samples/s over ALL ranks, against world x the per-GPU peak
                    whole_step_achieved=ALG_MFLOP[args.workload] * 1e6 * value / 1e12,
                    whole_step_frac=ALG_MFLOP[args.workload] * 1e6 * value / 1e12 / (pk["tflops"] * world),
                    top_entry_points_ms_per_step=top)

    cpu = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        v, ms, cores, kind, how = cpu_arm(args.workload, args.cpu_batch, 2, 1)
        cpu = dict(value=v, unit="samples/s", cores=cores, kind=kind,
                   sample=f"2 timed + 1 warm-up steps of batch {args.cpu_batch} of the same workload, fp32, torch CPU; {how}")
    stock = None
    if rank == 0 and world == 1 and not args.no_stock_torch and not args.no_cpu_baseline:
        torch.cuda.empty_cache()
        stock = stock_torch_leg(args.workload, B)
    if rank == 0:
        act_gb = B * 3 * (64 * 64 * 32 + 32 * 32 * 128 + 16 * 16 * 256 + 8 * 8 * 256) * 2 * 2 / 1e9 * (IMG / 64.0) ** 2
        line = dict(metric=METRIC, value=value, unit="samples/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_step, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="bf16",
                    data="synthetic", impl="ours",
                    config=dict(workload=(f"{args.workload} 64x64 z=128 (BASELINE.json {CONFIG_OF[args.workload]}: global batch {args.batch})"
                                          if args.resolution == 64 else
                                          f"{args.workload} 100x100 z=512 (the reference's ACTIVE configs/models_config.py block, "
                                          f"not a BASELINE.json config: global batch {args.batch})"),
                                global_batch=args.batch, per_gpu_batch=B, parallelism=f"dp{world}",
                                l2="inputs larger than L2: per-step activation working set ~%.1f GB per GPU >> 126 MB" % act_gb,
                                cuda_graph=bool(args.graph),
                                optimizer=("Adam (fused multi-tensor), betas (0.5, 0.999)" if "wae" in args.workload else
                                           "RMSprop (fused multi-tensor), equilibrium gate on device")
                                          + (" + Adam on the latent discriminator" if args.workload == "stage3_dual" else "")),
                    e2e=dict(value=e2e_value, unit="samples/s", ms_per_step=ms_e2e, h2d_bytes_per_step=h2d,
                             d2h_bytes_per_step=d2h), gpu_launches=launches, clocks=ck, roofline=roof, cpu_baseline=cpu, stock_torch=stock,
                    build_hash=build_hash(),
                    losses={k: (round(v, 4) if isinstance(v, float) else v) for k, v in losses.items()})
        print(json.dumps(line), flush=True)
    if world > 1:
        td.destroy_process_group()


def main():
    global METRIC
    sys.dont_write_bytecode = True   # the benchmark leaves the tree as build() left it: no __pycache__ of its imports
    args = parse()
    METRIC = f"{args.workload}_train_samples_per_sec_{args.resolution}x{args.resolution}"
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
