#!/usr/bin/env python
"""Device stimulus rescale (fmri_image_rescale) throughput: 375 x 375 x 3 uint8 stimuli (BOLD5000's native size) resized
to 100 x 100 and 64 x 64, with flip and shift, normalised.

  python scripts/rescale_bench.py [--batches 256,4096] [--res 100,64] [--reps 20] [--out profiles/r3_rescale_bench_1gpu.jsonl]

Per resolution and batch size, one JSON line (printed and written to --out) with images/s of
  resident   data.ResidentStimuli.batch over a store of --store distinct stimuli in HBM, a fresh random index draw per batch
             (descriptor table built on the host and copied, flip / shift drawn, one kernel); kernel_ms is the same call
             with the table prebuilt, timed with CUDA events. The store (1.7 GB at 4096 stimuli) is larger than the
             126 MB L2, so a batch mostly reads its sources from HBM;
  streamed   a pinned host batch [B, 375, 375, 3] copied to the device and rescaled (Prefetcher's work per batch, here
             without a step to overlap with);
  host       the fp64 scipy restatement (tests/rescale_reference.py) on ONE host core, images/s.
src_bytes_per_image / kernel time gives the kernel's source read rate (the bound named in DESIGN.md section 4), beside the
GPU's name, power limit and SM clocks (read-only nvidia-smi queries).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "scripts"))
sys.path.insert(2, os.path.join(ROOT, "tests"))

import bench  # noqa: E402  (clock sampler)
from loss_mix_bench import gpu_info  # noqa: E402  (read-only nvidia-smi query of name, power limit, clocks)

HS = 375


def events_ms(fn, reps):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_images_per_s(res, n=8):
    import numpy as np

    import rescale_reference as R

    rng = np.random.default_rng(0)
    imgs = rng.integers(0, 256, (n, HS, HS, 3), dtype=np.uint8)
    R.resize(imgs[0], (res, res))
    t = time.perf_counter()
    for im in imgs:
        R.resize(im, (res, res))
    return n / (time.perf_counter() - t)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--res", default="100,64")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--store", type=int, default=4096, help="distinct stimuli held in HBM")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_rescale_bench_1gpu.jsonl"))
    a = ap.parse_args()
    sys.dont_write_bytecode = True
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    import torch

    from thesis_fmri_reconstruction_b200 import data
    from thesis_fmri_reconstruction_b200 import lib as L

    if not torch.cuda.is_available():
        raise SystemExit("rescale_bench.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    info = gpu_info(0)
    g = torch.Generator().manual_seed(7)
    host_store = torch.randint(0, 256, (a.store, HS, HS, 3), generator=g, dtype=torch.uint8)
    stim = data.ResidentStimuli(host_store)
    lines = []
    for res in [int(v) for v in a.res.split(",")]:
        host_ips = host_images_per_s(res)
        for B in [int(v) for v in a.batches.split(",")]:
            pipe = data.DevicePipeline((0.5,) * 3, (0.5,) * 3, random_flip=True, max_shift=5, generator=g, size=(res, res))
            draws = [torch.randint(0, a.store, (B,), generator=g).tolist() for _ in range(a.reps)]
            out = torch.empty(B, 3, res, res, device="cuda")
            it = iter(range(10 ** 9))
            resident = lambda: stim.batch(draws[next(it) % a.reps], pipe, out)
            resident()
            # kernel alone: prebuilt table, fresh index draw per call
            tables = [L.image_src_table([stim.entries[i] for i in d]) for d in draws]
            flip, shift = (t.cuda() for t in pipe.draw(B))
            ws = torch.empty(L.image_rescale_workspace(B), dtype=torch.uint8, device="cuda")
            kt = iter(range(10 ** 9))
            kernel = lambda: L.image_rescale(stim.buf, tables[next(kt) % a.reps], flip, shift, pipe.mean, pipe.std, out, ws)
            kernel()
            pinned = host_store[:B].pin_memory()
            streamed = lambda: pipe(pinned.to("cuda", non_blocking=True), *pipe.draw(B), out)
            streamed()
            ck = bench.ClockSampler(0)
            ck.start()
            t_kernel = [events_ms(kernel, a.reps) for _ in range(2)]
            t_res = [events_ms(resident, a.reps) for _ in range(2)]
            t_str = [events_ms(streamed, a.reps) for _ in range(2)]
            clocks = ck.stop()
            ms_k, ms_r, ms_s = (min(t) for t in (t_kernel, t_res, t_str))
            src = HS * HS * 3
            line = dict(src=f"{HS}x{HS}x3", res=res, batch=B, reps=a.reps, store=a.store,
                        kernel_ms=round(ms_k, 4), kernel_ms_runs=[round(v, 4) for v in t_kernel],
                        kernel_images_per_s=round(B / ms_k * 1e3), resident_ms=round(ms_r, 4),
                        resident_images_per_s=round(B / ms_r * 1e3), streamed_ms=round(ms_s, 4),
                        streamed_images_per_s=round(B / ms_s * 1e3), host_scipy_images_per_s_per_core=round(host_ips, 1),
                        src_bytes_per_image=src, kernel_src_read_tb_per_s=round(B * src / (ms_k * 1e-3) / 1e12, 3),
                        sm_mhz=clocks.get("sm_mhz"), throttle=clocks.get("reasons"), **info)
            print(json.dumps(line), flush=True)
            lines.append(line)
            del pinned, out, ws
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
