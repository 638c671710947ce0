#!/usr/bin/env python
"""Device PIL-compatible resize (fmri_image_resample) throughput: COCO-shaped uint8 sources (a mix of 480 x 640 and
640 x 480, 3 channels) resized to 64 x 64 and 100 x 100 with BILINEAR and BICUBIC, flipped and shifted, normalised.

  python scripts/resample_bench.py [--batches 256,4096] [--res 64,100] [--reps 20] [--store 1024]
                                   [--out profiles/r3_resample_bench_1gpu.jsonl]

Per filter, resolution and batch size, one JSON line (printed and written to --out) with images/s of
  kernel     lib.image_resample with the descriptor table prebuilt, a fresh random index draw per call, timed with CUDA
             events;
  resident   data.ResidentStimuli.batch over a store of --store distinct images in HBM (descriptor table built on the
             host and copied, flip / shift drawn, one kernel). The store (0.94 GB at 1024 images) is larger than the
             126 MB L2, so a batch mostly reads its sources from HBM;
  host       PIL.Image.resize + torchvision ToTensor + Normalize on ONE host core, images/s.
src_bytes_per_image / kernel time gives the kernel's source read rate, beside the GPU's name, power limit and SM clocks
(read-only nvidia-smi queries).
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

import bench  # noqa: E402  (clock sampler)
from loss_mix_bench import gpu_info  # noqa: E402  (read-only nvidia-smi query of name, power limit, clocks)
from rescale_bench import events_ms  # noqa: E402

SHAPES = ((480, 640, 3), (640, 480, 3))


def host_images_per_s(res, filter, n=16):
    import numpy as np
    import torch
    from PIL import Image
    from torchvision import transforms as T

    rng = np.random.default_rng(0)
    imgs = [Image.fromarray(rng.integers(0, 256, SHAPES[i % 2], dtype=np.uint8)) for i in range(n)]
    f = {"bilinear": Image.Resampling.BILINEAR, "bicubic": Image.Resampling.BICUBIC}[filter]
    norm = T.Normalize((0.5,) * 3, (0.5,) * 3)
    torch.set_num_threads(1)
    step = lambda im: norm(T.functional.to_tensor(im.resize((res, res), f)))
    step(imgs[0])
    t = time.perf_counter()
    for im in imgs:
        step(im)
    return n / (time.perf_counter() - t)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--res", default="64,100")
    ap.add_argument("--filters", default="bilinear,bicubic")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--store", type=int, default=1024, help="distinct images held in HBM")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_resample_bench_1gpu.jsonl"))
    a = ap.parse_args()
    sys.dont_write_bytecode = True
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    import torch

    from thesis_fmri_reconstruction_b200 import data
    from thesis_fmri_reconstruction_b200 import lib as L

    if not torch.cuda.is_available():
        raise SystemExit("resample_bench.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    info = gpu_info(0)
    g = torch.Generator().manual_seed(7)
    stim = data.ResidentStimuli([torch.randint(0, 256, SHAPES[i % 2], generator=g, dtype=torch.uint8)
                                 for i in range(a.store)])
    lines = []
    for filter in a.filters.split(","):
        for res in [int(v) for v in a.res.split(",")]:
            host_ips = host_images_per_s(res, filter)
            for B in [int(v) for v in a.batches.split(",")]:
                pipe = data.DevicePipeline((0.5,) * 3, (0.5,) * 3, random_flip=True, max_shift=5, generator=g,
                                           size=(res, res), resample=filter)
                draws = [torch.randint(0, a.store, (B,), generator=g).tolist() for _ in range(a.reps)]
                out = torch.empty(B, 3, res, res, device="cuda")
                it = iter(range(10 ** 9))
                resident = lambda: stim.batch(draws[next(it) % a.reps], pipe, out)
                resident()
                tables = [L.image_window_table(data.resample_windows([stim.entries[i] for i in d], (res, res)))
                          for d in draws]
                flip, shift = (t.cuda() for t in pipe.draw(B))
                ws = torch.empty(L.image_resample_workspace(B), dtype=torch.uint8, device="cuda")
                kt = iter(range(10 ** 9))
                kernel = lambda: L.image_resample(stim.buf, tables[next(kt) % a.reps], filter, flip, shift, pipe.mean,
                                                  pipe.std, out, ws)
                kernel()
                ck = bench.ClockSampler(0)
                ck.start()
                t_kernel = [events_ms(kernel, a.reps) for _ in range(2)]
                t_res = [events_ms(resident, a.reps) for _ in range(2)]
                clocks = ck.stop()
                ms_k, ms_r = min(t_kernel), min(t_res)
                src = 480 * 640 * 3
                line = dict(src="480x640x3 / 640x480x3", filter=filter, res=res, batch=B, reps=a.reps, store=a.store,
                            kernel_ms=round(ms_k, 4), kernel_ms_runs=[round(v, 4) for v in t_kernel],
                            kernel_images_per_s=round(B / ms_k * 1e3), resident_ms=round(ms_r, 4),
                            resident_images_per_s=round(B / ms_r * 1e3),
                            host_pillow_totensor_normalize_images_per_s_per_core=round(host_ips, 1),
                            src_bytes_per_image=src, kernel_src_read_tb_per_s=round(B * src / (ms_k * 1e-3) / 1e12, 3),
                            sm_mhz=clocks.get("sm_mhz"), throttle=clocks.get("reasons"), **info)
                print(json.dumps(line), flush=True)
                lines.append(line)
                del out, ws
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
