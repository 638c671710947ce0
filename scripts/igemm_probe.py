"""Times the 32-channel implicit-GEMM launches of the batch-4096 step in isolation (CUDA events, 5 repetitions after warm-up).
With FMRI_IG_SKIP=1|2|4|8 one role of igemm_persistent_kernel is switched off (TMA loads / whole epilogue / MMAs / only the
epilogue's global stores): the role whose removal shortens the kernel most is the one that bounds it.
python scripts/igemm_probe.py [B]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from thesis_fmri_reconstruction_b200 import lib as L  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
BF = torch.bfloat16
F64 = torch.float64


def timeit(fn, n=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    dev = "cuda"
    rows = []
    # Discriminator block 1: Conv2d(32, 128, 5, s2) on 3B images of 64x64 (fprop with BN statistics; dgrad on 2B images)
    N3 = 3 * B
    d = L.conv_desc(N3, 64, 64, 32, 128, 2, False, 0, BF)
    w = torch.randn(128, 32, 5, 5, device=dev) * 0.05
    pf = torch.empty(L.conv_pack_elems(d), dtype=BF, device=dev)
    pd = torch.empty(L.conv_pack_elems(d), dtype=BF, device=dev)
    L.conv_pack_weights(d, w, pf, pd)
    x = torch.randn(N3, 64, 64, 32, device=dev).to(BF)
    y = torch.empty(N3, 32, 32, 128, dtype=BF, device=dev)
    s1, s2 = torch.zeros(128, dtype=F64, device=dev), torch.zeros(128, dtype=F64, device=dev)
    fl = 2.0 * N3 * 32 * 32 * 128 * 32 * 25
    rows.append(("D block 1 fprop 32->128 s2, 3B imgs, BN stats (gather)", lambda: L.conv_fprop(d, x, w, pf, None, L.ACT_NONE, y, s1, s2), fl))
    rows.append(("D block 1 fprop, no stats", lambda: L.conv_fprop(d, x, w, pf, None, L.ACT_NONE, y, None, None), fl))
    dx = torch.empty(N3, 64, 64, 32, dtype=BF, device=dev)
    rows.append(("D block 1 dgrad 128->32, 3B imgs (merged scatter)", lambda: L.conv_dgrad(d, y, w, pd, dx), fl))
    # Decoder block 3: ConvTranspose2d(128, 32, 5, s2) 32x32 -> 64x64 on B images
    dt = L.conv_desc(B, 32, 32, 128, 32, 2, True, 1, BF)
    wt = torch.randn(128, 32, 5, 5, device=dev) * 0.05
    tf = torch.empty(L.conv_pack_elems(dt), dtype=BF, device=dev)
    td = torch.empty(L.conv_pack_elems(dt), dtype=BF, device=dev)
    L.conv_pack_weights(dt, wt, tf, td)
    xt = torch.randn(B, 32, 32, 128, device=dev).to(BF)
    yt = torch.empty(B, 64, 64, 32, dtype=BF, device=dev)
    t1, t2 = torch.zeros(32, dtype=F64, device=dev), torch.zeros(32, dtype=F64, device=dev)
    flt = 2.0 * B * 32 * 32 * 128 * 32 * 25
    rows.append(("Decoder block 3 fprop 128->32 convT, B imgs, BN stats (merged scatter)", lambda: L.conv_fprop(dt, xt, wt, tf, None, L.ACT_NONE, yt, t1, t2), flt))
    dxt = torch.empty(B, 32, 32, 128, dtype=BF, device=dev)
    rows.append(("Decoder block 3 dgrad 32->128, B imgs (gather)", lambda: L.conv_dgrad(dt, yt, wt, td, dxt), flt))
    # a fat layer for scale: Discriminator block 2 Conv2d(128, 256, 5, s2) on 3B images of 32x32
    d2 = L.conv_desc(N3, 32, 32, 128, 256, 2, False, 0, BF)
    w2 = torch.randn(256, 128, 5, 5, device=dev) * 0.02
    p2 = torch.empty(L.conv_pack_elems(d2), dtype=BF, device=dev)
    L.conv_pack_weights(d2, w2, p2, None)
    y2 = torch.empty(N3, 16, 16, 256, dtype=BF, device=dev)
    u1, u2 = torch.zeros(256, dtype=F64, device=dev), torch.zeros(256, dtype=F64, device=dev)
    rows.append(("D block 2 fprop 128->256 s2, 3B imgs, BN stats", lambda: L.conv_fprop(d2, y, w2, p2, None, L.ACT_NONE, y2, u1, u2), 2.0 * N3 * 16 * 16 * 256 * 128 * 25))
    print(f"# FMRI_IG_SKIP={os.environ.get('FMRI_IG_SKIP', '0')} B={B}")
    for name, fn, flops in rows:
        ms = timeit(fn)
        print(f"{name:76s} {ms:8.3f} ms {flops / ms / 1e9:8.1f} TFLOP/s")


main()
