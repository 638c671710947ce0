"""Debug probe: wrap every lib entry point; after each call report the first tensor argument that became non-finite."""
import sys

import torch

sys.path.insert(0, __file__.rsplit("/", 2)[0])
from thesis_fmri_reconstruction_b200 import engine, hp, init, lib  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 512
seen = set()
count = [0]


def wrap(name, fn):
    def inner(*a, **k):
        r = fn(*a, **k)
        count[0] += 1
        torch.cuda.synchronize()
        ts = []
        for v in list(a) + list(k.values()):
            if torch.is_tensor(v):
                ts.append(v)
            elif isinstance(v, (list, tuple)):
                ts += [t for t in v if torch.is_tensor(t)]
        for i, t in enumerate(ts):
            if t.is_floating_point() and t.numel() and id(t) not in seen:
                tf = t.float() if t.dtype != torch.float64 else t
                if not torch.isfinite(tf).all():
                    seen.add(id(t))
                    print(f"call #{count[0]} {name}: tensor arg {i} shape {tuple(t.shape)} dtype {t.dtype} has "
                          f"{int((~torch.isfinite(tf)).sum())} non-finite values", flush=True)
        return r
    return inner


for n in dir(lib):
    f = getattr(lib, n)
    if callable(f) and not n.startswith("_") and n not in ("load", "ptr", "stream", "dt", "header_functions", "profile_begin",
                                                            "profile_end", "launch_count", "conv_desc", "edge_desc",
                                                            "linear_desc", "conv_out_hw", "conv_pack_elems",
                                                            "conv_wgrad_workspace", "edge_workspace", "FmriError", "ConvDesc",
                                                            "EdgeDesc", "LinearDesc", "ReluMask"):
        setattr(lib, n, wrap(n, f))

P, S = init.init_vaegan(hp.CFG64, 128, seed=12345)
tr = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.bfloat16)
g = torch.Generator().manual_seed(1234)
x = (torch.rand(B, 3, 64, 64, generator=g) * 2 - 1).cuda()
e = torch.randn(B, 128, generator=g).cuda()
zp = torch.randn(B, 128, generator=g).cuda()
tr.forward_backward(x, e, zp)
print("done, calls:", count[0])
