"""The pixel-NLE loss mixes of the fused Stage-I step (train_vgan_stage1.py:374-388: 'dcgan' and 'vae') against the oracle's
statement of them (oracle.stage1_vaegan_step(mode=...), pinned to the unmodified reference by tests/golden/stage1_vae_* and
stage1_dcgan_*), on the same seeded inputs and weights.

Tolerances are those of tests/test_engine_gpu.py (rel-L2 per tensor): fp32 exact path -- forward tensors, losses and BN
buffers 1e-4, gradient buckets against the fp64 oracle max(5e-3, 3 x the oracle's own fp32-vs-fp64 deviation); bf16 tensor
path -- forward 2e-2, gradient buckets reported and bounded at 0.5 (ReLU-mask flips under bf16 rounding, SURVEY.md 0-9).
Parameter deltas after the first RMSprop step are bounded at 0.15 on the fp32 path: that step moves every element by about
lr * sign(g) / sqrt(0.1) however small g is, so elements whose gradient is below the fp32 noise can move the other way
(the 'vae-gan' step's own fp32 report, profiles/parity/parity_stage1_B8_float32.json, shows 4e-2 .. 6e-2)."""
import json
import os
import subprocess
import sys

import pytest
import torch

from oracle import vaegan as O
from thesis_fmri_reconstruction_b200 import dp, engine, hp
from thesis_fmri_reconstruction_b200 import lib as L

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ("dcgan", "vae")
BUCKETS = ("encoder.", "decoder.", "discriminator.")
# mean bce values on both sides of equilibrium -/+ margin (0.33 and 1.03 at the default constants), never on a threshold
GATE_GRID = (0.05, 0.3, 0.36, 0.68, 1.0, 1.06, 2.5)


def rel(a, b):
    a, b = a.detach().double().cpu().reshape(-1), b.detach().double().cpu().reshape(-1)
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def nchw_flat(raw_nhwc):
    return raw_nhwc.float().permute(0, 3, 1, 2).reshape(raw_nhwc.shape[0], -1)


def _setup(res):
    return (O.CFG64, hp.CFG64, 128) if res == 64 else (O.CFG100, hp.CFG100, 512)


def _forward_errs(out, ref, lo):
    errs = dict(mu=rel(out["mu"], ref["mu"]), logvar=rel(out["logvar"], ref["logvar"]),
                x_tilde=rel(out["x_tilde"], ref["x_tilde"]), x_p=rel(out["x_p"], ref["x_p"]),
                disc_layer=rel(nchw_flat(out["disc_layer_nhwc"]), ref["disc_layer"]),
                disc_class=rel(out["disc_class"], ref["disc_class"].reshape(-1)), kl=rel(out["kl"], ref["kl"]),
                mse=rel(out["mse"], ref["mse"]), nle=rel(out["nle"], ref["nle"].sum(1)),   # oracle: nle per element
                bce=rel(out["bce"], torch.cat([ref["bce_o"], ref["bce_p"], ref["bce_s"]]).reshape(-1)))
    for k in ("loss_encoder", "loss_decoder", "loss_discriminator"):
        errs[k] = abs(lo[k] - ref[k].item()) / abs(ref[k].item())
    for k in ("nle", "kl", "mse", "bce_o", "bce_p", "bce_s"):   # the six logged sums of sc[0..5]
        errs["sum_" + k] = abs(lo[k] - ref[k].sum().item()) / abs(ref[k].sum().item())
    return errs


def run_mix_case(mode, B, adt, res=64, seed=4343):
    cfg_o, cfg, z = _setup(res)
    P, S = O.make_vaegan(cfg_o, seed=seed)
    x = O.synthetic_images(B, size=res, seed=seed)
    eps, z_p = O.synthetic_noise(B, z, seed=seed)
    S_ref = {k: v.clone() for k, v in S.items()}
    ref = O.stage1_vaegan_step(P, S_ref, x, eps, z_p, cfg=cfg_o, mode=mode)
    ref64 = None
    if adt == torch.float32:
        P64 = {k: v.double() for k, v in P.items()}
        S64 = {k: (v.double() if v.dtype.is_floating_point else v.clone()) for k, v in S.items()}
        ref64 = O.stage1_vaegan_step(P64, S64, x.double(), eps.double(), z_p.double(), cfg=cfg_o, mode=mode, update=False)
    tr = engine.VaeGanStage1(P, S, cfg, z, adt, mode=mode)
    be = tr.buckets["encoder."]
    enc_p0, enc_sq0 = be.flat_p.clone(), be.states[0].clone()
    out = tr.forward_backward(x.cuda(), eps.cuda(), z_p.cuda())
    grads = {k: v.clone() for k, v in tr.named_grads().items()}
    tr.update(B)
    torch.cuda.synchronize()
    lo = tr.losses()
    fwd = _forward_errs(out, ref, lo)
    gate_ok = (lo["train_dis"], lo["train_dec"]) == (ref["train_dis"], ref["train_dec"])
    gerr, gnoise = {}, {}
    for b in BUCKETS:
        ks = [k for k in grads if k.startswith(b)]
        if ks[0] not in ref["grads"]:   # 'dcgan': the oracle computes no encoder gradient (the encoder is not trained)
            continue
        a = torch.cat([grads[k].reshape(-1) for k in ks])
        gref = ref64 if ref64 is not None else ref
        gerr[b] = rel(a, torch.cat([gref["grads"][k].reshape(-1) for k in ks]))
        if ref64 is not None:
            gnoise[b] = rel(torch.cat([ref["grads"][k].reshape(-1) for k in ks]),
                            torch.cat([ref64["grads"][k].reshape(-1) for k in ks]))
    newP = tr.named_parameters()
    derr = {}
    for b in BUCKETS:
        ks = [k for k in newP if k.startswith(b)]
        derr[b] = rel(torch.cat([(newP[k].cpu() - P[k]).reshape(-1) for k in ks]),
                      torch.cat([(ref["params"][k] - P[k]).reshape(-1) for k in ks]))
    berr = {k: rel(v, S_ref[k]) for k, v in tr.named_buffers().items() if v.dtype.is_floating_point}
    nbt_ok = all(int(v) == int(S_ref[k]) for k, v in tr.named_buffers().items() if not v.dtype.is_floating_point)
    enc_grad_max = max(grads[k].abs().max().item() for k in grads if k.startswith("encoder."))
    enc_frozen = bool(torch.equal(be.flat_p, enc_p0) and torch.equal(be.states[0], enc_sq0))
    rep = dict(mode=mode, B=B, res=res, dtype=str(adt), forward=fwd, grad_bucket=gerr, grad_bucket_oracle_fp32_noise=gnoise,
               delta_bucket=derr, bn_worst=max(berr.items(), key=lambda t: t[1]), gate_ok=gate_ok, nbt_ok=nbt_ok,
               gate=(lo["train_dis"], lo["train_dec"]), enc_grad_max=enc_grad_max, enc_frozen=enc_frozen)
    out_dir = os.environ.get("FMRI_PARITY_DIR")   # optional: keep the per-case reports (profiles/parity/ holds such files)
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, f"parity_stage1_{mode}_res{res}_B{B}_{str(adt).split('.')[-1]}.json"), "w") as f:
            json.dump(rep, f, indent=1)
    print(json.dumps(rep, indent=1))
    return rep


def _check_case(rep, adt):
    if adt == torch.float32:
        assert max(rep["forward"].values()) < 1e-4, rep["forward"]
        for b, e in rep["grad_bucket"].items():
            assert e < max(5e-3, 3 * rep["grad_bucket_oracle_fp32_noise"][b]), (b, e, rep["grad_bucket_oracle_fp32_noise"])
        assert max(rep["delta_bucket"].values()) < 0.15, rep["delta_bucket"]
        assert rep["bn_worst"][1] < 1e-4
    else:
        assert max(rep["forward"].values()) < 2e-2, rep["forward"]
        assert max(rep["grad_bucket"].values()) < 0.5, rep["grad_bucket"]
        assert rep["bn_worst"][1] < 2e-2
    assert rep["gate_ok"] and rep["nbt_ok"], (rep["gate"], rep["nbt_ok"])
    if rep["mode"] == "dcgan":   # the encoder is not trained: zero gradient bucket, parameters and square_avg unchanged
        assert rep["enc_grad_max"] == 0.0 and rep["enc_frozen"]
    else:
        assert "encoder." in rep["grad_bucket"] and rep["enc_grad_max"] > 0.0


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("res,adt,B", [(64, torch.float32, 8), (64, torch.bfloat16, 16), (100, torch.float32, 4),
                                       (100, torch.bfloat16, 16)])
def test_loss_mix_step_matches_oracle(mode, res, adt, B):
    """64x64 / latent 128 and the reference's active 100x100 / latent 512 block (hp.CFG100: odd feature maps, stride_gan 2)."""
    _check_case(run_mix_case(mode, B, adt, res), adt)


def test_loss_mix_large_batch_bf16():
    """B = 256: the persistent, wave-split and merged-scatter kernel paths. The forward, the six loss sums and the BatchNorm
    buffers do not depend on the loss mix, so one fp32 oracle forward serves both modes; each mode's gate is the oracle's
    rule on those sums with the mode's pre-gate train_dis."""
    B, seed = 256, 9256
    P, S = O.make_vaegan(O.CFG64, seed=seed)
    x = O.synthetic_images(B, seed=seed)
    eps, z_p = O.synthetic_noise(B, 128, seed=seed)
    S_ref = {k: v.clone() for k, v in S.items()}
    ref = O.stage1_vaegan_step(P, S_ref, x, eps, z_p, mode="vae", update=False)
    for mode in MODES:
        tr = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.bfloat16, mode=mode)
        out = tr.forward_backward(x.cuda(), eps.cuda(), z_p.cuda())
        tr.update(B)
        torch.cuda.synchronize()
        lo = tr.losses()
        fwd = _forward_errs(out, {**ref, **_mode_losses(ref, mode)}, lo)
        berr = {k: rel(v, S_ref[k]) for k, v in tr.named_buffers().items() if v.dtype.is_floating_point}
        nbt_ok = all(int(v) == int(S_ref[k]) for k, v in tr.named_buffers().items() if not v.dtype.is_floating_point)
        for k, v in tr.named_grads().items():
            assert torch.isfinite(v).all(), (mode, k)
        bn_worst = max(berr.items(), key=lambda t: t[1])
        print(mode, "B=256 bf16 forward", fwd, "bn_worst", bn_worst)
        assert max(fwd.values()) < 2e-2, (mode, fwd)
        assert bn_worst[1] < 2e-2 and nbt_ok, (mode, bn_worst)
        want = O.gate(ref["bce_o"].mean().item(), ref["bce_p"].mean().item(), O.HP_VGAN["margin"], O.HP_VGAN["equilibrium"],
                      mode != "vae")
        assert (lo["train_dis"], lo["train_dec"]) == want, (mode, want)


def _mode_losses(ref, mode):
    """The three losses of `mode` from the mode-independent per-sample terms of an oracle step (train_vgan_stage1.py:374-387)."""
    lam = O.HP_VGAN["lambda_mse"]
    loss_dis = ref["bce_o"].sum() + ref["bce_s"].sum()
    loss_dec = (lam * ref["nle"]).sum() - ((1.0 - lam) * loss_dis if mode == "dcgan" else 0.0)
    return dict(loss_encoder=ref["kl"].sum() + ref["nle"].sum(), loss_discriminator=loss_dis, loss_decoder=loss_dec)


def test_gate_mix_kernel_matches_oracle_gate():
    """fmri_vgan_gate_mix on a grid of (mean bce_o, mean bce_p) covering both sides of every threshold, both pre-gate flags:
    the init weights rarely reach the 'vae' mode's "neither -> both" branch, so the grid is what exercises it."""
    B, margin, eq = 64, 0.35, 0.68
    gates = torch.full((2,), -1.0, device="cuda")
    seen = set()
    for dis_in in (0, 1):
        for mo in GATE_GRID:
            for mp in GATE_GRID:
                sums = torch.tensor([mo * B, mp * B], device="cuda")
                L.vgan_gate_mix(sums, B, margin, eq, dis_in, gates)
                got = tuple(bool(v) for v in gates.tolist())
                want = O.gate(mo, mp, margin, eq, bool(dis_in))
                assert got == want == dp.gate_from_sums(mo * B, mp * B, B, margin, eq, bool(dis_in)), (mo, mp, dis_in, got)
                if dis_in:
                    L.vgan_gate(sums, B, margin, eq, gates)   # the 'vae-gan' entry point is the same gate with 1
                    assert tuple(bool(v) for v in gates.tolist()) == got
                seen.add((dis_in, got))
    assert (0, (True, True)) in seen and (1, (True, False)) in seen and (0, (False, True)) in seen


@pytest.mark.parametrize("mode", MODES)
def test_loss_mix_five_bf16_steps_stay_finite(mode):
    B, seed = 16, 55
    P, S = O.make_vaegan(O.CFG64, seed=seed)
    tr = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.bfloat16, mode=mode)
    x = O.synthetic_images(B, seed=seed).cuda()
    eps, z_p = [t.cuda() for t in O.synthetic_noise(B, 128, seed=seed)]
    for step in range(5):
        tr.step(x, eps, z_p)
        torch.cuda.synchronize()
        for k, v in tr.losses().items():
            assert v == v and abs(v) != float("inf"), (step, k, v)
        for k, v in tr.named_parameters().items():
            assert torch.isfinite(v).all(), (step, k)


@pytest.mark.parametrize("mode", MODES)
def test_loss_mix_graphed_step_matches_eager(mode):
    """One CUDA-graph replay equals the eager step from the same loaded state (bounds of test_graphed_step_matches_eager)."""
    B, seed = 8, 37
    P, S = O.make_vaegan(O.CFG64, seed=seed)
    x = O.synthetic_images(B, seed=seed).cuda()
    eps, z_p = [t.cuda() for t in O.synthetic_noise(B, 128, seed=seed)]
    a = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.float32, mode=mode)
    b = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.float32, mode=mode)
    g = engine.GraphedStep(b, x, eps, z_p, warmup=2)
    for _ in range(3):
        a.step(x, eps, z_p)
    b.load_state_dict(a.state_dict())
    a.step(x, eps, z_p)
    out = g(x, eps, z_p)
    torch.cuda.synchronize()
    pa, pb = a.named_parameters(), b.named_parameters()
    worst = max(rel(pb[k], pa[k].cpu()) for k in pa)
    la, lb = a.losses(), b.losses()
    print(mode, "graphed vs eager: worst parameter rel", worst, "launches/replay", g.launches)
    assert worst < 1e-3, worst
    assert abs(la["loss_encoder"] - lb["loss_encoder"]) <= 1e-5 * abs(la["loss_encoder"])
    assert (la["train_dis"], la["train_dec"]) == (lb["train_dis"], lb["train_dec"])
    sa, sb = a.named_buffers(), b.named_buffers()
    assert all(int(sa[k]) == int(sb[k]) for k in sa if not sa[k].dtype.is_floating_point)
    assert max(rel(sb[k], sa[k].cpu()) for k in sa if sa[k].dtype.is_floating_point) < 1e-5
    assert g.launches > 100 and torch.isfinite(out["x_tilde"].float()).all()


@pytest.mark.parametrize("mode", MODES)
def test_loss_mix_checkpoint_round_trip(mode):
    """state_dict -> new trainer -> load_state_dict -> one step equals the original trainer's step (end_epoch included)."""
    B, seed = 8, 13
    x = O.synthetic_images(B, seed=seed).cuda()
    eps, z_p = [t.cuda() for t in O.synthetic_noise(B, 128, seed=seed)]
    P, S = O.make_vaegan(O.CFG64, seed=seed)
    a = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.float32, mode=mode)
    for _ in range(2):
        a.step(x, eps, z_p)
    a.end_epoch()
    sd = a.state_dict()
    b = engine.VaeGanStage1(P, S, hp.CFG64, 128, torch.float32, mode=mode)
    b.load_state_dict(sd)
    a.step(x, eps, z_p)
    b.step(x, eps, z_p)
    torch.cuda.synchronize()
    pa, pb = a.named_parameters(), b.named_parameters()
    worst = max(rel(pb[k], pa[k].cpu()) for k in pa)
    sa, sb = a.named_buffers(), b.named_buffers()
    assert worst < 1e-3, worst
    assert all(int(sa[k]) == int(sb[k]) for k in sa if not sa[k].dtype.is_floating_point)
    assert max(rel(sb[k], sa[k].cpu()) for k in sa if sa[k].dtype.is_floating_point) < 1e-5
    assert a.lr == b.lr and a.hp == b.hp
    if mode == "dcgan":
        for k in pa:
            if k.startswith("encoder."):
                assert torch.equal(pa[k].cpu(), P[k]), k


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dtype,B", [("f32", 8), ("bf16", 32)])
def test_loss_mix_two_rank_nccl_equals_sequential_shards(mode, dtype, B):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29531", os.path.join(ROOT, "tests", "dp_loss_mix_worker.py"), mode, dtype, str(B)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("DPRESULT ")][-1]
    res = json.loads(line[len("DPRESULT "):])
    print(res)
    for rr in res:
        assert max(rr["grad_err"].values()) < (1e-5 if dtype == "f32" else 0.2), rr
        assert rr["sum_err"] < 1e-5, rr
        assert tuple(rr["gate_dev"]) == tuple(rr["gate_host"]) == tuple(res[0]["gate_dev"]), rr
        if mode == "dcgan":
            assert rr["enc_grad_max"] == 0.0 and "encoder." not in rr["grad_err"], rr
        else:
            assert "encoder." in rr["grad_err"], rr
