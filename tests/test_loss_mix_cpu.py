"""CPU-side checks of the pixel-NLE loss mixes of the fused Stage-I step (train_vgan_stage1.py:374-388, modes 'dcgan' and
'vae'): the per-mode algorithmic-FLOP accounting of scripts/loss_mix_bench.py, the host restatement of the equilibrium gate
with the loss mix's pre-gate train_dis, and the refusal of an unknown mode before any device work."""
import importlib.util
import os

import pytest

from oracle import vaegan as O
from thesis_fmri_reconstruction_b200 import dp, engine, hp, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# mean bce values on both sides of equilibrium -/+ margin (0.33 and 1.03 at the default constants), never on a threshold
GATE_GRID = (0.05, 0.3, 0.36, 0.68, 1.0, 1.06, 2.5)


def _load(name, rel):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, rel))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_loss_mix_mflop_per_mode():
    mb = _load("loss_mix_bench_mod", os.path.join("scripts", "loss_mix_bench.py"))
    bench = _load("bench_mod", "bench.py")
    for cfg, z in ((hp.CFG64, 128), (hp.CFG100, 512)):
        assert mb.alg_mflop(cfg, z, "vae-gan") == pytest.approx(bench.stage1_alg_mflop(cfg, z), rel=1e-12)
    want = {(64, "vae-gan"): 16966.2, (64, "dcgan"): 13279.6, (64, "vae"): 12020.6,
            (100, "vae-gan"): 27815.4, (100, "dcgan"): 22254.4, (100, "vae"): 18106.0}
    for (res, mode), v in want.items():
        cfg, z = (hp.CFG64, 128) if res == 64 else (hp.CFG100, 512)
        assert round(mb.alg_mflop(cfg, z, mode), 1) == v, (res, mode, mb.alg_mflop(cfg, z, mode))
    with pytest.raises(ValueError):
        mb.alg_mflop(hp.CFG64, 128, "gan")


@pytest.mark.parametrize("train_dis_in", [False, True])
def test_gate_from_sums_matches_oracle_gate(train_dis_in):
    B, margin, eq = 64, 0.35, 0.68
    seen = set()
    for mo in GATE_GRID:
        for mp in GATE_GRID:
            got = dp.gate_from_sums(mo * B, mp * B, B, margin, eq, train_dis_in=train_dis_in)
            assert got == O.gate(mo, mp, margin, eq, train_dis_in), (mo, mp, train_dis_in)
            seen.add(got)
    # every reachable outcome; with train_dis_in False, (True, True) comes only from the "neither -> both" rule
    assert seen == ({(True, True), (False, True), (True, False)} if train_dis_in else {(True, True), (False, True)})
    # the default keeps the gate of the 'vae-gan' mix
    assert dp.gate_from_sums(0.5 * B, 0.5 * B, B, margin, eq) == (True, True)


@pytest.mark.parametrize("mode", ["gan", "VAE", "beta_vae", ""])
def test_unknown_mode_raises_before_device_work(mode):
    with pytest.raises(lib.FmriError, match="loss mix"):
        engine.VaeGanStage1({}, {}, hp.CFG64, 128, mode=mode)
