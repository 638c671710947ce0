"""The reference's UNCHANGED scripts on top of this repository's models (SURVEY.md 8f-1; VERDICT r1 "Next round" #2):

    train/train_vgan_stage1.py -> train_vgan_stage2.py -> train_vgan_stage3.py      (100x100 / latent 512: gan_config.py)
    train/train_wae_stage1.py  -> train_wae_stage2.py  -> train_wae_stage3.py       (64x64 / latent 128: wae_config.py)
    train/wae_vgan_stage1.py, inference/inference_gan.py

Each runs for one epoch of two iterations (batch 8) on a fabricated dataset tree, as a child process
`python <reference>/<script> -i <tree> -o <tree> -l <tree>/logs ...` with PYTHONPATH = harness stubs : this repo : the
reference (tests/script_harness/harness.py). Asserted per script: exit status 0; `models.vae_gan` and `configs.models_config`
were imported from THIS repository; libfmri_b200.so was loaded and launched kernels; every logged loss is finite; the
checkpoint the next stage loads was written (the stages hand over through `torch.save(model.state_dict())` files under the
names the reference's configs expect, so strict `load_state_dict` across stages is exercised by the scripts themselves).

The VAE/GAN scripts interleave `loss.backward(retain_graph=True)` with `optimizer.step()` (train_vgan_stage1.py:408-432),
which stock torch >= 1.5 rejects ON THE REFERENCE'S OWN MODULES (SURVEY.md 0-6); they run here because no Parameter is saved
for backward.

The reference's scripts are not part of this repository: these tests run against a checkout of the original project named by
$FMRI_REFERENCE_ROOT, and skip (and say so) without one.
"""
import math
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "script_harness"))
import harness as H  # noqa: E402

pytestmark = pytest.mark.gpu

REF = H.find_reference()
needs_ref = pytest.mark.skipif(REF is None, reason="FMRI_REFERENCE_ROOT names no checkout of the original project: the "
                               "unchanged-script harness needs the reference's scripts, which are not part of this repository")
COMMON = ["-b", 8, "-e", 1, "-nw", 0, "-d", "cuda:0"]
DRY = os.environ.get("FMRI_HARNESS_DRY") == "1"   # CPU dry run of the harness itself on the reference's own models (WAE chain)
if DRY:
    COMMON = ["-b", 8, "-e", 1, "-nw", 0, "-d", "cpu", "-im_size", 100, "-lat_dim", 512]


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    return H.make_tree(str(tmp_path_factory.mktemp("fmri_tree")))


def _run(script, tree, models_config, extra=()):
    r, rep = H.run_script(REF, script, tree, list(COMMON) + list(extra), models_config=models_config, repo_models=not DRY)
    tail = (r.stdout[-1500:] + "\n" + r.stderr[-4000:])
    assert r.returncode == 0, f"{script} exited {r.returncode}\n{tail}"
    assert rep is not None, f"{script}: no exit report\n{tail}"
    if not DRY:
        repo = H.REPO
        assert rep["models_file"] and os.path.abspath(rep["models_file"]).startswith(repo), rep
        assert rep["models_config_file"] and os.path.abspath(rep["models_config_file"]).startswith(repo), rep
        assert rep["lib_loaded"] and rep["launches"] > 100, rep
    losses = H.logged_losses(r.stderr)
    assert len(losses) >= 4, f"{script}: no per-step loss lines in the log\n{tail}"
    assert all(math.isfinite(v) for v in losses), losses
    print(f"{script}: rc 0, {rep['launches']} kernel launches, {len(losses)} logged loss values, all finite; first: {losses[:4]}")
    return r, rep


def _cfg(module):
    """A value the reference's config module holds (the names later stages load checkpoints by)."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("_ref_cfg_" + module, os.path.join(REF, "configs", module + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


# ------------------------------------------------------------------------------------------------ VAE/GAN chain (100x100)
@needs_ref
@pytest.mark.skipif(DRY, reason="the VAE/GAN scripts do not run on the reference's own modules under torch >= 1.5")
def test_train_vgan_stage1_unchanged(tree):
    _run("train/train_vgan_stage1.py", tree, 100)
    ck = H.newest_checkpoint(tree, "gan")
    assert ck is not None, "Stage I wrote no checkpoint"
    name, epoch = _cfg("gan_config").decoder_weights
    H.install_checkpoint(ck[1], tree, "gan", name, epoch)          # the name train_vgan_stage2.py:99-100 loads


@needs_ref
@pytest.mark.skipif(DRY, reason="see stage 1")
def test_train_vgan_stage2_unchanged(tree):
    name, epoch = _cfg("gan_config").decoder_weights
    if not os.path.exists(os.path.join(tree, "results", "gan", name, f"{name}_{epoch}.pth")):
        pytest.skip("Stage I checkpoint missing (stage 1 test did not run)")
    _run("train/train_vgan_stage2.py", tree, 100)
    ck = H.newest_checkpoint(tree, "gan_cog_2st")
    assert ck is not None, "Stage II wrote no checkpoint"
    name, epoch = _cfg("gan_config").cog_encoder_weights
    H.install_checkpoint(ck[1], tree, "gan_cog_2st", name, epoch)  # train_vgan_stage3.py:101-102


@needs_ref
@pytest.mark.skipif(DRY, reason="see stage 1")
def test_train_vgan_stage3_unchanged(tree):
    name, epoch = _cfg("gan_config").cog_encoder_weights
    if not os.path.exists(os.path.join(tree, "results", "gan_cog_2st", name, f"{name}_{epoch}.pth")):
        pytest.skip("Stage II checkpoint missing (stage 2 test did not run)")
    _run("train/train_vgan_stage3.py", tree, 100)
    assert H.newest_checkpoint(tree, "gan_cog_3st") is not None


@needs_ref
@pytest.mark.skipif(DRY, reason="see stage 1")
def test_wae_vgan_stage1_unchanged(tree):
    _run("train/wae_vgan_stage1.py", tree, 100)


# ------------------------------------------------------------------------------------------------ WAE/GAN chain (64x64)
@needs_ref
def test_train_wae_stage1_unchanged(tree):
    _run("train/train_wae_stage1.py", tree, 64)
    ck = H.newest_checkpoint(tree, "wae_gan")
    assert ck is not None, "WAE Stage I wrote no checkpoint"
    name, epoch = _cfg("wae_config").decoder_weights
    H.install_checkpoint(ck[1], tree, "wae_gan", name, epoch)      # train_wae_stage2.py:102-103


@needs_ref
def test_train_wae_stage2_unchanged(tree):
    name, epoch = _cfg("wae_config").decoder_weights
    if not os.path.exists(os.path.join(tree, "results", "wae_gan", name, f"{name}_{epoch}.pth")):
        pytest.skip("WAE Stage I checkpoint missing")
    _run("train/train_wae_stage2.py", tree, 64)
    ck = H.newest_checkpoint(tree, "waegan_cog")
    assert ck is not None, "WAE Stage II wrote no checkpoint"
    name, epoch = _cfg("wae_config").cog_encoder_weights
    H.install_checkpoint(ck[1], tree, "waegan_cog", name, epoch)   # train_wae_stage3.py:109-110


@needs_ref
def test_train_wae_stage3_unchanged(tree):
    name, epoch = _cfg("wae_config").cog_encoder_weights
    if not os.path.exists(os.path.join(tree, "results", "waegan_cog", name, f"{name}_{epoch}.pth")):
        pytest.skip("WAE Stage II checkpoint missing")
    _run("train/train_wae_stage3.py", tree, 64)
    assert H.newest_checkpoint(tree, "wae_3st") is not None


# ------------------------------------------------------------------------------------------------ inference
@needs_ref
@pytest.mark.skipif(DRY, reason="GPU only")
def test_inference_gan_unchanged(tree):
    """inference/inference_gan.py with its shipped configuration (configs/inference_config.py: dataset 'coco', mode
    'vae-gan', 100x100 / latent 512): eval-mode VaeGan forward on a training and a validation batch, PCC / SSIM / MSE."""
    r, rep = H.run_script(REF, "inference/inference_gan.py", tree, ["-b", 8, "-nw", 0, "-d", "cuda:0"], models_config=100)
    tail = r.stdout[-1500:] + "\n" + r.stderr[-4000:]
    assert r.returncode == 0, tail
    assert rep and rep["lib_loaded"] and rep["launches"] > 20 and os.path.abspath(rep["models_file"]).startswith(H.REPO), rep
    import re

    vals = [float(v) for v in re.findall(r"(?:PCC|SSIM|MSE):\s*(-?\d+\.\d+|nan|inf)", r.stderr)]
    assert len(vals) >= 6 and all(math.isfinite(v) for v in vals), (vals, tail)
    print(f"inference_gan.py: rc 0, {rep['launches']} kernel launches, metrics {vals[:6]}")
