"""Runs the reference's UNCHANGED train / inference scripts on top of this repository's models (SURVEY.md 8f-1).

    stubs/          stand-ins for the host-side packages this image lacks (matplotlib, skimage, nibabel, h5py)
    make_tree()     fabricates the dataset tree of the reference's configs/data_config.py:5-45 (random JPEGs for the COCO
                    folders and the BOLD5000 stimuli, random standardised 3620-voxel vectors in the pickles)
    run_script()    python <reference>/<script> ... in a child process with PYTHONPATH = stubs : this repo : reference, so
                    `models.vae_gan` and `configs.models_config` resolve HERE and everything else (configs.gan_config,
                    data_preprocessing, train.train_utils, the script itself) resolves in the untouched reference tree

The reference tree is a checkout of the original project named by $FMRI_REFERENCE_ROOT; this repository does not hold its
scripts, so without it the harness has nothing to run. Test infrastructure only.
"""
from __future__ import annotations

import json
import os
import pickle
import re
import shutil
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
STUBS = os.path.join(HERE, "stubs")
NEEDED = ("train/train_vgan_stage1.py", "configs/gan_config.py", "data_preprocessing/data_loader.py", "train/train_utils.py")


def find_reference():
    root = os.environ.get("FMRI_REFERENCE_ROOT")
    if root and all(os.path.exists(os.path.join(root, f)) for f in NEEDED):
        return root
    return None


def _jpeg(path, rng, px):
    from PIL import Image

    os.makedirs(os.path.dirname(path), exist_ok=True)
    # smooth random colour field (upsampled noise): compresses well and is not degenerate for PCC / SSIM
    small = rng.integers(0, 256, size=(12, 12, 3), dtype=np.uint8)
    Image.fromarray(small).resize((px, px), Image.BICUBIC).save(path, quality=85)


def make_tree(root, n_train=8, n_test=8, n_valid=8, n_bold_train=16, n_bold_valid=8, px=375, voxels=3620, seed=0):
    """Dataset tree under <root>/datasets/ (data_config.py: data_root, coco_*_data, train_data, valid_data; inference_config.py:
    train_data / valid_data). Image counts are multiples of the harness batch size, so one epoch is a whole number of steps."""
    rng = np.random.default_rng(seed)
    ds = os.path.join(root, "datasets")
    for sub, n in (("coco/coco_train2017/train2017", n_train), ("coco/coco_valid2017/val2017", n_valid),
                   ("coco/coco_test2017/test2017", n_test)):
        for i in range(n):
            _jpeg(os.path.join(ds, sub, f"{i:012d}.jpg"), rng, px)
    stim = os.path.join(ds, "BOLD5000/BOLD5000_Stimuli/Scene_Stimuli/Presented_Stimuli/COCO")
    sets = {}
    for name, n in (("train", n_bold_train), ("valid", n_bold_valid)):
        items = []
        for i in range(n):
            p = os.path.join(stim, f"{name}_{i:05d}.jpg")
            _jpeg(p, rng, px)
            v = rng.standard_normal(voxels).astype(np.float64)   # preprocessing.scale output is float64
            v[int(0.85 * voxels):] = 0.0
            items.append({"fmri": v, "image": p})
        sets[name] = items
    for rel, items in (("BOLD5000/bold_train/bold_train_all_fixed.pickle", sets["train"]),
                       ("BOLD5000/bold_valid/bold_valid_all_fixed.pickle", sets["valid"]),
                       ("BOLD5000/bold_train/bold_CSI4_pad.pickle", sets["train"])):
        p = os.path.join(ds, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        with open(p, "wb") as f:
            pickle.dump(items, f)
    # fixed stimulus split (data_config.py: train_stimuli_split / valid_stimuli_split): lists of image file names
    for rel, items in (("BOLD5000/bold_roi/stimuli_train.pickle", sets["train"]), ("BOLD5000/bold_roi/stimuli_valid.pickle", sets["valid"])):
        p = os.path.join(ds, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        with open(p, "wb") as f:
            pickle.dump([os.path.basename(it["image"]) for it in items], f)
    os.makedirs(os.path.join(root, "logs"), exist_ok=True)
    return root


def run_script(ref_root, script, root, extra_args=(), models_config=None, timeout=900, repo_models=True):
    """Run <ref_root>/<script> unchanged. models_config: 64 / 100 selects this repo's architecture preset for the child
    (the reference switches presets by editing configs/models_config.py). repo_models=False runs the reference's own models
    (CPU dry run of the harness itself). Returns (CompletedProcess, report dict or None)."""
    env = dict(os.environ)
    path = [STUBS] + ([REPO] if repo_models else []) + [ref_root]
    env["PYTHONPATH"] = os.pathsep.join(path)
    env["FMRI_HARNESS_REPORT"] = rep_path = os.path.join(root, "logs", "report_" + os.path.basename(script) + ".json")
    if models_config is not None:
        env["FMRI_MODELS_CONFIG"] = str(models_config)
    if os.path.exists(rep_path):
        os.remove(rep_path)
    cmd = [sys.executable, os.path.join(ref_root, script), "-i", root, "-o", root, "-l", os.path.join(root, "logs")] + \
        [str(a) for a in extra_args]
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=timeout)
    rep = None
    if os.path.exists(rep_path):
        with open(rep_path) as f:
            rep = json.load(f)
    return r, rep


_NUM = r"(-?(?:\d+\.\d+(?:e[-+]?\d+)?|nan|inf))"


def logged_losses(text):
    """All `<name> loss: <value>` / `<name>: <value>` numbers of the scripts' per-step logging lines, as floats."""
    vals = []
    for line in text.splitlines():
        if "loss" in line.lower() and ("Epoch" in line or "epoch" in line):
            vals += [float(v) for v in re.findall(r":\s*" + _NUM, line, flags=re.I)]
    return vals


def newest_checkpoint(root, folder):
    """(directory name, path of the newest *.pth) under <root>/results/<folder>/."""
    base = os.path.join(root, "results", folder)
    best = None
    for d in sorted(os.listdir(base)) if os.path.isdir(base) else []:
        for f in os.listdir(os.path.join(base, d)):
            if f.endswith(".pth"):
                p = os.path.join(base, d, f)
                if best is None or os.path.getmtime(p) >= os.path.getmtime(best[1]):
                    best = (d, p)
    return best


def install_checkpoint(src, root, folder, name, epoch):
    """Copy a checkpoint to the name a later stage's config expects: results/<folder>/<name>/<name>_<epoch>.pth."""
    dst = os.path.join(root, "results", folder, name, f"{name}_{epoch}.pth")
    os.makedirs(os.path.dirname(dst), exist_ok=True)
    shutil.copyfile(src, dst)
    return dst
