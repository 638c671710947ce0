"""All-pairs PCC / SSIM matrices and n-way identification on the GPU (inference.similarity_matrix / identification,
fmri_pairwise_similarity / fmri_identification):
  * every matrix entry against identification_reference.pairwise (a loop over the per-pair metrics of oracle/metrics.py,
    which the golden fixtures pin), 1e-5 absolute, at the four golden metric shapes with N != M, and a few entries
    against the single-pair kernels fmri_pearson / fmri_ssim;
  * N = M = 1000 at 3 x 64 x 64 (ragged against every tile): 256 seeded entries per metric, two calls bit-identical;
  * wins / acc against the closed form of identification_reference on a GPU matrix and on crafted ones (ties, NaN,
    perfect, worst);
  * end to end from Reconstructor(kind="cognitive") over a batch of 64;
  * every argument error raises FmriError before any launch.
"""
import numpy as np
import pytest
import torch

from oracle import metrics as M
from oracle import vaegan as O
from oracle.make_golden_metrics import CASES, inputs
from thesis_fmri_reconstruction_b200 import hp, inference
from thesis_fmri_reconstruction_b200 import lib as L

import identification_reference as R

pytestmark = pytest.mark.gpu
SHAPES = {"64": (20, 17), "100": (6, 5), "ragged": (7, 9), "grey": (8, 8)}


def pair_sets(case):
    _, Cc, H, W, seed = CASES[case]
    N, Mt = SHAPES[case]
    a, b = inputs(max(N, Mt), Cc, H, W, seed)      # b: a perturbed copy of a, so pair (i, i) is the similar one
    return a[:N].contiguous(), b[:Mt].contiguous()


@pytest.mark.parametrize("metric", ["pcc", "ssim"])
@pytest.mark.parametrize("case", list(SHAPES))
def test_matrix_matches_oracle(case, metric):
    pred, target = pair_sets(case)
    got = inference.similarity_matrix(pred.cuda(), target.cuda(), metric=metric)
    assert got.dtype == torch.float32 and tuple(got.shape) == (pred.shape[0], target.shape[0])
    ref = R.pairwise(pred, target, metric)
    err = (got.cpu().double() - ref).abs().max().item()
    print(case, metric, tuple(pred.shape), target.shape[0], "max |err|", err)
    assert err < 1e-5


def test_matrix_matches_single_pair_kernels():
    pred, target = pair_sets("64")
    P = inference.similarity_matrix(pred, target, metric="pcc").cpu()     # host tensors are moved like inference.pcc
    S = inference.similarity_matrix(pred, target, metric="ssim").cpu()
    for i, j in [(0, 0), (3, 11), (19, 16), (7, 7), (12, 2)]:
        p = float(inference.pcc(pred[i:i + 1].cuda(), target[j:j + 1].cuda()))
        s = float(inference.ssim(pred[i:i + 1].cuda(), target[j:j + 1].cuda()))
        assert abs(float(P[i, j]) - p) < 1e-5 and abs(float(S[i, j]) - s) < 1e-5, (i, j)


def test_large_ragged_sets_sampled_and_deterministic():
    N, Cc, H, W = 1000, 3, 64, 64
    g = torch.Generator().manual_seed(2026)
    pred = torch.rand(N, Cc, H, W, generator=g) * 2 - 1
    target = (pred + 0.5 * torch.randn(N, Cc, H, W, generator=g)).clamp(-1, 1)
    idx = torch.randint(0, N, (256, 2), generator=g)
    pc, tc = pred.cuda(), target.cuda()
    for metric in ("pcc", "ssim"):
        X1 = inference.similarity_matrix(pc, tc, metric=metric)
        X2 = inference.similarity_matrix(pc, tc, metric=metric)
        assert torch.equal(X1, X2), metric
        X = X1.cpu()
        err = 0.0
        for i, j in idx.tolist():
            if metric == "pcc":
                r = float(M.pearson(pred[i:i + 1].double(), target[j:j + 1].double()))
            else:
                r = float(M.ssim(pred[i:i + 1], target[j:j + 1]))
            err = max(err, abs(float(X[i, j]) - r))
        print(metric, "N = M = 1000 sampled max |err|", err)
        assert err < 1e-5


def check_identification(X, ns):
    wins, acc = inference.identification(X.cuda(), ns)
    assert wins.dtype == torch.int32 and acc.dtype == torch.float64 and wins.is_cuda and acc.is_cuda
    rw, ra = R.identification(X.cpu(), ns)
    assert wins.cpu().tolist() == rw.tolist()
    assert (acc.cpu() - ra).abs().max().item() < 1e-12, (acc.cpu(), ra)
    return acc.cpu()


def test_identification_on_gpu_matrix():
    _, Cc, H, W, seed = CASES["64"]
    a, b = inputs(16, Cc, H, W, seed)
    for metric in ("pcc", "ssim"):
        X = inference.similarity_matrix(a.cuda(), b.cuda(), metric=metric).cpu()
        check_identification(X, (2, 5, 10, 16))


def test_identification_crafted_matrices():
    g = torch.Generator().manual_seed(7)
    N = 12
    ns = list(range(2, N + 1))
    ties = torch.randint(0, 3, (N, N), generator=g).float()
    check_identification(ties, ns)
    nans = torch.rand(N, N, generator=g)
    nans[torch.rand(N, N, generator=g) < 0.2] = float("nan")
    nans[3, 3] = nans[8, 8] = float("nan")
    check_identification(nans, ns)
    diag_nan = torch.rand(N, N, generator=g)
    diag_nan.fill_diagonal_(float("nan"))
    assert check_identification(diag_nan, ns).tolist() == [0.0] * len(ns)
    perfect = torch.rand(N, N, generator=g)
    perfect.fill_diagonal_(2.0)
    assert check_identification(perfect, ns).tolist() == [1.0] * len(ns)
    worst = torch.rand(N, N, generator=g)
    worst.fill_diagonal_(-1.0)
    assert check_identification(worst, ns).tolist() == [0.0] * len(ns)
    big = torch.rand(1500, 1500, generator=g)
    big += 0.3 * torch.eye(1500)
    check_identification(big, (2, 5, 10, 100, 1500))


def test_end_to_end_cognitive_reconstructions():
    B, seed = 64, 91
    P, S = O.make_cognitive(O.CFG64, seed=seed)
    fmri = O.synthetic_fmri(B, seed=seed)
    r = inference.Reconstructor({**P, **S}, hp.CFG64, z=128, kind="cognitive", adt=torch.float32)
    recon = r(fmri.cuda(), sample=False)
    flat = recon.flatten(1).double()
    rms = torch.cdist(flat, flat) / flat.shape[1] ** 0.5
    rms.fill_diagonal_(float("inf"))
    scale = 0.01 * rms.min().item()
    noise = torch.randn(recon.shape, generator=torch.Generator().manual_seed(seed)).cuda()
    targets = recon + scale * noise
    print("smallest pairwise RMS difference", rms.min().item())
    for metric in ("ssim", "pcc"):
        X = inference.similarity_matrix(recon, targets, metric=metric)
        wins, acc = inference.identification(X, ns=(2, 5, 10, 64))
        assert acc.cpu().tolist() == [1.0] * 4, (metric, acc)
        rw, ra = R.identification(X.cpu(), (2, 5, 10, 64))
        assert wins.cpu().tolist() == rw.tolist() and (acc.cpu() - ra).abs().max().item() < 1e-12


def no_launch(fn):
    L.launch_count(reset=True)
    with pytest.raises(L.FmriError):
        fn()
    assert L.launch_count() == 0


def test_errors_before_any_device_work():
    a = torch.rand(4, 3, 16, 16, device="cuda")
    small = torch.rand(4, 3, 9, 16, device="cuda")
    no_launch(lambda: inference.similarity_matrix(small, small, metric="ssim"))
    no_launch(lambda: inference.similarity_matrix(a, torch.rand(4, 1, 16, 16, device="cuda")))
    no_launch(lambda: inference.similarity_matrix(a, torch.rand(4, 3, 16, 15, device="cuda"), metric="pcc"))
    no_launch(lambda: inference.similarity_matrix(a, a, metric="mse"))
    sq = torch.rand(6, 6, device="cuda")
    no_launch(lambda: inference.identification(torch.rand(6, 5, device="cuda")))
    no_launch(lambda: inference.identification(sq, ns=(1,)))
    no_launch(lambda: inference.identification(sq, ns=(2, 7)))
    # the library's own checks, through the bindings
    out = torch.empty(4, 4, device="cuda")
    for metric in (L.METRIC_PCC, L.METRIC_SSIM):
        need = L.pairwise_workspace(4, 4, 3, 16, 16, metric)
        assert need > 0
        ws = torch.empty(need - 1, dtype=torch.uint8, device="cuda")
        no_launch(lambda: L.pairwise_similarity(a, a, metric, out, ws))
        no_launch(lambda: L.pairwise_similarity(a.cpu(), a.cpu(), metric, out.cpu(), ws.cpu()))
    ws = torch.empty(L.pairwise_workspace(4, 4, 3, 9, 16, L.METRIC_SSIM), dtype=torch.uint8, device="cuda")
    no_launch(lambda: L.pairwise_similarity(small, small, L.METRIC_SSIM, out, ws))
    wins, acc = torch.empty(6, dtype=torch.int32, device="cuda"), torch.empty(2, dtype=torch.float64, device="cuda")
    no_launch(lambda: L.identification(sq, [2, 7], wins, acc))
    no_launch(lambda: L.identification(sq, [1, 3], wins, acc))
    no_launch(lambda: L.identification(sq[:1, :1], [2], wins, acc))
    no_launch(lambda: L.identification(sq.cpu(), [2, 3], wins.cpu(), acc.cpu()))
    assert np.isfinite(inference.similarity_matrix(a, a, metric="pcc").cpu().numpy()).all()
