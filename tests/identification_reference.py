"""CPU statement of the all-pairs similarity matrices and of the expected n-way identification accuracy (the exhaustive
form of objective_assessment, train/train_utils.py:752), built on the per-pair metrics of oracle/metrics.py that the
golden fixtures pin. TEST INFRASTRUCTURE ONLY.
"""
import math
from fractions import Fraction

import torch

from oracle import metrics as M


def pairwise(pred, target, metric):
    """[N, M] matrix of metric(pred[i:i+1], target[j:j+1]): pearson in fp64, ssim in fp32 (as the golden test uses them)."""
    N, Mt = pred.shape[0], target.shape[0]
    out = torch.empty(N, Mt, dtype=torch.float64)
    for i in range(N):
        for j in range(Mt):
            if metric == "pcc":
                out[i, j] = M.pearson(pred[i:i + 1].double(), target[j:j + 1].double())
            elif metric == "ssim":
                out[i, j] = M.ssim(pred[i:i + 1].float(), target[j:j + 1].float()).double()
            else:
                raise ValueError(f"unknown metric {metric!r}")
    return out


def identification(X, ns):
    """(wins [N] int64, acc [len(ns)] float64) of a square matrix X: wins[i] = #{j != i : X[i, i] > X[i, j]} (a NaN never
    wins) and acc[n] = (1/N) sum_i C(wins[i], n-1) / C(N-1, n-1), summed as exact rationals and rounded once."""
    X = torch.as_tensor(X).double()
    N = X.shape[0]
    beats = X.diagonal().unsqueeze(1) > X                    # comparisons with a NaN are False
    beats.fill_diagonal_(False)
    wins = beats.sum(1)
    acc = []
    for n in ns:
        tot = sum(Fraction(math.comb(int(w), n - 1), math.comb(N - 1, n - 1)) for w in wins)
        acc.append(float(tot / N))
    return wins, torch.tensor(acc, dtype=torch.float64)
