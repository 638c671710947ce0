"""The closed form of the expected n-way identification accuracy (tests/identification_reference.py) against brute force:
for every reconstruction i and every (n-1)-subset of the other targets, a trial counts when X[i, i] beats every
distractor of the subset; the accuracy is the mean over all trials of all rows. Matrices with ties (a tie is not a
win), for N <= 8 and every n."""
import itertools
import math

import pytest
import torch

import identification_reference as R


def brute_force(X, n):
    N = X.shape[0]
    tot = 0.0
    for i in range(N):
        others = [j for j in range(N) if j != i]
        hits = sum(all(bool(X[i, i] > X[i, j]) for j in sub) for sub in itertools.combinations(others, n - 1))
        tot += hits / math.comb(N - 1, n - 1)
    return tot / N


@pytest.mark.parametrize("N", [2, 3, 5, 8])
@pytest.mark.parametrize("seed", [0, 1])
def test_closed_form_equals_enumeration(N, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randint(0, 4, (N, N), generator=g).double()     # 4 levels: many ties, on and off the diagonal
    ns = list(range(2, N + 1))
    wins, acc = R.identification(X, ns)
    for i in range(N):
        assert int(wins[i]) == sum(1 for j in range(N) if j != i and X[i, i] > X[i, j])
    for q, n in enumerate(ns):
        assert abs(float(acc[q]) - brute_force(X, n)) < 1e-12, (N, n)


def test_closed_form_nan_and_extremes():
    X = torch.tensor([[1.0, 0.0, 0.0], [0.5, float("nan"), 0.0], [0.0, float("nan"), 2.0]])
    wins, acc = R.identification(X, [2, 3])
    assert wins.tolist() == [2, 0, 1]                # a NaN diagonal never wins; a NaN distractor is never beaten
    for q, n in enumerate([2, 3]):
        assert abs(float(acc[q]) - brute_force(X, n)) < 1e-12
    eye = torch.eye(6)
    assert R.identification(eye, range(2, 7))[1].tolist() == [1.0] * 5
    assert R.identification(-eye, range(2, 7))[1].tolist() == [0.0] * 5
