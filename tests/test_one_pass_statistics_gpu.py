"""class_statistics on one device in one pass over X: the Gram centres on a pilot shift (the first 32 rows
of each class) and writes the class sums on the way; the epilogue corrects by n d d^T. Checked class by class
against the float64 oracle, for the load paths, tile shapes, K splits and class-size edges of that pass."""

import pytest
import torch

from conftest import make_class_data, rel_err
from oracle import sqfa_oracle as O

pytestmark = pytest.mark.gpu

TOL_MEAN = 1e-6
TOL_COV = 1e-5


def _check(got, ref):
    for key, tol in (("means", TOL_MEAN), ("covariances", TOL_COV), ("second_moments", TOL_COV)):
        g, r = got[key].cpu(), ref[key]
        assert torch.equal(torch.isnan(g), torch.isnan(r)), key
        for c in range(r.shape[0]):
            ok = ~torch.isnan(r[c])
            if ok.any() and r[c][ok].norm() > 0:
                assert rel_err(g[c][ok], r[c][ok]) < tol, (key, c, rel_err(g[c][ok], r[c][ok]))
            else:
                assert torch.equal(g[c][ok], r[c][ok]), (key, c)


@pytest.mark.parametrize(
    "n,d,c,kw",
    [
        (3000, 4, 5, {}),
        (5000, 104, 7, {}),            # D <= 128: single-CTA Gram
        (6000, 784, 4, {}),            # ragged last tile
        (3000, 1027, 3, {}),           # D % 4 != 0: element loads, scalar sum slots
        (12000, 3072, 3, {}),
        (20000, 256, 3, {}),           # K split (test_gram_long_chains_and_k_split's shapes)
        (9000, 520, 7, {"skew": True}),
        (700, 2048, 2, {}),
        (4000, 300, 5, {"offset": 1e3}),  # uncentred data
    ],
)
def test_matches_float64_oracle(n, d, c, kw):
    from sqfa_b200.statistics import class_statistics

    X, y = make_class_data(n, d, c, seed=n + d, **kw)
    got = class_statistics(X.cuda(), y.cuda())
    _check(got, O.class_statistics(X.double(), y))


def _edge_labels(n, seed):
    """Class sizes 1500, 400, 31, 5, 1, 0, 33, rest: classes shorter than the pilot, a singleton, an empty one."""
    sizes = [1500, 400, 31, 5, 1, 0, 33]
    y = torch.cat([torch.full((s,), k, dtype=torch.int64) for k, s in enumerate(sizes)]
                  + [torch.full((n - sum(sizes),), len(sizes), dtype=torch.int64)])
    return y[torch.randperm(n, generator=torch.Generator().manual_seed(seed))]


@pytest.mark.parametrize("est", ["empirical", "oas"])
@pytest.mark.parametrize("d", [64, 520])
def test_small_singleton_and_empty_classes(d, est):
    from sqfa_b200.statistics import class_statistics

    n = 3000
    X, _ = make_class_data(n, d, 8, seed=d)
    y = _edge_labels(n, d)
    got = class_statistics(X.cuda(), y.cuda(), estimator=est)
    _check(got, O.class_statistics(X.double(), y, estimator=est))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("n,d,c", [(6000, 784, 4), (3000, 104, 9), (3000, 1027, 3)])
def test_half_inputs(n, d, c, dtype):
    from sqfa_b200.statistics import class_statistics

    X, y = make_class_data(n, d, c, seed=d, dtype=dtype)
    got = class_statistics(X.cuda(), y.cuda())
    _check(got, O.class_statistics(X.double(), y))
    ref32 = class_statistics(X.float().cuda(), y.cuda())
    for key in ("means", "covariances", "second_moments"):
        assert torch.equal(got[key], ref32[key]), key


@pytest.mark.parametrize("n,d,c", [(9000, 520, 7), (6000, 1027, 5), (5000, 104, 8)])
def test_reproducible_and_stepwise_equal(n, d, c):
    """Two calls give the same bits, and the step-by-step entry points give the single call's bits."""
    from sqfa_b200._stats_driver import CudaStatsOps, run_class_statistics

    X, y = make_class_data(n, d, c, seed=3 * d)
    y[5::11] = -1
    X, y = X.cuda(), y.cuda()
    ops = CudaStatsOps()
    a = run_class_statistics(ops, X, y, 0)
    b = run_class_statistics(ops, X, y, 0)
    ops.gram_events = []  # instrumented -> step by step
    s = run_class_statistics(ops, X, y, 0)
    ops.gram_events = None
    for i in range(3):
        assert torch.equal(a[i], b[i]) and torch.equal(a[i], s[i]), i


def test_pilot_shift_entry_point():
    """The pilot shift is the mean of each class's first min(n_c, 32) rows in bucket order, 0 when empty."""
    from sqfa_b200._stats_driver import CudaStatsOps

    X, _ = make_class_data(2000, 130, 8, seed=9)
    y = _edge_labels(2000, 9)
    ops = CudaStatsOps()
    perm, offsets, counts = ops.bucket(y.cuda(), 8)
    shift = ops.pilot_shift(X.cuda(), perm, offsets, 8).cpu()
    perm, offsets = perm.cpu().long(), offsets.cpu()
    for k in range(8):
        rows = perm[offsets[k]:offsets[k + 1]][:32]
        want = X[rows].double().mean(0) if rows.numel() else torch.zeros(130, dtype=torch.float64)
        assert torch.allclose(shift[k].double(), want, rtol=1e-6, atol=1e-6), k
