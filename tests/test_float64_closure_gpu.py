"""The native float64 fitting closure (affine-invariant and Fisher-Rao lower bound, `.double()` models) against
the float64 oracle: loss and gradient at the benchmark shapes and edge shapes, C = 1000, determinism, graph
replay, pair ranges, fits, the not-positive-definite guard and the cases that keep the composed path."""

import pytest
import torch

from conftest import rel_err
from oracle import sqfa_oracle as O
from test_bures_wasserstein_gpu import gauss_stats

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-10  # relative, against the float64 oracle
GRAD_TOL = 1e-8   # relative Frobenius norm of d loss / d raw filters
SHAPES = {"c1": (10, 784, 4), "c2": (10, 3072, 8), "c3": (19, 104, 8), "c5": (100, 1024, 32)}
# the models store their noise through float32 (as the reference does), so the oracle takes that value
NOISE = float(torch.tensor(0.01, dtype=torch.float32))
CLOSURES = [("second_moments", "affine_invariant"), ("second_moments", "affine_invariant_sq"),
            ("full", "fisher_rao_lower_bound"), ("full", "fisher_rao_lower_bound_sq")]


def _filters(k, D, seed):
    """Initial filters as the model stores them (its constructor takes them through float32), in float64."""
    return torch.randn(k, D, generator=torch.Generator().manual_seed(seed)).double()


def _model(kind, distance, D, k, F0, constraint="sphere", noise=0.01):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA, SecondMomentsSQFA

    cls = SecondMomentsSQFA if kind == "second_moments" else SQFA
    return cls(n_dim=D, feature_noise=noise, n_filters=k, filters=F0.clone(), distance_fun=getattr(Dn, distance),
               constraint=constraint).double().cuda()


def _stats_for(kind, stats):
    if kind == "second_moments":
        return stats["second_moments"].cuda()
    return {"means": stats["means"].cuda(), "covariances": stats["covariances"].cuda()}


def _case(kind, distance, C, D, k, seed=0, constraint="sphere"):
    stats = gauss_stats(C, D, seed=seed + C)
    F0 = _filters(k, D, seed + 3)
    return stats, F0, _model(kind, distance, D, k, F0, constraint), _stats_for(kind, stats)


def _check(kind, distance, C, D, k, seed=0, constraint="sphere"):
    stats, F0, model, sc = _case(kind, distance, C, D, k, seed, constraint)
    ostats = stats["second_moments"] if kind == "second_moments" else stats
    loss64, grad64, _ = O.loss_and_grad(kind, ostats, F0, noise=NOISE, constraint=constraint,
                                        distance=getattr(O, distance))
    direct = model._fused_direct_plan(sc)
    assert direct is not None
    out = direct().tolist()
    g = model.parametrizations.filters.original.grad.clone()
    assert g.dtype == torch.float64
    assert out[1] == 0.0
    assert abs(out[0] - float(loss64)) <= LOSS_TOL * abs(float(loss64)), (out[0], float(loss64))
    assert rel_err(g.cpu(), grad64) <= GRAD_TOL, rel_err(g.cpu(), grad64)
    assert out[2] == float(g.abs().max())
    return model, sc, direct, out, g


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind,distance", CLOSURES)
def test_closure_matches_oracle(kind, distance, shape):
    C, D, k = SHAPES[shape]
    _check(kind, distance, C, D, k)


@pytest.mark.parametrize("C,D,k", [(2, 16, 1), (2, 24, 3), (9, 40, 5), (13, 47, 7), (37, 64, 16), (21, 80, 32),
                                   (35, 41, 2), (53, 40, 4), (183, 24, 3), (301, 25, 4)])
@pytest.mark.parametrize("kind,distance", [CLOSURES[0], CLOSURES[2]])
def test_edge_shapes(kind, distance, C, D, k):
    """One pair, k = 1, odd k, k = 32 with Fisher-Rao (m = 33), odd D (scalar loads), and tiles of more than one
    pair over class counts that are not multiples of the tile edge: the tile edge is 1 below 16 384 pairs, 2 from
    there (C = 183: 16 653 pairs, R = 2, last block row half past C) and 3 from 36 864 pairs (C = 301: 45 150
    pairs, R = 3, last block row one class wide)."""
    _check(kind, distance, C, D, k, seed=11)


def test_unaligned_statistics_take_the_scalar_loads():
    """S starting 8 bytes past a 16-byte boundary: same loss and gradient as an aligned copy (bit for bit: the
    two load paths add the same products in the same order)."""
    from sqfa_b200 import _lib, _ops

    C, D, k = 7, 48, 5
    stats, F0, model, sc = _case("full", "fisher_rao_lower_bound", C, D, k, seed=2)
    S = sc["covariances"]
    buf = torch.empty(S.numel() + 1, dtype=torch.float64, device="cuda")
    S_odd = buf[1:].view_as(S)
    S_odd.copy_(S)
    assert S_odd.data_ptr() % 16 == 8
    lib = _lib.load()
    P = C * (C - 1) // 2
    res = []
    for s in (S, S_odd):
        ws = torch.empty(lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, 1, 0, P), dtype=torch.uint8, device="cuda")
        out = torch.zeros(3, dtype=torch.float64, device="cuda")
        grad = torch.zeros(k, D, dtype=torch.float64, device="cuda")
        noise = torch.full((1,), NOISE, dtype=torch.float64, device="cuda")
        _ops.closure_eval_f64_raw(F0.cuda(), s, sc["means"], noise, 1, True, 0, out, grad, ws)
        res.append((out.clone(), grad.clone()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


@pytest.mark.slow
def test_many_classes():
    _check("full", "fisher_rao_lower_bound", 1000, 64, 16, seed=1)


@pytest.mark.parametrize("C,D,k", [(45, 96, 8), (301, 24, 3)])
def test_deterministic_graph_replay_and_pair_ranges(C, D, k):
    """C = 301: the whole list runs with 3 x 3 tiles, its first third (15 050 pairs) with single pairs and the
    rest (30 100 pairs) with 2 x 2 tiles from the middle of block row 86 on."""
    from sqfa_b200 import _lib

    model, sc, direct, out, g = _check("full", "fisher_rao_lower_bound", C, D, k, seed=5)
    # second evaluation: a graph capture; third: its replay
    for _ in range(2):
        out2 = direct().tolist()
        assert out2 == out
        assert torch.equal(model.parametrizations.filters.original.grad, g)
    # two pair halves add up to the whole
    lib = _lib.load()
    S, M, dist = model._fused_inputs(sc)
    W = model.parametrizations.filters.original.detach()
    P = C * (C - 1) // 2
    noise = torch.full((1,), NOISE, dtype=torch.float64, device="cuda")
    parts = []
    for p0, p1 in ((0, P // 3), (P // 3, P)):
        ws = torch.empty(lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, dist, p0, p1), dtype=torch.uint8,
                         device="cuda")
        o = torch.zeros(3, dtype=torch.float64, device="cuda")
        gr = torch.zeros(k, D, dtype=torch.float64, device="cuda")
        _lib.check(lib.sqfa_closure_eval_f64(_lib.ptr(S), _lib.ptr(M), _lib.ptr(W), C, D, k, _lib.ptr(noise), dist, 1, 0,
                                             p0, p1, _lib.ptr(o), None, _lib.ptr(gr), _lib.ptr(ws), ws.numel(),
                                             _lib.stream_ptr()), "sqfa_closure_eval_f64")
        parts.append((o.clone(), gr.clone()))
    assert abs(float(parts[0][0][0] + parts[1][0][0]) - out[0]) <= 1e-13 * abs(out[0])
    assert rel_err(parts[0][1] + parts[1][1], g) <= 1e-13


@pytest.mark.parametrize("kind,distance", [CLOSURES[0], CLOSURES[2]])
def test_fit_matches_oracle_and_is_deterministic(kind, distance):
    C, D, k = 8, 40, 4
    stats = gauss_stats(C, D, seed=5)
    ostats = stats["second_moments"] if kind == "second_moments" else stats
    F0 = _filters(k, D, 9)
    _, losses_o, _ = O.fit_lbfgs(kind, ostats, F0, noise=NOISE, distance=getattr(O, distance), max_epochs=2,
                                 max_iter=5)
    filters = []
    for _ in range(2):
        model = _model(kind, distance, D, k, F0)
        assert model._fused_direct_plan(_stats_for(kind, stats)) is not None
        losses, _ = model.fit(data_statistics=_stats_for(kind, stats), max_epochs=2, show_progress=False,
                              return_loss=True, max_iter=5)
        # the fitting loop returns its loss history as float32 on every path: 1e-7 is above that rounding
        assert torch.allclose(losses.double(), losses_o.double(), rtol=1e-7, atol=0)
        filters.append(model.filters.detach().clone())
    assert torch.equal(filters[0], filters[1])


def test_frozen_filters_match_oracle():
    """FixedFilters on the first two rows (a later stage of the pairwise curriculum): zero gradient rows there,
    the oracle's gradient on the others."""
    C, D, k = 9, 40, 6
    stats, F0, model, sc = _case("full", "fisher_rao_lower_bound", C, D, k, seed=7)
    model._install_filters(model.filters.detach().clone(), n_frozen=2)
    raw = model.parametrizations.filters.original.detach().cpu()
    loss64, grad64, _ = O.loss_and_grad("full", stats, raw, noise=NOISE, distance=O.fisher_rao_lower_bound)
    direct = model._fused_direct_plan(sc)
    assert direct is not None
    out = direct().tolist()
    g = model.parametrizations.filters.original.grad.cpu()
    assert abs(out[0] - float(loss64)) <= LOSS_TOL * abs(float(loss64))
    assert torch.equal(g[:2], torch.zeros_like(g[:2]))
    assert rel_err(g[2:], grad64[2:]) <= GRAD_TOL
    assert out[2] == float(g.abs().max())


def test_pairwise_fit_on_double_model(monkeypatch):
    """Every stage of the curriculum takes the native float64 closure, the later ones with FixedFilters."""
    from sqfa_b200.constraints import FixedFilters
    from sqfa_b200.model import SecondMomentsSQFA

    taken = []
    plan = SecondMomentsSQFA._fused_direct_plan

    def spy(self, data_statistics):
        direct = plan(self, data_statistics)
        taken.append((direct is not None, any(type(m) is FixedFilters for m in self.parametrizations.filters)))
        return direct

    monkeypatch.setattr(SecondMomentsSQFA, "_fused_direct_plan", spy)
    C, D, k = 6, 32, 4
    stats = gauss_stats(C, D, seed=8)
    model = _model("full", "fisher_rao_lower_bound", D, k, _filters(k, D, 2))
    losses, _ = model.fit(data_statistics=_stats_for("full", stats), max_epochs=3, pairwise=True,
                          show_progress=False, return_loss=True)
    assert taken == [(True, False), (True, True)]
    assert losses.numel() >= 2 and torch.isfinite(losses).all()
    assert model.filters.dtype == torch.float64


def test_not_positive_definite_raises_the_reference_message():
    C, D, k = 5, 24, 3
    stats = gauss_stats(C, D, seed=3)
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    F0[1] = 0.0
    model = _model("second_moments", "affine_invariant", D, k, F0, constraint="none", noise=0.0)
    sc = _stats_for("second_moments", stats)
    assert model._fused_direct_plan(sc) is not None
    with pytest.raises(ValueError, match="Some distances between classes are NaN"):
        model.fit(data_statistics=sc, max_epochs=2, show_progress=False)


@pytest.mark.parametrize("case", ["log_euclidean", "orthogonal", "float32_stats", "bures_wasserstein"])
def test_out_of_scope_cases_keep_the_composed_path(case):
    C, D, k = 6, 32, 3
    stats = gauss_stats(C, D, seed=4)
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(6), dtype=torch.float64)
    constraint = "orthogonal" if case == "orthogonal" else "sphere"
    distance = case if case in ("log_euclidean", "bures_wasserstein") else "affine_invariant"
    model = _model("second_moments", distance, D, k, F0, constraint=constraint)
    sc = _stats_for("second_moments", stats)
    if case == "float32_stats":
        sc = sc.float()
    assert model._fused_direct_plan(sc) is None
    assert model._fused_loss_plan(sc) is None
    losses, _ = model.fit(data_statistics=sc, max_epochs=2, show_progress=False, return_loss=True, max_iter=3)
    assert torch.isfinite(losses).all()
