"""The native float64 fitting closure of the mean-covariance distances (Mahalanobis, squared Mahalanobis,
Bhattacharyya, Hellinger) on `.double()` SQFA models, against the float64 oracle: loss and gradient at the
benchmark shapes, edge shapes and tile-edge crossings, C = 1000, the composed path, determinism, graph replay,
pair ranges, fits, frozen filters, the not-positive-definite guard and the cases that keep the composed path."""

import pytest
import torch

from conftest import rel_err
from oracle import sqfa_oracle as O
from test_bures_wasserstein_gpu import gauss_stats

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-10  # relative, against the float64 oracle
GRAD_TOL = 1e-8   # relative Frobenius norm of d loss / d raw filters
NAMES = ["mahalanobis", "mahalanobis_sq", "bhattacharyya", "hellinger"]
SHAPES = {"c1": (10, 784, 4), "c2": (10, 3072, 8), "c3": (19, 104, 8), "c5": (100, 1024, 32)}
# the models store their noise through float32 (as the reference does), so the oracle takes that value
NOISE = float(torch.tensor(0.01, dtype=torch.float32))


def _filters(k, D, seed):
    """Initial filters as the model stores them (its constructor takes them through float32), in float64."""
    return torch.randn(k, D, generator=torch.Generator().manual_seed(seed)).double()


def _model(distance, D, k, F0, constraint="sphere", noise=0.01):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA

    fun = distance if callable(distance) else getattr(Dn, distance)
    return SQFA(n_dim=D, feature_noise=noise, n_filters=k, filters=F0.clone(), distance_fun=fun,
                constraint=constraint).double().cuda()


def _cuda(stats):
    return {"means": stats["means"].cuda(), "covariances": stats["covariances"].cuda()}


def _case(distance, C, D, k, seed=0, constraint="sphere"):
    stats = gauss_stats(C, D, seed=seed + C)
    F0 = _filters(k, D, seed + 3)
    return stats, F0, _model(distance, D, k, F0, constraint), _cuda(stats)


def _check(distance, C, D, k, seed=0, constraint="sphere"):
    stats, F0, model, sc = _case(distance, C, D, k, seed, constraint)
    loss64, grad64, _ = O.loss_and_grad("full", stats, F0, noise=NOISE, constraint=constraint,
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
@pytest.mark.parametrize("distance", NAMES)
def test_closure_matches_oracle_and_composed_path(distance, shape):
    C, D, k = SHAPES[shape]
    model, sc, direct, out, g = _check(distance, C, D, k)
    # the composed path on the same double model: get_class_distances -> -mean(tril) -> autograd
    model.parametrizations.filters.original.grad = None
    dmat = model.get_class_distances(sc, regularized=True)
    assert dmat.dtype == torch.float64
    i, j = torch.tril_indices(C, C, -1)
    loss = -dmat[i, j].mean()
    loss.backward()
    assert abs(float(loss.detach()) - out[0]) <= 1e-12 * abs(out[0])
    assert rel_err(model.parametrizations.filters.original.grad, g) <= 1e-10


@pytest.mark.parametrize("C,D,k", [(2, 16, 1), (7, 24, 1), (9, 40, 5), (13, 47, 7), (37, 64, 16), (21, 80, 32),
                                   (53, 40, 4)])
@pytest.mark.parametrize("distance", NAMES)
def test_edge_shapes(distance, C, D, k):
    """One pair, k = 1, odd k, odd D (the projection's scalar loads), k = 32, and class counts that are not
    multiples of the tile edge."""
    _check(distance, C, D, k, seed=11)


@pytest.mark.parametrize("C,D,k", [(183, 40, 32), (363, 40, 16), (363, 40, 32)])
@pytest.mark.parametrize("distance", ["mahalanobis", "hellinger"])
def test_tile_edge_crossings(distance, C, D, k):
    """Class counts just past the tile-edge thresholds: C = 183 at G = 32 (16 653 pairs, Q = 2, R = 2), C = 363
    at G = 16 (65 703 pairs, Q = 2, R = 4) and at G = 32 (Q = 4, R = 4; the largest pair-stage block)."""
    _check(distance, C, D, k, seed=13)


@pytest.mark.slow
@pytest.mark.parametrize("distance", NAMES)
def test_many_classes(distance):
    _check(distance, 1000, 64, 16, seed=1)


@pytest.mark.parametrize("distance", ["mahalanobis_sq", "bhattacharyya"])
def test_deterministic_graph_replay_and_pair_ranges(distance):
    from sqfa_b200 import _lib

    C, D, k = 45, 96, 8
    model, sc, direct, out, g = _check(distance, C, D, k, seed=5)
    # second evaluation: a graph capture; third: its replay
    for _ in range(2):
        assert direct().tolist() == out
        assert torch.equal(model.parametrizations.filters.original.grad, g)
    # two pair sub-ranges through the C entry add up to the whole
    lib = _lib.load()
    S, M, dist = model._fused_inputs(sc)
    W = model.parametrizations.filters.original.detach()
    P = C * (C - 1) // 2
    noise = torch.full((1,), NOISE, dtype=torch.float64, device="cuda")
    parts = []
    for p0, p1 in ((0, P // 3), (P // 3, P)):
        ws = torch.empty(lib.sqfa_gauss_closure_workspace_bytes_f64(C, D, k, dist, p0, p1), dtype=torch.uint8,
                         device="cuda")
        o = torch.zeros(3, dtype=torch.float64, device="cuda")
        gr = torch.zeros(k, D, dtype=torch.float64, device="cuda")
        _lib.check(lib.sqfa_gauss_closure_eval_f64(_lib.ptr(S), _lib.ptr(M), _lib.ptr(W), C, D, k, _lib.ptr(noise),
                                                   dist, 1, 0, p0, p1, _lib.ptr(o), None, _lib.ptr(gr), _lib.ptr(ws),
                                                   ws.numel(), _lib.stream_ptr()), "sqfa_gauss_closure_eval_f64")
        parts.append((o.clone(), gr.clone()))
    assert abs(float(parts[0][0][0] + parts[1][0][0]) - out[0]) <= 1e-13 * abs(out[0])
    assert rel_err(parts[0][1] + parts[1][1], g) <= 1e-13


@pytest.mark.parametrize("distance", ["mahalanobis", "hellinger"])
def test_fit_matches_oracle_and_is_deterministic(distance):
    C, D, k = 8, 40, 4
    stats = gauss_stats(C, D, seed=5)
    F0 = _filters(k, D, 9)
    _, losses_o, _ = O.fit_lbfgs("full", stats, F0, noise=NOISE, distance=getattr(O, distance), max_epochs=2,
                                 max_iter=5)
    filters = []
    for _ in range(2):
        model = _model(distance, D, k, F0)
        assert model._fused_direct_plan(_cuda(stats)) is not None
        losses, _ = model.fit(data_statistics=_cuda(stats), max_epochs=2, show_progress=False, return_loss=True,
                              max_iter=5)
        # the fitting loop returns its loss history as float32 on every path: 1e-7 is above that rounding
        assert torch.allclose(losses.double(), losses_o.double(), rtol=1e-7, atol=0)
        filters.append(model.filters.detach().clone())
    assert torch.equal(filters[0], filters[1])


def test_pairwise_fit_on_double_model(monkeypatch):
    """Every stage of the curriculum takes the native float64 closure, the later ones with FixedFilters."""
    from sqfa_b200.constraints import FixedFilters
    from sqfa_b200.model import SQFA

    taken = []
    plan = SQFA._fused_direct_plan

    def spy(self, data_statistics):
        direct = plan(self, data_statistics)
        taken.append((direct is not None, any(type(m) is FixedFilters for m in self.parametrizations.filters)))
        return direct

    monkeypatch.setattr(SQFA, "_fused_direct_plan", spy)
    C, D, k = 6, 32, 4
    stats = gauss_stats(C, D, seed=8)
    model = _model("bhattacharyya", D, k, _filters(k, D, 2))
    losses, _ = model.fit(data_statistics=_cuda(stats), max_epochs=3, pairwise=True, show_progress=False,
                          return_loss=True)
    assert len(taken) >= 2 and taken[0] == (True, False)
    assert all(t == (True, True) for t in taken[1:])
    assert torch.isfinite(losses).all()
    assert model.filters.dtype == torch.float64


def test_frozen_filters_match_oracle():
    """FixedFilters on the first two rows (a later stage of the pairwise curriculum): zero gradient rows there,
    the oracle's gradient on the others."""
    C, D, k = 9, 40, 6
    stats, F0, model, sc = _case("hellinger", C, D, k, seed=7)
    model._install_filters(model.filters.detach().clone(), n_frozen=2)
    raw = model.parametrizations.filters.original.detach().cpu()
    loss64, grad64, _ = O.loss_and_grad("full", stats, raw, noise=NOISE, distance=O.hellinger)
    direct = model._fused_direct_plan(sc)
    assert direct is not None
    out = direct().tolist()
    g = model.parametrizations.filters.original.grad.cpu()
    assert abs(out[0] - float(loss64)) <= LOSS_TOL * abs(float(loss64))
    assert torch.equal(g[:2], torch.zeros_like(g[:2]))
    assert rel_err(g[2:], grad64[2:]) <= GRAD_TOL
    assert out[2] == float(g.abs().max())


@pytest.mark.parametrize("distance", NAMES)
def test_not_positive_definite_raises_the_reference_message(distance):
    from sqfa_b200._optim import _INF_MSG, _NAN_MSG

    C, D, k = 5, 20, 3
    _, _, model, sc = _case(distance, C, D, k)
    # class 2 far from positive definite: the pair-mean covariances with it are negative definite too
    sc["covariances"][2] = -10 * sc["covariances"][2]
    assert model._fused_direct_plan(sc) is not None
    with pytest.raises(ValueError) as err:
        model.fit(data_statistics=sc, max_epochs=2, show_progress=False)
    assert str(err.value) in (_NAN_MSG, _INF_MSG)


@pytest.mark.parametrize("case", ["fisher_rao_same_cov", "lambda", "orthogonal", "float32_stats"])
def test_out_of_scope_cases_keep_the_composed_path(case):
    """These keep `_fused_direct_plan` None and, apart from fisher_rao_same_cov, still fit with finite losses."""
    from sqfa_b200 import distances as Dn

    C, D, k = 6, 32, 3
    stats = gauss_stats(C, D, seed=4)
    F0 = _filters(k, D, 6)
    distance = {"fisher_rao_same_cov": "fisher_rao_same_cov", "lambda": lambda a, b: Dn.hellinger(a, b)}.get(
        case, "hellinger")
    model = _model(distance, D, k, F0, constraint="orthogonal" if case == "orthogonal" else "sphere")
    sc = _cuda(stats)
    if case == "float32_stats":
        sc = {key: v.float() for key, v in sc.items()}
    assert model._fused_direct_plan(sc) is None
    assert model._fused_loss_plan(sc) is None
    if case == "fisher_rao_same_cov":
        return  # the reference's own closure gradient is NaN for it (DESIGN.md section 17), so it cannot fit
    losses, _ = model.fit(data_statistics=sc, max_epochs=2, show_progress=False, return_loss=True, max_iter=3)
    assert torch.isfinite(losses).all()
