"""Bures-Wasserstein (SPD) and 2-Wasserstein (Gaussian) distances on the device: values, gradients and the
composed path against float64 references, and the fused fitting closures of both models against the
oracle, including the sharded closure phases, determinism and the error paths of the C ABI."""

import ctypes

import pytest
import torch

from conftest import rel_err
from oracle import sqfa_oracle as O
from test_hp2_gpu import _bw_distance_sq

pytestmark = pytest.mark.gpu

GRAD_TOL = 2e-3  # gradient of the loss w.r.t. the raw filters, relative Frobenius vs fp64 oracle
LOSS_TOL = 1e-4


def sample_spd(n, m, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    ev = 2 * torch.rand(n, m, generator=g, dtype=dtype) ** 2 + 0.01
    low = torch.tril(torch.randn(n, m, m, generator=g, dtype=dtype), diagonal=-1)
    Q = torch.matrix_exp(low - low.transpose(1, 2))
    return torch.einsum("ijk,ik,ilk->ijl", Q, ev, Q)


def _sqrtm64(B):
    lam, V = torch.linalg.eigh(B)
    return torch.einsum("...ij,...j,...kj->...ik", V, torch.sqrt(lam), V)


def bw_sq64(A, B):
    """float64 reference, (n_A, n_B): tr A + tr B - 2 tr((B^1/2 A B^1/2)^1/2), clamped at 0."""
    A, B = O_batch(A), O_batch(B)
    R = _sqrtm64(B)
    inner = torch.linalg.eigvalsh(R[None] @ A[:, None] @ R[None]).clamp_min(0)
    tr_a = torch.diagonal(A, dim1=-2, dim2=-1).sum(-1)
    tr_b = torch.diagonal(B, dim1=-2, dim2=-1).sum(-1)
    return (tr_a[:, None] + tr_b[None] - 2 * torch.sqrt(inner).sum(-1)).clamp_min(0)


def O_batch(A):
    return A.unsqueeze(0) if A.dim() == 2 else A


def bw64(A, B):
    return torch.sqrt(bw_sq64(A, B) + 1e-6)


def w2_sq64(sa, sb):
    diff = sa["means"][:, None] - sb["means"][None]
    return (diff * diff).sum(-1) + bw_sq64(sa["covariances"], sb["covariances"])


def w264(sa, sb):
    return torch.sqrt(w2_sq64(sa, sb).clamp_min(0) + 1e-6)


REF64 = {"bures_wasserstein_sq": bw_sq64, "bures_wasserstein": bw64, "wasserstein_sq": w2_sq64,
         "wasserstein": w264}


def check_values(got, ref, trA, trB, abs_tol=1e-5):
    scale = (trA[:, None] + trB[None]).double()
    got, ref = got.double().cpu(), ref.double().cpu()
    err = (got - ref).abs()
    assert (err <= abs_tol * scale).all(), float((err / scale).max())
    big = ref >= 1e-2 * scale
    assert (err[big] <= 1e-4 * ref[big]).all(), float((err[big] / ref[big]).max())


# ------------------------------------------------------------------------------------------------
# distances
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [2, 4, 9, 17, 32, 33, 34])
def test_values_match_float64(m):
    from sqfa_b200 import distances as Dn
    from sqfa_b200 import linalg as Ln

    A = sample_spd(13, m, seed=m)
    B = sample_spd(6, m, seed=m + 50)
    trA, trB = torch.einsum("ijj->i", A), torch.einsum("ijj->i", B)
    Ac, Bc = A.float().cuda(), B.float().cuda()
    # A != B, unequal batch sizes
    got = Dn.bures_wasserstein_sq(Ac, Bc)
    assert got.shape == (13, 6) and got.dtype == torch.float32
    check_values(got, bw_sq64(A, B), trA, trB)
    # A is B: exact diagonal, symmetric
    same = Dn.bures_wasserstein_sq(Ac, Ac)
    check_values(same, bw_sq64(A, A).fill_diagonal_(0), trA, trA)
    assert torch.equal(torch.diagonal(same), torch.zeros(13, device="cuda"))
    assert torch.equal(same, same.T)
    d = Dn.bures_wasserstein(Ac, Ac)
    assert torch.equal(torch.diagonal(d), torch.full((13,), 1e-6, device="cuda").sqrt())
    assert torch.allclose(d, torch.sqrt(same + 1e-6))
    # the tutorial's composition with sqfa_b200.linalg, indexed [b, a]: its float32 eigvalsh of the
    # conjugated matrices leaves up to ~1e-5 (tr A + tr B) (1.03e-5 measured at m = 32), hence 2e-5
    tut = _bw_distance_sq(Ac, Bc, Ln).T
    check_values(tut.clamp_min(0), bw_sq64(A, B), trA, trB, abs_tol=2e-5)
    check_values(got, tut.clamp_min(0), trA, trB, abs_tol=2e-5)
    # squeezing like affine_invariant
    assert Dn.bures_wasserstein_sq(Ac[0], Bc[0]).shape == torch.Size([])


@pytest.mark.parametrize("m", [3, 9, 17, 32])
def test_distance_gradients_match_float64(m):
    from sqfa_b200 import distances as Dn

    A = sample_spd(7, m, seed=10 + m)
    B = sample_spd(5, m, seed=20 + m)
    Wt = torch.randn(7, 5, generator=torch.Generator().manual_seed(m), dtype=torch.float64)
    for name in ("bures_wasserstein_sq", "bures_wasserstein"):
        A64, B64 = A.clone().requires_grad_(True), B.clone().requires_grad_(True)
        (REF64[name](A64, B64) * Wt).sum().backward()
        Ac, Bc = A.float().cuda().requires_grad_(True), B.float().cuda().requires_grad_(True)
        (getattr(Dn, name)(Ac, Bc) * Wt.float().cuda()).sum().backward()
        sym = lambda g: 0.5 * (g + g.transpose(-2, -1))  # noqa: E731
        assert rel_err(sym(Ac.grad), sym(A64.grad)) <= 1e-4
        assert rel_err(sym(Bc.grad), sym(B64.grad)) <= 1e-4
    # Gaussian form: means and covariances
    g = torch.Generator().manual_seed(m)
    sa = {"means": torch.randn(7, m, generator=g, dtype=torch.float64), "covariances": A}
    sb = {"means": torch.randn(5, m, generator=g, dtype=torch.float64), "covariances": B}
    for name in ("wasserstein_sq", "wasserstein"):
        s64 = [{k: v.clone().requires_grad_(True) for k, v in s.items()} for s in (sa, sb)]
        (REF64[name](*s64) * Wt).sum().backward()
        s32 = [{k: v.float().cuda().requires_grad_(True) for k, v in s.items()} for s in (sa, sb)]
        out = getattr(Dn, name)(*s32)
        check_values(out if name == "wasserstein_sq" else out**2 - 1e-6, w2_sq64(sa, sb),
                     torch.einsum("ijj->i", A), torch.einsum("ijj->i", B))
        (out * Wt.float().cuda()).sum().backward()
        for a, b in zip(s32, s64):
            assert rel_err(a["means"].grad, b["means"].grad) <= 1e-4
            sym = lambda g: 0.5 * (g + g.transpose(-2, -1))  # noqa: E731
            assert rel_err(sym(a["covariances"].grad), sym(b["covariances"].grad)) <= 1e-4


def test_large_and_double_inputs_take_the_composed_path(monkeypatch):
    from sqfa_b200 import _ops, distances as Dn

    calls = []
    orig = _ops.PairDistance.apply
    monkeypatch.setattr(_ops.PairDistance, "apply", lambda *a: calls.append(a) or orig(*a))
    A = sample_spd(4, 40, seed=1)
    B = sample_spd(3, 40, seed=2)
    got = Dn.bures_wasserstein_sq(A.float().cuda(), B.float().cuda())
    assert got.dtype == torch.float32
    # float32 eigendecompositions: 1.1e-5 (tr A + tr B) measured, against < 1e-5 for the pair kernel
    check_values(got, bw_sq64(A, B), torch.einsum("ijj->i", A), torch.einsum("ijj->i", B), abs_tol=5e-5)
    A, B = sample_spd(5, 9, seed=3), sample_spd(4, 9, seed=4)
    A64 = A.cuda().requires_grad_(True)
    got = Dn.bures_wasserstein(A64, B.cuda())
    assert got.dtype == torch.float64
    assert (got.cpu() - bw64(A, B)).abs().max() <= 1e-12
    got.sum().backward()
    assert torch.isfinite(A64.grad).all()
    assert calls == []  # neither went through the pair kernel


# ------------------------------------------------------------------------------------------------
# fitting closures
# ------------------------------------------------------------------------------------------------
def gauss_stats(C, D, seed, rank=48):
    """Class means and low-rank-plus-diagonal covariances (float64), cheap at D = 3072."""
    g = torch.Generator().manual_seed(seed)
    G = torch.randn(C, D, rank, generator=g, dtype=torch.float64) / rank**0.5
    scale = 0.5 + 1.5 * torch.rand(C, 1, 1, generator=g, dtype=torch.float64)
    cov = scale * (G @ G.transpose(1, 2)) + 0.05 * torch.eye(D, dtype=torch.float64)
    means = 0.3 * torch.randn(C, D, generator=g, dtype=torch.float64) / D**0.5 * 4
    return {"means": means, "covariances": cov, "second_moments": cov + means[:, :, None] * means[:, None, :]}


SHAPES = {"c1": (10, 784, 4), "c2": (10, 3072, 8), "c3": (19, 104, 8), "c5": (100, 1024, 32)}
CLOSURES = [("second_moments", "bures_wasserstein"), ("second_moments", "bures_wasserstein_sq"),
            ("full", "wasserstein"), ("full", "wasserstein_sq")]


def _model(kind, distance, D, k, F0):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA, SecondMomentsSQFA

    cls = SecondMomentsSQFA if kind == "second_moments" else SQFA
    return cls(n_dim=D, feature_noise=0.01, n_filters=k, filters=F0.clone(), distance_fun=getattr(Dn, distance))


def _closure_case(kind, distance, C, D, k, seed=0):
    stats = gauss_stats(C, D, seed=seed + C)
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(seed + 3))
    model = _model(kind, distance, D, k, F0).cuda()
    sc = {kk: v.float().cuda() for kk, v in stats.items()}
    if kind == "full":
        sc = {"means": sc["means"], "covariances": sc["covariances"]}
    return stats, F0, model, sc


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind,distance", CLOSURES)
def test_fused_closure_matches_oracle(kind, distance, shape):
    C, D, k = SHAPES[shape]
    stats, F0, model, sc = _closure_case(kind, distance, C, D, k)
    loss64, grad64, _ = O.loss_and_grad(kind, stats, F0.double(), noise=0.01, distance=REF64[distance])
    direct = model._fused_direct_plan(sc)
    assert direct is not None
    out = direct().tolist()
    g = model.parametrizations.filters.original.grad.clone()
    assert out[1] == 0.0
    assert abs(out[0] - float(loss64)) <= LOSS_TOL * abs(float(loss64))
    assert rel_err(g, grad64) < GRAD_TOL
    # bit-identical on a second evaluation
    out2 = direct().tolist()
    assert out2[0] == out[0]
    assert torch.equal(model.parametrizations.filters.original.grad, g)
    # the autograd path through get_class_distances and the native distances agrees to 1e-5
    model.parametrizations.filters.original.grad = None
    dmat = model.get_class_distances(sc, regularized=True)
    i, j = torch.tril_indices(C, C, -1)
    loss = -dmat[i, j].mean()
    loss.backward()
    assert abs(float(loss.detach()) - out[0]) <= 1e-5 * abs(out[0])
    assert rel_err(model.parametrizations.filters.original.grad, g.double()) <= 1e-5


@pytest.mark.slow
@pytest.mark.parametrize("kind,distance", [("second_moments", "bures_wasserstein"), ("full", "wasserstein")])
def test_fused_closure_many_classes(kind, distance):
    C, D, k = 1000, 64, 16
    stats, F0, model, sc = _closure_case(kind, distance, C, D, k, seed=1)
    loss64, grad64, _ = O.loss_and_grad(kind, stats, F0.double(), noise=0.01, distance=REF64[distance])
    direct = model._fused_direct_plan(sc)
    out = direct().tolist()
    assert out[1] == 0.0
    assert abs(out[0] - float(loss64)) <= LOSS_TOL * abs(float(loss64))
    assert rel_err(model.parametrizations.filters.original.grad, grad64) < GRAD_TOL


@pytest.mark.parametrize("kind,distance", [("second_moments", "bures_wasserstein"), ("full", "wasserstein")])
def test_fit_matches_oracle_and_is_deterministic(kind, distance):
    C, D, k = 8, 40, 4
    stats = gauss_stats(C, D, seed=5)
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(9))
    _, losses_o, _ = O.fit_lbfgs(kind, stats, F0.double(), noise=0.01, distance=REF64[distance], max_epochs=2,
                                 max_iter=5)
    s32 = {kk: v.float() for kk, v in stats.items()}
    if kind == "full":
        s32 = {"means": s32["means"], "covariances": s32["covariances"]}
    filters = []
    for _ in range(2):
        model = _model(kind, distance, D, k, F0)
        losses, _ = model.fit(data_statistics=s32, max_epochs=2, show_progress=False, return_loss=True, max_iter=5)
        assert torch.allclose(losses.double(), losses_o.double(), rtol=1e-3)
        filters.append(model.filters.detach().clone())
    assert torch.equal(filters[0], filters[1])


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("kind,distance", [("second_moments", "bures_wasserstein"), ("full", "wasserstein_sq")])
def test_sharded_closure_phases_on_one_device(kind, distance, world):
    """sqfa_fused_loss_sharded with `world` emulated ranks on one device equals sqfa_fused_loss."""
    from sqfa_b200 import _lib, _ops
    from sqfa_b200._stats_driver import class_share

    lib = _lib.load()
    C, D, k = 23, 96, 6
    _, _, model, sc = _closure_case(kind, distance, C, D, k, seed=7)
    F = model.filters.detach().contiguous()
    S, M, dist = model._fused_inputs(sc)
    noise = model._noise_scalar()
    ref = _ops.fused_loss_raw(F, S, M, noise, dist)
    P = C * (C - 1) // 2
    ranks = []
    for r in range(world):
        p0, p1 = _ops.shard_pairs(P, C, r, world)
        c0, c1 = class_share(C, r, world)
        ws = torch.empty(lib.sqfa_fused_loss_workspace_bytes(C, D, k, dist, p0, p1), dtype=torch.uint8, device="cuda")
        spans = []
        for which in (0, 1):
            off, nb = ctypes.c_size_t(0), ctypes.c_size_t(0)
            _lib.check(lib.sqfa_fused_loss_exchange_span(C, D, k, dist, p0, p1, which, ctypes.byref(off),
                                                         ctypes.byref(nb)), "span")
            spans.append(ws[off.value:off.value + nb.value].view(torch.float32))
        ranks.append({"p": (p0, p1), "c": (c0, c1), "ws": ws, "spans": spans, "dF": torch.empty(k, D, device="cuda")})

    def phase(i):
        for q in ranks:
            _lib.check(lib.sqfa_fused_loss_sharded(i, _lib.ptr(S), _lib.ptr(M), _lib.ptr(F), C, D, k, float(noise), dist,
                                                   q["c"][0], q["c"][1], q["p"][0], q["p"][1], _lib.ptr(q["dF"]),
                                                   _lib.ptr(q["ws"]), q["ws"].numel(), _lib.stream_ptr()), "sharded")

    def all_reduce(which):
        total = torch.stack([q["spans"][which] for q in ranks]).sum(0)
        for q in ranks:
            q["spans"][which].copy_(total)

    phase(0)
    all_reduce(0)
    phase(1)
    all_reduce(1)
    phase(2)
    dF = torch.stack([q["dF"] for q in ranks]).sum(0)
    loss, bad = ranks[0]["spans"][1][-64:-62].tolist()
    assert bad == 0.0
    assert abs(loss - float(ref[0])) <= 1e-6 * abs(float(ref[0]))
    assert rel_err(dF, ref[4:].view(k, D)) < 1e-5


@pytest.mark.parametrize("kind,distance", CLOSURES)
def test_not_positive_definite_raises_reference_error(kind, distance):
    from sqfa_b200._optim import _INF_MSG, _NAN_MSG

    C, D, k = 5, 20, 3
    stats, F0, model, sc = _closure_case(kind, distance, C, D, k)
    sc["covariances"][2] = -sc["covariances"][2]  # both models build their class matrices from these
    with pytest.raises(ValueError) as err:
        model.fit(data_statistics=sc, max_epochs=2, show_progress=False)
    assert str(err.value) in (_NAN_MSG, _INF_MSG)


def test_abi_rejects_what_it_cannot_do():
    from sqfa_b200 import _lib, _ops

    E = sample_spd(3, 5, seed=1).float().cuda()
    with pytest.raises(_lib.SqfaNativeError, match="means"):
        _ops.class_factor_raw(E, _ops.DIST_W2)
    W, _ = _ops.class_factor_raw(E, _ops.DIST_BW)
    D = torch.empty(3, 3, device="cuda")
    with pytest.raises(_lib.SqfaNativeError, match="means"):
        _ops.pair_raw(W, W, 3, 3, 5, _ops.DIST_W2, True, dist_out=D)
    with pytest.raises(_lib.SqfaNativeError, match="eig_out"):
        _ops.pair_raw(W, W, 3, 3, 5, _ops.DIST_BW, False, dist_out=D, eig_out=torch.empty(3, 3, 5, device="cuda"))
    E35 = sample_spd(2, 35, seed=2).float().cuda()
    W35 = torch.empty(2, 2 * 35 * 35, device="cuda")
    with pytest.raises(_lib.SqfaNativeError, match="code -3"):
        _ops.class_factor_raw(E35, _ops.DIST_BW)
    with pytest.raises(_lib.SqfaNativeError, match="code -3"):
        _ops.pair_raw(W35, W35, 2, 2, 35, _ops.DIST_BW, True, dist_out=torch.empty(2, 2, device="cuda"))
    # the Gaussian closure needs the means
    lib = _lib.load()
    S = sample_spd(3, 8, seed=3).float().cuda()
    F = torch.randn(2, 8, device="cuda")
    nb = lib.sqfa_fused_loss_workspace_bytes(3, 8, 2, _ops.DIST_W2, 0, 3)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    out = torch.empty(4 + 16, device="cuda")
    rc = lib.sqfa_fused_loss(_lib.ptr(S), _lib.ptr(None), _lib.ptr(F), 3, 8, 2, 0.01, _ops.DIST_W2, 0, 3, _lib.ptr(out),
                             ctypes.c_void_p(out.data_ptr() + 16), _lib.ptr(ws), nb, _lib.stream_ptr())
    assert rc == -1
