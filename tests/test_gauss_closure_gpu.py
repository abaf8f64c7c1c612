"""The native fitting closure of the mean-covariance distances (Mahalanobis, squared Mahalanobis,
Bhattacharyya, Hellinger) against the float64 oracle: loss and gradient at the benchmark shapes, edge
shapes, determinism, the generic path, fits, the orthogonal constraint, the sharded phases, the
not-positive-definite guard and the C ABI's rejections."""

import ctypes
import os

import pytest
import torch

from conftest import rel_err
from oracle import sqfa_oracle as O
from test_bures_wasserstein_gpu import gauss_stats

pytestmark = pytest.mark.gpu

GRAD_TOL = 2e-3  # gradient of the loss w.r.t. the raw filters, relative Frobenius vs fp64 oracle
LOSS_TOL = 1e-4
NAMES = ["mahalanobis", "mahalanobis_sq", "bhattacharyya", "hellinger"]
SHAPES = {"c1": (10, 784, 4), "c2": (10, 3072, 8), "c3": (19, 104, 8), "c5": (100, 1024, 32)}


def _model(distance, D, k, F0, constraint="sphere"):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA

    fun = distance if callable(distance) else getattr(Dn, distance)
    return SQFA(n_dim=D, feature_noise=0.01, n_filters=k, filters=F0.clone(), distance_fun=fun, constraint=constraint)


def _case(distance, C, D, k, seed=0, constraint="sphere"):
    stats = gauss_stats(C, D, seed=seed + C)
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(seed + 3))
    model = _model(distance, D, k, F0, constraint).cuda()
    sc = {"means": stats["means"].float().cuda(), "covariances": stats["covariances"].float().cuda()}
    return stats, F0, model, sc


def _check_closure(distance, C, D, k, seed=0):
    stats, F0, model, sc = _case(distance, C, D, k, seed)
    loss64, grad64, _ = O.loss_and_grad("full", stats, F0.double(), noise=0.01, distance=getattr(O, distance))
    direct = model._fused_direct_plan(sc)
    assert direct is not None
    out = direct().tolist()
    g = model.parametrizations.filters.original.grad.clone()
    assert out[1] == 0.0
    assert abs(out[0] - float(loss64)) <= LOSS_TOL * abs(float(loss64))
    assert rel_err(g, grad64) < GRAD_TOL
    return model, sc, out, g


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("distance", NAMES)
def test_fused_closure_matches_oracle(distance, shape):
    C, D, k = SHAPES[shape]
    model, sc, out, g = _check_closure(distance, C, D, k)
    direct = model._fused_direct_plan(sc)
    out2 = direct().tolist()
    assert out2[0] == out[0]
    assert torch.equal(model.parametrizations.filters.original.grad, g)
    # the generic path (get_class_distances -> -mean(tril) -> autograd) agrees to 1e-5
    model.parametrizations.filters.original.grad = None
    dmat = model.get_class_distances(sc, regularized=True)
    i, j = torch.tril_indices(C, C, -1)
    loss = -dmat[i, j].mean()
    loss.backward()
    assert abs(float(loss.detach()) - out[0]) <= 1e-5 * abs(out[0])
    assert rel_err(model.parametrizations.filters.original.grad, g.double()) <= 1e-5


@pytest.mark.parametrize("C,D,k", [(2, 16, 3), (7, 24, 1), (9, 40, 5), (13, 48, 7), (37, 64, 16), (21, 80, 32),
                                   (35, 40, 2), (53, 40, 4)])
@pytest.mark.parametrize("distance", NAMES)
def test_edge_shapes(distance, C, D, k):
    """One pair, k = 1, odd k, k = 32, and class counts that are not multiples of the tile edge."""
    _check_closure(distance, C, D, k, seed=11)


@pytest.mark.slow
@pytest.mark.parametrize("distance", NAMES)
def test_many_classes(distance):
    _check_closure(distance, 1000, 64, 16, seed=1)


@pytest.mark.parametrize("distance", ["mahalanobis", "hellinger"])
def test_fit_matches_oracle_deterministic_and_unpipelined(distance, monkeypatch):
    C, D, k = 8, 40, 4
    stats = gauss_stats(C, D, seed=5)
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(9))
    _, losses_o, _ = O.fit_lbfgs("full", stats, F0.double(), noise=0.01, distance=getattr(O, distance), max_epochs=2,
                                 max_iter=5)
    s32 = {"means": stats["means"].float(), "covariances": stats["covariances"].float()}
    filters = []
    for pipeline in ("1", "1", "0"):
        monkeypatch.setenv("SQFA_LBFGS_PIPELINE", pipeline)
        model = _model(distance, D, k, F0)
        losses, _ = model.fit(data_statistics=s32, max_epochs=2, show_progress=False, return_loss=True, max_iter=5)
        assert torch.allclose(losses.double(), losses_o.double(), rtol=1e-3)
        filters.append(model.filters.detach().clone())
    assert torch.equal(filters[0], filters[1])
    assert torch.equal(filters[0], filters[2])


@pytest.mark.parametrize("distance", NAMES)
def test_orthogonal_constraint_takes_fused_loss(distance):
    C, D, k = 12, 48, 6
    _, _, model, sc = _case(distance, C, D, k, seed=4, constraint="orthogonal")
    assert model._fused_direct_plan(sc) is None
    fused = model._fused_loss_plan(sc)
    assert fused is not None
    out = fused()
    out[0].backward()
    g = model.parametrizations.filters.original.grad.clone()
    model.parametrizations.filters.original.grad = None
    dmat = model.get_class_distances(sc, regularized=True)
    i, j = torch.tril_indices(C, C, -1)
    loss = -dmat[i, j].mean()
    loss.backward()
    assert abs(float(loss.detach()) - float(out[0].detach())) <= 1e-5 * abs(float(out[0].detach()))
    assert rel_err(model.parametrizations.filters.original.grad, g.double()) <= 1e-5


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("distance", ["mahalanobis_sq", "bhattacharyya", "hellinger"])
def test_sharded_closure_phases_on_one_device(distance, world):
    """sqfa_fused_loss_sharded with `world` emulated ranks on one device equals sqfa_fused_loss."""
    from sqfa_b200 import _lib, _ops
    from sqfa_b200._stats_driver import class_share

    lib = _lib.load()
    C, D, k = 23, 96, 6
    _, _, model, sc = _case(distance, C, D, k, seed=7)
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


def _nccl_worker(rank, world, port, distance, result):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        stats = gauss_stats(16, 40, seed=3)
        F0 = torch.randn(4, 40, generator=torch.Generator().manual_seed(2))
        s32 = {"means": stats["means"].float().cuda(), "covariances": stats["covariances"].float().cuda()}
        model = _model(distance, 40, 4, F0)
        losses, _ = model.fit(data_statistics=s32, max_epochs=2, show_progress=False, return_loss=True, max_iter=5,
                              process_group=dist.group.WORLD)
        if rank == 0:
            result.put(losses.tolist())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("distance", ["bhattacharyya"])
def test_two_rank_nccl_fit(distance):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    result = ctx.Queue()
    mp.spawn(_nccl_worker, args=(2, port, distance, result), nprocs=2, join=True)
    got = torch.tensor(result.get())
    stats = gauss_stats(16, 40, seed=3)
    F0 = torch.randn(4, 40, generator=torch.Generator().manual_seed(2))
    _, losses_o, _ = O.fit_lbfgs("full", stats, F0.double(), noise=0.01, distance=getattr(O, distance), max_epochs=2,
                                 max_iter=5)
    assert torch.allclose(got.double(), losses_o.double(), rtol=1e-3)


@pytest.mark.parametrize("distance", NAMES)
def test_not_positive_definite_raises_reference_error(distance):
    from sqfa_b200._optim import _INF_MSG, _NAN_MSG

    C, D, k = 5, 20, 3
    _, _, model, sc = _case(distance, C, D, k)
    # class 2 far from positive definite: the pair-mean covariances with it are negative definite too
    sc["covariances"][2] = -10 * sc["covariances"][2]
    assert model._fused_direct_plan(sc) is not None
    with pytest.raises(ValueError) as err:
        model.fit(data_statistics=sc, max_epochs=2, show_progress=False)
    assert str(err.value) in (_NAN_MSG, _INF_MSG)


def test_fisher_rao_same_cov_and_custom_functions_stay_generic():
    from sqfa_b200 import distances as Dn

    _, _, model, sc = _case("fisher_rao_same_cov", 6, 20, 3)
    assert model._fused_direct_plan(sc) is None
    assert model._fused_loss_plan(sc) is None
    _, _, model, sc = _case(lambda a, b: Dn.hellinger(a, b), 6, 20, 3)
    assert model._fused_direct_plan(sc) is None


def test_abi_rejects_what_it_cannot_do():
    from sqfa_b200 import _lib, _ops

    lib = _lib.load()
    E = torch.eye(3, device="cuda").expand(2, 3, 3).contiguous()
    W = torch.empty(2, 18, device="cuda")
    flag = torch.empty(1, dtype=torch.int32, device="cuda")
    for code in (_ops.DIST_MAHA, _ops.DIST_BHATT, _ops.DIST_HELL, _ops.DIST_MAHA | _ops.SQUARED):
        rc = lib.sqfa_class_factor(_lib.ptr(E), 2, 3, code, _lib.ptr(W), _lib.ptr(flag), _lib.stream_ptr())
        assert rc == -1 and b"sqfa_gauss_pair_distances" in lib.sqfa_last_error()
        with pytest.raises(_lib.SqfaNativeError, match="sqfa_gauss_pair_distances"):
            _ops.pair_raw(W, W, 2, 2, 3, code, True, dist_out=torch.empty(2, 2, device="cuda"))
        with pytest.raises(_lib.SqfaNativeError, match="sqfa_gauss_pair_distances"):
            _ops.embed_fwd_raw(E, torch.zeros(2, 3, device="cuda"), 0.0, code)
        with pytest.raises(_lib.SqfaNativeError, match="sqfa_gauss_pair_distances"):
            _ops.embed_bwd_raw(E, torch.zeros(2, 3, device="cuda"), 3, code)
        with pytest.raises(_lib.SqfaNativeError, match="sqfa_gauss_pair_distances"):
            _ops.class_factor_bwd_raw(W, E, 3, code, torch.zeros_like(E))
    # closures: means required, no squared Bhattacharyya / Hellinger, no code 8, n_filters <= 32
    S = torch.eye(8, device="cuda").expand(3, 8, 8).contiguous()
    Mn = torch.zeros(3, 8, device="cuda")
    F = torch.randn(2, 8, device="cuda")
    out = torch.empty(4 + 16, device="cuda")
    nb = lib.sqfa_fused_loss_workspace_bytes(3, 8, 2, _ops.DIST_BHATT, 0, 3)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")

    def call(Mptr, code, k=2):
        return lib.sqfa_fused_loss(_lib.ptr(S), Mptr, _lib.ptr(F), 3, 8, k, 0.01, code, 0, 3, _lib.ptr(out),
                                   ctypes.c_void_p(out.data_ptr() + 16), _lib.ptr(ws), nb, _lib.stream_ptr())

    assert call(_lib.ptr(None), _ops.DIST_MAHA) == -1
    for code in (_ops.DIST_BHATT | _ops.SQUARED, _ops.DIST_HELL | _ops.SQUARED, 8):
        assert call(_lib.ptr(Mn), code) == -1
        assert lib.sqfa_fused_loss_workspace_bytes(3, 8, 2, code, 0, 3) == 256
    assert call(_lib.ptr(Mn), _ops.DIST_HELL, k=33) == -3
    assert call(_lib.ptr(Mn), _ops.DIST_HELL) == 0
