"""The class- and pair-sharded float64 closure (sqfa_fused_loss_sharded_f64) and float64 fits over a process group.

* Emulated ranks on one device: every rank runs the three phases on its own workspace, the two exchange spans and
  dF are summed over the ranks the way the all-reduces would sum them. Loss and dLoss/dF equal the single-device
  float64 closure at the same filters and the float64 oracle, for all eight float64 closure codes, more ranks than
  classes and pair cuts inside a pair tile; a workspace full of NaN changes nothing; two runs are bit-identical.
* 2 ranks over NCCL (skipped on a single-GPU box): the sharded plans of `.double()` models against the single-GPU
  float64 closure, and float64 fits with `process_group` against the single-GPU float64 fit.
"""

import os
import socket

import pytest
import torch

from conftest import rel_err
from oracle import sqfa_oracle as O
from test_bures_wasserstein_gpu import gauss_stats

pytestmark = pytest.mark.gpu

# the models store their noise through float32 (as the reference does), so the oracle takes that value
NOISE = float(torch.tensor(0.01, dtype=torch.float32))
CODES = [("second_moments", "affine_invariant"), ("second_moments", "affine_invariant_sq"),
         ("full", "fisher_rao_lower_bound"), ("full", "fisher_rao_lower_bound_sq"), ("full", "mahalanobis"),
         ("full", "mahalanobis_sq"), ("full", "bhattacharyya"), ("full", "hellinger")]


def _model(kind, distance, D, k, F0):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA, SecondMomentsSQFA

    cls = SecondMomentsSQFA if kind == "second_moments" else SQFA
    return cls(n_dim=D, feature_noise=0.01, n_filters=k, filters=F0.clone(), distance_fun=getattr(Dn, distance),
               constraint="sphere").double().cuda()


def _stats_for(kind, stats):
    if kind == "second_moments":
        return stats["second_moments"].cuda()
    return {"means": stats["means"].cuda(), "covariances": stats["covariances"].cuda()}


def _unit_filters(k, D, seed, device="cpu"):
    F = torch.randn(k, D, generator=torch.Generator().manual_seed(seed)).double()
    return (F / F.norm(dim=1, keepdim=True)).to(device).contiguous()


def _single(S, M, F, dist):
    """The single-device float64 closure at the constrained filters F (no constraint): loss, #bad, dF."""
    from sqfa_b200 import _ops

    C, D, _ = S.shape
    k = F.shape[0]
    P = C * (C - 1) // 2
    ws = torch.empty(_ops.closure_workspace_bytes_f64(C, D, k, dist, 0, P), dtype=torch.uint8, device="cuda")
    out = torch.zeros(3, dtype=torch.float64, device="cuda")
    grad = torch.zeros(k, D, dtype=torch.float64, device="cuda")
    noise = torch.full((1,), NOISE, dtype=torch.float64, device="cuda")
    gauss = (dist & 15) in (_ops.DIST_MAHA, _ops.DIST_BHATT, _ops.DIST_HELL)
    run = _ops.gauss_closure_eval_f64_raw if gauss else _ops.closure_eval_f64_raw
    run(F, S, M, noise, dist, False, 0, out, grad, ws)
    return out[0].item(), out[1].item(), grad


def _emulated(S, M, F, dist, world, nan_fill=False):
    """sqfa_fused_loss_sharded_f64 with `world` ranks on one device; the all-reduces are sums in rank order."""
    from sqfa_b200 import _lib, _ops
    from sqfa_b200._stats_driver import class_share

    lib = _lib.load()
    C, D, _ = S.shape
    k = F.shape[0]
    P = C * (C - 1) // 2
    noise = torch.full((1,), NOISE, dtype=torch.float64, device="cuda")
    ranks = []
    for r in range(world):
        p0, p1 = _ops.shard_pairs(P, C, r, world)
        c0, c1 = class_share(C, r, world)
        ws = torch.empty(_ops.closure_workspace_bytes_f64(C, D, k, dist, p0, p1), dtype=torch.uint8, device="cuda")
        dF = torch.empty(k, D, dtype=torch.float64, device="cuda")
        if nan_fill:
            ws.view(torch.float64).fill_(float("nan"))
            dF.fill_(float("nan"))
        spans = _ops._exchange_spans("sqfa_fused_loss_exchange_span_f64", C, D, k, dist, p0, p1, ws, torch.float64)
        ranks.append({"p": (p0, p1), "c": (c0, c1), "ws": ws, "spans": spans, "dF": dF})

    def phase(i):
        for q in ranks:
            _lib.check(lib.sqfa_fused_loss_sharded_f64(i, _lib.ptr(S), _lib.ptr(M), _lib.ptr(F), C, D, k,
                                                       _lib.ptr(noise), dist, q["c"][0], q["c"][1], q["p"][0],
                                                       q["p"][1], _lib.ptr(q["dF"]), _lib.ptr(q["ws"]),
                                                       q["ws"].numel(), _lib.stream_ptr()), "sharded_f64")

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
    red = ranks[0]["spans"][1][-64:]
    assert torch.equal(red[2:], torch.zeros_like(red[2:]))
    loss, bad = red[:2].tolist()
    return loss, bad, dF


def _inputs(kind, distance, C, D, k, seed):
    stats = gauss_stats(C, D, seed=seed + C)
    F = _unit_filters(k, D, seed + 3)
    model = _model(kind, distance, D, k, F)
    S, M, dist = model._fused_inputs(_stats_for(kind, stats))
    return stats, F.cuda(), S, M, dist


# (C, D, k, world): a cut of shard_pairs inside a pair tile of the mean-covariance closure (C = 37, k = 3: tile edge
# 8, cut after row 20), more ranks than classes, odd D, k = 32 (Fisher-Rao: m = 33)
CASES = [(37, 64, 3, 3), (12, 40, 5, 5), (3, 24, 4, 5), (19, 33, 8, 2), (21, 80, 32, 3)]


@pytest.mark.parametrize("C,D,k,world", CASES)
@pytest.mark.parametrize("kind,distance", CODES)
def test_emulated_ranks_match_single_device_and_oracle(kind, distance, C, D, k, world):
    stats, F, S, M, dist = _inputs(kind, distance, C, D, k, seed=world)
    ref_loss, ref_bad, ref_dF = _single(S, M, F, dist)
    loss, bad, dF = _emulated(S, M, F, dist, world)
    assert bad == 0.0 and ref_bad == 0.0
    assert abs(loss - ref_loss) <= 1e-12 * abs(ref_loss), (loss, ref_loss)
    assert rel_err(dF, ref_dF) <= 1e-10, rel_err(dF, ref_dF)
    ostats = stats["second_moments"] if kind == "second_moments" else stats
    loss64, grad64, _ = O.loss_and_grad(kind, ostats, F.cpu(), noise=NOISE, constraint="none",
                                        distance=getattr(O, distance))
    assert abs(loss - float(loss64)) <= 1e-10 * abs(float(loss64)), (loss, float(loss64))
    assert rel_err(dF.cpu(), grad64) <= 1e-8, rel_err(dF.cpu(), grad64)
    # a workspace (and dF) full of NaN before phase 0 changes nothing, and two runs are bit-identical
    loss2, bad2, dF2 = _emulated(S, M, F, dist, world, nan_fill=True)
    assert (loss2, bad2) == (loss, bad) and torch.equal(dF2, dF)


@pytest.mark.parametrize("kind,distance", [CODES[0], CODES[3]])
def test_pair_cut_inside_an_affine_invariant_tile(kind, distance):
    """C = 400 on 2 ranks: about 40 000 pairs per rank give the affine-invariant / Fisher-Rao pair stage a tile edge
    of 3, and shard_pairs cuts after row 280, inside the tile of rows 279-281."""
    stats, F, S, M, dist = _inputs(kind, distance, 400, 24, 3, seed=1)
    ref_loss, _, ref_dF = _single(S, M, F, dist)
    loss, bad, dF = _emulated(S, M, F, dist, 2)
    assert bad == 0.0
    assert abs(loss - ref_loss) <= 1e-12 * abs(ref_loss)
    assert rel_err(dF, ref_dF) <= 1e-10


@pytest.mark.slow
@pytest.mark.parametrize("kind,distance", [("full", "fisher_rao_lower_bound"), ("full", "mahalanobis")])
def test_c4_on_eight_emulated_ranks(kind, distance):
    """The c4 shape (C = 1000, D = 512, k = 16) on 8 emulated ranks against the single-device float64 closure.
    Statistics are generated on the device (the host generator would take minutes at this size)."""
    C, D, k, r = 1000, 512, 16, 48
    g = torch.Generator(device="cuda").manual_seed(4)
    G = torch.randn(C, D, r, generator=g, dtype=torch.float64, device="cuda") / r**0.5
    cov = G @ G.transpose(1, 2) + 0.05 * torch.eye(D, dtype=torch.float64, device="cuda")
    del G
    means = 0.3 * torch.randn(C, D, generator=g, dtype=torch.float64, device="cuda") / D**0.5 * 4
    F = _unit_filters(k, D, 7, "cuda")
    model = _model(kind, distance, D, k, F.cpu())
    S, M, dist = model._fused_inputs({"means": means, "covariances": cov})
    ref_loss, _, ref_dF = _single(S, M, F, dist)
    loss, bad, dF = _emulated(S, M, F, dist, 8)
    assert bad == 0.0
    assert abs(loss - ref_loss) <= 1e-12 * abs(ref_loss)
    assert rel_err(dF, ref_dF) <= 1e-10


# ------------------------------------------------------------------------------------------------------------------
WORLD = 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _fit(model, stats, group, **kw):
    losses, _ = model.fit(data_statistics=stats, show_progress=False, return_loss=True, process_group=group, **kw)
    return losses, model.filters.detach().clone()


def _worker(rank, world, port, out_dir, slow):
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import torch.distributed as dist

    from test_bures_wasserstein_gpu import gauss_stats

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    group = dist.group.WORLD
    try:
        res = {}
        C, D, k = 40, 64, 6
        stats = gauss_stats(C, D, seed=9)
        sc = {"means": stats["means"].cuda(), "covariances": stats["covariances"].cuda()}
        F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(0)).double()
        for distance in ("fisher_rao_lower_bound", "mahalanobis"):
            model = _model("full", distance, D, k, F0)
            grad = lambda: model.parametrizations.filters.original.grad.clone()  # noqa: E731
            rep = model._fused_direct_plan(sc)().clone()
            g_rep = grad()
            model._process_group = group
            plan = model._fused_direct_plan(sc)
            res[f"{distance}_plan_dtype"] = float(plan is not None and plan.dtype == torch.float64)
            sh = plan().clone()
            g_sh = grad()
            os.environ["SQFA_SHARD_CLASSES"] = "0"
            sh_p = model._fused_direct_plan(sc)().clone()
            g_sh_p = grad()
            os.environ["SQFA_SHARD_CLASSES"] = "1"
            model._process_group = None
            for tag, out, g in (("classes", sh, g_sh), ("pairs", sh_p, g_sh_p)):
                res[f"{distance}_{tag}_dtype"] = float(out.dtype == torch.float64 and g.dtype == torch.float64)
                res[f"{distance}_{tag}_bad"] = float(out[1])
                res[f"{distance}_{tag}_loss_rel"] = abs(float(out[0]) - float(rep[0])) / abs(float(rep[0]))
                res[f"{distance}_{tag}_grad_rel"] = float((g - g_rep).norm() / g_rep.norm())
            # a float64 fit with the group against the single-GPU float64 fit
            l1, f1 = _fit(_model("full", distance, D, k, F0), sc, None, max_epochs=2, max_iter=6)
            l2, f2 = _fit(_model("full", distance, D, k, F0), sc, group, max_epochs=2, max_iter=6)
            res[f"{distance}_fit_loss_rel"] = float(((l1 - l2).abs() / l1.abs()).max())
            res[f"{distance}_fit_filter_rel"] = float((f1 - f2).norm() / f1.norm())
            fo = f2.cuda().clone()
            dist.broadcast(fo, src=0)
            res[f"{distance}_fit_rank_divergence"] = float((f2.cuda() - fo).abs().max())
        # the pairwise curriculum (frozen rows) under the group
        Cp, kp = 8, 4
        sp = gauss_stats(Cp, D, seed=2)
        scp = {"means": sp["means"].cuda(), "covariances": sp["covariances"].cuda()}
        Fp = torch.randn(kp, D, generator=torch.Generator().manual_seed(1)).double()
        l1, f1 = _fit(_model("full", "fisher_rao_lower_bound", D, kp, Fp), scp, None, max_epochs=3, pairwise=True)
        l2, f2 = _fit(_model("full", "fisher_rao_lower_bound", D, kp, Fp), scp, group, max_epochs=3, pairwise=True)
        res["pairwise_finite"] = float(torch.isfinite(l2).all())
        res["pairwise_loss_rel"] = float(((l1 - l2).abs() / l1.abs()).max())
        res["pairwise_filter_rel"] = float((f1 - f2).norm() / f1.norm())
        if slow:
            # C = 1000: the composed float64 path fails here (a batched eigvalsh of 10^6 problems)
            sl = gauss_stats(1000, D, seed=5)
            scl = {"means": sl["means"].cuda(), "covariances": sl["covariances"].cuda()}
            Fl = torch.randn(8, D, generator=torch.Generator().manual_seed(2)).double()
            ll, _ = _fit(_model("full", "fisher_rao_lower_bound", D, 8, Fl), scl, group, max_epochs=2, max_iter=4)
            res["c1000_finite"] = float(len(ll) > 0 and torch.isfinite(ll).all())
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.barrier()
        dist.destroy_process_group()


def _run_nccl(tmp_path, slow):
    import torch.multiprocessing as mp

    mp.spawn(_worker, args=(WORLD, _free_port(), str(tmp_path), slow), nprocs=WORLD, join=True)
    return [torch.load(os.path.join(str(tmp_path), f"rank{r}.pt")) for r in range(WORLD)]


@pytest.mark.skipif(torch.cuda.device_count() < WORLD, reason="needs 2 GPUs")
def test_two_ranks_over_nccl(tmp_path):
    for rank, res in enumerate(_run_nccl(tmp_path, slow=False)):
        print(rank, res)
        for distance in ("fisher_rao_lower_bound", "mahalanobis"):
            assert res[f"{distance}_plan_dtype"] == 1.0
            for tag in ("classes", "pairs"):
                assert res[f"{distance}_{tag}_dtype"] == 1.0 and res[f"{distance}_{tag}_bad"] == 0.0
                assert res[f"{distance}_{tag}_loss_rel"] <= 1e-12, (rank, distance, tag, res)
                assert res[f"{distance}_{tag}_grad_rel"] <= 1e-10, (rank, distance, tag, res)
            assert res[f"{distance}_fit_loss_rel"] <= 1e-10, (rank, distance, res)
            assert res[f"{distance}_fit_filter_rel"] <= 1e-8, (rank, distance, res)
            assert res[f"{distance}_fit_rank_divergence"] == 0.0
        assert res["pairwise_finite"] == 1.0
        assert res["pairwise_loss_rel"] <= 1e-8 and res["pairwise_filter_rel"] <= 1e-6, res


@pytest.mark.slow
@pytest.mark.skipif(torch.cuda.device_count() < WORLD, reason="needs 2 GPUs")
def test_two_ranks_many_classes_fit(tmp_path):
    for res in _run_nccl(tmp_path, slow=True):
        assert res["c1000_finite"] == 1.0
