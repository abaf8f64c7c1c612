"""GPU: bfloat16 / float16 points in class_statistics, the streaming accumulator, the derived paths and
transform. The kernels widen every element to float32 as they load it, so the results are those of the
float32 path on `X.float()`: the same bits where that path is deterministic (class sums, means, epilogue,
Grams without a K split), float32 rounding elsewhere."""

import ctypes
import os
import socket

import pytest
import torch

from conftest import make_class_data, rel_err
from oracle import sqfa_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5
HALF = [torch.bfloat16, torch.float16]
KEYS = ("means", "covariances", "second_moments")


def _stepwise(X, y):
    """class_statistics through the driver's separate steps (bucket, sums, means, Gram, epilogue)."""
    from sqfa_b200 import _lib
    from sqfa_b200._stats_driver import CudaStatsOps, run_class_statistics

    ops = CudaStatsOps(_lib.ELEM_CODES.get(X.dtype, 0))
    ops.gram_events = []  # events around the Gram keep the driver off the one-call path
    means, cov, sm, _ = run_class_statistics(ops, X, y, 0)
    return {"means": means, "covariances": cov, "second_moments": sm}


@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("n,d,c", [(50000, 3072, 10), (60000, 104, 200)])
def test_bit_identical_to_float32_path(n, d, c, dtype):
    """c2 (780 tiles >= 6 x 74 CTA pairs, 5 000 rows x 12 KB per class: no K split) and a D <= 128 shape
    with C >= 148 (single-CTA Gram, one job per class): one-call entry and stepwise driver."""
    from sqfa_b200 import _lib
    from sqfa_b200.statistics import class_statistics

    lib = _lib.load()
    if d > 128:  # one job per (class, tile): the plan holds C x 78 jobs
        for elem in (1, 2):
            assert lib.sqfa_class_gram_workspace_bytes_h(n, d, c, elem) == c * 78 * 16 + 256
        assert lib.sqfa_class_gram_workspace_bytes(n, d, c) == c * 78 * 16 + 256
    X, y = make_class_data(n, d, c, seed=d, dtype=dtype)
    Xh, yd = X.cuda(), y.cuda()
    X32 = Xh.float()
    got, ref = class_statistics(Xh, yd), class_statistics(X32, yd)
    step, ref_step = _stepwise(Xh, yd), _stepwise(X32, yd)
    for key in KEYS:
        assert got[key].dtype == torch.float32 and step[key].dtype == torch.float32
        assert torch.equal(got[key], ref[key]), key
        assert torch.equal(step[key], ref_step[key]), key


def _assert_per_class(got, ref):
    for key in KEYS:
        g, r = got[key].double().cpu(), ref[key]
        assert g.shape == r.shape, key
        assert torch.equal(torch.isnan(g), torch.isnan(r)), key
        for cc in range(r.shape[0]):
            if torch.isnan(r[cc]).any():
                continue
            assert rel_err(g[cc], r[cc]) < TOL, (key, cc)


def _place(X, layout):
    """X on the device in the given memory layout (same values)."""
    n, d = X.shape
    if layout == "contiguous":
        return X.cuda()
    if layout == "offset1":  # one element past an 8-byte boundary: element loads everywhere
        buf = torch.zeros(n * d + 1, dtype=X.dtype, device="cuda")
        buf[1:] = X.reshape(-1).cuda()
        return buf[1:].view(n, d)
    pad = int(layout[len("pitch"):])  # row stride d + pad
    buf = torch.zeros(n, d + pad, dtype=X.dtype, device="cuda")
    buf[:, :d] = X.cuda()
    return buf[:, :d]


@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize(
    "n,d,c,kw,est,layout",
    [
        (3000, 1027, 4, {}, "empirical", "contiguous"),           # D % 4 != 0: element loads in the last tile
        (3000, 104, 19, {}, "empirical", "contiguous"),           # D <= 128: single-CTA Gram
        (4000, 512, 40, {"skew": True}, "empirical", "contiguous"),
        (2500, 300, 5, {"offset": 3.0}, "empirical", "contiguous"),  # cancellation stress
        (6000, 784, 10, {}, "oas", "contiguous"),
        (30000, 64, 1000, {}, "empirical", "contiguous"),         # C = 1000
        (4000, 512, 6, {}, "empirical", "pitch8"),                # row stride > D, still 8-byte aligned rows
        (4000, 300, 6, {}, "empirical", "pitch5"),                # row stride > D, unaligned rows
        (4000, 512, 6, {}, "empirical", "offset1"),               # X starts 2 bytes past an 8-byte boundary
    ],
)
def test_matches_oracle(n, d, c, kw, est, layout, dtype):
    from sqfa_b200.statistics import class_statistics

    X, y = make_class_data(n, d, c, seed=d + c, dtype=dtype, **kw)
    y[::17] = -1  # rows no class selects
    got = class_statistics(_place(X, layout), y.cuda(), estimator=est)
    _assert_per_class(got, O.class_statistics(X.double(), y, estimator=est))


@pytest.mark.parametrize("dtype", HALF)
def test_host_resident_input(dtype):
    from sqfa_b200.statistics import class_statistics

    X, y = make_class_data(5000, 256, 7, seed=2, dtype=dtype)
    got = class_statistics(X, y)
    assert got["means"].device.type == "cpu" and got["covariances"].dtype == torch.float32
    ref = class_statistics(X.float(), y)
    for key in KEYS:
        assert torch.equal(got[key], ref[key]), key


@pytest.mark.parametrize("dtype", HALF)
def test_streaming_half_chunks_equal_float32_chunks(dtype):
    """Same state after every chunk as float32 chunks of the same values: first-chunk shift with a class
    absent from it, and a recentring (rows grow 4x) on the third chunk. C = 12 keeps every chunk's Gram
    free of a K split (the streaming Gram adds into the state with one red.add per element)."""
    from sqfa_b200.statistics import StreamingClassStatistics

    d, c = 256, 12
    sizes = [4000, 4000, 8000, 8000]
    X, y = make_class_data(sum(sizes), d, c, seed=13, dtype=dtype)
    first = y[: sizes[0]]
    first[first == 11] = 10  # class 11 is absent from the first chunk
    a, b = StreamingClassStatistics(d, c), StreamingClassStatistics(d, c)
    lo = 0
    for s in sizes:
        a.update(X[lo:lo + s].cuda(), y[lo:lo + s].cuda())
        b.update(X[lo:lo + s].float().cuda(), y[lo:lo + s].cuda())
        lo += s
        for name in ("shift", "counts", "sums", "gram"):
            assert torch.equal(getattr(a, name), getattr(b, name)), (name, lo)
    ra, rb = a.finalize(), b.finalize()
    for key in KEYS:
        assert torch.equal(ra[key], rb[key]), key
    _assert_per_class(ra, O.class_statistics(X.double(), y))


@pytest.mark.parametrize("dtype", HALF)
def test_derived_paths_equal_float32(dtype):
    """sample_covariance, pca, fit_pca and fit at shapes whose Grams have no K split (one class: < 1024 rows;
    fit: 10 classes of about 200 rows): the same bits as on X.float()."""
    from sqfa_b200 import statistics as S
    from sqfa_b200.model import SQFA

    X, y = make_class_data(1000, 256, 1, seed=21, dtype=dtype)
    Xh = X.cuda()
    assert torch.equal(S.sample_covariance(Xh), S.sample_covariance(Xh.float()))
    assert torch.equal(S.sample_covariance(Xh, assume_centered=True),
                       S.sample_covariance(Xh.float(), assume_centered=True))
    assert torch.equal(S.pca(Xh, 4), S.pca(Xh.float(), 4))
    ma, mb = SQFA(n_dim=256, n_filters=4).cuda(), SQFA(n_dim=256, n_filters=4).cuda()
    ma.fit_pca(Xh)
    mb.fit_pca(Xh.float())
    assert torch.equal(ma.filters, mb.filters)

    X, y = make_class_data(2000, 256, 10, seed=22, dtype=dtype)
    X = X / (X.float().std() * 256**0.5)
    Xh, yd = X.cuda(), y.cuda()
    torch.manual_seed(0)
    F0 = torch.randn(4, 256)
    ma = SQFA(n_dim=256, n_filters=4, feature_noise=0.01, filters=F0.clone()).cuda()
    mb = SQFA(n_dim=256, n_filters=4, feature_noise=0.01, filters=F0.clone()).cuda()
    ma.fit(X=Xh, y=yd, max_epochs=5, show_progress=False)
    mb.fit(X=Xh.float(), y=yd, max_epochs=5, show_progress=False)
    assert torch.equal(ma.filters, mb.filters)


@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("k", [3, 8, 16, 32])
@pytest.mark.parametrize("d,layout", [(520, "contiguous"), (520, "pitch8"), (520, "pitch3"), (520, "offset1"),
                                      (517, "contiguous")])
def test_transform(d, layout, k, dtype):
    """Z = X F^T (float32) and dZ/dF within 1e-6 of the float32 kernel on X.float(): aligned rows (shared-memory
    tile kernel, X staged as bf16 / fp16), strided rows, unaligned rows and D % 4 != 0 (row kernel)."""
    from sqfa_b200.model import SQFA, _Transform

    n = 5000
    g = torch.Generator().manual_seed(k + d)
    X = torch.randn(n, d, generator=g).to(dtype)
    Xd = _place(X, layout)
    model = SQFA(n_dim=d, n_filters=k).cuda()
    Z, ref = model.transform(Xd), model.transform(Xd.float())
    assert Z.dtype == torch.float32 and Z.shape == (n, k)
    assert float((Z - ref).norm()) <= 1e-6 * float(ref.norm())
    G = torch.randn(n, k, generator=g).cuda()
    Fa = torch.randn(k, d, generator=g).cuda().requires_grad_()
    Fb = Fa.detach().clone().requires_grad_()
    (_Transform.apply(Fa, Xd) * G).sum().backward()
    (_Transform.apply(Fb, Xd.float()) * G).sum().backward()
    assert Fa.grad.dtype == torch.float32
    assert float((Fa.grad - Fb.grad).norm()) <= 1e-6 * float(Fb.grad.norm())


@pytest.mark.parametrize("n,d,c,world", [(6000, 512, 10, 8), (9000, 520, 7, 2)])
def test_reduce_scatter_building_blocks_on_one_device(n, d, c, world):
    """The pieces of the multi-GPU sharded-output path with bf16 rows on ONE device (`world` emulated ranks):
    packed Gram partials with completion counters in owner order, pushes into the owners' slots, and the
    epilogue that sums the slots in rank order -- the statistics of the union."""
    from sqfa_b200 import _lib
    from sqfa_b200._stats_driver import CudaStatsOps, class_share, peer_push_schedule

    lib = _lib.load()
    X, y = make_class_data(n, d, c, seed=3 * d, dtype=torch.bfloat16)
    X, y = X.cuda(), y.cuda()
    ops = CudaStatsOps(_lib.ELEM_CODES[torch.bfloat16])
    perm_all, off_all, cnt_all = ops.bucket(y, c)
    counts = cnt_all[:c].clone()
    means = ops.class_means(ops.class_sums(X, perm_all, off_all, c), counts)
    assert torch.equal(means, CudaStatsOps().class_means(CudaStatsOps().class_sums(X.float(), perm_all, off_all, c),
                                                         counts))
    shares = [class_share(c, r, world) for r in range(world)]
    per_class = lib.sqfa_gram_packed_floats(d, c) // c
    stride = max(hi - lo for lo, hi in shares) * per_class
    cuts = [(n * r) // world for r in range(world + 1)]
    slots = torch.full((world, world, stride), float("nan"), device="cuda")
    partials = []
    for r in range(world):
        Xr, yr = X[cuts[r]:cuts[r + 1]], y[cuts[r]:cuts[r + 1]]
        perm, offsets, _ = ops.bucket(yr, c)
        done = torch.zeros(world, dtype=torch.int32, device="cuda")
        rotated = ops.class_gram(Xr, perm, offsets, means, c, packed=True, done=done, n_groups=world,
                                 first_class=shares[r][1] % c)
        expected = [lib.sqfa_class_gram_group_signals_h(Xr.shape[0], d, c, world, g, 1) for g in range(world)]
        assert done.tolist() == expected
        partials.append(rotated)
        for g, lo, hi in peer_push_schedule(r, world, shares):
            _lib.check(lib.sqfa_peer_push(ctypes.c_void_p(slots[g, r].data_ptr()),
                                          ctypes.c_void_p(rotated.data_ptr() + 4 * lo * per_class),
                                          4 * (hi - lo) * per_class, _lib.stream_ptr()), "sqfa_peer_push")
    ref = O.class_statistics(X.double().cpu(), y.cpu())
    for r in range(world):
        lo, hi = shares[r]
        nc = hi - lo
        if nc == 0:
            continue
        cov = torch.empty(nc, d, d, device="cuda")
        sm = torch.empty(nc, d, d, device="cuda")
        ws = torch.empty(lib.sqfa_stats_epilogue_workspace_bytes(nc), dtype=torch.uint8, device="cuda")
        own = partials[r].data_ptr() + 4 * lo * per_class
        _lib.check(lib.sqfa_stats_epilogue_reduce(
            ctypes.c_void_p(own), _lib.ptr(slots[r]), stride, world, r, _lib.ptr(means[lo:hi]), None,
            _lib.ptr(counts[lo:hi]), d, nc, 0, 1, _lib.ptr(cov), _lib.ptr(sm), _lib.ptr(ws), ws.numel(),
            _lib.stream_ptr()), "sqfa_stats_epilogue_reduce")
        assert rel_err(cov, ref["covariances"][lo:hi]) < TOL
        assert rel_err(sm, ref["second_moments"][lo:hi]) < TOL


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out_dir):
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import torch.distributed as dist

    from conftest import make_class_data
    from sqfa_b200 import statistics as S

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        n, d, c = 9001, 512, 12
        X, y = make_class_data(n, d, c, seed=4, dtype=torch.bfloat16)
        cut = [0, 4000, n]
        Xs, ys = X[cut[rank]:cut[rank + 1]].cuda(), y[cut[rank]:cut[rank + 1]].cuda()
        res = {"full": S.class_statistics(X.float().cuda(), y.cuda()),
               "rep": S.class_statistics(Xs, ys, group=dist.group.WORLD),
               "rep32": S.class_statistics(Xs.float(), ys, group=dist.group.WORLD),
               "shard": S.class_statistics(Xs, ys, group=dist.group.WORLD, shard_output=True)}
        torch.save({k: {kk: (vv.cpu() if torch.is_tensor(vv) else vv) for kk, vv in v.items()} for k, v in res.items()},
                   os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_bf16_shards(tmp_path):
    import torch.multiprocessing as mp

    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for rank in range(2):
        res = torch.load(os.path.join(tmp_path, f"rank{rank}.pt"))
        full, rep, rep32, shard = res["full"], res["rep"], res["rep32"], res["shard"]
        lo, hi = shard["class_range"]
        for key in KEYS:
            assert torch.equal(rep[key], rep32[key]), key  # bf16 shards == their float32 copies, exchange included
            assert rel_err(rep[key], full[key]) < TOL, key
            part = full[key] if key == "means" else full[key][lo:hi]
            assert rel_err(shard[key], part) < TOL, key


@pytest.mark.parametrize("dtype", [torch.int32, torch.int64, torch.uint8] +
                         [getattr(torch, n) for n in ("float8_e4m3fn", "float8_e5m2") if hasattr(torch, n)])
def test_other_dtypes_still_raise(dtype):
    from sqfa_b200.statistics import class_statistics

    X = torch.zeros(100, 8).to(dtype).cuda()
    y = torch.zeros(100, dtype=torch.int64).cuda()
    with pytest.raises(TypeError, match="float32, float64, bfloat16 or float16"):
        class_statistics(X, y)


def test_unknown_element_code_is_an_error():
    from sqfa_b200 import _lib

    lib = _lib.load()
    X = torch.zeros(64, 8, dtype=torch.bfloat16, device="cuda")
    F = torch.zeros(2, 8, device="cuda")
    Z = torch.zeros(64, 2, device="cuda")
    assert lib.sqfa_transform_h(_lib.ptr(X), 8, 3, _lib.ptr(F), 64, 8, 2, _lib.ptr(Z), _lib.stream_ptr()) == -1
    assert b"unknown element code" in lib.sqfa_last_error()
    assert lib.sqfa_transform_h(_lib.ptr(X), 8, 1, _lib.ptr(F), 64, 8, 2, _lib.ptr(Z), _lib.stream_ptr()) == 0
