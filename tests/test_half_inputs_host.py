"""CPU: the bfloat16 / float16 entry points of the C ABI (prototypes, host-only queries, element-code
errors), the dtype dispatch of the statistics module, and the sample-sharded driver on bf16 shards under
gloo with oracle-backed ops (float32 sums / counts exchange, same result as the float32 shards)."""

import os
import re
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HALF_ENTRIES = ("sqfa_class_sums_h", "sqfa_class_gram_workspace_bytes_h", "sqfa_class_gram_h",
                "sqfa_class_gram_group_signals_h", "sqfa_class_statistics_workspace_bytes_h",
                "sqfa_class_statistics_h", "sqfa_transform_h")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from sqfa_b200 import _lib

    return _lib.load()


def test_half_prototypes_match_header(lib):
    from test_abi import _ctype_of, header_prototypes

    from sqfa_b200 import _lib

    protos = header_prototypes()
    for name in HALF_ENTRIES:
        assert hasattr(lib, name), name
        ret, args = protos[name]
        restype, argtypes = _lib.SIGNATURES[name]
        assert restype is _ctype_of(ret), name
        assert [_ctype_of(a) for a in args] == list(argtypes), name
        assert args[2] == "int32_t" or name.endswith("bytes_h") or name.endswith("signals_h"), name  # (X, ldx, elem)
    header = open(os.path.join(ROOT, "include", "sqfa_b200.h")).read()
    codes = dict(re.findall(r"#define SQFA_ELEM_(BF16|F16) (\d+)", header))
    assert _lib.ELEM_CODES == {torch.bfloat16: int(codes["BF16"]), torch.float16: int(codes["F16"])}


def test_half_workspace_queries(lib):
    # no K split at c2: the same job plan for every element type
    n, d, c = 50000, 3072, 10
    for elem in (1, 2):
        assert lib.sqfa_class_gram_workspace_bytes_h(n, d, c, elem) == lib.sqfa_class_gram_workspace_bytes(n, d, c)
    # the K-split rule counts bytes: the c5 shard (125 000 rows x 1024 per class) splits half as often in bf16
    n, d, c = 12500000, 1024, 100
    f32 = lib.sqfa_class_gram_workspace_bytes(n, d, c)
    bf16 = lib.sqfa_class_gram_workspace_bytes_h(n, d, c, 1)
    assert bf16 == lib.sqfa_class_gram_workspace_bytes_h(n, d, c, 2)
    assert (bf16 - 256) * 2 == f32 - 256  # plan entries: C x tiles x K parts
    groups = 4
    sig = [lib.sqfa_class_gram_group_signals_h(n, d, c, groups, g, 1) for g in range(groups)]
    assert sum(sig) == lib.sqfa_class_gram_group_signals_h(n, d, c, 1, 0, 1)
    assert sum(sig) * 2 == lib.sqfa_class_gram_group_signals(n, d, c, 1, 0)
    # the one-call workspace covers its parts, with the half Gram plan
    total = lib.sqfa_class_statistics_workspace_bytes_h(n, d, c, 1)
    parts = (lib.sqfa_bucket_workspace_bytes(n, c) + lib.sqfa_class_sums_workspace_bytes(n, d, c) + c * d * 4
             + bf16 + lib.sqfa_stats_epilogue_workspace_bytes(c))
    assert parts <= total <= parts + 5 * 256


def test_unknown_element_code(lib):
    for elem in (0, 3, -1):
        assert lib.sqfa_class_gram_workspace_bytes_h(1000, 64, 3, elem) == 0
        assert b"unknown element code" in lib.sqfa_last_error()
        assert lib.sqfa_class_statistics_workspace_bytes_h(1000, 64, 3, elem) == 0
        assert lib.sqfa_class_gram_group_signals_h(1000, 64, 3, 1, 0, elem) == 0
        assert lib.sqfa_class_sums_h(None, 64, elem, None, None, None, 1000, 64, 3, None, 0, None, 0, None) == -1
        assert b"sqfa_class_sums_h: unknown element code" in lib.sqfa_last_error()
        assert lib.sqfa_class_gram_h(None, 64, elem, None, None, None, 1000, 64, 3, None, 0, 0, None, 0, 0, 0, None, 0,
                                     None) == -1
        assert lib.sqfa_class_statistics_h(None, 64, elem, None, 1000, 64, 3, 0, 1, None, None, None, None, None, None,
                                           None, 0, None) == -1
        assert lib.sqfa_transform_h(None, 64, elem, None, 10, 64, 2, None, None) == -1
    # a known code with bad arguments is an argument error, named after the entry point
    assert lib.sqfa_class_sums_h(None, 64, 1, None, None, None, 1000, 64, 3, None, 0, None, 0, None) == -1
    assert b"sqfa_class_sums_h: bad argument" in lib.sqfa_last_error()


def test_dtype_dispatch_without_gpu(lib):
    from sqfa_b200 import statistics as S

    assert S._cuda_ops(torch.float32).elem == 0
    for dtype, code in ((torch.bfloat16, 1), (torch.float16, 2)):
        ops = S._cuda_ops(dtype)
        assert ops.elem == code and S._cuda_ops(dtype) is ops
        fn, xa = ops._x_fn("sqfa_class_gram")
        assert fn is lib.sqfa_class_gram_h
        X = torch.zeros(5, 3, dtype=dtype)
        assert len(xa(X)) == 3 and xa(X)[1:] == (3, code)
        assert ops._query("sqfa_class_gram_workspace_bytes", 50000, 3072, 10) == \
            lib.sqfa_class_gram_workspace_bytes(50000, 3072, 10)
    cpu = torch.device("cpu")
    for dtype in (torch.bfloat16, torch.float16):
        assert S._as_device_points(torch.ones(4, 3, dtype=dtype), cpu).dtype == dtype
    for dtype in (torch.int32, torch.int64, torch.uint8, torch.bool):
        with pytest.raises(TypeError, match="float32, float64, bfloat16 or float16"):
            S._as_device_points(torch.zeros(4, 3).to(dtype), cpu)
    with pytest.raises(TypeError):
        S._as_device_points([[1.0, 2.0]], cpu)


class HalfOracleOps:
    """CPU stand-ins for CudaStatsOps' local steps on bf16 / fp16 rows: elements widened to float32, then
    float32 arithmetic (what the kernels do). Records the dtype of the buffer the driver exchanges."""

    def __init__(self):
        self.sums_out_dtypes = []

    def label_max(self, y):
        return y.max().reshape(1).clone()

    def bucket(self, y, C):
        key = torch.where((y < 0) | (y >= C), torch.full_like(y, C), y)
        perm = torch.sort(key, stable=True).indices.to(torch.int32)
        counts = torch.bincount(key, minlength=C + 1)
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(counts, 0)])
        return perm, offsets, counts

    def class_sums(self, X, perm, offsets, C, out=None):
        sums = torch.stack([X[perm[offsets[c]:offsets[c + 1]].long()].float().sum(0) for c in range(C)])
        self.sums_out_dtypes.append(None if out is None else out.dtype)
        if out is None:
            return sums
        out.copy_(sums)
        return out

    def class_means(self, sums, counts):
        return sums / counts[:, None].to(sums.dtype)

    def class_gram(self, X, perm, offsets, centre, C):
        out = []
        for c in range(C):
            Z = X[perm[offsets[c]:offsets[c + 1]].long()].float() - centre[c]
            out.append(Z.T @ Z)
        return torch.stack(out)

    def finalize(self, gram, means, counts, estimator_id, ddof, want_sm, class_range=None):
        c0, c1 = (0, means.shape[0]) if class_range is None else class_range
        cov = gram[c0:c1] / (counts[c0:c1, None, None].to(gram.dtype) - ddof)
        return cov, cov + means[c0:c1, :, None] * means[c0:c1, None, :]


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sqfa_b200._stats_driver import run_class_statistics

    g = torch.Generator().manual_seed(1)
    X = (torch.randn(900, 7, generator=g) + 0.5).to(torch.bfloat16)
    y = torch.randint(0, 5, (900,), generator=g)
    cuts = [0, 250, 600, 900] if world == 3 else [0, 400, 900]
    lo, hi = cuts[rank], cuts[rank + 1]
    ops = HalfOracleOps()
    half = run_class_statistics(ops, X[lo:hi], y[lo:hi], 0, group=dist.group.WORLD)
    f32 = run_class_statistics(HalfOracleOps(), X[lo:hi].float(), y[lo:hi], 0, group=dist.group.WORLD)
    ret[rank] = (half[:3], f32[:3], ops.sums_out_dtypes)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_driver_on_bf16_shards(world):
    sys.path.insert(0, ROOT)
    from oracle import sqfa_oracle as O

    port = 29500 + (os.getpid() % 2000) + 7 * world
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
        results = [ret[r] for r in range(world)]
    g = torch.Generator().manual_seed(1)
    X = (torch.randn(900, 7, generator=g) + 0.5).to(torch.bfloat16)
    y = torch.randint(0, 5, (900,), generator=g)
    ref = O.class_statistics(X.double(), y)
    for half, f32, dtypes in results:
        assert dtypes == [torch.float32]  # the [sums | counts] exchange buffer is float32 for bf16 rows
        for a, b, key in zip(half, f32, ("means", "covariances", "second_moments")):
            assert a.dtype == torch.float32
            assert torch.equal(a, b), key
            assert torch.allclose(a.double(), ref[key], rtol=1e-5, atol=1e-6), key
