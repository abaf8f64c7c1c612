"""Class statistics of labeled data points -- B200-native drop-in for `sqfa.statistics`.

Same public names and semantics as /root/reference/src/sqfa/statistics.py (`class_statistics`,
`oas_covariance`, `sample_covariance`, `pca`, `pca_from_scatter`); the arithmetic runs in the
sm_100a kernels of libsqfa_b200.so (label bucketing, segmented column sums, tcgen05 3xTF32 Gram,
statistics epilogue). Inputs may live on the CPU or on a CUDA device; outputs are returned on the
device of `points`. There is no CPU compute path.
"""

import torch

from . import _lib
from ._stats_driver import CudaStatsOps, CudaStatsOps64, run_class_statistics

__all__ = ["class_statistics", "oas_covariance", "pca", "pca_from_scatter"]  # the reference's; extensions below

_ESTIMATORS = {"empirical": 0, "oas": 1}
_POINT_DTYPES = (torch.float32, torch.float64, torch.bfloat16, torch.float16)
_ops_singleton = None
_ops64_singleton = None
_ops_half = {}


def _cuda_ops(dtype=torch.float32):
    """The local kernels for the dtype of the points: float32 (tcgen05 3xTF32), float64 (DFMA), or
    bfloat16 / float16 (the float32 kernels, every element widened to float32 as it is loaded)."""
    global _ops_singleton, _ops64_singleton
    if dtype == torch.float64:
        if _ops64_singleton is None:
            _ops64_singleton = CudaStatsOps64()
        return _ops64_singleton
    if dtype in _lib.ELEM_CODES:
        if dtype not in _ops_half:
            _ops_half[dtype] = CudaStatsOps(_lib.ELEM_CODES[dtype])
        return _ops_half[dtype]
    if _ops_singleton is None:
        _ops_singleton = CudaStatsOps()
    return _ops_singleton


def _as_device_points(points, dev):
    if not isinstance(points, torch.Tensor):
        raise TypeError("points must be a torch.Tensor")
    if points.dim() != 2:
        raise ValueError("points must have shape (n_points, n_dim)")
    if points.dtype not in _POINT_DTYPES:
        raise TypeError("points must be float32, float64, bfloat16 or float16 (the output follows their dtype; "
                        f"float32 for bfloat16 / float16); got {points.dtype}")
    X = points.detach().to(dev, non_blocking=True)
    if X.stride(1) != 1 or X.stride(0) < X.shape[1]:
        X = X.contiguous()
    return X


def _as_device_labels(labels, dev):
    """int64 labels on `dev`. Rows whose label equals no integer class (negative or non-integral
    values) get -1: the reference's `labels == i` (statistics.py:37) never selects them."""
    y = torch.as_tensor(labels).detach().reshape(-1)
    if y.dtype.is_floating_point:
        y = y.to(dev, non_blocking=True)
        yi = y.to(torch.int64)
        yi = torch.where(yi.to(y.dtype) == y, yi, torch.full_like(yi, -1))
        return yi.contiguous()
    if y.dtype == torch.bool:
        y = y.to(torch.int64)
    return y.to(dev, dtype=torch.int64, non_blocking=True).contiguous()


def bucket_labels(labels, n_classes=None):
    """Stable bucketing of row ids by label on the device (kernel K1).

    Returns (perm int32 [n], offsets int64 [C+2], counts int64 [C+1]) as CUDA tensors; entry C of
    counts / offsets is the bucket of rows whose label is outside [0, C). `perm[:offsets[C]]`
    equals `torch.sort(labels, stable=True).indices` for in-range labels (bit-exact).
    """
    dev = _lib.compute_device(labels)
    y = _as_device_labels(labels, dev)
    ops = _cuda_ops()
    with torch.cuda.device(dev):
        if n_classes is None:
            n_classes = ops.label_max_host(y) + 1
        return ops.bucket(y, int(n_classes))


def class_statistics(points, labels, estimator="empirical", keep_on_device=False, group=None, shard_output=False):
    """
    Compute the mean, covariance and second moment matrix of each class.

    Drop-in for `sqfa.statistics.class_statistics` (reference statistics.py:8-54).

    Parameters
    ----------
    points : torch.Tensor
        Data points with shape (n_points, n_dim), float32 or float64 (the statistics have the dtype of
        the points, like the reference's), on the CPU or a CUDA device.
        (extension) bfloat16 and float16 points are accepted too, and their statistics are FLOAT32: the
        reference would accumulate them in bf16, whose 8-bit mantissa loses the small eigenvalues the
        affine-invariant distance depends on, and the fitting closure takes float32 or float64 only.
        Every element is widened to float32 as the kernels load it, so the result is what
        `class_statistics(points.float(), labels)` returns -- bit for bit where that path is
        deterministic -- while half the bytes are read and no float32 copy of the points is made.
    labels : torch.Tensor
        Class labels of each point with shape (n_points).
    estimator:
        Covariance estimator to use. Options are "empirical" and "oas". Default is "empirical".
    keep_on_device : bool
        (extension) leave the result on the CUDA device even if `points` lives on the CPU.
    group : torch.distributed process group
        (extension) `points` / `labels` are this rank's shard of the samples; the statistics of the
        union over all ranks are returned on every rank (two small all-reduces and the all-reduce of
        the packed Gram partials, see _stats_driver).
    shard_output : bool
        (extension, with `group`) every rank returns the means of all classes but the covariances and
        second moments of ITS share of the classes only -- rows `class_range[0]:class_range[1]`, the
        range is added to the dict as "class_range". The ranks' results together are the statistics;
        nobody computes or moves the same matrix twice: the Gram partials are reduce-scattered by class
        inside the Gram kernel (copy-engine pushes into peer-mapped slots) and summed by the epilogue.

    Returns
    -------
    statistics_dict : dict
        "means" (n_classes, n_dim), "covariances" and "second_moments" (n_classes, n_dim, n_dim),
        on the device of `points`.
    """
    if estimator not in _ESTIMATORS:
        raise ValueError(f"estimator must be 'empirical' or 'oas', got {estimator!r}")
    dev = _lib.compute_device(points, labels)
    out_dev = points.device if isinstance(points, torch.Tensor) else dev
    X = _as_device_points(points, dev)
    y = _as_device_labels(labels, dev)
    if y.numel() != X.shape[0]:
        raise ValueError("labels must have one entry per row of points")
    if y.numel() == 0 and group is None:
        raise RuntimeError("class_statistics: empty input (max() of an empty labels tensor)")
    with torch.cuda.device(dev):
        means, cov, sm, _ = run_class_statistics(_cuda_ops(X.dtype), X, y, _ESTIMATORS[estimator], group=group,
                                                 shard_output=shard_output and group is not None)
    stats = {"means": means, "covariances": cov, "second_moments": sm}
    if out_dev != dev and not keep_on_device:
        stats = {k: v.to(out_dev) for k, v in stats.items()}
    if shard_output and group is not None:
        import torch.distributed as dist

        from ._stats_driver import class_share

        stats["class_range"] = class_share(means.shape[0], dist.get_rank(group), dist.get_world_size(group))
    return stats


class StreamingClassStatistics:
    """Out-of-core `class_statistics`: chunks of labeled rows are folded into the additive per-class
    state (count, sum (x - s), sum (x - s)(x - s)^T) with a fixed shift s, and `finalize` returns the
    reference's statistics dict (statistics.py:8-54) for all rows seen so far.

    This is BASELINE config 5 (N = 100 M rows do not exist as one tensor) and SURVEY section 8(f)
    row 2; it uses the same kernels as `class_statistics` with their `accumulate` / `shift`
    arguments. The shift only has to be near the class means (it keeps the accumulated Gram
    well-conditioned; the epilogue removes it exactly): by default it is the class means of the
    first chunk. With `group`, every rank streams its own rows, the shift of rank 0 is broadcast at
    the first update and `finalize` all-reduces the state.

    >>> acc = StreamingClassStatistics(n_dim=1024, n_classes=100)
    >>> for X_chunk, y_chunk in loader: acc.update(X_chunk, y_chunk)
    >>> stats = acc.finalize()            # {"means", "covariances", "second_moments"}
    """

    def __init__(self, n_dim, n_classes, shift=None, device=None, group=None):
        self.D, self.C = int(n_dim), int(n_classes)
        if self.D <= 0 or self.C <= 0:
            raise ValueError("n_dim and n_classes must be positive")
        self.dev = _lib.compute_device() if device is None else torch.device(device)
        self.group = group
        self.lib = _lib.load()
        self.shift = None if shift is None else torch.as_tensor(shift, dtype=torch.float32).to(self.dev).contiguous()
        if self.shift is not None and tuple(self.shift.shape) != (self.C, self.D):
            raise ValueError("shift must have shape (n_classes, n_dim)")
        with torch.cuda.device(self.dev):
            self.counts = torch.zeros(self.C, dtype=torch.int64, device=self.dev)
            self.sums = torch.zeros(self.C, self.D, dtype=torch.float32, device=self.dev)
            self.gram = torch.zeros(self.C, self.D, self.D, dtype=torch.float32, device=self.dev)
        self.n_rows = 0
        self._auto_shift = shift is None and group is None  # ranks must keep identical shifts
        self._rows_at_shift = 0

    def _first_shift(self, X, perm, offsets, counts):
        ops = _cuda_ops(X.dtype)
        m = ops.class_means(ops.class_sums(X, perm, offsets, self.C), counts[: self.C].clone())
        # classes absent from the first chunk. Computed on the chunk's float32 values (a copy of the first
        # chunk only, for bf16 / fp16) with the same reduction a float32 stream runs, so that a bf16 / fp16
        # stream and a float32 stream of the same values hold identical state
        fallback = X.float().mean(dim=0, keepdim=True).expand_as(m)
        shift = torch.where(torch.isfinite(m), m, fallback).contiguous()
        if self.group is not None:
            import torch.distributed as dist

            dist.broadcast(shift, src=dist.get_global_rank(self.group, 0), group=self.group)
        return shift

    def update(self, points, labels):
        """Fold a chunk of rows (n, n_dim) float32 (or bfloat16 / float16, widened to float32 as they are
        loaded: the same state as the chunk's float32 copy would give) with labels (n,) into the state.
        Rows whose label is outside [0, n_classes) are ignored, like rows no `labels == i` selects in
        the reference."""
        dev, C, D = self.dev, self.C, self.D
        X = _as_device_points(points, dev)
        y = _as_device_labels(labels, dev)
        if X.dtype == torch.float64:
            raise TypeError("StreamingClassStatistics accumulates float32, bfloat16 or float16 chunks")
        if X.shape[1] != D or y.numel() != X.shape[0]:
            raise ValueError("chunk must have shape (n, n_dim) and one label per row")
        n = X.shape[0]
        if n == 0:
            return self
        with torch.cuda.device(dev):
            ops = _cuda_ops(X.dtype)
            perm, offsets, counts = ops.bucket(y, C)
            if self.shift is None:
                self.shift = self._first_shift(X, perm, offsets, counts)
                self._rows_at_shift = n
            elif self._auto_shift and self.n_rows + n >= 4 * self._rows_at_shift:
                self._recentre(X, perm, offsets, counts)
            st = _lib.stream_ptr(dev)
            nb = self.lib.sqfa_class_sums_workspace_bytes(n, D, C)
            ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
            fn, xa = ops._x_fn("sqfa_class_sums")
            _lib.check(
                fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), _lib.ptr(self.shift), n, D, C, _lib.ptr(self.sums), 1,
                   _lib.ptr(ws), nb, st),
                "sqfa_class_sums",
            )
            nb = ops._query("sqfa_class_gram_workspace_bytes", n, D, C)
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            fn, xa = ops._x_fn("sqfa_class_gram")
            _lib.check(
                fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), _lib.ptr(self.shift), n, D, C, _lib.ptr(self.gram), 1, 0,
                   None, 0, 0, 0, _lib.ptr(ws), nb, st),
                "sqfa_class_gram",
            )
            self.counts += counts[:C]
            self.n_rows += n
        return self

    def _recentre(self, X, perm, offsets, counts):
        """Move the shift to the class means of (rows so far + the incoming chunk) BEFORE the chunk is
        accumulated. Exact algebra: with m = s' - s the old state becomes G - m u^T - u m^T + n m m^T,
        u - n m. Done every time the number of rows grows 4x, so the shift stays within a few
        standard errors of the means whatever the first chunk looked like -- a shift far from the
        mean inflates the accumulated Gram by n d d^T and with it the fp32 rounding error."""
        ops = _cuda_ops(X.dtype)
        u_c = ops.class_sums_shifted(X, perm, offsets, self.shift, self.C)
        n_old = self.counts.to(torch.float32)[:, None]
        n_all = n_old + counts[: self.C].to(torch.float32)[:, None]
        m = torch.where(n_all > 0, (self.sums + u_c) / n_all.clamp_min(1.0), torch.zeros_like(self.sums))
        u = self.sums
        self.gram.addcmul_(m.unsqueeze(2), u.unsqueeze(1), value=-1.0)  # elementwise fp32, no temporaries
        self.gram.addcmul_(u.unsqueeze(2), m.unsqueeze(1), value=-1.0)
        self.gram.addcmul_((m * n_old).unsqueeze(2), m.unsqueeze(1), value=1.0)
        self.sums = (u - n_old * m).contiguous()
        self.shift = (self.shift + m).contiguous()
        self._rows_at_shift = self.n_rows + X.shape[0]

    def finalize(self, estimator="empirical"):
        """Statistics of all rows folded in so far (the state is left untouched: more chunks may follow)."""
        if estimator not in _ESTIMATORS:
            raise ValueError(f"estimator must be 'empirical' or 'oas', got {estimator!r}")
        if self.shift is None:
            raise RuntimeError("StreamingClassStatistics.finalize: no rows were folded in")
        lib, dev, C, D = self.lib, self.dev, self.C, self.D
        with torch.cuda.device(dev):
            counts, sums, gram = self.counts, self.sums, self.gram
            if self.group is not None:
                import torch.distributed as dist

                counts, sums, gram = counts.clone(), sums.clone(), gram.clone()
                for t in (counts, sums, gram):
                    dist.all_reduce(t, group=self.group)
            st = _lib.stream_ptr(dev)
            means = torch.empty(C, D, dtype=torch.float32, device=dev)
            _lib.check(
                lib.sqfa_class_means(_lib.ptr(sums), _lib.ptr(counts), _lib.ptr(self.shift), D, C, _lib.ptr(means), st),
                "sqfa_class_means",
            )
            cov = torch.empty(C, D, D, dtype=torch.float32, device=dev)
            sm = torch.empty(C, D, D, dtype=torch.float32, device=dev)
            nb = lib.sqfa_stats_epilogue_workspace_bytes(C)
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            _lib.check(
                lib.sqfa_stats_epilogue(_lib.ptr(gram), _lib.ptr(means), _lib.ptr(self.shift), _lib.ptr(counts), D, C,
                                        _ESTIMATORS[estimator], 1, _lib.ptr(cov), _lib.ptr(sm), _lib.ptr(ws), nb, st),
                "sqfa_stats_epilogue",
            )
        return {"means": means, "covariances": cov, "second_moments": sm}


def _single_class(points, estimator_id, assume_centered):
    dev = _lib.compute_device(points)
    X = _as_device_points(points, dev)
    n, D = X.shape
    with torch.cuda.device(dev):
        y = torch.zeros(n, dtype=torch.int64, device=dev)
        # the centring vector has the dtype of the statistics: float32 for bf16 / fp16 points
        centre = torch.zeros(1, D, dtype=torch.float64 if X.dtype == torch.float64 else torch.float32,
                             device=dev) if assume_centered else None
        _, cov, _, _ = run_class_statistics(
            _cuda_ops(X.dtype), X, y, estimator_id, n_classes=1, ddof=0 if assume_centered else 1, centre=centre,
            want_sm=False,
        )
    cov = cov[0]
    return cov if points.device == dev else cov.to(points.device)


def sample_covariance(points, assume_centered=False):
    """Sample covariance matrix of the given points (reference statistics.py:97-124)."""
    return _single_class(points, 0, assume_centered)


def oas_covariance(points, assume_centered=False):
    """OAS shrinkage covariance of the given points (reference statistics.py:57-94)."""
    return _single_class(points, 1, assume_centered)


def pca(points, n_components=None):
    """
    Principal components of the given points, shape (n_components, n_dim), descending variance
    (reference statistics.py:127-160). The D x D `eigh` is a one-off library call on the device.
    """
    n_points, n_dim = points.shape
    if n_components is None:
        n_components = min(n_points, n_dim)
    if n_components > n_dim:
        raise ValueError("n_components must be less than or equal to n_dim.")
    covariance = sample_covariance(points)
    dev = _lib.compute_device(covariance)
    _, components = torch.linalg.eigh(covariance.to(dev))
    components = components[:, -n_components:]
    components = torch.flip(components, dims=[1]).T
    return components.to(points.device)


def pca_from_scatter(scatters, n_components=None):
    """
    Principal components from class scatter matrices (reference statistics.py:163-192). As in the
    reference, the mean scatter matrix is handed to `pca` as if it were a point cloud.
    """
    n_classes, n_dim, _ = scatters.shape
    if n_components is None:
        n_components = n_dim
    if n_components > n_dim:
        raise ValueError("n_components must be less than or equal to n_dim.")
    average_scatter = torch.mean(scatters, dim=0)
    return pca(average_scatter, n_components=n_components)
