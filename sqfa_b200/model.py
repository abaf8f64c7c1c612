"""Supervised Quadratic Feature Analysis models -- B200-native drop-in for `sqfa.model`.

`SecondMomentsSQFA` and `SQFA` keep the constructor, method names, defaults, module state names
(`parametrizations.filters.original`, `noise_mat`) and error behaviour of the reference
(/root/reference/src/sqfa/model.py); `fit`, `fit_pca`, `transform`, `transform_scatters` and
`get_class_distances` dispatch to the sm_100a kernels. Models and data may live on the CPU: `fit`
moves the model to the CUDA device for the duration of the optimisation and back afterwards, and
every method returns results on the device of its inputs.
"""

import contextlib
import os

import torch
import torch.nn as nn
from torch.nn.utils.parametrizations import orthogonal
from torch.nn.utils.parametrize import is_parametrized as parametrize_is_parametrized
from torch.nn.utils.parametrize import register_parametrization, remove_parametrizations

from . import _lib, _ops, distances
from ._optim import fitting_loop
from .constraints import FixedFilters, Identity, Sphere
from .distances import affine_invariant, fisher_rao_lower_bound
from .linalg import conjugate_matrix
from .statistics import class_statistics, pca, pca_from_scatter

__all__ = ["SecondMomentsSQFA", "SQFA"]


def __dir__():
    return __all__


# built-in distance callables -> native distance selector (SecondMoments models: tensors in)
_TENSOR_DISTANCES = {
    distances.affine_invariant: _ops.DIST_AI,
    distances.affine_invariant_sq: _ops.DIST_AI | _ops.SQUARED,
    distances.log_euclidean: _ops.DIST_LE,
    distances.log_euclidean_sq: _ops.DIST_LE | _ops.SQUARED,
    distances.bures_wasserstein: _ops.DIST_BW,
    distances.bures_wasserstein_sq: _ops.DIST_BW | _ops.SQUARED,
}
# full models: dicts {"means", "covariances"} in
_DICT_DISTANCES = {
    distances.fisher_rao_lower_bound: _ops.DIST_FR,
    distances.fisher_rao_lower_bound_sq: _ops.DIST_FR | _ops.SQUARED,
    distances.wasserstein: _ops.DIST_W2,
    distances.wasserstein_sq: _ops.DIST_W2 | _ops.SQUARED,
    distances.mahalanobis: _ops.DIST_MAHA,
    distances.mahalanobis_sq: _ops.DIST_MAHA | _ops.SQUARED,
    distances.bhattacharyya: _ops.DIST_BHATT,
    distances.hellinger: _ops.DIST_HELL,
}
# fisher_rao_same_cov stays on the generic path on purpose: with the reference's closure its gradient is NaN
# (acosh' is infinite at the diagonal's x = 0, and 0 * inf = NaN), so those fits fail. A native closure
# that only touches the pairs i > j would turn such a fit into a working one.


_GRAPH_CLOSURE = os.environ.get("SQFA_GRAPH_CLOSURE", "1") != "0"


def _capture_graph(launch, device):
    """Capture one closure evaluation (8 kernel launches from one C call) into a CUDA graph; None if the
    capture is not possible here (the caller keeps launching directly)."""
    try:
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            launch()  # warm-up on the capture stream (sets per-kernel attributes outside the capture)
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        with torch.cuda.graph(graph, stream=side):
            launch()
        return graph
    except Exception:  # e.g. capture unsupported in this context
        torch.cuda.synchronize(device)
        return None


def _stats_to_scatter(statistics):
    """Scatter (second-moment) matrices from either input format (reference model.py:24-53):
    a dict gives covariances + mean outer products, a tensor is passed through."""
    if isinstance(statistics, dict):
        _check_statistics(statistics)
        means = statistics["means"]
        return statistics["covariances"] + torch.einsum("ni,nj->nij", means, means)
    return statistics


def _check_statistics(data_statistics, needs_dict=False):
    """Validate `data_statistics` (reference model.py:56-94): a dict needs the keys 'means' and
    'covariances' (ValueError otherwise); anything that is neither a dict nor tensor-like, or a
    tensor when a dict is required, is a TypeError."""
    if isinstance(data_statistics, dict):
        required_keys = {"means", "covariances"}
        missing_keys = required_keys - set(data_statistics.keys())
        if missing_keys:
            raise ValueError(
                f"`data_statistics` dictionary must contain the keys {required_keys}. "
                f"Missing keys: {missing_keys}"
            )
    elif not hasattr(data_statistics, "shape"):
        raise TypeError(
            "`data_statistics` must be either a dict with 'means' and 'covariances' "
            "or a torch.Tensor of shape (n_classes, n_dim, n_dim)."
        )
    elif needs_dict:
        raise TypeError(
            "`data_statistics` must be a dictionary with 'means' and 'covariances' "
            "when `needs_dict` is True."
        )


def _statistics_to(data_statistics, dev, dtype=torch.float32):
    """The statistics on the compute device in the model's dtype (no copy if already so). float32 models
    run the native closure; a model converted with `.double()` -- the reference's remedy for NaN / inf
    distances, _optim.py:28-30 -- keeps float64 statistics; its affine-invariant / Fisher-Rao closure and its
    Mahalanobis / Bhattacharyya / Hellinger closure are native (closure64.cu, gauss.cu) on one device, every
    other float64 closure uses float64 device-side library calls (SURVEY.md 8(f) row 3)."""

    def put(t):
        return t.detach().to(device=dev, dtype=dtype).contiguous()

    if isinstance(data_statistics, dict):
        return {k: put(v) for k, v in data_statistics.items() if isinstance(v, torch.Tensor)}
    return put(torch.as_tensor(data_statistics))


class _Transform(torch.autograd.Function):
    """Z = X F^T with the native skinny-GEMM kernel (reference model.py:236)."""

    @staticmethod
    def forward(ctx, F, X):
        Fc = _ops.f32c(F, X.device)
        ctx.save_for_backward(Fc, X)
        return _ops.transform_raw(X, Fc)

    @staticmethod
    def backward(ctx, gZ):
        Fc, X = ctx.saved_tensors
        dF = gZ.t() @ X.float() if ctx.needs_input_grad[0] else None  # bf16 / fp16 X: float32 like Z
        dX = (gZ @ Fc).to(X.dtype) if ctx.needs_input_grad[1] else None
        return dF, dX


class _PairwiseCurriculum:
    """`fit(pairwise=True)` (reference model.py:348-409): the filters are learned two at a time.
    Stage s optimises a model that holds the 2 s filters learned so far, frozen, followed by rows
    [2 s, 2 s + 2) of the initial filters; the noise buffer is resized with it. One object owns the
    swaps of parameter, constraint and buffer so that `fit` only sees a sequence of stages."""

    def __init__(self, model):
        n_filters = model.filters.shape[0]
        if n_filters % 2 != 0:
            raise ValueError("Number of filters must be even for pairwise training.")
        self.model = model
        self.n_stages = n_filters // 2
        self.start = model.filters.detach().clone()
        self.noise_level = model.noise_mat.detach()[0, 0].clone()
        self.loss, self.seconds = torch.tensor([]), torch.tensor([])

    @contextlib.contextmanager
    def stage(self, s):
        model, lo, hi = self.model, 2 * s, 2 * s + 2
        learned = model.filters.detach()[:lo].clone()
        model._install_filters(torch.cat((learned, self.start[lo:hi])).contiguous(), n_frozen=lo)
        model.register_buffer("noise_mat", self.noise_level * torch.eye(hi, device=self.start.device))
        try:
            yield
        finally:
            model._install_filters(model.filters.detach().clone())  # drops the freeze, keeps the constraint

    def log(self, stage_loss, stage_seconds):
        """Append a stage's per-epoch losses; its clock continues where the previous stage stopped."""
        offset = self.seconds[-1] if self.seconds.numel() > 0 else 0.0
        self.loss = torch.cat((self.loss, stage_loss))
        self.seconds = torch.cat((self.seconds, stage_seconds + offset))


class SecondMomentsSQFA(nn.Module):
    """
    Second-moments Supervised Quadratic Feature Analysis (SQFA) model: uses only the second
    moment matrices of the classes and distances in the SPD manifold.
    """

    def __init__(
        self,
        n_dim,
        feature_noise=0,
        n_filters=2,
        filters=None,
        distance_fun=None,
        constraint="sphere",
    ):
        """
        Parameters
        ----------
        n_dim : int
            Dimension of the input data space.
        feature_noise : float
            Diagonal term added to the feature covariances (regularisation). Default 0.
        n_filters : int
            Number of filters, used when `filters` is None (random initialisation). Default 2.
        filters : torch.Tensor
            Initial filters of shape (n_filters, n_dim). Default None.
        distance_fun : callable
            Takes two tensors (n_classes, n_filters, n_filters) and returns the (n_classes,
            n_classes) matrix of pairwise distances. Default: affine invariant distance.
        constraint : str
            'none', 'sphere' or 'orthogonal'. Default 'sphere'.
        """
        super().__init__()

        if filters is None:
            filters = torch.randn(n_filters, n_dim)
        else:
            filters = torch.as_tensor(filters, dtype=torch.float32)

        self.filters = nn.Parameter(filters)

        if self.filters.shape[0] > self.filters.shape[1]:
            raise ValueError("Number of filters must be less than or equal to the data dimension.")

        # built from the n_filters ARGUMENT, like the reference (model.py:159-161)
        feature_noise_mat = torch.as_tensor(feature_noise, dtype=torch.float32) * torch.eye(n_filters)
        self.register_buffer("noise_mat", feature_noise_mat)

        self.distance_fun = affine_invariant if distance_fun is None else distance_fun
        self.constraint = constraint
        self._add_constraint(constraint=self.constraint)
        self._process_group = None

    # ------------------------------------------------------------------ feature space maps
    def transform_scatters(self, data_scatters):
        """Feature-space scatter matrices F S_c F^T, shape (n_classes, n_filters, n_filters)
        (reference model.py:172-188). Native projection kernel, differentiable w.r.t. filters."""
        return conjugate_matrix(data_scatters, self.filters)

    def transform(self, data_points):
        """Project data points (n_samples, n_dim) to feature space (n_samples, n_filters)
        (reference model.py:222-237)."""
        dev = _lib.compute_device(data_points, self.filters)
        # float32, bf16 and fp16 points run the native kernel (Z is float32); float64 stays with torch
        if data_points.dim() != 2 or data_points.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            return torch.einsum("ij,nj->ni", self.filters.to(dev), data_points.to(dev)).to(data_points.device)
        with torch.cuda.device(dev):
            X = data_points.to(dev)
            if X.stride(1) != 1:
                X = X.contiguous()
            Z = _Transform.apply(self.filters.to(dev), X)
        return Z.to(data_points.device)

    def get_class_distances(self, data_statistics, regularized=False):
        """Pairwise distances (n_classes, n_classes) between the feature scatter matrices of the
        classes (reference model.py:190-220)."""
        data_scatters = _stats_to_scatter(data_statistics)
        feature_scatters = self.transform_scatters(data_scatters)
        if regularized:
            feature_scatters = feature_scatters + self.noise_mat.to(feature_scatters.device)[None, :, :]
        return self.distance_fun(feature_scatters, feature_scatters)

    # ------------------------------------------------------------------ fused closure
    def _noise_scalar(self):
        nm = self.noise_mat
        val = float(nm[0, 0]) if nm.numel() > 0 else 0.0
        if not torch.equal(nm, val * torch.eye(nm.shape[0], device=nm.device, dtype=nm.dtype)):
            return None  # not a multiple of the identity: use the generic path
        if nm.shape[0] != self.filters.shape[0]:
            raise RuntimeError(
                f"noise_mat is {tuple(nm.shape)} but the model has {self.filters.shape[0]} filters"
            )
        return val

    def _fused_inputs(self, data_statistics):
        """(S, M, dist) for the fused native loss, or None if distance_fun is not built in."""
        dist = _TENSOR_DISTANCES.get(self.distance_fun)
        if dist is None:
            return None
        return _stats_to_scatter(data_statistics).contiguous(), None, dist

    def _fused_loss_plan(self, data_statistics):
        """Callable evaluating [loss, #non-finite] natively at the current filters, or None."""
        if (not self.filters.is_cuda or self.filters.dtype != torch.float32
                or self.filters.shape[0] > _ops.MAX_FILTERS):
            return None
        plan = self._fused_inputs(data_statistics)
        noise = self._noise_scalar()
        if plan is None or noise is None:
            return None
        S, M, dist = plan
        if S.dtype != torch.float32 or (M is not None and M.dtype != torch.float32):
            return None
        group = self._process_group
        rank, world = 0, 1
        if group is not None:
            import torch.distributed as dist_mod

            rank, world = dist_mod.get_rank(group), dist_mod.get_world_size(group)
        C, D, k = S.shape[0], S.shape[1], self.filters.shape[0]
        p0, p1 = _ops.shard_pairs(C * (C - 1) // 2, C, rank, world)
        nbytes = _lib.load().sqfa_fused_loss_workspace_bytes(C, D, k, dist, p0, p1)
        ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=S.device)  # reused by every evaluation
        return lambda: _ops.FusedLoss.apply(self.filters, S, M, noise, dist, group, ws)

    def _fused_direct_plan(self, data_statistics):
        """Like `_fused_loss_plan`, without an autograd graph: the callable evaluates the loss at the
        current raw parameter, stores dLoss/d(raw parameter) in its `.grad` and returns the device
        vector [loss, #non-finite distances, max|grad|]. Available when every constraint on the
        filters has a closed-form adjoint (Sphere: (I - f f^T)/|w| per row; Identity; FixedFilters:
        zero rows) -- torch's `orthogonal` keeps the autograd path. Saves the ~15 micro-kernels and
        the autograd engine round trip per evaluation that dominate small-C fits. A float64 parameter with
        float64 statistics takes a float64 closure for the affine-invariant / Fisher-Rao distances and for the
        mean-covariance distances (Mahalanobis, Bhattacharyya, Hellinger), on one device or sharded over a
        process group like float32, and None otherwise."""
        if not parametrize_is_parametrized(self, "filters"):
            return None
        chain = list(self.parametrizations.filters)
        if any(type(m) not in (Sphere, Identity, FixedFilters) for m in chain):
            return None
        p = self.parametrizations.filters.original
        if not (p.is_cuda and p.dtype in (torch.float32, torch.float64)) or p.shape[0] > _ops.MAX_FILTERS:
            return None
        plan = self._fused_inputs(data_statistics)
        noise = self._noise_scalar()
        if plan is None or noise is None:
            return None
        S, M, dist = plan
        if S.dtype != p.dtype or (M is not None and M.dtype != p.dtype):
            return None
        f64 = p.dtype == torch.float64
        # float64 (a `.double()` model): the native closures cover affine-invariant / Fisher-Rao and the
        # mean-covariance distances
        gauss64 = f64 and (dist & 15) in (_ops.DIST_MAHA, _ops.DIST_BHATT, _ops.DIST_HELL)
        if f64 and (dist & 15) not in (_ops.DIST_AI, _ops.DIST_FR) and not gauss64:
            return None
        group = self._process_group
        k, D = p.shape
        C = S.shape[0]
        sphere = any(type(m) is Sphere for m in chain)
        n_fixed = max([m.n_row_fixed for m in chain if type(m) is FixedFilters], default=0)
        lib = _lib.load()

        if group is not None:
            # pair list sharded over the ranks: [loss, flag, -, dF] of this rank's pairs, ONE all-reduce,
            # then the (linear) constraint adjoint on every rank
            import torch.distributed as dist_mod

            rank, world = dist_mod.get_rank(group), dist_mod.get_world_size(group)
            p0, p1 = _ops.shard_pairs(C * (C - 1) // 2, C, rank, world)
            nbytes = (_ops.closure_workspace_bytes_f64(C, D, k, dist, p0, p1) if f64
                      else lib.sqfa_fused_loss_workspace_bytes(C, D, k, dist, p0, p1))
            ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=S.device)
            # AI / FR with at least one class per rank: the projection shards with the classes as well
            # (three small all-reduces per evaluation instead of one; SQFA_SHARD_CLASSES=0: pairs only)
            shard_classes = ((dist & 15) != _ops.DIST_LE and C >= world
                             and os.environ.get("SQFA_SHARD_CLASSES", "1") == "1")
            if f64:
                # the float64 closures read the noise from the device
                noise_arg = torch.full((1,), noise, dtype=torch.float64, device=S.device)
                eval_sharded = _ops.fused_loss_sharded_f64_raw if shard_classes else _ops.fused_loss_f64_raw
            else:
                noise_arg = noise
                eval_sharded = _ops.fused_loss_sharded_raw if shard_classes else _ops.fused_loss_raw

            @torch.no_grad()
            def run_sharded():
                W = p.detach()
                if sphere:
                    nrm = W.norm(dim=-1, keepdim=True)
                    F = W / nrm
                else:
                    F = W
                packed = eval_sharded(F, S, M, noise_arg, dist, group, ws)
                dF = packed[4:].view(k, D)
                if n_fixed:
                    dF[:n_fixed] = 0.0  # frozen rows are detached in FixedFilters.forward
                dW = (dF - (dF * F).sum(dim=-1, keepdim=True) * F) / nrm if sphere else dF
                p.grad = dW
                return torch.cat([packed[:2], dW.abs().max().view(1)])

            run_sharded.dtype = p.dtype  # a float64 fit hands its loss to the optimiser in float64
            return run_sharded

        # single device: ONE native call per evaluation (constraint and its adjoint included), all
        # buffers static, captured in a CUDA graph after the first evaluations
        P = C * (C - 1) // 2
        if gauss64:
            ws_query, eval_f64 = lib.sqfa_gauss_closure_workspace_bytes_f64, _ops.gauss_closure_eval_f64_raw
        elif f64:
            ws_query, eval_f64 = lib.sqfa_fused_loss_workspace_bytes_f64, _ops.closure_eval_f64_raw
        else:
            ws_query = lib.sqfa_fused_loss_workspace_bytes
        ws_bytes = ws_query(C, D, k, dist, 0, P)
        ws = torch.empty(max(int(ws_bytes), 1), dtype=torch.uint8, device=S.device)
        out = torch.zeros(_ops.N_OUT, dtype=p.dtype, device=S.device)
        out_host = torch.zeros(_ops.N_OUT, dtype=p.dtype).pin_memory()  # mirror, filled by every evaluation
        grad = torch.zeros(k, D, dtype=p.dtype, device=S.device)
        state = {"calls": 0, "graph": None, "param_ptr": None}
        if f64:
            noise_dev = torch.full((1,), noise, dtype=torch.float64, device=S.device)

            def launch():
                eval_f64(p.detach(), S, M, noise_dev, dist, sphere, n_fixed, out, grad, ws, out_host)
        else:
            def launch():
                _ops.closure_eval_raw(p.detach(), S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host)

        @torch.no_grad()
        def enqueue():
            """One evaluation enqueued on the current stream, no host wait: the result lands in `out`
            (device) and `host_out` (pinned host memory, valid once the stream has been waited for)."""
            if not p.is_contiguous():
                raise RuntimeError("filter parameter must be contiguous")
            state["calls"] += 1
            if state["graph"] is not None and state["param_ptr"] == p.data_ptr():
                state["graph"].replay()
            else:
                launch()
                if state["calls"] == 2 and _GRAPH_CLOSURE and state["graph"] is None:
                    state["graph"], state["param_ptr"] = _capture_graph(launch, S.device), p.data_ptr()
            p.grad = grad  # static buffer: the optimiser reads it before the next evaluation overwrites it

        def run():
            enqueue()
            return out

        run.enqueue, run.host_out, run.dtype = enqueue, out_host, p.dtype
        return run

    # ------------------------------------------------------------------ training
    def fit_pca(self, X=None, data_statistics=None):
        """Set the filters to the leading principal components of the data (or of the mean
        scatter matrix, with the reference's `pca_from_scatter` semantics); reference
        model.py:239-268."""
        if X is None and data_statistics is None:
            raise ValueError("Either X or data_statistics must be provided.")

        n_components = self.filters.shape[0]
        if data_statistics is None:
            pca_filters = pca(X, n_components)
        else:
            pca_filters = pca_from_scatter(_stats_to_scatter(data_statistics), n_components)

        device = self.filters.device
        self._install_filters(pca_filters.detach().to(device=device, dtype=self.filters.dtype).contiguous())

    def fit(
        self,
        X=None,
        y=None,
        data_statistics=None,
        max_epochs=300,
        lr=0.1,
        estimator="empirical",
        pairwise=False,
        show_progress=True,
        return_loss=False,
        atol=1e-6,
        process_group=None,
        **kwargs,
    ):
        """
        Fit the model with the LBFGS optimizer (reference model.py:270-414).

        Parameters are those of the reference; `process_group` (optional, extension) shards the
        class-pair list of every loss evaluation over the ranks of a torch.distributed group.
        Extra keyword arguments go to `torch.optim.LBFGS`.
        """
        if data_statistics is None:
            if X is None or y is None:
                raise ValueError("Either data_statistics or X and y must be provided.")
            data_statistics = class_statistics(X, y, estimator=estimator, keep_on_device=True)

        _check_statistics(data_statistics)

        dev = _lib.compute_device(
            *(data_statistics.values() if isinstance(data_statistics, dict) else [data_statistics])
        )
        home = self.filters.device
        self._process_group = process_group
        self._last_fit_evaluations = 0
        with torch.cuda.device(dev):
            stats_dev = _statistics_to(data_statistics, dev, self.filters.dtype)
            self.to(dev)
            try:
                loss, training_time = self._fit_on_device(
                    stats_dev, max_epochs, lr, pairwise, show_progress, atol, **kwargs
                )
            finally:
                self._process_group = None
                self.to(home)

        if return_loss:
            return loss, training_time
        return None

    def _fit_on_device(self, data_statistics, max_epochs, lr, pairwise, show_progress, atol, **kwargs):
        def run_optimiser():
            return fitting_loop(
                model=self, data_statistics=data_statistics, max_epochs=max_epochs, lr=lr,
                show_progress=show_progress, return_loss=True, atol=atol, **kwargs,
            )

        if not pairwise:
            return run_optimiser()
        curriculum = _PairwiseCurriculum(self)
        for stage in range(curriculum.n_stages):
            with curriculum.stage(stage):
                curriculum.log(*run_optimiser())
        return curriculum.loss, curriculum.seconds

    def _install_filters(self, value, n_frozen=0):
        """Make `value` (k, n_dim) the raw filter parameter under the model's constraint; the first
        `n_frozen` rows receive no gradient (FixedFilters stacked on top of the constraint)."""
        if parametrize_is_parametrized(self, "filters"):
            remove_parametrizations(self, "filters")
        self.filters = nn.Parameter(value)
        self._add_constraint(constraint=self.constraint)
        if n_frozen > 0:
            register_parametrization(self, "filters", FixedFilters(n_row_fixed=n_frozen))

    def _add_constraint(self, constraint="none"):
        """Register the filter parametrization: 'none', 'sphere' or 'orthogonal'
        (reference model.py:416-431)."""
        if constraint == "none":
            register_parametrization(self, "filters", Identity())
        elif constraint == "sphere":
            register_parametrization(self, "filters", Sphere())
        elif constraint == "orthogonal":
            orthogonal(self, "filters")

    def __dir__(self):
        return [
            "filters",
            "noise_mat",
            "distance_fun",
            "constraint",
            "transform_scatters",
            "get_class_distances",
            "transform",
            "fit_pca",
        ]


class SQFA(SecondMomentsSQFA):
    """
    Supervised Quadratic Feature Analysis (SQFA) model: uses the class means and covariances and
    distances (or bounds) in the manifold of normal distributions.
    """

    def __init__(
        self,
        n_dim,
        feature_noise=0,
        n_filters=2,
        filters=None,
        distance_fun=None,
        constraint="sphere",
    ):
        """Same parameters as `SecondMomentsSQFA`; `distance_fun` takes two dicts with 'means'
        (n_classes, n_filters) and 'covariances' (n_classes, n_filters, n_filters). Default: the
        Calvo-Oller lower bound of the Fisher-Rao distance."""
        if distance_fun is None:
            distance_fun = fisher_rao_lower_bound
        super().__init__(
            n_dim=n_dim,
            feature_noise=feature_noise,
            n_filters=n_filters,
            filters=filters,
            distance_fun=distance_fun,
            constraint=constraint,
        )

    def get_class_distances(self, data_statistics, regularized=False):
        """Pairwise distances between the feature-space class Gaussians (reference
        model.py:508-546). `data_statistics` must be a dict with 'means' and 'covariances'."""
        if not isinstance(data_statistics, dict):
            raise TypeError("data_statistics must be a dictionary with 'means' and 'covariances' keys.")
        means, covs = data_statistics["means"], data_statistics["covariances"]
        native = (
            covs.dim() == 3 and covs.dtype == torch.float32 and means.dtype == torch.float32
            and self.filters.shape[0] <= _ops.MAX_FILTERS
        )
        if native:
            # one pass over the covariances gives both F S F^T and F m
            dev = _lib.compute_device(covs, means, self.filters)
            with torch.cuda.device(dev):
                feature_covariances, feature_means = _ops.Project.apply(
                    self.filters.to(dev), covs.to(dev).contiguous(), means.to(dev).contiguous()
                )
            feature_covariances = feature_covariances.to(covs.device)
            feature_means = feature_means.to(means.device)
        else:
            feature_means = self.transform(means)
            feature_covariances = self.transform_scatters(covs)

        if regularized:
            feature_covariances = feature_covariances + self.noise_mat.to(feature_covariances.device)[None, :, :]

        feature_statistics = {"means": feature_means, "covariances": feature_covariances}
        return self.distance_fun(feature_statistics, feature_statistics)

    def _fused_inputs(self, data_statistics):
        dist = _DICT_DISTANCES.get(self.distance_fun)
        if dist is None or not isinstance(data_statistics, dict):
            return None
        return data_statistics["covariances"].contiguous(), data_statistics["means"].contiguous(), dist

    def fit(
        self,
        X=None,
        y=None,
        data_statistics=None,
        max_epochs=300,
        lr=0.1,
        estimator="empirical",
        pairwise=False,
        show_progress=True,
        return_loss=False,
        atol=1e-6,
        process_group=None,
        **kwargs,
    ):
        """Fit the SQFA model with the LBFGS optimizer (reference model.py:548-630);
        `data_statistics`, when given, must be a dict with 'means' and 'covariances'."""
        if data_statistics is None:
            if X is None or y is None:
                raise ValueError("Either data_statistics or X and y must be provided.")
            data_statistics = class_statistics(X, y, estimator=estimator, keep_on_device=True)
        else:
            _check_statistics(data_statistics, needs_dict=True)

        loss, training_time = super().fit(
            X=None,
            y=None,
            data_statistics=data_statistics,
            max_epochs=max_epochs,
            lr=lr,
            estimator=estimator,
            pairwise=pairwise,
            show_progress=show_progress,
            return_loss=True,
            atol=atol,
            process_group=process_group,
            **kwargs,
        )
        if return_loss:
            return loss, training_time
        return None
