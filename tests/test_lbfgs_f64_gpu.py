"""GPU: the float64 device L-BFGS direction update against torch.optim.LBFGS in float64 -- on a quadratic, through
the fall-through configurations, in fits on the native float64 closures and on a composed float64 closure, and
pipelined against waited iterations. Both optimisers do the same arithmetic in the same order; only the summation
order inside each dot product differs, which a short float64 run keeps far below the bounds used here."""

import pytest
import torch

from test_bures_wasserstein_gpu import gauss_stats
from test_float64_closure_gpu import _model, _stats_for

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-10     # relative, loss per epoch of a fit
FILTER_TOL = 1e-8    # relative Frobenius norm of the fitted filters
QUAD_TOL = 1e-12     # relative, iterates and losses on the quadratic


def _filters(k, D, seed):
    """Unit-norm initial rows, as a PCA start has. From rows of norm ~sqrt(D) the gradient is sqrt(D) times
    smaller and y.s stays below 1e-10 for many iterations: no pair would enter the history."""
    F = torch.randn(k, D, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    return F / F.norm(dim=1, keepdim=True)


def _quadratic(n, seed):
    """The quadratic of test_lbfgs_gpu.py (condition number ~3000), in float64."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    diag = torch.exp(torch.empty(n, device="cuda", dtype=torch.float64).uniform_(-4.0, 4.0, generator=g))
    U = torch.randn(n, 8, generator=g, device="cuda", dtype=torch.float64) / n**0.5
    b = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)

    def f(x):  # 0.5 x^T (diag + U U^T) x - b^T x
        return 0.5 * (x * diag * x).sum() + 0.5 * ((x @ U) ** 2).sum() - (b * x).sum()

    return f


def _run(opt_cls, f, n, steps, **kw):
    x = torch.nn.Parameter(torch.zeros(n, device="cuda", dtype=torch.float64))
    opt = opt_cls([x], **kw)
    losses = []

    def closure():
        opt.zero_grad()
        loss = f(x)
        loss.backward()
        return loss

    for _ in range(steps):
        losses.append(float(opt.step(closure)))
    return x.detach().clone(), losses, opt


@pytest.mark.parametrize("n,hist", [(3000, 5), (20000, 100), (65536, 7)])
def test_direction_update_matches_torch_lbfgs(n, hist):
    from sqfa_b200._lbfgs import LBFGS

    f = _quadratic(n, n)
    kw = dict(lr=0.3, history_size=hist, max_iter=12)
    x_ref, l_ref, opt_ref = _run(torch.optim.LBFGS, f, n, 3, **kw)
    x_got, l_got, opt = _run(LBFGS, f, n, 3, **kw)
    st, st_ref = opt.state[opt._params[0]], opt_ref.state[opt_ref._params[0]]
    assert "sqfa_native" in st, "the native path was not taken"
    assert st["sqfa_native"]["S"].dtype == torch.float64
    assert st["n_iter"] == st_ref["n_iter"] == 36 and st["func_evals"] == st_ref["func_evals"]
    assert float((x_got - x_ref).norm() / x_ref.norm()) <= QUAD_TOL
    for a, b in zip(l_got, l_ref):
        assert abs(a - b) <= QUAD_TOL * abs(b), (a, b)
    assert int(st["sqfa_native"]["meta"][1]) == len(st_ref["old_dirs"]) == min(hist, 35)  # the ring wrapped


@pytest.mark.parametrize("case", ["too_long", "strong_wolfe", "history"])
def test_unsupported_configurations_fall_back_to_torch(case):
    from sqfa_b200 import _lib
    from sqfa_b200._lbfgs import LBFGS

    lib = _lib.load()
    n = lib.sqfa_lbfgs_max_n_f64() + 1 if case == "too_long" else 500
    kw = {"lr": 0.3, "max_iter": 6}
    if case == "strong_wolfe":
        kw.update(lr=1.0, line_search_fn="strong_wolfe")
    if case == "history":
        kw.update(history_size=lib.sqfa_lbfgs_max_history() + 1)
    f = _quadratic(n, 1)
    x_ref, l_ref, _ = _run(torch.optim.LBFGS, f, n, 2, **kw)
    x_got, l_got, opt = _run(LBFGS, f, n, 2, **kw)
    assert "sqfa_native" not in opt.state[opt._params[0]]
    assert torch.equal(x_ref, x_got) and l_ref == l_got


def _fit(monkeypatch, base, make, sc, epochs=3, **kw):
    """Fit with `base` as the fitting loop's optimiser; the loss of every epoch in float64 (the fitting loop
    returns its history in float32), the filters and the optimiser's state."""
    import sqfa_b200._optim as optim_mod

    record = {"losses": []}

    class Recording(base):
        def step(self, closure):
            record["opt"] = self
            loss = super().step(closure)
            record["losses"].append(float(loss))
            return loss

    monkeypatch.setattr(optim_mod, "LBFGS", Recording)
    model = make()
    model.fit(data_statistics=sc, max_epochs=epochs, atol=0.0, show_progress=False, **kw)
    opt = record["opt"]
    return torch.tensor(record["losses"], dtype=torch.float64), model.filters.detach().clone(), opt.state[opt._params[0]]


def _compare_with_torch(monkeypatch, make, sc, pairs_pushed=True, **kw):
    from sqfa_b200._lbfgs import LBFGS

    runs = [_fit(monkeypatch, LBFGS, make, sc, max_iter=8, **kw) for _ in range(2)]
    l_ref, F_ref, st_ref = _fit(monkeypatch, torch.optim.LBFGS, make, sc, max_iter=8, **kw)
    (l_got, F_got, st), (l_again, F_again, _) = runs
    assert "sqfa_native" in st and "sqfa_native" not in st_ref
    assert F_got.dtype == torch.float64
    assert torch.equal(l_got, l_again) and torch.equal(F_got, F_again)  # two device runs: the same bits
    assert st["n_iter"] == st_ref["n_iter"] and st["func_evals"] == st_ref["func_evals"]
    assert int(st["sqfa_native"]["meta"][1]) == len(st_ref["old_dirs"])
    assert (len(st_ref["old_dirs"]) > 0) == pairs_pushed  # whether the two-loop recursion ran
    assert float(((l_got - l_ref).abs() / l_ref.abs()).max()) <= LOSS_TOL, (l_got, l_ref)
    assert float((F_got - F_ref).norm() / F_ref.norm()) <= FILTER_TOL


NATIVE_FITS = {
    "fr_small": ("full", "fisher_rao_lower_bound", 8, 40, 4),
    "ai_small": ("second_moments", "affine_invariant", 9, 48, 5),
    "maha_small": ("full", "mahalanobis", 8, 40, 4),
    "fr_c5": ("full", "fisher_rao_lower_bound", 100, 1024, 32),
    "ai_c5": ("second_moments", "affine_invariant", 100, 1024, 32),
    "maha_c5": ("full", "mahalanobis", 100, 1024, 32),
}


@pytest.mark.parametrize("case", list(NATIVE_FITS))
def test_fit_on_native_float64_closure_matches_torch_lbfgs(monkeypatch, case):
    """A `.double()` model on a native float64 closure: the device optimiser (pipelined with the closure) against
    torch.optim.LBFGS. The c5 shape has k D = 32 768, 4 elements per thread."""
    kind, distance, C, D, k = NATIVE_FITS[case]
    stats = gauss_stats(C, D, seed=C + k)
    sc = _stats_for(kind, stats)
    F0 = _filters(k, D, 11)

    def make():
        model = _model(kind, distance, D, k, F0)
        assert model._fused_direct_plan(sc) is not None
        return model

    # the c5 Mahalanobis fit keeps y.s below 1e-10 for its first 24 iterations: no pair enters the history
    _compare_with_torch(monkeypatch, make, sc, pairs_pushed=case != "maha_c5")


def test_fit_on_composed_float64_closure_matches_torch_lbfgs(monkeypatch):
    """`.double()` log-Euclidean keeps the composed closure; its float64 parameter still takes the device
    direction update, without the pipeline."""
    C, D, k = 6, 32, 3
    stats = gauss_stats(C, D, seed=4)
    sc = _stats_for("second_moments", stats)
    F0 = _filters(k, D, 6)

    def make():
        model = _model("second_moments", "log_euclidean", D, k, F0)
        assert model._fused_direct_plan(sc) is None
        return model

    _compare_with_torch(monkeypatch, make, sc)


def test_pipelined_iterations_equal_waited_ones(monkeypatch):
    """With SQFA_LBFGS_PIPELINE=1 the float64 evaluation at the new iterate is enqueued behind the direction
    kernel and each iteration waits once; with 0 it waits after each kernel. Same kernels on the same data in the
    same order: identical losses, filters and evaluation counts, in a fixed-length fit and in one that converges
    inside an epoch."""
    C, D, k = 15, 64, 5
    stats = gauss_stats(C, D, seed=21)
    sc = _stats_for("full", stats)
    F0 = _filters(k, D, 2)
    for fit_kw in ({"max_epochs": 4, "atol": 0.0, "max_iter": 9},
                   {"max_epochs": 40, "atol": 1e-9, "tolerance_change": 1e-9, "tolerance_grad": 1e-6}):
        runs = []
        for pipe in ("1", "0"):
            monkeypatch.setenv("SQFA_LBFGS_PIPELINE", pipe)
            model = _model("full", "fisher_rao_lower_bound", D, k, F0)
            assert model._fused_direct_plan(sc) is not None
            loss, _ = model.fit(data_statistics=sc, show_progress=False, return_loss=True, **fit_kw)
            runs.append((loss, model.filters.detach().clone(), model._last_fit_evaluations))
        assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
        assert runs[0][2] == runs[1][2]
