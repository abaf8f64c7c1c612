"""CPU: the float64 device L-BFGS direction update -- its C ABI (size query, argument validation before any
launch) and the host optimiser's fall-through for a float64 CPU parameter."""

import ctypes

import pytest
import torch

BENCH_KD = {"c1": 3136, "c2": 24576, "c3": 832, "c4": 8192, "c5": 32768}  # k * D of the benchmark shapes


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from sqfa_b200 import _lib

    return _lib.load()


def test_prototypes_are_bound(lib):
    from sqfa_b200 import _lib
    from test_abi import header_prototypes

    for name in ("sqfa_lbfgs_max_n_f64", "sqfa_lbfgs_direction_f64"):
        assert name in _lib.SIGNATURES and hasattr(lib, name) and name not in lib.sqfa_missing_symbols
    args = header_prototypes()["sqfa_lbfgs_direction_f64"][1]
    assert len(args) == 15
    assert all(t.endswith("*") for t in args if "double" in t)  # no double by value: ctypes has no c_double here


def test_max_n_covers_every_benchmark_shape(lib):
    assert lib.sqfa_lbfgs_max_n_f64() >= 65536
    assert lib.sqfa_lbfgs_max_n_f64() >= max(BENCH_KD.values())
    assert lib.sqfa_lbfgs_max_n_f64() <= lib.sqfa_lbfgs_max_n()  # a double takes two registers


def test_argument_validation_without_a_launch(lib):
    """Every rejection happens before anything touches the device (the pointers below are not device memory)."""
    fake = ctypes.c_void_p(4096)
    scalars = (ctypes.c_double * 3)(0.0, 1.0, 1e-9)
    max_n, max_hist = lib.sqfa_lbfgs_max_n_f64(), lib.sqfa_lbfgs_max_history()

    def call(n=1000, history=10, scalars=scalars, **ptrs):
        p = {k: ptrs.get(k, fake) for k in ("g", "prev_g", "d", "S", "Y", "ro", "hdiag", "meta", "param", "out")}
        return lib.sqfa_lbfgs_direction_f64(p["g"], p["prev_g"], p["d"], p["S"], p["Y"], p["ro"], p["hdiag"],
                                            p["meta"], n, history, scalars, 0, p["param"], p["out"], None)

    for name in ("g", "prev_g", "d", "S", "Y", "ro", "hdiag", "meta", "out"):
        lib.sqfa_last_error()
        assert call(**{name: None}) == -1, name
        assert b"sqfa_lbfgs_direction_f64" in lib.sqfa_last_error() and b"bad argument" in lib.sqfa_last_error()
    assert call(scalars=None) == -1 and b"bad argument" in lib.sqfa_last_error()
    for n, history in ((0, 10), (-5, 10), (1000, 0), (1000, -1)):
        assert call(n=n, history=history) == -1, (n, history)
        assert b"bad argument" in lib.sqfa_last_error()
    for n, history in ((max_n + 1, 10), (1000, max_hist + 1)):
        assert call(n=n, history=history) == -3, (n, history)
        msg = lib.sqfa_last_error()
        assert b"sqfa_lbfgs_direction_f64" in msg and b"too large" in msg


def test_float64_cpu_parameter_is_torch_lbfgs():
    """A float64 CPU parameter takes torch.optim.LBFGS.step: the same iterates and no device state."""
    from sqfa_b200._lbfgs import LBFGS

    def run(cls, **kw):
        torch.manual_seed(0)
        x = torch.nn.Parameter(torch.randn(50, dtype=torch.float64))
        A = torch.diag(torch.linspace(0.5, 5.0, 50, dtype=torch.float64))
        opt = cls([x], lr=0.5, history_size=6, **kw)

        def closure():
            opt.zero_grad()
            loss = 0.5 * x @ A @ x - x.sum()
            loss.backward()
            return loss

        losses = [opt.step(closure).item() for _ in range(3)]
        return x.detach().clone(), losses, opt.state[opt._params[0]]

    for kw in ({}, {"line_search_fn": "strong_wolfe"}):
        x_ref, l_ref, st_ref = run(torch.optim.LBFGS, **kw)
        x_got, l_got, state = run(LBFGS, **kw)
        assert torch.equal(x_ref, x_got) and l_ref == l_got
        assert "sqfa_native" not in state
        assert state["n_iter"] == st_ref["n_iter"] and state["func_evals"] == st_ref["func_evals"]
