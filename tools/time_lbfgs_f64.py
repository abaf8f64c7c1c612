"""The float64 device L-BFGS (sqfa_lbfgs_direction_f64) on one GPU and in ONE process.

1. The direction kernel alone, float32 against float64 (alternated), at n = 3 136, 24 576, 32 768 and 65 536 with
   a full history of 100 pairs: device events over enough launches for a window of at least a second.
2. Fits of `.double()` SQFA models (Fisher-Rao lower bound and Mahalanobis) at c1, c2, c3 and the c5 shape in
   epochs/s, the device L-BFGS (pipelined behind the native float64 closure) against `torch.optim.LBFGS`,
   alternated, from unit-norm random filters. Tolerances 0, so every epoch runs its 20 iterations; 5 warm-up
   epochs fill the history, the next 10 are timed. Also recorded: the pair count at the end, the first-epoch loss of each optimiser, and the closure's
   graph-replay time, so that the optimiser's cost per iteration is epoch time / 20 - closure.
Card name, power limit and maximum SM clock are read in the same run.

Usage: python tools/time_lbfgs_f64.py --out DIR [--shapes c1,c2,c3,c5] [--rounds 2]
Writes DIR/lbfgs_f64.json."""

import argparse
import ctypes
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_bures_wasserstein import SHAPES, card, time_calls  # noqa: E402

KERNEL_N = (3136, 24576, 32768, 65536)
HISTORY = 100
ITERS = 20          # torch.optim.LBFGS's default max_iter: evaluations and direction updates per epoch
WARM_EPOCHS, TIMED_EPOCHS = 5, 10


def time_direction(dtype, n, dev, window_s=1.0):
    """Mean time of one direction update at a full history (device events), and the number of launches."""
    from sqfa_b200 import _lib

    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(n)
    rnd = lambda *shape: torch.randn(*shape, device=dev, generator=g, dtype=dtype)  # noqa: E731
    grad, prev_g, d = rnd(n), rnd(n), rnd(n)
    S, Y = rnd(HISTORY + 1, n), rnd(HISTORY + 1, n)
    ro = torch.rand(HISTORY + 1, device=dev, generator=g, dtype=dtype) + 0.5
    hdiag = torch.ones(1, device=dev, dtype=dtype)
    meta = torch.tensor([0, HISTORY], dtype=torch.int32, device=dev)  # a full ring
    out = torch.zeros(8, device=dev, dtype=dtype)
    bufs = (_lib.ptr(grad), _lib.ptr(prev_g), _lib.ptr(d), _lib.ptr(S), _lib.ptr(Y), _lib.ptr(ro), _lib.ptr(hdiag),
            _lib.ptr(meta), n, HISTORY)
    stream = _lib.stream_ptr(dev)
    scalars = (ctypes.c_double * 3)(0.1, 0.1, 0.0)

    def launch():
        # after the first launch prev_g = g, so y = 0 and no pair is pushed: every launch walks all 100 pairs
        if dtype == torch.float64:
            code = lib.sqfa_lbfgs_direction_f64(*bufs, scalars, 0, None, _lib.ptr(out), stream)
        else:
            code = lib.sqfa_lbfgs_direction(*bufs, 0.1, 0, None, 0.1, 0.0, _lib.ptr(out), stream)
        _lib.check(code, "direction")

    ms, _ = time_calls(launch, 20)
    reps = max(int(math.ceil(window_s * 1e3 / ms)), 20)
    ms, _ = time_calls(launch, reps)
    assert int(meta[1]) == HISTORY
    return ms, reps


def make_stats(C, D, dev, rank=48):
    """Well-separated float64 classes (low rank plus diagonal covariances with a scale per class, and means of
    norm ~1), as in the tests' `gauss_stats`: the fit keeps moving for hundreds of iterations, so the L-BFGS
    history fills (a pair is kept only when y.s > 1e-10)."""
    g = torch.Generator(device=dev).manual_seed(C + D)
    G = torch.randn(C, D, rank, device=dev, generator=g, dtype=torch.float64) / rank**0.5
    scale = 0.5 + 1.5 * torch.rand(C, 1, 1, device=dev, generator=g, dtype=torch.float64)
    cov = scale * (G @ G.transpose(1, 2)) + 0.05 * torch.eye(D, device=dev, dtype=torch.float64)
    means = 1.2 * torch.randn(C, D, device=dev, generator=g, dtype=torch.float64) / D**0.5
    return {"means": means, "covariances": cov.contiguous()}


def model(name, D, k, dev):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA

    torch.manual_seed(0)
    F0 = torch.randn(k, D)
    F0 = F0 / F0.norm(dim=1, keepdim=True)  # unit rows, as a PCA start has: with raw rows of norm ~sqrt(D) the
    # gradient is sqrt(D) times smaller, y.s stays below 1e-10 and the history never fills
    return SQFA(n_dim=D, feature_noise=0.01, n_filters=k, filters=F0,
                distance_fun=getattr(Dn, name)).to(dev).double()


def fit(name, D, k, dev, stats, optimiser):
    """One fit of WARM_EPOCHS + TIMED_EPOCHS epochs with `optimiser` as the fitting loop's L-BFGS."""
    import sqfa_b200._optim as optim_mod

    seen = {}

    class Recording(optimiser):
        def step(self, closure):
            seen["opt"] = self
            loss = super().step(closure)
            seen.setdefault("losses", []).append(float(loss))
            return loss

    saved = optim_mod.LBFGS
    optim_mod.LBFGS = Recording
    try:
        m = model(name, D, k, dev)
        assert m._fused_direct_plan(stats) is not None
        _, seconds = m.fit(data_statistics=stats, max_epochs=WARM_EPOCHS + TIMED_EPOCHS, show_progress=False,
                           atol=0.0, return_loss=True, tolerance_grad=0.0, tolerance_change=0.0)
    finally:
        optim_mod.LBFGS = saved
    opt = seen["opt"]
    state = opt.state[opt._params[0]]
    native = "sqfa_native" in state
    pairs = int(state["sqfa_native"]["meta"][1]) if native else len(state["old_dirs"])
    timed = float(seconds[-1] - seconds[WARM_EPOCHS - 1])  # each epoch ends in a host read of its loss
    return {"native": native, "epochs_per_s": TIMED_EPOCHS / timed, "epoch_ms": timed / TIMED_EPOCHS * 1e3,
            "pairs": pairs, "n_iter": int(state["n_iter"]), "first_epoch_loss": seen["losses"][0],
            "last_loss": seen["losses"][-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default="c1,c2,c3,c5", help="fit shapes (comma separated, may be empty)")
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the two arms")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from sqfa_b200._lbfgs import LBFGS

    dev = torch.device("cuda")
    res = {"card": card(), "history": HISTORY, "kernel_us": {}, "fits": {}}
    for n in KERNEL_N:
        row = {}
        for _ in range(args.rounds):
            for arm, dtype in (("float32", torch.float32), ("float64", torch.float64)):
                ms, reps = time_direction(dtype, n, dev)
                row.setdefault(arm, []).append(ms * 1e3)
                row[f"{arm}_launches"] = reps
        res["kernel_us"][str(n)] = row
        print("direction n", n, row, flush=True)

    for cfg in [c for c in args.shapes.split(",") if c]:
        C, D, k = SHAPES[cfg]
        stats = make_stats(C, D, dev)
        for name in ("fisher_rao_lower_bound", "mahalanobis"):
            key = f"{cfg}_{name}"
            row = {"C": C, "D": D, "k": k, "n": k * D}
            plan = model(name, D, k, dev)._fused_direct_plan(stats)
            row["closure_ms"] = time_calls(plan, 200 if C * D < 50000 else 50)[0]
            del plan
            for _ in range(args.rounds):
                for arm, cls in (("device", LBFGS), ("torch", torch.optim.LBFGS)):
                    try:
                        r = fit(name, D, k, dev, stats, cls)
                    except Exception as e:  # recorded, not hidden
                        r = {"error": f"{type(e).__name__}: {e}"[:2000]}
                    row.setdefault(arm, []).append(r)
            for arm in ("device", "torch"):
                ok = [r for r in row[arm] if "error" not in r]
                if ok:
                    best = min(r["epoch_ms"] for r in ok)
                    row[f"{arm}_optimiser_ms_per_iter"] = [r["epoch_ms"] / ITERS - row["closure_ms"] for r in ok]
                    row[f"{arm}_best_epochs_per_s"] = 1e3 / best
            res["fits"][key] = row
            print("fit", key, json.dumps(row), flush=True)
            torch.cuda.empty_cache()
        del stats
        torch.cuda.empty_cache()

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "lbfgs_f64.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
