"""Fitting closures of the mean-covariance distances (Mahalanobis, squared Mahalanobis, Bhattacharyya,
Hellinger) on one GPU, in ONE process: the native closure evaluation (CUDA-graph replay of
`_fused_direct_plan`) against the generic path the same distance takes when wrapped in a lambda
(`get_class_distances` on all C^2 pairs, the NaN/inf check, -mean(tril), autograd backward), at the closure
shapes c1-c4 and the c5 shape (C = 100, D = 1024, k = 32), next to the affine-invariant closure of
SecondMomentsSQFA at the same shapes; and fit epochs per second at c2, native against generic. Device
events around many evaluations after warm-up; card name and power limit are read in the same run.

Usage: python tools/time_gauss_closure.py --out DIR [--reps 50] [--shapes c1,c2,...]
Writes DIR/gauss_closure.json."""

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_bures_wasserstein import SHAPES, card, make_stats, time_calls  # noqa: E402

NAMES = ("mahalanobis", "mahalanobis_sq", "bhattacharyya", "hellinger")


def generic_closure(model, stats, C, dev):
    """The fitting loop's closure body for a distance_fun without a native closure (_optim.py)."""
    from sqfa_b200._optim import check_distances_valid

    i, j = torch.tril_indices(C, C, -1, device=dev)

    def run():
        model.zero_grad()
        d = model.get_class_distances(stats, regularized=True)
        check_distances_valid(d)
        loss = -d[i, j].mean()
        loss.backward()
        return loss.detach().view(1)

    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--shapes", default=",".join(SHAPES), help="closure shapes to time (comma separated, may be empty)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA, SecondMomentsSQFA

    dev = torch.device("cuda")
    res = {"card": card(), "closure_ms": {}, "fit_c2": {}}
    for cfg in [c for c in args.shapes.split(",") if c]:
        C, D, k = SHAPES[cfg]
        stats = make_stats(C, D, dev)
        reps = args.reps if C < 500 else max(args.reps // 5, 5)
        row = {}
        plans = {}
        for name in NAMES:
            torch.manual_seed(0)
            model = SQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=getattr(Dn, name)).to(dev)
            plans[name] = model._fused_direct_plan(stats)
            assert plans[name] is not None, name
        torch.manual_seed(0)
        ai = SecondMomentsSQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=Dn.affine_invariant).to(dev)
        plans["affine_invariant"] = ai._fused_direct_plan(stats["covariances"])
        for _ in range(2):  # alternate, so that every closure sees the same machine state
            for name, plan in plans.items():
                ms, out = time_calls(plan, reps)
                row.setdefault(name, []).append(ms)
                row[name + "_loss"] = float(out[0])
        del plans
        for name in NAMES:
            fun = getattr(Dn, name)
            torch.manual_seed(0)
            model = SQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=lambda a, b, f=fun: f(a, b)).to(dev)
            assert model._fused_direct_plan(stats) is None
            ms, out = time_calls(generic_closure(model, stats, C, dev), max(reps // 5, 3), warm=2)
            row[name + "_generic"] = ms
            row[name + "_generic_loss"] = float(out[0])
        res["closure_ms"][cfg] = row
        del stats
        torch.cuda.empty_cache()
        print(cfg, row, flush=True)

    # fit epochs per second at c2 (pipelined L-BFGS on the graph-captured closure against the generic closure).
    # Tolerances 0: every epoch runs its 20 L-BFGS iterations, so epochs/s compares the cost of equal work.
    C, D, k = SHAPES["c2"]
    stats = make_stats(C, D, dev)
    stats["covariances"] = stats["covariances"] * D
    lbfgs = {"tolerance_grad": 0.0, "tolerance_change": 0.0}
    for name in NAMES:
        fun = getattr(Dn, name)
        for kind, dfun in (("native", fun), ("generic", lambda a, b, f=fun: f(a, b))):
            epochs = 20 if kind == "native" else 5
            torch.manual_seed(0)
            model = SQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=dfun).to(dev)
            model.fit(data_statistics=stats, max_epochs=2, show_progress=False, atol=0.0, **lbfgs)  # warm-up
            torch.manual_seed(0)
            model = SQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=dfun).to(dev)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss, _ = model.fit(data_statistics=stats, max_epochs=epochs, show_progress=False, atol=0.0,
                                return_loss=True, **lbfgs)
            e1.record()
            torch.cuda.synchronize()
            s = e0.elapsed_time(e1) / 1e3
            res["fit_c2"].setdefault(name, {})[kind] = {
                "epochs": int(loss.numel()), "seconds": s, "epochs_per_s": loss.numel() / s,
                "first_last_loss": [float(loss[0]), float(loss[-1])]}
            print("fit c2", name, kind, res["fit_c2"][name][kind], flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "gauss_closure.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
