"""The float64 fitting closure of `.double()` models on one GPU, in ONE process: the native closure (CUDA-graph
replay of `_fused_direct_plan`) against the composed float64 closure the fitting loop runs when there is no
native one (`get_class_distances` through the library's float64 linear algebra, the NaN/inf check,
-mean(tril), autograd backward), with the native float32 closure for context. Fisher-Rao lower bound (SQFA) and
affine-invariant (SecondMomentsSQFA) at the closure shapes c1-c4 and the c5 shape (C = 100, D = 1024, k = 32);
a failure of the composed path is recorded with its exception text. Then fit epochs per second at c2, native
against composed float64. Device events around many evaluations after warm-up; card name, power limit and
maximum SM clock are read in the same run.

Usage: python tools/time_float64_closure.py --out DIR [--reps 30] [--shapes c1,c2,...]
Writes DIR/float64_closure.json."""

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_bures_wasserstein import SHAPES, card, make_stats, time_calls  # noqa: E402
from time_gauss_closure import generic_closure  # noqa: E402

# S (float64) fits in the 126 MB L2 at c1 (49 MB) and c3 (1.6 MB): those timings read S from L2 after warm-up
L2_RESIDENT = {"c1", "c3"}


def models(kind, D, k, dev, composed=False):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA, SecondMomentsSQFA

    torch.manual_seed(0)
    if kind == "fisher_rao_lower_bound":
        dfun = Dn.fisher_rao_lower_bound
        cls = SQFA
    else:
        dfun = Dn.affine_invariant
        cls = SecondMomentsSQFA
    if composed:  # a wrapped distance has no native closure: the fitting loop composes it
        dfun = (lambda a, b, f=dfun: f(a, b))
    return cls(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=dfun).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--shapes", default=",".join(SHAPES), help="closure shapes to time (comma separated, may be empty)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    dev = torch.device("cuda")
    res = {"card": card(), "l2_resident_shapes": sorted(L2_RESIDENT), "closure_ms": {}, "fit_c2": {}}
    for cfg in [c for c in args.shapes.split(",") if c]:
        C, D, k = SHAPES[cfg]
        s32 = make_stats(C, D, dev)
        s64 = {key: v.double() for key, v in s32.items()}
        reps = args.reps if C < 500 else max(args.reps // 5, 3)
        row = {}
        for kind in ("fisher_rao_lower_bound", "affine_invariant"):
            st32 = s32 if kind == "fisher_rao_lower_bound" else s32["covariances"]
            st64 = s64 if kind == "fisher_rao_lower_bound" else s64["covariances"]
            native64 = models(kind, D, k, dev).double()._fused_direct_plan(st64)
            native32 = models(kind, D, k, dev)._fused_direct_plan(st32)
            assert native64 is not None and native32 is not None
            for _ in range(2):  # alternate, so that both see the same machine state
                for name, plan in (("native64", native64), ("native32", native32)):
                    ms, out = time_calls(plan, reps)
                    row.setdefault(f"{kind}_{name}", []).append(ms)
                    row[f"{kind}_{name}_loss"] = float(out[0])
            del native64, native32
            model = models(kind, D, k, dev, composed=True).double()
            assert model._fused_direct_plan(st64) is None
            try:
                ms, out = time_calls(generic_closure(model, st64, C, dev), max(reps // 5, 2), warm=1)
                row[f"{kind}_composed64"] = ms
                row[f"{kind}_composed64_loss"] = float(out[0])
            except Exception as e:  # recorded, not hidden: at c4 the batched eigvalsh is expected to fail
                row[f"{kind}_composed64"] = None
                row[f"{kind}_composed64_error"] = f"{type(e).__name__}: {e}"[:2000]
            del model
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
        res["closure_ms"][cfg] = row
        del s32, s64
        torch.cuda.empty_cache()
        print(cfg, row, flush=True)

    # fit epochs per second at c2; tolerances 0, so every epoch runs its 20 L-BFGS iterations (equal work)
    C, D, k = SHAPES["c2"]
    stats = {key: v.double() for key, v in make_stats(C, D, dev).items()}
    stats["covariances"] = stats["covariances"] * D
    lbfgs = {"tolerance_grad": 0.0, "tolerance_change": 0.0}
    for kind, composed, epochs in (("native64", False, 10), ("composed64", True, 3)):
        model = models("fisher_rao_lower_bound", D, k, dev, composed).double()
        model.fit(data_statistics=stats, max_epochs=1, show_progress=False, atol=0.0, **lbfgs)  # warm-up
        model = models("fisher_rao_lower_bound", D, k, dev, composed).double()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss, _ = model.fit(data_statistics=stats, max_epochs=epochs, show_progress=False, atol=0.0,
                            return_loss=True, **lbfgs)
        e1.record()
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        res["fit_c2"][kind] = {"epochs": int(loss.numel()), "seconds": s, "epochs_per_s": loss.numel() / s,
                               "losses": [float(v) for v in loss]}
        print("fit c2", kind, res["fit_c2"][kind], flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "float64_closure.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
