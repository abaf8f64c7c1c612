"""The float64 fitting closure of the mean-covariance distances (Mahalanobis, squared Mahalanobis, Bhattacharyya,
Hellinger) on `.double()` SQFA models, on one GPU and in ONE process. Three arms per shape and distance:
  native64    CUDA-graph replay of `_fused_direct_plan` (sqfa_gauss_closure_eval_f64)
  composed64  the same distance wrapped in a lambda on the `.double()` model: `get_class_distances` through the
              composed float64 branch of distances._gauss_pairs, the NaN/inf check, -mean(tril), autograd backward
              (what a float64 fit of these distances ran before the native closure)
  native32    the float32 closure, alternated with native64 in the same run
at the closure shapes c1-c4 and the c5 shape (C = 100, D = 1024, k = 32). A failure of the composed arm is
recorded with its exception text. Then fit epochs per second at c2, native against composed float64. Device
events around many evaluations after warm-up; card name, power limit and maximum SM clock are read in the same
run, and each shape states whether its float64 S fits in the 126 MB L2 (then the timings read S from L2).

Usage: python tools/time_gauss_closure_f64.py --out DIR [--reps 30] [--shapes c1,c2,...]
Writes DIR/gauss_closure_f64.json."""

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

NAMES = ("mahalanobis", "mahalanobis_sq", "bhattacharyya", "hellinger")
L2_BYTES = 126 * 2**20


def model(name, D, k, dev, composed=False):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA

    torch.manual_seed(0)
    dfun = getattr(Dn, name)
    if composed:  # a wrapped distance has no native closure: the fitting loop composes it
        dfun = (lambda a, b, f=dfun: f(a, b))
    return SQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=dfun).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--shapes", default=",".join(SHAPES), help="closure shapes to time (comma separated, may be empty)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    dev = torch.device("cuda")
    res = {"card": card(), "shapes": {}, "closure_ms": {}, "fit_c2": {}}
    for cfg in [c for c in args.shapes.split(",") if c]:
        C, D, k = SHAPES[cfg]
        s_bytes = C * D * D * 8
        res["shapes"][cfg] = {"C": C, "D": D, "k": k, "S_float64_MB": s_bytes / 1e6, "S_l2_resident": s_bytes <= L2_BYTES}
        s32 = make_stats(C, D, dev)
        s64 = {key: v.double() for key, v in s32.items()}
        reps = args.reps if C < 500 else max(args.reps // 5, 3)
        row = {}
        for name in NAMES:
            native64 = model(name, D, k, dev).double()._fused_direct_plan(s64)
            native32 = model(name, D, k, dev)._fused_direct_plan(s32)
            assert native64 is not None and native32 is not None
            for _ in range(2):  # alternate, so that both see the same machine state
                for arm, plan in (("native64", native64), ("native32", native32)):
                    ms, out = time_calls(plan, reps)
                    row.setdefault(f"{name}_{arm}", []).append(ms)
                    row[f"{name}_{arm}_loss"] = float(out[0])
            del native64, native32
            m = model(name, D, k, dev, composed=True).double()
            assert m._fused_direct_plan(s64) is None
            try:
                ms, out = time_calls(generic_closure(m, s64, C, dev), max(reps // 5, 2), warm=1)
                row[f"{name}_composed64"] = ms
                row[f"{name}_composed64_loss"] = float(out[0])
            except Exception as e:  # recorded, not hidden: at c4 the (C, C, k, k) float64 tensors take 2 GB each
                row[f"{name}_composed64"] = None
                row[f"{name}_composed64_error"] = f"{type(e).__name__}: {e}"[:2000]
            del m
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
        res["closure_ms"][cfg] = row
        del s32, s64
        torch.cuda.empty_cache()
        print(cfg, res["shapes"][cfg], row, flush=True)

    # fit epochs per second at c2; tolerances 0, so every epoch runs its 20 L-BFGS iterations (equal work)
    C, D, k = SHAPES["c2"]
    stats = {key: v.double() for key, v in make_stats(C, D, dev).items()}
    stats["covariances"] = stats["covariances"] * D
    lbfgs = {"tolerance_grad": 0.0, "tolerance_change": 0.0}
    for name in ("mahalanobis", "hellinger"):
        for arm, composed, epochs in (("native64", False, 10), ("composed64", True, 3)):
            m = model(name, D, k, dev, composed).double()
            m.fit(data_statistics=stats, max_epochs=1, show_progress=False, atol=0.0, **lbfgs)  # warm-up
            m = model(name, D, k, dev, composed).double()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss, _ = m.fit(data_statistics=stats, max_epochs=epochs, show_progress=False, atol=0.0,
                            return_loss=True, **lbfgs)
            e1.record()
            torch.cuda.synchronize()
            s = e0.elapsed_time(e1) / 1e3
            res["fit_c2"][f"{name}_{arm}"] = {"epochs": int(loss.numel()), "seconds": s,
                                             "epochs_per_s": loss.numel() / s, "losses": [float(v) for v in loss]}
            print("fit c2", name, arm, res["fit_c2"][f"{name}_{arm}"], flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "gauss_closure_f64.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
