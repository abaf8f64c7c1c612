"""Bures-Wasserstein / Gaussian 2-Wasserstein closures on one GPU, in ONE process: the fused closure
evaluation (CUDA-graph replay of `_fused_direct_plan`) of SecondMomentsSQFA with native Bures-Wasserstein
against native affine-invariant, and of SQFA with native 2-Wasserstein against Fisher-Rao, at the closure
shapes c1-c4 and the c5 shape (C = 100, D = 1024, k = 32); the reference tutorial's Bures-Wasserstein
`distance_fun` (spd_sqrt per class, (C, C, k, k) conjugations, eigvalsh, autograd backward) at the same
shapes where it fits; and fit epochs per second at c2. Device events around many evaluations after
warm-up; card name and power limit are read in the same run.

Usage: python tools/time_bures_wasserstein.py --out DIR [--reps 50]
Writes DIR/bures_wasserstein.json."""

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c1": (10, 784, 4), "c2": (10, 3072, 8), "c3": (19, 104, 8), "c4": (1000, 512, 16), "c5": (100, 1024, 32)}


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:  # the numbers are still tied to the torch device name
        info["nvidia_smi"] = f"unavailable: {e!r}"
    return info


def tutorial_bw(A, B):
    """The reference tutorial's Bures-Wasserstein distance_fun (docs/source/tutorials/distances.md)."""
    from sqfa_b200 import linalg

    tr_A = torch.einsum("ijj->i", A)
    tr_B = torch.einsum("ijj->i", B)
    C = linalg.conjugate_matrix(B, linalg.spd_sqrt(A))
    tr_C = torch.sum(torch.sqrt(torch.linalg.eigvalsh(C)), dim=-1)
    return torch.sqrt(torch.abs(tr_A[None, :] + tr_B[:, None] - 2 * tr_C) + 1e-6)


def make_stats(C, D, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    A = torch.randn(C, D, D + 8, device=dev, generator=g)
    cov = ((A @ A.transpose(1, 2)) / (D + 8) / D).contiguous()
    del A
    means = 0.05 * torch.randn(C, D, device=dev, generator=g) / D**0.5
    return {"means": means, "covariances": cov}


def time_calls(fn, reps, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


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
    res = {"card": card(), "closure_ms": {}, "tutorial_ms": {}, "fit_c2": {}}
    for cfg in [c for c in args.shapes.split(",") if c]:
        C, D, k = SHAPES[cfg]
        stats = make_stats(C, D, dev)
        reps = args.reps if C < 500 else max(args.reps // 5, 5)
        row = {}
        # alternate the native distances so that both see the same machine state
        pairs = [("bw", SecondMomentsSQFA, Dn.bures_wasserstein, stats["covariances"]),
                 ("ai", SecondMomentsSQFA, Dn.affine_invariant, stats["covariances"]),
                 ("w2", SQFA, Dn.wasserstein, stats),
                 ("fr", SQFA, Dn.fisher_rao_lower_bound, stats)]
        plans = {}
        for name, cls, fun, st in pairs:
            torch.manual_seed(0)
            model = cls(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=fun).to(dev)
            plans[name] = (model, model._fused_direct_plan(st))
            assert plans[name][1] is not None, name
        for _ in range(2):
            for name in plans:
                ms, out = time_calls(plans[name][1], reps)
                row.setdefault(name, []).append(ms)
                row[name + "_loss"] = float(out[0])
        res["closure_ms"][cfg] = row
        del plans
        # tutorial distance_fun: generic autograd path (get_class_distances + backward)
        try:
            torch.manual_seed(0)
            model = SecondMomentsSQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=tutorial_bw).to(dev)
            i, j = torch.tril_indices(C, C, -1, device=dev)

            def generic():
                model.zero_grad()
                d = model.get_class_distances(stats["covariances"], regularized=True)
                loss = -d[i, j].mean()
                loss.backward()
                return loss.detach().view(1)

            ms, out = time_calls(generic, max(reps // 5, 3), warm=2)
            res["tutorial_ms"][cfg] = {"ms": ms, "loss": float(out[0])}
        except (torch.cuda.OutOfMemoryError, RuntimeError) as e:  # e.g. a batch the library call rejects
            res["tutorial_ms"][cfg] = {"error": f"{type(e).__name__}: {e}"[:300]}
        del stats
        torch.cuda.empty_cache()
        print(cfg, res["closure_ms"][cfg], res["tutorial_ms"][cfg], flush=True)

    # fit epochs per second at c2 (pipelined L-BFGS on the graph-captured closure). The covariances are scaled
    # to eigenvalues of order 1 (above the feature noise) and the tolerances are 0, so that every epoch runs
    # its 20 L-BFGS iterations whatever the distance: epochs/s then compares the cost of equal work.
    C, D, k = SHAPES["c2"]
    scat = make_stats(C, D, dev)["covariances"] * D
    lbfgs = {"tolerance_grad": 0.0, "tolerance_change": 0.0}
    for name, fun in (("bw", Dn.bures_wasserstein), ("ai", Dn.affine_invariant), ("tutorial_bw", tutorial_bw)):
        epochs = 20
        torch.manual_seed(0)
        model = SecondMomentsSQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=fun).to(dev)
        model.fit(data_statistics=scat, max_epochs=2, show_progress=False, atol=0.0, **lbfgs)  # warm-up
        torch.manual_seed(0)
        model = SecondMomentsSQFA(n_dim=D, feature_noise=0.01, n_filters=k, distance_fun=fun).to(dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss, _ = model.fit(data_statistics=scat, max_epochs=epochs, show_progress=False, atol=0.0, return_loss=True,
                            **lbfgs)
        e1.record()
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        res["fit_c2"][name] = {"epochs": int(loss.numel()), "seconds": s, "epochs_per_s": loss.numel() / s,
                               "first_last_loss": [float(loss[0]), float(loss[-1])]}
        print("fit c2", name, res["fit_c2"][name], flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bures_wasserstein.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
