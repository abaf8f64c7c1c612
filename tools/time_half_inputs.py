"""bfloat16 vs float32 points on one GPU, in ONE process, on identical values (the float32 tensor is the
bf16 tensor widened): class_statistics at the BASELINE configs c1-c4 and the c5 shard with device- and
host-resident inputs, class_sums and the Gram kernel alone, and transform at 50 000 x 3072 (k = 8, 16, 32).
The two dtypes alternate call by call; a 256 MB buffer is overwritten before every timed call so that no
input is read from the 126 MB L2. Reports ms, samples/s, achieved HBM bytes/s of the HBM-bound kernels
against 7.7 TB/s (algorithmic bytes: one read of X, plus Z for transform) and the peak device memory a
call allocates beyond its resident input; card name and power limit are read in the same run.

Usage: python tools/time_half_inputs.py --out DIR [--reps 5] [--skip-c5]
Writes DIR/half_inputs.json."""

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12
CONFIGS = {"c1": (60000, 784, 10), "c2": (50000, 3072, 10), "c3": (200000, 104, 19), "c4": (1280000, 512, 1000),
           "c5_shard": (12500000, 1024, 100)}


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:  # the numbers are still tied to the torch device name
        info["nvidia_smi"] = f"unavailable: {e!r}"
    return info


class Timer:
    def __init__(self):
        self.flush_buf = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device="cuda")  # 256 MB > L2

    def __call__(self, fn, reps):
        """median ms of `reps` calls, L2 overwritten before each; peak bytes allocated during one call."""
        fn()  # warm-up: module load, workspace sizes, class-count guess
        torch.cuda.synchronize()
        times = []
        for _ in range(reps):
            self.flush_buf.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b))
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        times.sort()
        return {"ms": times[len(times) // 2], "ms_all": times, "peak_extra_bytes": int(peak)}


def alternate(timer, fns, reps):
    """{name: result}, the callables interleaved rep by rep (one call each per round)."""
    out = {k: [] for k in fns}
    peaks = {}
    for _ in range(reps):
        for k, fn in fns.items():
            r = timer(fn, 1)
            out[k].append(r["ms"])
            peaks[k] = max(peaks.get(k, 0), r["peak_extra_bytes"])
    return {k: {"ms": sorted(v)[len(v) // 2], "ms_all": v, "peak_extra_bytes": peaks[k]} for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives half_inputs.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-c5", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_half_inputs.py needs a CUDA device")
    from sqfa_b200 import _ops
    from sqfa_b200._stats_driver import CudaStatsOps
    from sqfa_b200.statistics import class_statistics

    torch.cuda.set_device(0)
    res = {"card": card(), "hbm_peak_bytes_per_s": HBM_PEAK, "reps": args.reps,
           "l2": "256 MB buffer overwritten before every timed call", "class_statistics": {}, "kernels": {},
           "transform": {}}
    timer = Timer()
    g = torch.Generator(device="cuda").manual_seed(0)
    for name, (n, d, c) in CONFIGS.items():
        if name == "c5_shard" and args.skip_c5:
            res["class_statistics"][name] = "not measured (--skip-c5)"
            continue
        Xb = torch.randn(n, d, generator=g, device="cuda").to(torch.bfloat16)
        X32 = Xb.float()
        y = torch.randint(0, c, (n,), generator=g, device="cuda")
        r = alternate(timer, {"float32": lambda: class_statistics(X32, y), "bfloat16": lambda: class_statistics(Xb, y)},
                      args.reps)
        for k, bpe in (("float32", 4), ("bfloat16", 2)):
            r[k]["samples_per_s"] = n / (r[k]["ms"] * 1e-3)
            r[k]["input_bytes"] = n * d * bpe
        row = {"n": n, "d": d, "c": c, "device_resident": r}
        if name != "c5_shard":  # host-resident (pinned) input: the copy is part of the call
            Xb_h, X32_h, y_h = Xb.cpu().pin_memory(), X32.cpu().pin_memory(), y.cpu().pin_memory()
            h = alternate(timer, {"float32": lambda: class_statistics(X32_h, y_h),
                                  "bfloat16": lambda: class_statistics(Xb_h, y_h)}, args.reps)
            for k in h:
                h[k]["samples_per_s"] = n / (h[k]["ms"] * 1e-3)
            row["host_resident_pinned"] = h
            del Xb_h, X32_h, y_h
        else:
            row["host_resident_pinned"] = "not measured (51 GB of float32 rows do not fit pinned host memory here)"
        # the kernels alone: class sums (HBM-bound, one read of X) and the Gram (tensor-bound except c5)
        if name in ("c2", "c4", "c5_shard"):
            kern = {}
            for k, X in (("float32", X32), ("bfloat16", Xb)):
                ops = CudaStatsOps(0 if k == "float32" else 1)
                perm, offsets, counts = ops.bucket(y, c)
                means = ops.class_means(ops.class_sums(X, perm, offsets, c), counts[:c].clone())
                s = timer(lambda: ops.class_sums(X, perm, offsets, c), args.reps)
                s["bytes"] = X.numel() * X.element_size() + 4 * n
                s["achieved_bytes_per_s"] = s["bytes"] / (s["ms"] * 1e-3)
                s["share_of_hbm_peak"] = s["achieved_bytes_per_s"] / HBM_PEAK
                gk = timer(lambda: ops.class_gram(X, perm, offsets, means, c), args.reps)
                gk["bytes_one_read"] = X.numel() * X.element_size()
                kern[k] = {"class_sums": s, "gram": gk}
            res["kernels"][name] = kern
        res["class_statistics"][name] = row
        print(name, json.dumps({k: v["ms"] for k, v in r.items()}), flush=True)
        del Xb, X32, y
        torch.cuda.empty_cache()
    n, d = 50000, 3072
    Xb = torch.randn(n, d, generator=g, device="cuda").to(torch.bfloat16)
    X32 = Xb.float()
    for k in (8, 16, 32):
        F = torch.randn(k, d, generator=g, device="cuda")
        r = alternate(timer, {"float32": lambda: _ops.transform_raw(X32, F), "bfloat16": lambda: _ops.transform_raw(Xb, F)},
                      args.reps)
        for key, X in (("float32", X32), ("bfloat16", Xb)):
            r[key]["bytes"] = X.numel() * X.element_size() + 4 * n * k
            r[key]["achieved_bytes_per_s"] = r[key]["bytes"] / (r[key]["ms"] * 1e-3)
            r[key]["share_of_hbm_peak"] = r[key]["achieved_bytes_per_s"] / HBM_PEAK
        res["transform"][f"n{n}_d{d}_k{k}"] = r
        print("transform", k, json.dumps({kk: v["ms"] for kk, v in r.items()}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "half_inputs.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
