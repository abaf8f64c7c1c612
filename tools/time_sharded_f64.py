"""The class- and pair-sharded float64 closure (sqfa_fused_loss_sharded_f64) of `.double()` models.

Run as `torchrun --nproc-per-node W tools/time_sharded_f64.py --out DIR` (W = 1, 2, 4, 8), or plainly for one
rank. At c4 (1000, 512, 16) and the c5 shape (100, 1024, 32), for Fisher-Rao, affine-invariant and Mahalanobis:

1. group: the sharded plan of `_fused_direct_plan` at the launch's world size W, float64 against float32 (same
   statistics, alternated): device events around one evaluation including its all-reduces, median over the
   timed evaluations after warm-up, reported as the max over the ranks.
2. composed: the composed float64 closure (get_class_distances, -mean, autograd), which ignores the group and runs
   in full on every rank (median of 3 calls after 1); a failure is recorded with its exception text.
3. fit: a c4 Fisher-Rao `.double()` fit with `process_group`, in epochs/s (tolerance 0, 20 iterations an epoch).
4. With W = 1 only, emulated ranks: for W' = 2, 4, 8 the three phases of every rank on this one GPU (the spans and
   dF summed between phases as the all-reduces would), device events around each rank's phases, max over the
   ranks -- per-rank work without collectives, not a multi-GPU time.
Card name, power limit and maximum SM clock are read in the same run. Writes DIR/sharded_f64_w{W}.json."""

import argparse
import json
import os
import statistics
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_bures_wasserstein import card, make_stats  # noqa: E402

SHAPES = {"c4": (1000, 512, 16), "c5": (100, 1024, 32)}
DISTANCES = (("full", "fisher_rao_lower_bound"), ("second_moments", "affine_invariant"), ("full", "mahalanobis"))
WARM, TIMED = 3, 15


def model_for(kind, distance, D, k, dtype, dev):
    from sqfa_b200 import distances as Dn
    from sqfa_b200.model import SQFA, SecondMomentsSQFA

    cls = SecondMomentsSQFA if kind == "second_moments" else SQFA
    F0 = torch.randn(k, D, generator=torch.Generator().manual_seed(1))
    return cls(n_dim=D, feature_noise=0.01, n_filters=k, filters=F0, distance_fun=getattr(Dn, distance)).to(dev, dtype)


def stats_for(kind, stats):
    if kind == "second_moments":
        return stats["covariances"] + stats["means"][:, :, None] * stats["means"][:, None, :]
    return stats


def event_ms(fn, warm=WARM, timed=TIMED):
    """Median device time of one call over `timed` calls after `warm` (events around each call)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(timed):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times)


def max_over_ranks(x, dev):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def emulated_phases_ms(S, M, F, dist_code, world, dev):
    """Per-rank time of the three phases of `world` emulated ranks on this GPU (no collectives): for every rank the
    median over TIMED rounds of its summed phase times; returns the max over the ranks and the loss."""
    from sqfa_b200 import _lib, _ops
    from sqfa_b200._stats_driver import class_share

    lib = _lib.load()
    C, D, _ = S.shape
    k = F.shape[0]
    P = C * (C - 1) // 2
    noise = torch.full((1,), 0.01, dtype=torch.float64, device=dev)
    ranks = []
    for r in range(world):
        p0, p1 = _ops.shard_pairs(P, C, r, world)
        c0, c1 = class_share(C, r, world)
        ws = torch.empty(_ops.closure_workspace_bytes_f64(C, D, k, dist_code, p0, p1), dtype=torch.uint8, device=dev)
        spans = _ops._exchange_spans("sqfa_fused_loss_exchange_span_f64", C, D, k, dist_code, p0, p1, ws,
                                     torch.float64)
        ranks.append({"p": (p0, p1), "c": (c0, c1), "ws": ws, "spans": spans,
                      "dF": torch.empty(k, D, dtype=torch.float64, device=dev)})
    stream = _lib.stream_ptr(dev)

    def one_round():
        times = [0.0] * world
        for i in range(3):
            for r, q in enumerate(ranks):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _lib.check(lib.sqfa_fused_loss_sharded_f64(i, _lib.ptr(S), _lib.ptr(M), _lib.ptr(F), C, D, k,
                                                           _lib.ptr(noise), dist_code, q["c"][0], q["c"][1],
                                                           q["p"][0], q["p"][1], _lib.ptr(q["dF"]),
                                                           _lib.ptr(q["ws"]), q["ws"].numel(), stream), "phase")
                e1.record()
                torch.cuda.synchronize()
                times[r] += e0.elapsed_time(e1)
            if i < 2:
                total = torch.stack([q["spans"][i] for q in ranks]).sum(0)
                for q in ranks:
                    q["spans"][i].copy_(total)
        return times

    for _ in range(WARM):
        one_round()
    rounds = [one_round() for _ in range(TIMED)]
    per_rank = [statistics.median(r[i] for r in rounds) for i in range(world)]
    return max(per_rank), float(ranks[0]["spans"][1][-64])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--fit-epochs", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29517")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD
    rank, world = dist.get_rank(), dist.get_world_size()
    result = {"world": world, "card": card(), "rows": []}
    try:
        for shape in [s for s in args.shapes.split(",") if s]:
            C, D, k = SHAPES[shape]
            stats32 = make_stats(C, D, dev)
            stats64 = {key: v.double() for key, v in stats32.items()}
            for kind, distance in DISTANCES:
                row = {"shape": shape, "distance": distance}
                s64, s32 = stats_for(kind, stats64), stats_for(kind, stats32)
                m64 = model_for(kind, distance, D, k, torch.float64, dev)
                m32 = model_for(kind, distance, D, k, torch.float32, dev)
                m64._process_group = m32._process_group = group
                plan64, plan32 = m64._fused_direct_plan(s64), m32._fused_direct_plan(s32)
                row["loss64"], row["loss32"] = float(plan64()[0]), float(plan32()[0])
                # alternated: float64, float32, float64, float32
                t64, t32 = [], []
                for _ in range(2):
                    t64.append(event_ms(plan64))
                    t32.append(event_ms(plan32))
                row["group_f64_ms"] = max_over_ranks(min(t64), dev)
                row["group_f32_ms"] = max_over_ranks(min(t32), dev)
                del plan64, plan32
                m64._process_group = None
                try:
                    i, j = torch.tril_indices(C, C, -1, device=dev)

                    def composed():
                        m64.zero_grad()
                        dmat = m64.get_class_distances(s64, regularized=True)
                        loss = -dmat[i, j].mean()
                        loss.backward()
                        return loss

                    row["composed_f64_ms"] = event_ms(composed, warm=1, timed=3)  # up to seconds a call
                except Exception as e:  # recorded, not hidden: at c4 the batched eigvalsh fails
                    row["composed_f64_ms"] = None
                    row["composed_f64_error"] = f"{type(e).__name__}: {e}"[:600]
                torch.cuda.empty_cache()
                if world == 1:
                    S, M, code = m64._fused_inputs(s64)
                    p = m64.parametrizations.filters.original.detach()
                    F = (p / p.norm(dim=1, keepdim=True)).contiguous()
                    for w in (2, 4, 8):
                        ms, loss = emulated_phases_ms(S, M, F, code, w, dev)
                        row[f"emulated_w{w}_per_rank_ms"] = ms
                        row[f"emulated_w{w}_loss"] = loss
                    del S, M, F
                    torch.cuda.empty_cache()
                if rank == 0:
                    print(json.dumps(row), flush=True)
                result["rows"].append(row)
                del m64, m32
            del stats32, stats64
            torch.cuda.empty_cache()
        if "c4" in args.shapes.split(","):
            C, D, k = SHAPES["c4"]
            stats = {key: v.double() for key, v in make_stats(C, D, dev).items()}
            m = model_for("full", "fisher_rao_lower_bound", D, k, torch.float64, dev)
            m.fit(data_statistics=stats, max_epochs=1, show_progress=False, atol=0.0, tolerance_grad=0.0,
                  tolerance_change=0.0, process_group=group)  # warm-up
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            losses, _ = m.fit(data_statistics=stats, max_epochs=args.fit_epochs, show_progress=False, atol=0.0,
                              tolerance_grad=0.0, tolerance_change=0.0, return_loss=True, process_group=group)
            torch.cuda.synchronize()
            secs = max_over_ranks(time.perf_counter() - t0, dev)
            result["fit_c4_fr64"] = {"epochs": len(losses), "epochs_per_s": len(losses) / secs,
                                     "last_loss": float(losses[-1])}
            if rank == 0:
                print(json.dumps(result["fit_c4_fr64"]), flush=True)
    finally:
        if rank == 0:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"sharded_f64_w{world}.json"), "w") as f:
                json.dump(result, f, indent=1)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
