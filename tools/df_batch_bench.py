"""Batched distance fields against a Python loop of single fields (K6), on three workloads:
  (a) 256 distinct 256^2 maps      -- many small fields: the loop pays launch and host-look overheads per field
  (b) one 1024^2 map, 64 goals     -- a heuristic table: one map shared by many goals
  (c) eight 4096^2 maps            -- few deep fields: the loop is already mostly wavefront depth
Each workload: batch and loop outputs are checked to be bit-identical first (exit 1 if not), then the loop of
ops.distance_field and one ops.distance_field_batch are timed alternately with CUDA events (one synchronisation at the
end of each timed call), after a warm-up, median of REPS.  Grids are on the device before timing.  With --profile, one
more call of each under torch.profiler gives the GPU time per kernel (the rest of the wall time is launch gaps and host
looks).  Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from headland_trajectory_planning_b200 import ops  # noqa: E402
from headland_trajectory_planning_b200.utils.occupancy_grid_utils import synthetic_grid  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [v.strip() for v in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def workloads(dev):
    rng = np.random.default_rng(0)
    a = [synthetic_grid(256, seed=s) for s in range(256)]
    occ_b, _ = synthetic_grid(1024, seed=1)
    free = np.argwhere(~occ_b)
    goals_b = [tuple(int(v) for v in free[k]) for k in rng.choice(len(free), 64, replace=False)]
    c = [synthetic_grid(4096, seed=s) for s in range(1, 9)]
    up = lambda o: torch.from_numpy(o.astype(np.uint8)).to(dev)  # noqa: E731
    d_b = up(occ_b)
    return [("a_256x256_maps", [up(o) for o, _ in a], [g for _, g in a], False),
            ("b_1024x1024_map_64_goals", d_b, goals_b, True),
            ("c_4096x4096_maps", [up(o) for o, _ in c], [g for _, g in c], False)]


def run_loop(occs, goals, shared):
    outs, launches = [], 0
    for k, g in enumerate(goals):
        o, s = ops.distance_field(occs if shared else occs[k], g, "King")
        outs.append(o)
        launches += s
    return outs, launches


def run_batch(occs, goals, shared):
    return ops.distance_field_batch(occs, goals, "King")


def timed(fn, *args, keep=False):
    """(ms, outputs if keep, launches).  Timed calls drop their outputs before the next call starts, so the caching
    allocator hands the same blocks back instead of mapping a new 0.5-1 GB output buffer inside the timed window."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    outs, launches = fn(*args)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), (outs if keep else None), launches


def kernel_times(fn, *args):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(*args)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            per[e.key[:60]] = {"ms": round(t / 1e3, 3), "calls": e.count}
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "df_batch_bench needs a CUDA device"
    dev = torch.device("cuda", 0)
    res = {"metric": "distance_field_batch_speedup", "gpu": gpu_info(), "motion_type": "King",
           "timing": f"CUDA events around each call, median of {args.reps}, loop and batch alternating", "workloads": []}
    ok = True
    for name, occs, goals, shared in workloads(dev):
        shapes = [tuple(occs.shape)] * len(goals) if shared else [tuple(o.shape) for o in occs]
        cells = int(sum(w * h for w, h in shapes))
        _, lo, _ = timed(run_loop, occs, goals, shared, keep=True)            # warm-up, and the outputs to compare
        _, bo, _ = timed(run_batch, occs, goals, shared, keep=True)
        same = all(torch.equal(x, y) for x, y in zip(lo, bo)) and len(lo) == len(bo)
        ok &= same
        del lo, bo
        timed(run_loop, occs, goals, shared)
        timed(run_batch, occs, goals, shared)
        t_loop, t_batch = [], []
        for _ in range(args.reps):
            t, _, n_loop = timed(run_loop, occs, goals, shared)
            t_loop.append(t)
            t, _, n_batch = timed(run_batch, occs, goals, shared)
            t_batch.append(t)
        ml, mb = float(np.median(t_loop)), float(np.median(t_batch))
        side = lambda ms, n: {"ms": round(ms, 3), "fields_per_s": round(len(goals) / (ms * 1e-3), 1),  # noqa: E731
                              "cells_per_s": round(cells / (ms * 1e-3)), "relaxation_launches": int(n)}
        w = {"workload": name, "fields": len(goals), "cells": cells, "bit_identical": bool(same),
             "loop": dict(side(ml, n_loop), ms_all=[round(t, 3) for t in t_loop]),
             "batch": dict(side(mb, n_batch), ms_all=[round(t, 3) for t in t_batch]),
             "speedup_batch_over_loop": round(ml / mb, 2)}
        if args.profile:
            w["loop"]["kernel_ms"] = kernel_times(run_loop, occs, goals, shared)
            w["batch"]["kernel_ms"] = kernel_times(run_batch, occs, goals, shared)
        res["workloads"].append(w)
        torch.cuda.empty_cache()
    res["bit_identical"] = bool(ok)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
