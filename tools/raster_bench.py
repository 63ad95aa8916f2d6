"""K12 occupancy-grid rasteriser (hl_env_rasterize) on config-5 environments.

For N environments (scenarios.scenario_spec(i), i < N, default 4096) and each resolution (default 0.1 and 0.2 m), every
environment's grid covers its field ring's bounding box grown by --margin (ops.raster_window), all grids in one
pooled buffer and one call.  Before timing, the tool checks the grids of the first 8 environments against the CPU
oracle rasteriser (tests/raster_oracle.py) byte for byte and two runs for byte identity; it exits 1 if either fails.
Timed, with CUDA events around work that ends in a device synchronisation, after a warm-up, median of --reps:
  * rasterise: the hl_env_rasterize call alone (table and output buffer prepared outside the window);
  * rasterise + grid_pack: the same call followed by one hl_grid_pack per grid (K7's bit-packed grids);
  * rasterise + distance_field_batch: the same call followed by one K6 batch, a King field per grid with the goal
    cell = the cell holding the scenario's goal (host looks of the wavefront included);
  * the CPU oracle rasteriser on the first 8 environments (one process), for comparison.
The pooled output of 4096 environments is larger than the 126 MB L2 at both default resolutions (each row reports
its size in bytes as "output_bytes"), so every pass writes to HBM.  Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import raster_oracle as RO  # noqa: E402
from headland_trajectory_planning_b200 import _lib, ops, scenarios  # noqa: E402
from headland_trajectory_planning_b200.car_model import CarModel  # noqa: E402
from headland_trajectory_planning_b200.env_batch import EnvBatch, make_record  # noqa: E402
from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [v.strip() for v in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def events_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-env", type=int, default=4096)
    ap.add_argument("--res", type=float, nargs="+", default=[0.1, 0.2])
    ap.add_argument("--margin", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "raster_bench needs a CUDA device"
    torch.cuda.set_device(0)
    info = gpu_info()
    lib = _lib.load_library()
    scns = scenarios.make_scenarios_gpu(range(args.n_env))
    recs, quads, rings = [], [], []
    for s in scns:
        env = OrchardGeometryEnvironment(s["rows"], [], tree_width=s["tree_width"], headland_width=s["headland_width"])
        rec = make_record(env, CarModel(**s["car"]))
        recs.append(rec); quads.append(rec.obs); rings.append(rec.field)
    envs = EnvBatch(recs)
    flags = ops.CHECK_OBSTACLES | ops.CHECK_BOUNDARY
    result = {"metric": "env_rasterize", "gpu": info, "n_env": args.n_env, "margin_m": args.margin, "flags": flags,
              "timing": f"CUDA events, device synchronised, median of {args.reps} after one warm-up", "resolutions": []}
    ok = True
    for res in args.res:
        wins = [ops.raster_window(f, res, args.margin) for f in rings]
        table = (_lib.HlRasterGrid * len(wins))()
        base = 0
        for k, (i0, j0, w, h) in enumerate(wins):
            table[k] = _lib.HlRasterGrid(base, k, w, h, i0, j0)
            base += w * h
        out = torch.empty(base, dtype=torch.uint8, device="cuda")
        n_exact = torch.zeros(1, dtype=torch.int64, device="cuda")
        ctx, st = envs.ctx, _lib.stream_ptr()

        def raster(count=False):
            _lib.check(lib.hl_env_rasterize(ctx, envs.handle, table, len(wins), res, flags, _lib.ptr(out), base,
                                            _lib.ptr(n_exact) if count else None, st), "hl_env_rasterize")
            return out

        views = [out[table[k].out_offset:table[k].out_offset + w * h].view(w, h) for k, (_, _, w, h) in enumerate(wins)]
        # correctness before timing: 8 environments against the oracle, then run-to-run byte identity
        raster(count=True)
        torch.cuda.synchronize()
        escalated = int(n_exact.item())
        first = out.clone()
        t0 = time.perf_counter()
        oracle = [RO.rasterize(quads[k], rings[k], *wins[k], res, flags) for k in range(min(8, args.n_env))]
        t_oracle = time.perf_counter() - t0
        oracle_cells = int(sum(o.size for o in oracle))
        match = all(np.array_equal(views[k].cpu().numpy(), oracle[k]) for k in range(len(oracle)))
        raster()
        torch.cuda.synchronize()
        same = bool(torch.equal(first, out))
        ok &= match and same
        del first
        bits = [torch.empty((w * h + 31) // 32, dtype=torch.int32, device="cuda") for (_, _, w, h) in wins]

        def pack():
            raster()
            for v, b, (_, _, w, h) in zip(views, bits, wins):
                _lib.check(lib.hl_grid_pack(ctx, _lib.ptr(v), w, h, _lib.ptr(b), st), "hl_grid_pack")

        goals = []
        for s, (i0, j0, w, h) in zip(scns, wins):
            gi = ops._cell_range(s["goal"][0], s["goal"][0], res)[0] - i0
            gj = ops._cell_range(s["goal"][1], s["goal"][1], res)[0] - j0
            goals.append((gi, gj))
        df_info = {}

        def with_df():
            raster()
            try:
                fields, sweeps = ops.distance_field_batch(views, goals, "King")
            except _lib.HeadlandError as e:                    # report the limit instead of failing the whole run
                df_info["error"] = str(e)
                return
            df_info["relaxation_launches"] = int(sweeps)
            del fields

        row = {"res_m": res, "grids": len(wins), "cells": int(base), "output_bytes": int(base),
               "oracle_match_8_envs": bool(match), "run_to_run_identical": same,
               "escalated_cells": escalated, "escalated_fraction": escalated / base}
        for name, fn in (("rasterize", raster), ("rasterize_plus_grid_pack", pack), ("rasterize_plus_distance_field_batch", with_df)):
            events_ms(fn)                                      # warm-up
            if "error" in df_info and name.endswith("batch"):
                row[name] = {"error": df_info["error"]}
                continue
            ts = [events_ms(fn)[0] for _ in range(args.reps)]
            m = float(np.median(ts))
            row[name] = {"ms": round(m, 3), "ms_all": [round(t, 3) for t in ts], "cells_per_s": round(base / (m * 1e-3))}
            if name.endswith("batch"):
                row[name].update(fields=len(goals), fields_per_s=round(len(goals) / (m * 1e-3), 1), **df_info)
        row["cpu_oracle_8_envs"] = {"cells": oracle_cells, "s": round(t_oracle, 3), "cells_per_s": round(oracle_cells / t_oracle)}
        result["resolutions"].append(row)
        del views, bits, out
        torch.cuda.empty_cache()
    result["ok"] = bool(ok)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
