"""K7 batch (hl_grid_pack_batch, hl_grid_footprint_check_batch) against a loop of per-grid K7 calls, and the grid check
against K1 on the same poses.

(a) pack: the rasters of N config-5 environments (scenarios.scenario_spec(i), i < N, default 4096; margin 2 m, flags 3,
    as tools/raster_bench.py makes them) at each resolution (default 0.1 and 0.2 m), one hl_grid_pack per grid against
    one hl_grid_pack_batch over all of them.
(b) check: the Y-park candidate paths of S config-5 scenarios (default 256; bench.py's Y-park sweep: 858 candidates,
    step 0.1 m, pose_idx = index within the path), each scenario's car plus one rear implement rectangle (the config-2
    mower's aux [[-1.84, 0.5], 1.0, 1.1]: config-5 cars have none), grids at 0.1 m.  Three checks of the same poses:
    K1 (hl_collision_check, flags 3 | HL_CHECK_AUX, per-pose environment ids), a loop of one hl_grid_footprint_check_batch
    call per scenario (one map, that scenario's poses), and one hl_grid_footprint_check_batch over all maps.
Before timing, the tool asserts that batch and loop agree byte for byte on both workloads and counts K1-hit /
grid-free poses (must be 0: the grid is conservative) and grid-only hits.  Timed with CUDA events around work that ends
in a device synchronisation (tables and buffers are prepared outside the window); the loop and the batch (and K1)
alternate in the same process, median of --reps after one warm-up of each.  Prints one JSON line (and writes --out)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
import numpy as np  # noqa: E402
import torch  # noqa: E402

from headland_trajectory_planning_b200 import _lib, ops, scenarios  # noqa: E402
from headland_trajectory_planning_b200 import headland_path_planning as HP  # noqa: E402
from headland_trajectory_planning_b200.car_model import CarModel  # noqa: E402
from headland_trajectory_planning_b200.env_batch import EnvBatch, EnvRecord, make_record  # noqa: E402
from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment  # noqa: E402

L2_BYTES = 126 * 2**20
MOWER_AUX = np.array([[-1.84, -1.84 + 1.1, 0.5 - 1.0, 0.5]])          # CarModel's extents of [[-1.84, 0.5], 1.0, 1.1]
YPARK = (0.35, 0.55, 2.0, 2.5, 1.4, 0.7, 0.22, 0.50)                  # bench.py's Y-park sweep parameters


def C_void(p):
    return ctypes.c_void_p(p)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [v.strip() for v in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def events_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def alternate(fns, reps):
    """one warm-up of each, then `reps` rounds running each once per round; median ms per name"""
    for fn in fns.values():
        events_ms(fn)
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            ts[k].append(events_ms(fn))
    return {k: (float(np.median(v)), [round(x, 3) for x in v]) for k, v in ts.items()}


def records(n):
    recs, specs = [], []
    for i in range(n):
        sp = scenarios.scenario_spec(i)
        env = OrchardGeometryEnvironment(sp["rows"], [], tree_width=sp["tree_width"], headland_width=sp["headland_width"])
        recs.append(make_record(env, CarModel(**sp["car"])))
        specs.append(sp)
    return recs, specs


def pack_workload(lib, ctx, st, recs, envs, res, margin, reps):
    wins = [(k,) + tuple(ops.raster_window(r.field, res, margin)) for k, r in enumerate(recs)]
    grids = ops.rasterize(envs, wins, res, 3)
    storage = grids[0].untyped_storage()
    base = storage.data_ptr()
    shapes = [(w, h) for (_, _, _, w, h) in wins]
    words = np.array([(w * h + 31) // 32 for w, h in shapes], dtype=np.int64)
    woff = np.concatenate([[0], np.cumsum(words)])[:-1]
    total = int(words.sum())
    loop_bits = torch.empty(total, dtype=torch.int32, device="cuda")
    batch_bits = torch.empty(total, dtype=torch.int32, device="cuda")
    table = (_lib.HlGridPack * len(grids))(*[_lib.HlGridPack(g.data_ptr() - base, int(o), w, h)
                                              for g, o, (w, h) in zip(grids, woff, shapes)])
    args = [(_lib.ptr(g), w, h, C_void(loop_bits.data_ptr() + 4 * int(o))) for g, o, (w, h) in zip(grids, woff, shapes)]

    def loop():
        for a in args:
            _lib.check(lib.hl_grid_pack(ctx, a[0], a[1], a[2], a[3], st), "hl_grid_pack")

    def batch():
        _lib.check(lib.hl_grid_pack_batch(ctx, C_void(base), storage.nbytes(), table, len(grids), _lib.ptr(batch_bits), total, st),
                   "hl_grid_pack_batch")

    loop_bits.fill_(-1); batch_bits.fill_(0)
    loop(); batch()
    torch.cuda.synchronize()
    assert torch.equal(loop_bits, batch_bits), f"pack: batch differs from the loop at res {res}"
    t = alternate({"loop": loop, "batch": batch}, reps)
    cells = int(sum(w * h for w, h in shapes))
    row = {"res_m": res, "grids": len(grids), "cells": cells, "byte_grid_bytes": cells, "packed_bytes": 4 * total,
           "byte_grids_larger_than_l2": cells > L2_BYTES, "packed_larger_than_l2": 4 * total > L2_BYTES,
           "batch_equals_loop": True}
    for k, (ms, all_) in t.items():
        row[k] = {"ms": round(ms, 3), "ms_all": all_, "cells_per_s": round(cells / (ms * 1e-3))}
    row["loop_over_batch"] = round(t["loop"][0] / t["batch"][0], 2)
    return row


def check_workload(lib, ctx, st, recs, specs, res, margin, reps):
    n = len(recs)
    vrecs = [EnvRecord(r.obs, r.field, r.body_ext, MOWER_AUX) for r in recs]
    envs = EnvBatch(vrecs)
    # the sweep's candidate paths, as bench.py's Y-park stage builds them
    ends, bdirs, wbs = [], [], []
    for i, sp in enumerate(specs):
        end = np.array(sp["end"], dtype=np.float64)
        shift = (0.0, 1.5, 3.0)[i % 3]
        end[0] -= shift * np.cos(end[2]); end[1] -= shift * np.sin(end[2])
        ends.append(end)
        bdirs.append(float(HP.get_backward_steer_dir_for_y_type_parking(sp["start"], end)))
        wbs.append(CarModel(**sp["car"]).WHEEL_BASE)
    cands = HP.y_park_candidates(*YPARK)
    c = len(cands)
    rows = np.empty((n, c, 8))
    rows[:, :, :2] = cands[None, :, :2]
    rows[:, :, 2] = cands[None, :, 2] * np.array(bdirs)[:, None]
    rows[:, :, 3] = cands[None, :, 3] * -np.array(bdirs)[:, None]
    rows[:, :, 4:7] = np.array(ends)[:, None, :]
    rows[:, :, 7] = np.array(wbs)[:, None]
    poses, offsets = ops.ypark_paths(rows.reshape(-1, 8), 0.1)
    offsets_d = torch.from_numpy(offsets).cuda()
    counts = offsets_d[1:] - offsets_d[:-1]
    path_of = torch.repeat_interleave(torch.arange(n * c, device="cuda"), counts)
    pose_idx = (torch.arange(poses.shape[0], device="cuda") - offsets_d[path_of]).to(torch.int32)
    map_id = (path_of // c).to(torch.int32)
    n_poses = int(poses.shape[0])
    # grids, packed in one batch
    wins = [(k,) + tuple(ops.raster_window(r.field, res, margin)) for k, r in enumerate(vrecs)]
    grids = ops.rasterize(envs, wins, res, 3)
    bits, woff = ops.grid_pack_batch(grids)
    maps = (_lib.HlGridMap * n)()
    for k, ((_, i0, j0, w, h), r) in enumerate(zip(wins, vrecs)):
        m = maps[k]
        m.bits_offset, m.w, m.h, m.i0, m.j0 = int(woff[k]), w, h, i0, j0
        m.body_ext[:] = [float(v) for v in r.body_ext]
        m.aux_first, m.n_aux = 0, 1
    aux = np.ascontiguousarray(MOWER_AUX)
    scen_first = offsets[np.arange(n) * c]                 # pose range of scenario k (its candidates are contiguous)
    scen_end = np.append(scen_first[1:], n_poses)
    out_k1 = torch.empty(n_poses, dtype=torch.uint8, device="cuda")
    out_loop = torch.empty_like(out_k1)
    out_batch = torch.empty_like(out_k1)
    flags = ops.CHECK_OBSTACLES | ops.CHECK_BOUNDARY | ops.CHECK_AUX
    one = [(_lib.HlGridMap * 1)(maps[k]) for k in range(n)]
    loop_args = [(one[k], C_void(poses.data_ptr() + 24 * int(a)), C_void(pose_idx.data_ptr() + 4 * int(a)),
                  int(b - a), C_void(out_loop.data_ptr() + int(a))) for k, (a, b) in enumerate(zip(scen_first, scen_end))]

    def k1():
        _lib.check(lib.hl_collision_check(envs.ctx, envs.handle, _lib.ptr(map_id), _lib.ptr(poses), _lib.ptr(pose_idx), n_poses,
                                          flags, _lib.ptr(out_k1), None, st), "hl_collision_check")

    def loop():
        for t, p, q, m, o in loop_args:
            _lib.check(lib.hl_grid_footprint_check_batch(ctx, _lib.ptr(bits), bits.numel(), t, 1, _lib.dptr(aux), 1, res, None,
                                                         p, q, m, ops.CHECK_AUX, o, st), "hl_grid_footprint_check_batch")

    def batch():
        _lib.check(lib.hl_grid_footprint_check_batch(ctx, _lib.ptr(bits), bits.numel(), maps, n, _lib.dptr(aux), 1, res,
                                                     _lib.ptr(map_id), _lib.ptr(poses), _lib.ptr(pose_idx), n_poses, ops.CHECK_AUX,
                                                     _lib.ptr(out_batch), st), "hl_grid_footprint_check_batch")

    out_loop.fill_(7); out_batch.fill_(9)
    k1(); loop(); batch()
    torch.cuda.synchronize()
    assert torch.equal(out_loop, out_batch), "check: batch differs from the loop"
    a, g = out_k1.bool(), out_batch.bool()
    k1_only, grid_only = int((a & ~g).sum()), int((g & ~a).sum())
    assert k1_only == 0, f"{k1_only} poses K1 finds infeasible are free on the grid"
    t = alternate({"k1": k1, "loop": loop, "batch": batch}, reps)
    path_bad = ops.path_reduce(envs, out_batch, offsets_d)
    row = {"res_m": res, "scenarios": n, "candidates_per_scenario": c, "paths": n * c, "poses": n_poses,
           "implements_per_vehicle": 1, "packed_bytes": 4 * bits.numel(), "pose_bytes": 24 * n_poses + 4 * n_poses,
           "working_set_larger_than_l2": 4 * bits.numel() + 28 * n_poses > L2_BYTES, "batch_equals_loop": True,
           "k1_hits": int(a.sum()), "grid_hits": int(g.sum()), "k1_hit_grid_free": k1_only, "grid_only_hits": grid_only,
           "paths_free_on_grid": int((path_bad == 0).sum())}
    for k, (ms, all_) in t.items():
        row[k] = {"ms": round(ms, 3), "ms_all": all_, "checks_per_s": round(n_poses / (ms * 1e-3))}
    row["loop_over_batch"] = round(t["loop"][0] / t["batch"][0], 2)
    row["k1_over_batch"] = round(t["k1"][0] / t["batch"][0], 2)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-env", type=int, default=4096)
    ap.add_argument("--res", type=float, nargs="+", default=[0.1, 0.2])
    ap.add_argument("--scenarios", type=int, default=256)
    ap.add_argument("--check-res", type=float, default=0.1)
    ap.add_argument("--margin", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "grid_batch_bench needs a CUDA device"
    torch.cuda.set_device(0)
    info = gpu_info()
    lib = _lib.load_library()
    ctx, st = _lib.get_ctx(), _lib.stream_ptr()
    recs, specs = records(max(args.n_env, args.scenarios))
    envs = EnvBatch(recs[:args.n_env])
    result = {"metric": "grid_batch", "gpu": info, "l2_bytes": L2_BYTES,
              "timing": f"CUDA events, device synchronised, loop / batch alternating, median of {args.reps} after one warm-up",
              "pack": [], "check": None}
    for res in args.res:
        result["pack"].append(pack_workload(lib, ctx, st, recs[:args.n_env], envs, res, args.margin, args.reps))
        torch.cuda.empty_cache()
    result["check"] = check_workload(lib, ctx, st, recs[:args.scenarios], specs[:args.scenarios], args.check_res,
                                     args.margin, args.reps)
    result["ok"] = True
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
