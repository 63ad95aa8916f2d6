#!/usr/bin/env python
"""bench.py -- warm-start plans/sec on B200 (BASELINE.json metric), config 5:
synthetic headland scenarios (varied row spacing, headland width, vehicle length), King
mode, step 0.2 m, max_nodes 400, sharded over the GPUs of one box.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU reference arm

One "step" = one pass of the batched Hybrid A* search over this rank's scenarios.
`value` = scenarios of ALL ranks / max-over-ranks device time with environments and
scenarios already resident in HBM; `e2e` = the same through the host-buffer API (H2D of
environment geometry + scenario records, search, D2H of result records, expanded-key
sequences and paths, plus the NCCL gather to rank 0 when N > 1).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "warm_start_plans_per_sec"
UNIT = "plans/s"
WORKLOAD = "config5: synthetic headland scenarios (8 rows, row spacing U(2.2,4.0) m, headland U(5,9) m, " \
           "axle_to_front U(2.85,4.5) m), King, step 0.2 m, max_nodes 400"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenarios-per-gpu", type=int, default=4096)
    ap.add_argument("--cpu-sample", type=int, default=0, help="scenarios in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--collision-poses", type=int, default=1 << 24)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed search step computed as DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU search's outputs: it needs --impl ours")
    return args


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run_nvml(self):
        """Dense sampling through NVML (a few ms per sample) so that even a 150 ms timed region gets a median."""
        nv, h, mx = self._nvml
        bits = [(0x8, 2), (0x40, 3), (0x20, 4), (0x4, 5)]      # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        while not self._stop.is_set():
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            row = [str(sm), str(mx), "", "", "", ""]
            for mask, col in bits:
                row[col] = "Active" if (r & mask) else "Not Active"
            self.rows.append(row)
            self._stop.wait(0.005)

    def _run(self):
        if self._nvml is not None:
            try:
                self._run_nvml()
                return
            except Exception as exc:           # fall back to nvidia-smi below
                print(f"[bench] NVML sampling failed ({exc!r}); using nvidia-smi", file=sys.stderr)
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._nvml = None
        try:                                   # initialise NVML BEFORE the timed region starts
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self._nvml = (nv, h, nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def scenario_indices(args, rank, world):
    total = args.scenarios_per_gpu * world
    return list(range(rank, total, world)), total


def cpu_sample_size(args, cores):
    return args.cpu_sample if args.cpu_sample > 0 else int(min(128, max(8, 4 * cores)))


def run_reference(args, rank, world):
    """CPU arm: the oracle port of the reference's Python path on the host cores."""
    if rank != 0:
        return
    from oracle import baseline as OB
    from headland_trajectory_planning_b200 import scenarios as SC
    cores = os.cpu_count() or 1
    # size the per-step sample so that the whole run stays within a few minutes:
    # ~6 s of search per scenario on average, spread over `cores` workers
    # At least 4 scenarios per core and step: with one scenario per core the wall of every step is the ONE slowest
    # (401-pop, ~30 s) scenario and the pool idles -- that understated the CPU arm 3.7x in round 1.
    # (64 scenarios take ~7.5 s on 16 cores, so the driver's 20 + 5 steps stay within ~3 minutes.)
    n = args.cpu_sample if args.cpu_sample > 0 else int(min(128, max(32, 4 * cores)))
    specs = [SC.scenario_spec(i) for i in range(n)]
    scns = [SC.finalize(sp, OB.candidate_feasibility(sp)) for sp in specs]
    for _ in range(args.warmup):
        OB.run_pool(scns[: max(1, n // 8)], cores)
    wall = 0.0
    for _ in range(args.steps):
        _, dt, used = OB.run_pool(scns, cores)
        wall += dt
    value = n * args.steps / wall
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": f"scenarios 0..{n - 1} per step ({n / used:.1f} per core)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port",
                             "sample": f"scenarios 0..{n - 1} of the workload, oracle port (shapely/heapdict "
                                       f"unavailable), multiprocessing.Pool({used})"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_JSON_FD = None


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything libraries print to fd 1 meanwhile (NCCL's
    version banner, worker chatter) has been diverted to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    args = parse()
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    from headland_trajectory_planning_b200 import _lib, ops, scenarios as SC, sweep
    from headland_trajectory_planning_b200.env_batch import EnvBatch, pack_structs
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    # ---------------- setup (untimed): scenarios, host geometry, resident copies
    idx, total = scenario_indices(args, rank, world)
    t_setup = time.time()
    scns = SC.make_scenarios_gpu(idx)
    recs, scen, car = sweep.build_records(scns)
    params = sweep.search_params(car)
    envs = EnvBatch(recs)
    n = len(scns)
    path_cap = 1024 * n
    d_scen = torch.from_numpy(scen.view(np.uint8).reshape(-1)).to(dev)
    setup_s = time.time() - t_setup
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # untimed: bring the SM clocks out of idle (a cold GPU ramps from ~120 MHz over several hundred ms)
    t_ramp = time.time()
    while time.time() - t_ramp < 1.0:
        ops.hybrid_astar_batch(envs, d_scen, params, path_capacity=path_cap, to_host=False)
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident steps
    for _ in range(args.warmup):
        out = ops.hybrid_astar_batch(envs, d_scen, params, path_capacity=path_cap, to_host=False)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clocks:
        barrier()
        for s in range(args.steps):
            flush.fill_(s & 0xFF)                       # L2 flush between timed iterations
            ev[s][0].record()
            out = ops.hybrid_astar_batch(envs, d_scen, params, path_capacity=path_cap, to_host=False)
            ev[s][1].record()
        barrier()
    kernel_ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    value = total * args.steps / (max_ms * 1e-3)

    # strong scaling (N > 1 only): the SAME 4096 scenarios split over the N ranks; every rank searches the first
    # 4096 / N scenarios of its interleaved shard.  One 401-pop scenario alone takes ~15 ms, so this cannot scale
    # like the weak run: the floor is the latency of the slowest scenario, and the line says so.
    strong = None
    if world > 1:
        m = max(1, args.scenarios_per_gpu // world)
        d_sub = d_scen[: m * _lib.SCENARIO_DTYPE.itemsize]
        for _ in range(2):
            ops.hybrid_astar_batch(envs, d_sub, params, path_capacity=path_cap, to_host=False)
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for s in range(args.steps):
            flush.fill_(s & 0xFF)
            evs[s][0].record()
            ops.hybrid_astar_batch(envs, d_sub, params, path_capacity=path_cap, to_host=False)
            evs[s][1].record()
        barrier()
        ts = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], dtype=torch.float64, device=dev)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        strong = {"scaling": "strong", "total_scenarios": m * world, "scenarios_per_gpu": m,
                  "ms_per_step": float(ts.item()) / args.steps, "value": m * world * args.steps / (float(ts.item()) * 1e-3),
                  "unit": UNIT, "floor": "one max_nodes scenario alone on a GPU takes ~10 ms and ~13-17 ms next to others on its SM (profiles/r2u_k4_lockstep_probe.txt): "
                                         "with the sweep's 546 such scenarios the step time cannot drop below that however many GPUs share them"}

    res = out["results"].cpu().numpy().view(_lib.RESULT_DTYPE)
    flops = sweep.algorithmic_flops(recs, res)                              # reference-equivalent checks x F_check
    flops_exec = sweep.algorithmic_flops(recs, res, field="n_pose_checks")   # what the kernel actually executed
    n_checks = int(res["n_pose_checks"].sum())
    n_checks_ref = int(res["n_pose_checks_ref"].sum())
    n_exact = int(res["n_exact"].sum())
    status_hist = {_lib.STATUS_NAMES[int(k)]: int(v) for k, v in zip(*np.unique(res["status"], return_counts=True))}
    expansions = int(res["n_expanded"].sum())

    # ---------------- end-to-end steps: host buffers in, host buffers out
    host_scen = torch.from_numpy(scen.view(np.uint8).reshape(-1).copy()).pin_memory()
    host_structs = pack_structs(recs)          # HlEnvHost records over the host geometry buffers
    h2d = int(sum(r.obs.nbytes + r.field.nbytes + r.seg_xy.nbytes + r.seg_polys.nbytes + r.seg_len.nbytes +
                  r.crit.nbytes + r.guide.nbytes + r.aux.nbytes + 32 for r in recs) + host_scen.numel())
    d2h = 0
    def e2e_steps(pf, dl, k_steps):
        """k_steps pipelined steps.  Every step uploads its own inputs from host memory (environment geometry through
        hl_env_upload, scenario records) and downloads its own results (records, key sequences, paths; over NCCL to
        rank 0 when N > 1) into host memory; the upload of step k+1 (worker thread, the context's copy stream) and the
        device -> host copy + merge of step k-1 (side stream, copy engine) overlap the search of step k."""
        nbytes = 0
        pending = None
        pf.submit(recs, host_structs)                                       # H2D environment geometry of step 0
        for s in range(k_steps):
            envs_e = pf.result()
            if s + 1 < k_steps:
                pf.submit(recs, host_structs)                               # ... of step s+1, behind step s's search
            d_s = host_scen.to(dev, non_blocking=True)                      # H2D scenario records
            o = ops.hybrid_astar_batch(envs_e, d_s, params, path_capacity=path_cap, to_host=False)   # queued
            done = dl.finish(pending, total) if pending is not None else None                      # step s-1 on the host
            # size exchange (returns when search s is finished), NVLink gatherv to rank 0, D2H queued on the side stream
            pending = dl.begin(o, release=envs_e.close)
            if done is not None:
                nbytes = int(done["results"].nbytes + done["expanded"].nbytes + sum(done[k].nbytes for k in ("x", "y", "yaw", "k", "dir")))
        done = dl.finish(pending, total)
        if done is not None:
            nbytes = int(done["results"].nbytes + done["expanded"].nbytes + sum(done[k].nbytes for k in ("x", "y", "yaw", "k", "dir")))
            assert len(done["results"]) == total and int((done["results"]["status"] >= 0).sum()) == total
        return nbytes

    pf = sweep.UploadPrefetcher()
    dl = sweep.SweepDownloader(world, rank)
    e2e_steps(pf, dl, max(3, args.warmup))                                  # untimed warm-up of the very same path
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d2h = e2e_steps(pf, dl, args.steps)                                     # EXACTLY K timed steps
    torch.cuda.synchronize()
    barrier()
    e2e_wall = time.perf_counter() - t0
    pf.close()
    t = torch.tensor([e2e_wall, float(h2d)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t[:1], op=dist.ReduceOp.MAX)
        dist.all_reduce(t[1:], op=dist.ReduceOp.SUM)
    e2e_value = total * args.steps / float(t[0].item())
    h2d = int(t[1].item())                                                  # whole job: every rank uploads its shard

    # ---------------- secondary: stand-alone collision kernel (M2) on the canonical scenario
    coll = None
    coll_paths = None
    ypark = None
    rs_sweep = None
    refpath = None
    dfield = None
    single = None
    fp32_peak = None
    if rank == 0:
        fp32_peak = ops.measure_fp32_peak(local_rank)
        coll = collision_microbench(args, dev, fp32_peak)
        args.collision_mode = "paths"
        args.collision_poses = min(args.collision_poses, 1 << 23)
        coll_paths = collision_microbench(args, dev, fp32_peak)
        ypark = ypark_microbench(args, dev, world == 1 and not args.no_cpu_baseline)
        rs_sweep = rs_microbench(args, dev, world == 1 and not args.no_cpu_baseline)
        refpath = refpath_microbench(out, car.WHEEL_BASE, world == 1 and not args.no_cpu_baseline)
        dfield = distance_field_microbench(dev, world == 1 and not args.no_cpu_baseline)
        single = single_scenario_microbench(dev)

    # ---------------- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import baseline as OB
        cores = os.cpu_count() or 1
        m = min(n, cpu_sample_size(args, cores))
        _, dt, used = OB.run_pool(scns[:m], cores)
        cpu = {"value": m / dt, "unit": UNIT, "cores": used, "kind": "port",
               "sample": f"first {m} scenarios of rank 0's shard, oracle port of the reference's Python path "
                         f"(shapely/heapdict unavailable), multiprocessing.Pool({used}), search time only"}

    if rank == 0 and args.dump_outputs:                # with N > 1 GPUs: rank 0's shard
        dump_outputs(args.dump_outputs, out, res, idx)

    if rank == 0:
        ms_per_launch = max_ms / args.steps
        achieved = flops / (kernel_ms / args.steps * 1e-3) * 1e-12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_launch, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "scenarios_per_gpu": args.scenarios_per_gpu, "total_scenarios": total,
                       "sharding": "scenario i -> rank i mod N", "l2": "flushed (256 MiB fill) between timed iterations",
                       "setup_s_untimed": round(setup_s, 1)},
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": args.steps * ops.astar_launches_per_call(envs, n),
            "roofline": {"bound": "alu_fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp32_peak if fp32_peak else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one k_hybrid_astar_s launch on this very
                         # workload (4096 scenarios; the search launch of the two-phase sweep), ncu --set full,
                         # profiles/r2u_k4_ncu_full_summary.txt (170.2 MB read + 281.5 MB written: node / hash /
                         # open-list scratch of 740 scenario slots)
                         "traffic": 451706112 if args.scenarios_per_gpu == 4096 else None,
                         "kernel": "k_hybrid_astar_s",
                         # the same launch against the HBM roof (SURVEY 8d: this path is not bandwidth-bound): algorithmic
                         # bytes = environments + scenario records in, result records + key sequences + paths out
                         "hbm": hbm_view(h2d + d2h, kernel_ms / args.steps),
                         "executed_frac": (flops_exec / (kernel_ms / args.steps * 1e-3) * 1e-12 / fp32_peak) if fp32_peak else None,
                         "note": "no tensor cores on this path; algorithmic flop = pose checks the REFERENCE performs "
                                 "for the same searches (poses of every Reeds-Shepp word tried + of every primitive "
                                 "rolled out; HlPlanResult.n_pose_checks_ref, equal to the oracle's tally) x F_check "
                                 "(SURVEY 8d); executed_frac counts only the checks the kernel ran after its early "
                                 "exits; peak = FFMA micro-benchmark measured in this run; the kernel is a "
                                 "latency-bound search, see kernels.k_collision for the ALU-bound kernel"},
            "kernels": {"k_collision": coll, "k_collision_path_ordered": coll_paths, "ypark_sweep": ypark, "rs_sweep": rs_sweep, "ref_path": refpath,
                        "distance_field": dfield, "single_scenario": single},
            "search": {"expansions": expansions, "pose_checks": n_checks, "pose_checks_algorithmic": n_checks_ref,
                       "exact_escalations": n_exact,
                       "status": status_hist},
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if strong:
            line["strong_scaling"] = strong
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_BUDGET = (64 << 20) - (64 << 10)          # array bytes; the rest of 64 MB is room for the .npy headers
# Fields of HlPlanResult that describe the plan.  Left out because they change from run to run: path_offset and
# keys_offset (positions in the pools, handed out by atomics), cycles (a clock reading), n_pose_checks and n_exact
# (checks executed after the early exits, which depend on the order warps finish in).
DUMP_FIELDS = ("status", "counter", "n_expanded", "arrival", "path_len", "rs_word", "goal_cost", "n_pose_checks_ref")


def _ragged(starts, lens):
    """Row indices starts[i] .. starts[i] + lens[i] - 1 for every i, concatenated."""
    ends = np.cumsum(lens)
    return np.repeat(starts - (ends - lens), lens) + np.arange(int(ends[-1]) if len(ends) else 0)


def dump_outputs(dirname, out, res, scenario_index):
    """Write one hybrid_astar_batch output as float64 ``dirname/<name>.npy``, scenario by scenario: the result fields,
    the expanded keys [rows, 3] and the path arrays, both pools regrouped in scenario order.  If everything would
    exceed DUMP_BUDGET, scenarios are taken in a fixed seeded order until the budget is spent; ``scenario_index`` names
    the scenarios written, in the order their rows appear."""
    n_exp = res["n_expanded"].astype(np.int64)
    n_path = res["path_len"].astype(np.int64)
    nbytes = 8 * (len(DUMP_FIELDS) + 1 + 3 * n_exp + 5 * n_path)
    sel = np.arange(len(res))
    if nbytes.sum() > DUMP_BUDGET:
        order = np.random.default_rng(0).permutation(len(res))
        sel = np.sort(order[:int(np.searchsorted(np.cumsum(nbytes[order]), DUMP_BUDGET, side="right"))])
    kused, used = (int(v) for v in np.concatenate([out["kcursor"].cpu().numpy(), out["cursor"].cpu().numpy()]))
    arrays = {"scenario_index": np.asarray(scenario_index)[sel]}
    arrays.update({"result_" + f: res[f][sel] for f in DUMP_FIELDS})
    arrays["expanded_keys"] = out["expanded"][:kused].cpu().numpy()[_ragged(res["keys_offset"][sel], n_exp[sel])]
    rows = _ragged(res["path_offset"][sel], n_path[sel])
    for name in ("x", "y", "yaw", "k", "dir"):
        arrays["path_" + name] = out[name][:used].cpu().numpy()[rows]
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a, dtype=np.float64))


def collision_microbench(args, dev, fp32_peak):
    """Footprint collision checks/sec (metric M2) of hl_collision_check on the canonical
    scenario (8 tree rows, 16-vertex field polygon, 4-segment lane; obstacles + boundary +
    lane, body only), poses resident in HBM, CUDA-event timed, L2 flushed."""
    import math
    import torch
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.car_model import CarModel
    from headland_trajectory_planning_b200.env_batch import EnvBatch, make_record
    from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment
    from headland_trajectory_planning_b200.reference_line_heuristic import ReferenceLineHeuristic
    from headland_trajectory_planning_b200.utils import map_utils
    np.random.seed(1)
    rows = map_utils.create_tree_rows(8, 2.5, 20, slope_angle=math.radians(10), l_std=0.0)
    env = OrchardGeometryEnvironment(rows, [], tree_width=0.3, headland_width=6.0)
    car = CarModel(max_steer=0.55, axle_to_front=3, axle_to_back=0.55, width=1.48)
    ends = rows[:, 0, :]
    way = np.vstack(([0.88, 3.75], [[ends[i, 0] - 4.5, ends[i, 1]] for i in (2, 3, 4)], [-1.2, 11.25]))
    heur = ReferenceLineHeuristic(way, [-1.2, 11.25, 0.0], car)
    envs = EnvBatch([make_record(env, car, heur)])
    n = args.collision_poses
    g = torch.Generator(device=dev).manual_seed(0)
    if getattr(args, "collision_mode", "random") == "paths":
        # poses in PATH order (what check_path_feasibility sees): Reeds-Shepp words between random headland
        # poses, sampled on the GPU at 0.1 m (hl_rs_all_paths + hl_rs_sample), concatenated
        rng = np.random.default_rng(0)
        n_pairs = max(1024, n // 640)
        sg = np.empty((n_pairs, 6))
        sg[:, [0, 3]] = rng.uniform(-8.0, 1.0, (n_pairs, 2))
        sg[:, [1, 4]] = rng.uniform(0.0, 18.0, (n_pairs, 2))
        sg[:, [2, 5]] = rng.uniform(-math.pi, math.pi, (n_pairs, 2))
        words, count, _ = ops.rs_all_paths(sg, car.curvature, 0.1, want_order=False)
        w = ops.rs_words_to_host(words)
        cnt = count.cpu().numpy()
        sel = [(i, k) for i in range(n_pairs) for k in range(cnt[i])]
        starts = np.array([sg[i, :3] for i, _ in sel])
        wsel = np.array([w[i, k] for i, k in sel])
        _, px, py, pyaw, _, _ = ops.rs_sample(starts, wsel, car.curvature, 0.1)
        poses = torch.from_numpy(np.stack([px, py, pyaw], axis=1)[:n].copy()).to(dev)
        n = poses.shape[0]
    else:
        poses = torch.empty((n, 3), dtype=torch.float64, device=dev)
        poses[:, 0] = torch.rand(n, generator=g, device=dev, dtype=torch.float64) * 14.0 - 10.0
        poses[:, 1] = torch.rand(n, generator=g, device=dev, dtype=torch.float64) * 22.0 - 2.0
        poses[:, 2] = (torch.rand(n, generator=g, device=dev, dtype=torch.float64) * 2.0 - 1.0) * math.pi
    flags = int(os.environ.get("HL_K1_FLAGS", ops.CHECK_OBSTACLES | ops.CHECK_BOUNDARY | ops.CHECK_LANE))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        out, nex = ops.collision_check(envs, poses, flags=flags, count_exact=True)
    torch.cuda.synchronize()
    ms = 0.0
    reps = 5
    for r in range(reps):
        flush.fill_(r)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = ops.collision_check(envs, poses, flags=flags)
        b.record()
        torch.cuda.synchronize()
        ms += a.elapsed_time(b)
    ms /= reps
    f_check = 32 + 128 * 8 + 80 * 16 + 48 * 4
    checks = n / (ms * 1e-3)
    achieved = checks * f_check * 1e-12
    return {"metric": "footprint_collision_checks_per_sec", "value": checks, "unit": "checks/s", "poses": n,
            "pose_order": getattr(args, "collision_mode", "random"),
            "ms_per_launch": ms, "f_check_flop": f_check, "infeasible_frac": float(out.float().mean().item()),
            "exact_escalation_frac": float(nex.item()) / n,
            "roofline": {"bound": "alu_fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp32_peak if fp32_peak else None,
                         "hbm_GBps": checks * 25 * 1e-9,
                         # 30.6 B of DRAM traffic per pose (ncu --set full, 4 Mi poses, profiles/r2s_k1_ncu_full_summary.txt:
                         # 103.1 MB read + 25.4 MB written) against 25 B algorithmic (24 B pose in + 1 B flag out)
                         "traffic": int(30.6 * n)}}


def hbm_view(bytes_per_launch, ms_per_launch):
    peak = None
    try:
        peak = float(json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        peak = 6549.1                   # the pool's measured copy bandwidth (MEASURED_PEAKS.json at build time)
    achieved = bytes_per_launch / (ms_per_launch * 1e-3) * 1e-9
    return {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak}


def refpath_microbench(out, wheel_base, with_cpu):
    """SURVEY 8(f) rank 4: the sweep's paths (still on the GPU) -> OBCA initial guesses (K8)."""
    import time
    import torch
    from headland_trajectory_planning_b200 import _lib, obca_util as GU
    GU.get_init_ref_path_batch(out, wheel_base)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        traj, off, status = GU.get_init_ref_path_batch(out, wheel_base)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    n_paths = int((np.diff(off) > 0).sum())
    res = {"metric": "ref_paths_per_sec", "value": n_paths / dt, "unit": "paths/s", "paths": n_paths,
           "rows": int(off[-1]), "ms_per_batch": dt * 1e3, "scenarios_without_rows": int(status.sum())}
    if with_cpu:
        from oracle import obca_util as OU
        r = out["results"].cpu().numpy().view(_lib.RESULT_DTYPE)
        x, y, d = out["x"].cpu().numpy(), out["y"].cpu().numpy(), out["dir"].cpu().numpy()
        picks = [i for i in range(len(r)) if r["path_len"][i] > 4][:32]
        t0 = time.perf_counter()
        done = 0
        for i in picks:
            a, b = int(r["path_offset"][i]), int(r["path_offset"][i] + r["path_len"][i])
            try:
                OU.get_init_ref_path(wheel_base, x[a:b], y[a:b], x[a:b] * 0, x[a:b] * 0, d[a:b].astype(np.float64))
            except ValueError:
                pass
            done += 1
        res["cpu_baseline"] = {"value": done / (time.perf_counter() - t0), "unit": "paths/s", "cores": 1, "kind": "port",
                               "sample": f"first {done} paths, oracle (scipy CubicSpline like the reference)"}
    return res


def distance_field_microbench(dev, with_cpu):
    """BASELINE config 4: holonomic grid distance field of a 4096 x 4096 occupancy grid (0.05 m cells), King moves
    (hl_distance_field).  Algorithmic bytes per cell: 1 B occupancy in + 8 B float64 cost out (float64 keeps the result
    bit-identical to the reference's sequential sums).  The kernel is bound by the dependency depth of the wavefront
    (thousands of frontier steps), not by HBM -- the line reports both."""
    import time
    import torch
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.utils.occupancy_grid_utils import synthetic_grid
    n = 4096
    occ, goal = synthetic_grid(n, seed=1)
    d_occ = torch.from_numpy(occ.astype(np.uint8)).to(dev)
    ops.distance_field(d_occ, goal, "King")
    torch.cuda.synchronize()
    sweeps, times = 0, []
    for _ in range(5):          # median of 5: the call looks at the host between launch batches, a busy host shows up
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out, sweeps = ops.distance_field(d_occ, goal, "King")
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = sorted(times)[len(times) // 2]
    cells = n * n
    res = {"metric": "distance_field_cells_per_sec", "value": cells / (ms * 1e-3), "unit": "cells/s", "grid": f"{n}x{n}",
           "motion_type": "King", "ms_per_field": ms, "ms_per_field_min": min(times), "timing": "median of 5 fields",
           "relaxation_launches": int(sweeps),
           "reachable_cells": int(torch.isfinite(out).sum().item()),
           "roofline": dict(hbm_view(9 * cells, ms), bound="hbm (nominal; really the wavefront's dependency depth)",
                            algorithmic_bytes=9 * cells)}
    if with_cpu:
        from oracle import distance_field as DF
        rates = {}
        for m in (128, 256):
            o2, g2 = DF.synthetic_grid(m, seed=1)
            t0 = time.perf_counter()
            DF.holonomic_costs_with_obstacles(g2, o2, "King")
            rates[m] = m * m / (time.perf_counter() - t0)
        res["cpu_baseline"] = {"value": rates[256], "unit": "cells/s", "cores": 1, "kind": "port",
                               "sample": "256 x 256 instance of the same generator (128 x 128: "
                                         f"{rates[128]:.0f} cells/s), oracle port pinned bit for bit on the reference's a_star_utils.py",
                               "extrapolated_4096x4096_s": cells / rates[256]}
    return res


def single_scenario_microbench(dev):
    """BASELINE config 2: ONE mower scenario (test/obca.ipynb: 8 rows, tractor + mower implement, King, step 0.2 m,
    max_nodes 400) through the drop-in class -- HybridAStarSearch(...).hybrid_a_star_search(max_nodes=400) -- host
    geometry in, path lists out: environment upload, search and download included.  Latency, not throughput."""
    import contextlib
    import io
    import math
    import time
    import torch
    from headland_trajectory_planning_b200.car_model import CarModel
    from headland_trajectory_planning_b200.hybrid_a_star_search import HybridAStarSearch
    from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment
    from headland_trajectory_planning_b200.reference_line_heuristic import ReferenceLineHeuristic
    from headland_trajectory_planning_b200.utils import map_utils
    np.random.seed(1)
    rows = map_utils.create_tree_rows(8, 2.5, 20, slope_angle=math.radians(10), l_std=0.0)
    env = OrchardGeometryEnvironment(rows, [], tree_width=0.3, headland_width=6.0)
    car = CarModel(max_steer=0.55, axle_to_front=3, axle_to_back=0.55, width=1.48,
                   aux_poly_features=[[[-1.84, 0.5], 1.0, 1.1]], with_aux=True)
    out = {"metric": "single_scenario_latency_ms", "unit": "ms", "config": "mower, King, step 0.2 m, max_nodes 400"}
    for name, start, goal in (("rs_shot_first_pop", map_utils.get_base_pose(1, rows, -1.0, side=map_utils.NEAR_SIDE, pose_type=map_utils.LEAVE_POSE),
                               np.array([-2.11713892, 8.75, 0.0])),
                              ("multi_expansion", map_utils.get_base_pose(1, rows, 0.0, side=map_utils.NEAR_SIDE, pose_type=map_utils.LEAVE_POSE),
                               map_utils.get_base_pose(4, rows, 2.0, side=map_utils.NEAR_SIDE, pose_type=map_utils.ENTER_POSE))):
        ends = rows[:, 0, :]
        way = np.vstack((start[:2], [[ends[i, 0] - 4.5, ends[i, 1]] for i in (2, 3)], goal[:2]))
        heur = ReferenceLineHeuristic(way, goal, car)
        lat = []
        counter = 0
        for rep in range(6):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                r = HybridAStarSearch(start, goal, env, car, heur, motion_type="King", plan_resolution=0.2).hybrid_a_star_search(max_nodes=400)
            lat.append((time.perf_counter() - t0) * 1e3)
            counter = r[5]
        out[name] = {"counter": int(counter), "first_call_ms": lat[0], "warm_ms_median": sorted(lat[1:])[len(lat[1:]) // 2],
                     "path_poses": len(r[0])}
    out["value"] = out["multi_expansion"]["warm_ms_median"]
    return out


def rs_microbench(args, dev, with_cpu):
    """SURVEY 8(d) config 3: Reeds-Shepp words of 1 Mi random pose pairs, every word sampled at 0.1 m and
    collision-checked against the canonical orchard (k_rs_all_paths)."""
    import math
    import time
    import torch
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.car_model import CarModel
    from headland_trajectory_planning_b200.env_batch import EnvBatch, make_record
    from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment
    from headland_trajectory_planning_b200.utils import map_utils
    n = 1 << 20
    rng = np.random.default_rng(0)
    sg = np.empty((n, 6))
    sg[:, [0, 1, 3, 4]] = rng.uniform(-10, 10, (n, 4))
    sg[:, [2, 5]] = rng.uniform(-math.pi, math.pi, (n, 2))
    np.random.seed(1)
    rows = map_utils.create_tree_rows(8, 2.5, 20, slope_angle=math.radians(10), l_std=0.0)
    env = OrchardGeometryEnvironment(rows, [], tree_width=0.3, headland_width=6.0)
    car = CarModel(max_steer=0.55, axle_to_front=3, axle_to_back=0.55, width=1.48)
    envs = EnvBatch([make_record(env, car)])
    d_sg = torch.from_numpy(sg).to(dev)
    # warm-up at full size: the 5.4 GB word table is then served by torch's caching allocator in the timed launches
    words, count, _ = ops.rs_all_paths(d_sg, car.curvature, 0.1, envs=envs, flags=ops.CHECK_OBSTACLES, want_order=False)
    del words
    torch.cuda.synchronize()
    times = []
    for _ in range(3):          # median of 3: a launch that has to cudaMalloc its 5.4 GB word table again shows up as an outlier
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        words, count, _ = ops.rs_all_paths(d_sg, car.curvature, 0.1, envs=envs, flags=ops.CHECK_OBSTACLES, want_order=False)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
        if len(times) < 3:
            del words
    ms = sorted(times)[1]
    out = {"metric": "rs_pairs_per_sec", "value": n / (ms * 1e-3), "unit": "pairs/s", "pairs": n, "ms_per_launch": ms,
           "ms_per_launch_all": [round(t, 2) for t in times], "words": int(count.sum().item())}
    del words
    if with_cpu:
        from oracle import planner as OP
        from oracle import rs_port
        o_env = OP.OrchardGeometryEnvironment(rows, [], tree_width=0.3, headland_width=6.0)
        o_car = OP.CarModel(max_steer=0.55, axle_to_front=3, axle_to_back=0.55, width=1.48)
        m = 128
        t0 = time.perf_counter()
        for i in range(m):
            for p in rs_port.calc_all_paths(*sg[i], o_car.curvature, 0.1):
                o_env.check_path_feasibility(o_car, np.array([p.x, p.y, p.yaw]).T, boundary_check=False)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": m / dt, "unit": "pairs/s", "cores": 1, "kind": "port",
                               "sample": f"first {m} pairs: rs_port.calc_all_paths (bit-equal to the reference's "
                                         "reeds_shepp.py) + oracle collision check of every word"}
    return out


def ypark_microbench(args, dev, with_cpu):
    """SURVEY 8(f) rank 1: the Y-type parking sweep that produces the search goal, as a batch stage
    (hl_ypark_paths + hl_collision_check + hl_path_reduce) over 256 config-5 environments with the defaults of
    headland_planner_y_type_park (858 candidates each, step 0.1 m); host arrays in, chosen candidates out."""
    import time
    import torch
    from headland_trajectory_planning_b200 import headland_path_planning as HP, scenarios as SC
    from headland_trajectory_planning_b200.car_model import CarModel
    from headland_trajectory_planning_b200.env_batch import EnvBatch, make_record
    from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment
    n = 256
    ps = (0.35, 0.55, 2.0, 2.5, 1.4, 0.7, 0.22, 0.50)
    step = 0.1
    specs = [SC.scenario_spec(i) for i in range(n)]
    recs, ends, bdirs, wbs = [], [], [], []
    for i, sp in enumerate(specs):
        env = OrchardGeometryEnvironment(sp["rows"], [], tree_width=sp["tree_width"], headland_width=sp["headland_width"])
        car = CarModel(**sp["car"])
        recs.append(make_record(env, car))
        end = np.array(sp["end"], dtype=np.float64)
        shift = (0.0, 1.5, 3.0)[i % 3]
        end[0] -= shift * np.cos(end[2]); end[1] -= shift * np.sin(end[2])
        ends.append(end)
        bdirs.append(float(HP.get_backward_steer_dir_for_y_type_parking(sp["start"], end)))
        wbs.append(car.WHEEL_BASE)
    envs = EnvBatch(recs)
    cands = HP.y_park_candidates(*ps)
    for _ in range(2):
        first, feas, goal = HP.search_y_type_parking_path_batch(envs, np.arange(n), np.array(ends), bdirs, wbs, cands, step)
    torch.cuda.synchronize()
    reps, ms = 3, 0.0
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        first, feas, goal = HP.search_y_type_parking_path_batch(envs, np.arange(n), np.array(ends), bdirs, wbs, cands, step)
        b.record()
        torch.cuda.synchronize()
        ms += a.elapsed_time(b)
    ms /= reps
    poses = int(((np.rint(cands[:, 0] / step) + np.rint(cands[:, 1] / step) + 2).sum()) * n)
    out = {"metric": "ypark_sweeps_per_sec", "value": n / (ms * 1e-3), "unit": "sweeps/s", "sweeps": n,
           "candidates_per_sweep": int(len(cands)), "poses_checked": poses, "ms_per_batch": ms,
           "candidates_per_sec": n * len(cands) / (ms * 1e-3), "found": int((first >= 0).sum())}
    if with_cpu:
        from oracle import planner as OP
        import contextlib
        import io
        m = 6
        t0 = time.perf_counter()
        agree = 0
        for i in range(m):
            sp = specs[i]
            env = OP.OrchardGeometryEnvironment(sp["rows"], [], tree_width=sp["tree_width"], headland_width=sp["headland_width"])
            car = OP.CarModel(**sp["car"])
            with contextlib.redirect_stdout(io.StringIO()):
                _, par = OP.search_y_type_parking_path(car, env, ends[i], bdirs[i], -bdirs[i], *ps, step_size=step, debug=True)
            agree += int((len(par) > 0) == (first[i] >= 0) and (len(par) == 0 or np.array_equal(np.array(par), cands[first[i]])))
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": m / dt, "unit": "sweeps/s", "cores": 1, "kind": "port",
                               "sample": f"first {m} sweeps, oracle port (stops at the first feasible candidate)",
                               "agree_with_gpu": agree}
    return out


if __name__ == "__main__":
    try:
        main()
    except BaseException as exc:                    # torchrun swallows child tracebacks: say which rank died and why
        if not isinstance(exc, SystemExit) or exc.code not in (0, None):
            import traceback
            sys.stderr.write(f"[bench] rank {os.environ.get('RANK', '0')} (local {os.environ.get('LOCAL_RANK', '0')}) failed:\n")
            traceback.print_exc()
            sys.stderr.flush()
        raise
