"""Thin Python wrappers over the C ABI (device tensors in, device tensors out)."""
import ctypes as C
import math

import numpy as np

from . import _lib
from ._lib import CHECK_AUX, CHECK_BOUNDARY, CHECK_LANE, CHECK_OBSTACLES  # noqa: F401


def _torch():
    import torch
    return torch


def _device(envs=None, *tensors):
    """Current CUDA device; without one every op fails loudly (no CPU fallback).  An environment batch or a CUDA
    tensor that lives on ANOTHER device than the calling thread's current one raises instead of launching across
    devices (the C ABI checks the same thing again, ``hl_enter``)."""
    import torch
    if not torch.cuda.is_available():
        raise _lib.HeadlandError("no CUDA device: headland_trajectory_planning_b200 has no CPU fallback")
    cur = torch.cuda.current_device()
    if envs is not None and getattr(envs, "device", cur) != cur:
        raise _lib.HeadlandError(f"environment batch was uploaded to cuda:{envs.device} but the current device of this "
                                 f"thread is cuda:{cur} (torch.cuda.set_device / EnvBatch(device=...))")
    for t in tensors:
        if torch.is_tensor(t) and (not t.is_cuda or t.device.index != cur):
            raise _lib.HeadlandError(f"tensor on {t.device} passed to an op running on cuda:{cur}")
    return torch.device("cuda", cur)


def collision_check(envs, poses, env_id=None, pose_idx=None, flags=CHECK_OBSTACLES | CHECK_BOUNDARY,
                    count_exact=False):
    """Per-pose infeasibility flags (uint8 CUDA tensor).  ``poses``: [N,3] float64
    (CUDA tensor, or host array which is copied).  ``pose_idx``: index of each pose
    within its path (implement rectangles are tested at even indices only)."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(envs, poses, env_id, pose_idx)
    if not torch.is_tensor(poses):
        poses = torch.from_numpy(np.ascontiguousarray(np.asarray(poses, dtype=np.float64)[:, :3])).to(dev)
    poses = poses.contiguous()
    n = poses.shape[0]
    if env_id is not None and not torch.is_tensor(env_id):
        env_id = torch.from_numpy(np.ascontiguousarray(env_id, dtype=np.int32)).to(dev)
    if pose_idx is not None and not torch.is_tensor(pose_idx):
        pose_idx = torch.from_numpy(np.ascontiguousarray(pose_idx, dtype=np.int32)).to(dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    n_exact = torch.zeros(1, dtype=torch.int64, device=dev) if count_exact else None
    if n == 0:
        return (out, n_exact) if count_exact else out
    _lib.check(lib.hl_collision_check(envs.ctx, envs.handle, _lib.ptr(env_id), _lib.ptr(poses),
                                      _lib.ptr(pose_idx), n, flags, _lib.ptr(out), _lib.ptr(n_exact),
                                      _lib.stream_ptr()), "hl_collision_check")
    if count_exact:
        return out, n_exact
    return out


def path_reduce(envs, pose_bad, path_start):
    torch = _torch()
    lib = _lib.load_library()
    n_paths = path_start.shape[0] - 1
    out = torch.empty(n_paths, dtype=torch.uint8, device=pose_bad.device)
    _lib.check(lib.hl_path_reduce(envs.ctx, _lib.ptr(pose_bad), _lib.ptr(path_start), n_paths,
                                  _lib.ptr(out), _lib.stream_ptr()), "hl_path_reduce")
    return out


def ypark_paths(cand, step):
    """Candidate paths of the Y-type parking sweep (K5, ``hl_ypark_paths``).  ``cand``: [n,8] float64 rows
    (backward_length, forward_length, signed backward_steer, signed forward_steer, end_x, end_y, end_yaw,
    wheel_base).  Returns (poses [total,3] float64 CUDA tensor, offsets [n+1] int64).  A host array gives host offsets;
    a CUDA tensor stays on the device (pose counts and offsets are computed there, one scalar read for the pool size)
    and gives a CUDA offsets tensor -- the batched sweep builds its candidate table on the device."""
    torch = _torch()
    lib = _lib.load_library()
    if torch.is_tensor(cand) and cand.is_cuda:
        dev = _device(None, cand)
        d_cand = cand.to(torch.float64).reshape(-1, 8).contiguous()
        n = d_cand.shape[0]
        # Python round() == rint (ties to even) == torch.round; the same IEEE division as on the host
        counts = (torch.round(d_cand[:, 0] / step) + torch.round(d_cand[:, 1] / step) + 2).to(torch.int64)
        d_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        if n:
            d_off[1:] = torch.cumsum(counts, 0)
        total = int(d_off[-1].item()) if n else 0
        poses = torch.empty((total, 3), dtype=torch.float64, device=dev)
        if n:
            _lib.check(lib.hl_ypark_paths(_lib.get_ctx(dev.index), _lib.ptr(d_cand), _lib.ptr(d_off), n, float(step),
                                          _lib.ptr(poses), _lib.stream_ptr()), "hl_ypark_paths")
        return poses, d_off
    dev = _device()
    cand = np.ascontiguousarray(np.asarray(cand, dtype=np.float64).reshape(-1, 8))
    n = cand.shape[0]
    counts = (np.rint(cand[:, 0] / step) + np.rint(cand[:, 1] / step) + 2).astype(np.int64)   # Python round()
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    poses = torch.empty((int(offsets[-1]), 3), dtype=torch.float64, device=dev)
    if n == 0:
        return poses, offsets
    d_cand = torch.from_numpy(cand).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    _lib.check(lib.hl_ypark_paths(_lib.get_ctx(dev.index), _lib.ptr(d_cand), _lib.ptr(d_off), n, float(step),
                                  _lib.ptr(poses), _lib.stream_ptr()), "hl_ypark_paths")
    return poses, offsets


def arc_paths(cand, step):
    """Single-arc rollouts (``hl_arc_paths``, CarModel.calculate_motion_path).  ``cand``: [n,8] float64 rows
    (init_x, init_y, init_yaw, signed steer, direction, search_length, wheel_base, unused).
    Returns (poses [total,3] CUDA tensor, offsets [n+1] int64 host array)."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device()
    cand = np.ascontiguousarray(np.asarray(cand, dtype=np.float64).reshape(-1, 8))
    n = cand.shape[0]
    counts = (np.rint(cand[:, 5] / step) + 1).astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    poses = torch.empty((int(offsets[-1]), 3), dtype=torch.float64, device=dev)
    if n == 0:
        return poses, offsets
    d_cand = torch.from_numpy(cand).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    _lib.check(lib.hl_arc_paths(_lib.get_ctx(dev.index), _lib.ptr(d_cand), _lib.ptr(d_off), n, float(step),
                                _lib.ptr(poses), _lib.stream_ptr()), "hl_arc_paths")
    return poses, offsets


def ref_path_batch(x, y, direction, in_offsets, wheel_base, desired_v=0.5, ds=0.1):
    """OBCA initial guesses of many planner paths (K8, ``hl_ref_path_count`` + ``hl_ref_path_fill``).
    ``x, y`` float64 and ``direction`` int8 pooled pose arrays (CUDA tensors or host arrays), ``in_offsets`` [n+1].
    Returns (traj [T,5] float64 CUDA tensor: x, y, v, yaw, steer; out_offsets [n+1] int64 host; status [n] int32 host,
    1 = a direction piece with fewer than two distinct poses, no rows)."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device()
    def dev_t(a, dt):
        if torch.is_tensor(a):
            return a.to(dev).to(dt).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev).to(dt).contiguous()
    x, y = dev_t(x, torch.float64), dev_t(y, torch.float64)
    direction = dev_t(direction, torch.int8)
    in_off = dev_t(np.asarray(in_offsets, dtype=np.int64), torch.int64)
    n = in_off.numel() - 1
    counts = torch.zeros(max(n, 1), dtype=torch.int64, device=dev)
    status = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)
    ctx = _lib.get_ctx(dev.index)
    if n > 0:
        _lib.check(lib.hl_ref_path_count(ctx, _lib.ptr(x), _lib.ptr(y), _lib.ptr(direction), _lib.ptr(in_off), n, float(ds),
                                         _lib.ptr(counts), _lib.ptr(status), _lib.stream_ptr()), "hl_ref_path_count")
    out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    if n > 0:
        out_off[1:] = torch.cumsum(counts[:n], 0)
    total = int(out_off[-1].item())
    traj = torch.empty((total, 5), dtype=torch.float64, device=dev)
    if n > 0 and total > 0:
        ws = torch.empty(8 * max(int(x.numel()), 1), dtype=torch.float64, device=dev)
        _lib.check(lib.hl_ref_path_fill(ctx, _lib.ptr(x), _lib.ptr(y), _lib.ptr(direction), _lib.ptr(in_off), _lib.ptr(out_off),
                                        _lib.ptr(status), n, float(wheel_base), float(desired_v), float(ds), _lib.ptr(ws),
                                        _lib.ptr(traj), _lib.stream_ptr()), "hl_ref_path_fill")
    return traj, out_off.cpu().numpy(), status[:n].cpu().numpy()


def min_boundary_distance(envs, poses, path_start, env_id=None, with_aux=True):
    """``get_min_distance_to_boundary`` of many paths (K10).  ``poses`` pooled [N,3] float64 (CUDA tensor or host),
    ``path_start`` [n+1] int64 (host array or CUDA tensor).  Returns a float64 CUDA tensor [n]."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(envs, poses, env_id)
    if not torch.is_tensor(poses):
        poses = torch.from_numpy(np.ascontiguousarray(np.asarray(poses, dtype=np.float64)[:, :3])).to(dev)
    poses = poses.contiguous()
    if not torch.is_tensor(path_start):
        path_start = torch.from_numpy(np.ascontiguousarray(path_start, dtype=np.int64)).to(dev)
    if env_id is not None and not torch.is_tensor(env_id):
        env_id = torch.from_numpy(np.ascontiguousarray(env_id, dtype=np.int32)).to(dev)
    n = path_start.numel() - 1
    out = torch.empty(max(n, 0), dtype=torch.float64, device=dev)
    if n > 0:
        _lib.check(lib.hl_min_boundary_distance(envs.ctx, envs.handle, _lib.ptr(env_id), _lib.ptr(poses), _lib.ptr(path_start),
                                                n, 1 if with_aux else 0, _lib.ptr(out), _lib.stream_ptr()),
                   "hl_min_boundary_distance")
    return out


def corridor_hits(envs, points, line_start, radius, env_id=None):
    """Does the flat-capped, round-joined buffer of each polyline meet an obstacle?  (K11.)  ``points`` pooled [N,2],
    ``line_start`` [n+1].  Returns a uint8 CUDA tensor [n]."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(envs, points, env_id)
    if not torch.is_tensor(points):
        points = torch.from_numpy(np.ascontiguousarray(np.asarray(points, dtype=np.float64).reshape(-1, 2))).to(dev)
    points = points.contiguous()
    if not torch.is_tensor(line_start):
        line_start = torch.from_numpy(np.ascontiguousarray(line_start, dtype=np.int64)).to(dev)
    if env_id is not None and not torch.is_tensor(env_id):
        env_id = torch.from_numpy(np.ascontiguousarray(env_id, dtype=np.int32)).to(dev)
    n = line_start.numel() - 1
    out = torch.zeros(max(n, 0), dtype=torch.uint8, device=dev)
    if n > 0:
        _lib.check(lib.hl_corridor_hits(envs.ctx, envs.handle, _lib.ptr(env_id), _lib.ptr(points), _lib.ptr(line_start), n,
                                        float(radius), _lib.ptr(out), _lib.stream_ptr()), "hl_corridor_hits")
    return out


def dubins_course_batch(pairs, turning_radius, step=0.1, ds=0.1, append_goal=False, want_samples=False):
    """Dubins shortest paths of many (start, end) pose pairs + their cubic-spline course (K9).  ``pairs``: [n,6] float64
    (sx, sy, syaw, ex, ey, eyaw), host array or CUDA tensor.  Returns (rows [T,4] float64 CUDA tensor: x, y, yaw,
    curvature; row_offsets [n+1] int64 host; word [n] int32 host (0..5 = LSL LSR RSL RSR RLR LRL, -1 none);
    length [n] float64 host) -- plus, with ``want_samples``, the raw ``sample_many`` configurations [slots,3] and the
    slot offsets.  A pair whose course cannot be built (coincident poses) has no rows."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(None, pairs)
    if not torch.is_tensor(pairs):
        pairs = torch.from_numpy(np.ascontiguousarray(np.asarray(pairs, dtype=np.float64).reshape(-1, 6))).to(dev)
    pairs = pairs.contiguous()
    n = pairs.shape[0]
    ctx = _lib.get_ctx(dev.index)
    rho, step, ds, ag = float(turning_radius), float(step), float(ds), 1 if append_goal else 0
    slots = torch.zeros(max(n, 1), dtype=torch.int64, device=dev)
    word = torch.full((max(n, 1),), -1, dtype=torch.int32, device=dev)
    length = torch.zeros(max(n, 1), dtype=torch.float64, device=dev)
    if n == 0:
        return torch.empty((0, 4), dtype=torch.float64, device=dev), np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0)
    _lib.check(lib.hl_dubins_count(ctx, _lib.ptr(pairs), n, rho, step, ds, ag, _lib.ptr(slots), _lib.ptr(word),
                                   _lib.ptr(length), _lib.stream_ptr()), "hl_dubins_count")
    slot_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    slot_off[1:] = torch.cumsum(slots[:n], 0)
    total_slots = int(slot_off[-1].item())
    ws = torch.empty(9 * max(total_slots, 1), dtype=torch.float64, device=dev)
    n_knots = torch.zeros(n, dtype=torch.int32, device=dev)
    n_rows = torch.zeros(n, dtype=torch.int64, device=dev)
    samples = torch.empty((max(total_slots, 1), 3), dtype=torch.float64, device=dev) if want_samples else None
    _lib.check(lib.hl_dubins_knots(ctx, _lib.ptr(pairs), n, rho, step, ds, ag, _lib.ptr(slot_off), _lib.ptr(ws),
                                   _lib.ptr(n_knots), _lib.ptr(n_rows), _lib.ptr(samples), _lib.stream_ptr()), "hl_dubins_knots")
    row_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    row_off[1:] = torch.cumsum(n_rows, 0)
    total = int(row_off[-1].item())
    out = torch.empty((max(total, 1), 4), dtype=torch.float64, device=dev)
    _lib.check(lib.hl_dubins_fill(ctx, n, ds, _lib.ptr(slot_off), _lib.ptr(row_off), _lib.ptr(n_knots), _lib.ptr(ws),
                                  _lib.ptr(out), _lib.stream_ptr()), "hl_dubins_fill")
    res = (out[:total], row_off.cpu().numpy(), word[:n].cpu().numpy(), length[:n].cpu().numpy())
    if want_samples:                      # raw sample_many configurations: pair p owns slots slot_off[p] .. slot_off[p+1]-2
        return res + (samples, slot_off.cpu().numpy())
    return res


def measure_fp32_peak(device=None):
    lib = _lib.load_library()
    v = C.c_double()
    _lib.check(lib.hl_measure_fp32_peak(_lib.get_ctx(device), C.byref(v)), "hl_measure_fp32_peak")
    return v.value


def rs_all_paths(start_goal, maxc, step, max_steer=0.55, envs=None, env_id=None,
                 flags=CHECK_OBSTACLES, want_order=True):
    """Batched Reeds-Shepp words.  Returns (words [N,46] structured CUDA bytes viewed on
    the host on demand, count [N] int32, order [N,46] int32) as CUDA tensors; use
    ``rs_words_to_host`` to view the word records."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(envs, start_goal, env_id)
    if not torch.is_tensor(start_goal):
        start_goal = torch.from_numpy(np.ascontiguousarray(start_goal, dtype=np.float64)).to(dev)
    start_goal = start_goal.contiguous()
    n = start_goal.shape[0]
    if env_id is not None and not torch.is_tensor(env_id):
        env_id = torch.from_numpy(np.ascontiguousarray(env_id, dtype=np.int32)).to(dev)
    words = torch.zeros((n, _lib.HL_RS_CANDIDATES, _lib.RSWORD_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    count = torch.empty(n, dtype=torch.int32, device=dev)
    order = torch.empty((n, _lib.HL_RS_CANDIDATES), dtype=torch.int32, device=dev) if want_order else None
    ctx = envs.ctx if envs is not None else _lib.get_ctx()
    _lib.check(lib.hl_rs_all_paths(ctx, envs.handle if envs is not None else None, _lib.ptr(env_id),
                                   _lib.ptr(start_goal), n, float(maxc), float(step), float(max_steer),
                                   flags, _lib.ptr(words), _lib.ptr(count), _lib.ptr(order),
                                   _lib.stream_ptr()), "hl_rs_all_paths")
    return words, count, order


def rs_words_to_host(words):
    """[N,46,112] uint8 CUDA tensor -> numpy structured array [N,46] (RSWORD_DTYPE)."""
    a = words.cpu().numpy()
    return a.view(_lib.RSWORD_DTYPE).reshape(a.shape[0], a.shape[1])


def rs_sample(starts, words_host, maxc, step):
    """Sample M words.  ``starts`` [M,3] float64 host, ``words_host`` structured [M].
    Returns host arrays (offset [M+1], x, y, yaw, cs, dir)."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device()
    m = len(words_host)
    offset = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(words_host["npts"], out=offset[1:])
    total = int(offset[-1])
    d_start = torch.from_numpy(np.ascontiguousarray(starts, dtype=np.float64)).to(dev)
    d_words = torch.from_numpy(np.ascontiguousarray(words_host).view(np.uint8).reshape(m, -1)).to(dev)
    d_off = torch.from_numpy(offset).to(dev)
    x = torch.empty(max(total, 1), dtype=torch.float64, device=dev)
    y = torch.empty_like(x); yaw = torch.empty_like(x); cs = torch.empty_like(x)
    dr = torch.empty(max(total, 1), dtype=torch.int8, device=dev)
    _lib.check(lib.hl_rs_sample(_lib.get_ctx(), _lib.ptr(d_start), _lib.ptr(d_words), m, float(maxc),
                                float(step), _lib.ptr(d_off), _lib.ptr(x), _lib.ptr(y), _lib.ptr(yaw),
                                _lib.ptr(cs), _lib.ptr(dr), _lib.stream_ptr()), "hl_rs_sample")
    return (offset, x[:total].cpu().numpy(), y[:total].cpu().numpy(), yaw[:total].cpu().numpy(),
            cs[:total].cpu().numpy(), dr[:total].cpu().numpy())


def hybrid_astar_batch(envs, scenarios, params, path_capacity=None, to_host=True):
    """Run ``hl_hybrid_astar_batch`` on a batch of scenarios.

    ``scenarios``: numpy structured array (``_lib.SCENARIO_DTYPE``) on the host (it is
    copied to the device inside this call) or a uint8 CUDA tensor of the same bytes.
    Returns a dict with ``results`` (structured), the pooled ``expanded`` keys [rows, 3] int32 (slice
    of scenario i: ``expanded_of(out, i)``) and the pooled path arrays (host numpy when ``to_host``)."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(envs, scenarios)
    _lib.apply_astar_variant(envs.ctx)
    if torch.is_tensor(scenarios):
        d_scen = scenarios
        n = d_scen.numel() // _lib.SCENARIO_DTYPE.itemsize
    else:
        n = len(scenarios)
        d_scen = torch.from_numpy(np.ascontiguousarray(scenarios).view(np.uint8).reshape(-1)).to(dev, non_blocking=True)
    if path_capacity is None:
        path_capacity = max(4096, 1024 * n)
    mn = params.max_nodes
    results = torch.empty(n * _lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    keys_cap = n * (mn + 2)
    expanded = torch.empty((keys_cap, 3), dtype=torch.int32, device=dev)
    kcursor = torch.zeros(1, dtype=torch.int64, device=dev)
    px = torch.empty(path_capacity, dtype=torch.float64, device=dev)
    py = torch.empty_like(px); pyaw = torch.empty_like(px); pk = torch.empty_like(px)
    pdir = torch.empty(path_capacity, dtype=torch.int8, device=dev)
    cursor = torch.zeros(1, dtype=torch.int64, device=dev)
    _lib.check(lib.hl_hybrid_astar_batch(envs.ctx, envs.handle, _lib.ptr(d_scen), n, C.byref(params),
                                         _lib.ptr(results), _lib.ptr(expanded), keys_cap, _lib.ptr(kcursor),
                                         _lib.ptr(px), _lib.ptr(py),
                                         _lib.ptr(pyaw), _lib.ptr(pk), _lib.ptr(pdir), path_capacity,
                                         _lib.ptr(cursor), _lib.stream_ptr()), "hl_hybrid_astar_batch")
    out = dict(results=results, expanded=expanded, x=px, y=py, yaw=pyaw, k=pk, dir=pdir, cursor=cursor,
               kcursor=kcursor, n=n)
    if to_host:
        both = torch.cat([cursor, kcursor]).cpu().numpy()
        used, kused = int(both[0]), int(both[1])
        out["results"] = results.cpu().numpy().view(_lib.RESULT_DTYPE)
        out["expanded"] = expanded[:min(kused, keys_cap)].cpu().numpy()
        out["keys_used"] = kused
        for key in ("x", "y", "yaw", "k", "dir"):
            out[key] = out[key][:min(used, path_capacity)].cpu().numpy()
        out["used"] = used
    return out


def astar_launches_per_call(envs, n_scenarios):
    """Kernel launches one ``hybrid_astar_batch`` call makes (the default two-warp variant runs sweeps several times
    larger than the resident scenario slots in two launches: first shots only, then the scenarios they left over)."""
    import os
    sm = int(_lib.load_library().hl_ctx_sm_count(envs.ctx))
    if os.environ.get("HL_ASTAR_VARIANT", "spec") == "spec" and n_scenarios > 2 * sm * 5:
        return 2
    return 1


def distance_field(occ, goal, motion_type="King"):
    """Grid distance field from ``goal`` (hl_distance_field).  ``occ``: [W,H] bool/uint8
    (host array or CUDA tensor).  Returns (float64 CUDA tensor [W,H], relaxation launches)."""
    torch = _torch()
    lib = _lib.load_library()
    dev = _device()
    if not torch.is_tensor(occ):
        occ = torch.from_numpy(np.ascontiguousarray(np.asarray(occ).astype(np.uint8))).to(dev)
    occ = occ.to(torch.uint8).contiguous()
    w, h = occ.shape
    out = torch.empty((w, h), dtype=torch.float64, device=dev)
    sweeps = C.c_int32(0)
    mt = {"King": 0, "Pawn": 1}[motion_type]
    _lib.check(lib.hl_distance_field(_lib.get_ctx(), _lib.ptr(occ), w, h, int(goal[0]), int(goal[1]), mt,
                                     _lib.ptr(out), C.byref(sweeps), _lib.stream_ptr()), "hl_distance_field")
    return out, sweeps.value


def distance_field_batch(occs, goals, motion_type="King"):
    """Distance fields of many (grid, goal) pairs in one wavefront (hl_distance_field_batch).  ``occs``: one [W,H]
    bool/uint8 grid shared by every goal (uploaded once), or a sequence of B grids, one per goal, of any shapes (host
    arrays or CUDA tensors).  ``goals``: B pairs (i, j).  Returns (list of B float64 CUDA tensors [W_b, H_b], views of
    one pooled buffer, relaxation launches); each field equals ``distance_field`` of its grid and goal bit for bit."""
    torch = _torch()
    lib = _lib.load_library()
    if motion_type not in ("King", "Pawn"):
        raise _lib.HeadlandError(f"unknown motion type {motion_type!r} (King or Pawn)")
    goals = [(int(g[0]), int(g[1])) for g in goals]
    shared = (torch.is_tensor(occs) or isinstance(occs, np.ndarray)) and occs.ndim == 2
    grids = [g if torch.is_tensor(g) else np.asarray(g) for g in ([occs] if shared else occs)]
    if not shared and len(grids) != len(goals):
        raise _lib.HeadlandError(f"distance_field_batch: {len(grids)} grids for {len(goals)} goals")
    dev = _device(None, *grids)
    if not goals:
        return [], 0
    if any(g.ndim != 2 for g in grids):
        raise _lib.HeadlandError("distance_field_batch: every grid must be 2-D [W, H]")
    shapes = [tuple(int(v) for v in g.shape) for g in grids]
    if any(torch.is_tensor(g) for g in grids):
        occ = torch.cat([(g if torch.is_tensor(g) else torch.from_numpy(g.astype(np.uint8))).to(dev, torch.uint8).reshape(-1)
                         for g in grids])
    else:                                  # host grids: one upload
        occ = torch.from_numpy(np.concatenate([g.astype(np.uint8).reshape(-1) for g in grids])).to(dev)
    occ_base = np.concatenate([[0], np.cumsum([w * h for w, h in shapes])])
    fields = (_lib.HlGridField * len(goals))()
    out_base = 0
    for k, (gi, gj) in enumerate(goals):
        s = 0 if shared else k
        w, h = shapes[s]
        fields[k] = _lib.HlGridField(int(occ_base[s]), out_base, w, h, gi, gj)
        out_base += w * h
    out = torch.empty(out_base, dtype=torch.float64, device=dev)
    sweeps = C.c_int32(0)
    mt = {"King": 0, "Pawn": 1}[motion_type]
    _lib.check(lib.hl_distance_field_batch(_lib.get_ctx(), _lib.ptr(occ), occ.numel(), fields, len(goals), mt,
                                           _lib.ptr(out), out.numel(), C.byref(sweeps), _lib.stream_ptr()),
               "hl_distance_field_batch")
    views = [out[f.out_offset:f.out_offset + f.w * f.h].view(f.w, f.h) for f in fields]
    return views, sweeps.value


def grid_pack(occ):
    torch = _torch()
    lib = _lib.load_library()
    dev = _device()
    if not torch.is_tensor(occ):
        occ = torch.from_numpy(np.ascontiguousarray(np.asarray(occ).astype(np.uint8))).to(dev)
    occ = occ.to(torch.uint8).contiguous()
    w, h = occ.shape
    bits = torch.empty((w * h + 31) // 32, dtype=torch.int32, device=dev)
    _lib.check(lib.hl_grid_pack(_lib.get_ctx(), _lib.ptr(occ), w, h, _lib.ptr(bits), _lib.stream_ptr()), "hl_grid_pack")
    return bits


def _int32(v, what):
    """``v`` as a Python int that fits an int32 ABI slot; ctypes would wrap a larger value silently, so the C side's
    range checks would see a different number."""
    v = int(v)
    if not -2**31 <= v < 2**31:
        raise _lib.HeadlandError(f"{what} = {v} does not fit int32")
    return v


def grid_footprint_check(bits, shape, res, poses, body_ext, origin=(0, 0)):
    """K7: 1 where the body rectangle at a pose meets an occupied cell of the bit-packed grid (``grid_pack``).  The
    grid's cell (0, 0) has the global index ``origin`` = (i0, j0): cell (i, j) covers [fl((i0+i)*res),
    fl((i0+i+1)*res)] x [fl((j0+j)*res), fl((j0+j+1)*res)], as ``rasterize`` lays its grids out."""
    w, h = _int32(shape[0], "grid_footprint_check: w"), _int32(shape[1], "grid_footprint_check: h")
    i0, j0 = _int32(origin[0], "grid_footprint_check: origin i0"), _int32(origin[1], "grid_footprint_check: origin j0")
    torch = _torch()
    lib = _lib.load_library()
    dev = _device()
    if not torch.is_tensor(poses):
        poses = torch.from_numpy(np.ascontiguousarray(np.asarray(poses, dtype=np.float64)[:, :3])).to(dev)
    poses = poses.contiguous()
    n = poses.shape[0]
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    if n == 0:
        return out
    ext = (C.c_double * 4)(*[float(v) for v in body_ext])
    _lib.check(lib.hl_grid_footprint_check_at(_lib.get_ctx(), _lib.ptr(bits), w, h, i0, j0, float(res), _lib.ptr(poses), n, ext, _lib.ptr(out),
                                              _lib.stream_ptr()), "hl_grid_footprint_check_at")
    return out


def _cell_range(vmin, vmax, res):
    """Cells lo..hi whose closed interval [fl(i*res), fl((i+1)*res)] meets [vmin, vmax] (K7's cell_range rule, not
    clamped to a grid): the floor() estimate stepped by the float64 edge comparisons themselves."""
    lo = int(math.floor(vmin / res))
    while float(lo) * res >= vmin:
        lo -= 1
    while (float(lo) + 1.0) * res < vmin:
        lo += 1
    hi = int(math.floor(vmax / res))
    while (float(hi) + 1.0) * res <= vmax:
        hi += 1
    while float(hi) * res > vmax:
        hi -= 1
    return lo, hi


def raster_window(field_ring, res, margin):
    """(i0, j0, w, h) of the cells whose closed intervals meet the float64 bounding box of ``field_ring`` grown by
    ``margin`` metres on every side (computed on the host)."""
    ring = np.asarray(field_ring, dtype=np.float64).reshape(-1, 2)
    if len(ring) == 0:
        raise _lib.HeadlandError("raster_window: the field ring has no vertices")
    res, margin = float(res), float(margin)
    if not (math.isfinite(res) and res > 0) or not (math.isfinite(margin) and margin >= 0):
        raise _lib.HeadlandError(f"raster_window: res must be finite and positive and margin finite and >= 0 "
                                 f"(res={res}, margin={margin})")
    i0, i1 = _cell_range(float(ring[:, 0].min()) - margin, float(ring[:, 0].max()) + margin, res)
    j0, j1 = _cell_range(float(ring[:, 1].min()) - margin, float(ring[:, 1].max()) + margin, res)
    return i0, j0, i1 - i0 + 1, j1 - j0 + 1


def rasterize(envs, grids, res, flags=CHECK_OBSTACLES | CHECK_BOUNDARY, count_exact=False):
    """K12 (``hl_env_rasterize``): occupancy grids of environments of ``envs``, all in one launch.  ``grids`` is a
    sequence of (env_id, i0, j0, w, h); cell (i, j) of a grid is the closed square [fl((i0+i)*res), fl((i0+i+1)*res)]
    x [fl((j0+j)*res), fl((j0+j+1)*res)], occupied (1) when it meets an obstacle quad (CHECK_OBSTACLES) or is not
    contained in the field polygon (CHECK_BOUNDARY).  Returns a list of uint8 CUDA tensors [w, h], views of one pooled
    buffer, in ``distance_field``'s layout; with ``count_exact`` also the int64 CUDA counter of cells the float64
    predicates decided."""
    grids = [tuple(g) for g in grids]
    if any(len(g) != 5 for g in grids):
        raise _lib.HeadlandError("rasterize: every grid is (env_id, i0, j0, w, h)")
    names = ("env_id", "i0", "j0", "w", "h")
    grids = [tuple(_int32(v, f"rasterize: grid {k}: {nm}") for v, nm in zip(g, names)) for k, g in enumerate(grids)]
    if not 0 <= int(flags) < 2**32:
        raise _lib.HeadlandError(f"rasterize: flags = {int(flags)} does not fit uint32")
    torch = _torch()
    lib = _lib.load_library()
    dev = _device(envs)
    table = (_lib.HlRasterGrid * max(len(grids), 1))()
    base = 0
    for k, (env_id, i0, j0, w, h) in enumerate(grids):
        if w < 1 or h < 1:
            raise _lib.HeadlandError(f"rasterize: grid {k}: a {w}x{h} grid (w and h must be at least 1)")
        table[k] = _lib.HlRasterGrid(base, env_id, w, h, i0, j0)
        base += w * h
    out = torch.empty(max(base, 1), dtype=torch.uint8, device=dev)
    n_exact = torch.zeros(1, dtype=torch.int64, device=dev)
    _lib.check(lib.hl_env_rasterize(envs.ctx, envs.handle, table, len(grids), float(res), int(flags), _lib.ptr(out), base,
                                    _lib.ptr(n_exact) if count_exact else None, _lib.stream_ptr()), "hl_env_rasterize")
    views = [out[table[k].out_offset:table[k].out_offset + w * h].view(w, h) for k, (_, _, _, w, h) in enumerate(grids)]
    return (views, n_exact) if count_exact else views


PHASE_NAMES = ["pop", "rs_candidates", "rs_select", "rs_plan", "rs_sample", "arrival", "rollout", "filter", "exact",
               "cost_heuristic", "merge", "setup", "output"]


def astar_phase_cycles(reset=True, device=None):
    """Per-phase cycles of the search kernel summed over scenarios since the last reset."""
    lib = _lib.load_library()
    buf = (C.c_uint64 * len(PHASE_NAMES))()
    _lib.check(lib.hl_astar_phase_cycles(_lib.get_ctx(device), buf, len(PHASE_NAMES), 1 if reset else 0),
               "hl_astar_phase_cycles")
    return dict(zip(PHASE_NAMES, [int(v) for v in buf]))


def expanded_of(out, i):
    """Popped grid keys [n_expanded, 3] of scenario ``i`` from a host result dict."""
    r = out["results"][i]
    a = int(r["keys_offset"])
    return out["expanded"][a:a + int(r["n_expanded"])]
