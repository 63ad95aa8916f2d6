"""K4 outputs: what the three search-kernel variants write at the end of a search.

The default kernel (two warps per scenario with the analytic shot decoupled), the one-warp-per-scenario kernel and
the level-synchronous graph each write the expanded keys, the path and the result record of a finished scenario.
They must write the same bytes for the same scenario, including for a blocked start or goal, and they must handle
a keys pool that is too small the same way: a scenario whose keys do not fit reports HL_STATUS_CAPACITY with no
keys and no path, never a truncated key list."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VARIANTS = ("spec", "warp", "level")
RECORD_FIELDS = ("status", "counter", "n_expanded", "arrival", "path_len", "rs_word", "goal_cost")
PATH_FIELDS = ("x", "y", "yaw", "k", "dir")


def _golden_records():
    """The 512 golden scenarios, then three copies whose start and one whose goal lies 100 m off the field."""
    from headland_trajectory_planning_b200 import scenarios as SC, sweep
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "astar_golden.npz"))
    specs = [SC.scenario_spec(int(i)) for i in g["index"]]
    scns = [SC.finalize(sp, f) for sp, f in zip(specs, g["feas"])]
    recs, scen, car = sweep.build_records(scns)
    off = scen[[0, 7, 40, 3]].copy()
    off["start"][:3, 1] -= 100.0
    off["goal"][3, 1] -= 100.0
    return recs, np.concatenate([scen, off]), car, len(scen)


@pytest.fixture(scope="module")
def golden_batch(built_library):
    from headland_trajectory_planning_b200 import sweep
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    recs, scen, car, n_golden = _golden_records()
    return EnvBatch(recs), scen, sweep.search_params(car), n_golden


def _run(envs, scen, params, variant, monkeypatch, keys_capacity=None):
    """hl_hybrid_astar_batch with a chosen keys-pool capacity (ops.hybrid_astar_batch always sizes it for the
    worst case).  Returns host arrays in the layout of ops.hybrid_astar_batch's result dict."""
    import torch
    from headland_trajectory_planning_b200 import _lib
    monkeypatch.setenv("HL_ASTAR_VARIANT", variant)
    lib = _lib.load_library()
    _lib.apply_astar_variant(envs.ctx)
    dev = torch.device("cuda", envs.device)
    n = len(scen)
    path_capacity = 2048 * n
    if keys_capacity is None:
        keys_capacity = n * (params.max_nodes + 2)
    d_scen = torch.from_numpy(np.ascontiguousarray(scen).view(np.uint8).reshape(-1)).to(dev)
    results = torch.empty(n * _lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    expanded = torch.empty((keys_capacity, 3), dtype=torch.int32, device=dev)
    kcursor = torch.zeros(1, dtype=torch.int64, device=dev)
    cursor = torch.zeros(1, dtype=torch.int64, device=dev)
    px, py, pyaw, pk = (torch.empty(path_capacity, dtype=torch.float64, device=dev) for _ in range(4))
    pdir = torch.empty(path_capacity, dtype=torch.int8, device=dev)
    _lib.check(lib.hl_hybrid_astar_batch(envs.ctx, envs.handle, _lib.ptr(d_scen), n, C.byref(params),
                                         _lib.ptr(results), _lib.ptr(expanded), keys_capacity, _lib.ptr(kcursor),
                                         _lib.ptr(px), _lib.ptr(py), _lib.ptr(pyaw), _lib.ptr(pk), _lib.ptr(pdir),
                                         path_capacity, _lib.ptr(cursor), _lib.stream_ptr()), "hl_hybrid_astar_batch")
    used, kused = (int(v) for v in torch.cat([cursor, kcursor]).cpu())
    out = dict(results=results.cpu().numpy().view(_lib.RESULT_DTYPE), keys_used=kused,
               expanded=expanded[:min(kused, keys_capacity)].cpu().numpy())
    for name, t in zip(PATH_FIELDS, (px, py, pyaw, pk, pdir)):
        out[name] = t[:min(used, path_capacity)].cpu().numpy()
    return out


def _keys(out, i):
    r = out["results"][i]
    a = int(r["keys_offset"])
    return out["expanded"][a:a + int(r["n_expanded"])]


def _path(out, i, field):
    r = out["results"][i]
    a = int(r["path_offset"])
    return out[field][a:a + int(r["path_len"])]


def test_variants_write_identical_outputs(golden_batch, monkeypatch):
    """Per scenario, every variant writes bit-identical records, key rows and paths (the algorithmic pose-check
    tally too, except at a tolerance arrival, where only the default kernel also counts that pop's shot)."""
    envs, scen, params, n_golden = golden_batch
    outs = {v: _run(envs, scen, params, v, monkeypatch) for v in VARIANTS}
    ref = outs["spec"]
    res = ref["results"]
    assert (res["status"][n_golden:] == 1).all()                      # HL_STATUS_START_GOAL_BLOCKED
    assert (res["counter"][n_golden:] == 0).all() and (res["n_pose_checks_ref"][n_golden:] == 0).all()
    assert (res["arrival"] == 1).any() and (res["path_len"] > 0).any()
    for v in VARIANTS[1:]:
        got = outs[v]["results"]
        for f in RECORD_FIELDS:
            bad = np.nonzero(res[f] != got[f])[0]
            assert len(bad) == 0, (v, f, bad[:10])
        sel = res["arrival"] != 2
        assert np.array_equal(res["n_pose_checks_ref"][sel], got["n_pose_checks_ref"][sel]), v
        for i in range(len(scen)):
            assert np.array_equal(_keys(ref, i), _keys(outs[v], i)), (v, i)
            for f in PATH_FIELDS:
                assert np.array_equal(_path(ref, i, f), _path(outs[v], i, f)), (v, i, f)


@pytest.mark.parametrize("variant", VARIANTS)
def test_keys_pool_overflow(golden_batch, variant, monkeypatch):
    """A keys pool of half the size the batch needs: each record is either the full-capacity one or
    HL_STATUS_CAPACITY with no keys and no path.  Which scenarios overflow depends on the order in which they
    finish, so only that both kinds occur is asserted."""
    envs, scen, params, _ = golden_batch
    full = _run(envs, scen, params, variant, monkeypatch)
    need = full["keys_used"]
    small = _run(envs, scen, params, variant, monkeypatch, keys_capacity=need // 2)
    rf, rs = full["results"], small["results"]
    same = 0
    lost = 0
    for i in range(len(scen)):
        if rs["status"][i] == 4 and rs["n_expanded"][i] == 0 and rf["n_expanded"][i] > 0:
            assert rs["path_len"][i] == 0, i                          # HL_STATUS_CAPACITY, nothing written
            lost += 1
            continue
        for f in ("status", "counter", "n_expanded", "path_len"):
            assert rs[f][i] == rf[f][i], (i, f)
        assert np.array_equal(_keys(small, i), _keys(full, i)), i
        same += rf["n_expanded"][i] > 0
    assert lost > 0 and same > 0, (lost, same)
    assert int((rs["n_expanded"].astype(np.int64)).sum()) <= need // 2
