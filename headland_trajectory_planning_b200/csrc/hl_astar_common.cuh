// hl_astar_common.cuh -- shared pieces of the K4 search kernels (parameters, per-scenario workspace, output block,
// grid keys, hash set, heapdict replay, pose filter, heuristic, rollout, start node, result write-out).
//
// Replaces HybridAStarSearch.hybrid_a_star_search (path_planner/hybrid_a_star_search.py:497-607,
// King mode): every popped node first gets a Reeds-Shepp analytic shot over all words
// (:232-287), then the 14 motion primitives are rolled out (:357-410), collision-checked
// against obstacles + field polygon + guide lane (:412-427), costed (:306-329) and merged
// into the open list (:580-596).  The pop->expand->push chain of ONE scenario is sequential;
// the parallelism is (a) scenarios across CTAs (persistent CTAs pull scenario ids from an
// atomic counter), (b) inside an expansion: 46 word solvers, the poses of a word, the
// 14 x (n+1) primitive poses, the guide-point argmin.
//
// Exactness: everything that feeds a discrete decision (rollout, grid keys, g-cost,
// heuristic, priorities, word validity/dedup/cost, heap order, sample counts) is float64 in
// the reference's operation order; the open list replays heapdict's tie behaviour
// (oracle/heapdict_port.py).  Footprint tests go through the float32 filter first and
// escalate to the float64 predicates only inside the error band, and only when no other
// pose of the same path already decided it.
// The search kernel runs many different phases on different warps/CTAs at once; with every helper
// inlined its SASS was 460 KB and 73 % of the non-barrier stall samples were instruction-fetch misses
// (profiles/r1b).  HL_SHARED_CODE makes the heavy helpers out-of-line so the kernel keeps one copy.
#define HL_SHARED_CODE 1
#pragma once
#include <cstring>
#include "hl_geom.cuh"
#include "hl_rs.cuh"
#include "hl_dubins.cuh"

#define AS_ROLL (HL_MAX_ROLLOUT + 1)
#define AS_ENV_FLOATS 512       // staged float32 environment of one scenario (canonical: 8x28 + 16x12 + 4x4 = 432 floats)
#define KEY_EMPTY (-1LL)
#define FULL 0xffffffffu
enum { ST_IDLE = 0, ST_SEARCH = 1, ST_DONE = 2 };   // scenario slot of the persistent kernels
// phase timers (cycles of lane 0 between phases), the device analogue of the reference's three
// accumulating timers (hybrid_a_star_search.py:91-94): summed over scenarios into ctx->d_counters
enum { PH_POP = 0, PH_RS_CAND, PH_RS_SELECT, PH_RS_PLAN, PH_RS_SAMPLE, PH_ARRIVE, PH_ROLLOUT, PH_FILTER, PH_EXACT,
       PH_COST_HEUR, PH_MERGE, PH_SETUP, PH_OUTPUT, AS_N_PHASES };

struct AsParams {
    double res, yaw_res, maxc, max_steer, wheel_base;
    int n_prims;
    double steer[HL_MAX_PRIMS], dir[HL_MAX_PRIMS], yaw_step[HL_MAX_PRIMS], curv[HL_MAX_PRIMS], steer_eff[HL_MAX_PRIMS];
    double steer_cost, delta_steer_cost, dir_change_cost, reverse_cost, hybrid_cost, min_len_goal;
    int max_nodes, max_path_poses;
    int cap_nodes, hash_size;
    int pawn;                 // motion_type "Pawn": forward-only primitives, Dubins goal extension (:184-230, :289-304)
    int dub_cap;              // capacity (samples / course rows) of the Dubins scratch of one scenario slot
};

// per-CTA workspace in global memory (L2 resident while the scenario runs)
struct AsWs {
    double* nx; double* ny; double* nyaw; double* ng;
    long long* nkey;
    int* nparent; int* nheap; int* nhpos;
    signed char* nprim; signed char* nsteps; signed char* nstate;
    long long* hkey; int* hval;
    double* hprio; int* hslot;
    int* corder;
    long long* cref;          // algorithmic primitive-pose checks done BEFORE pop i was expanded
    double* dub;              // Pawn mode: 13 x dub_cap doubles (ts kx ky ks dx dy cp bx by | rx ry ryaw rk), else unused
};

// where a search writes its results (pools are shared by the batch and claimed with the cursors)
struct AsOut {
    HlPlanResult* results;
    int32_t* expanded_keys;
    long long keys_capacity;
    unsigned long long* keys_cursor;
    double* path_x; double* path_y; double* path_yaw; double* path_k;
    int8_t* path_dir;
    long long path_capacity;
    unsigned long long* path_cursor;
    unsigned long long* phase_cycles;
    // two-phase sweeps (k_hybrid_astar_s): `order` lists the scenarios to run (NULL = 0 .. n-1; `order_count` then holds
    // their number on the device); with `first_only` a scenario whose FIRST analytic shot fails is not searched but
    // appended to `defer_list` for the second launch
    const int* order; const int* order_count;
    int* defer_list; int* defer_count;
    int first_only;
};

__host__ __device__ inline size_t as_align(size_t x) { return (x + 255) & ~(size_t)255; }

__host__ __device__ inline size_t as_ws_bytes(int cap, int hsize, int max_nodes, int dub_cap = 0) {
    size_t b = 0;
    b += 4 * as_align(sizeof(double) * cap);           // nx ny nyaw ng
    b += as_align(sizeof(long long) * cap);            // nkey
    b += 3 * as_align(sizeof(int) * cap);              // nparent nheap nhpos
    b += 3 * as_align(cap);                            // nprim nsteps nstate
    b += as_align(sizeof(long long) * hsize) + as_align(sizeof(int) * hsize);
    b += as_align(sizeof(double) * cap) + as_align(sizeof(int) * cap);
    b += as_align(sizeof(int) * (max_nodes + 4));
    b += as_align(sizeof(long long) * (max_nodes + 4));
    b += as_align(sizeof(double) * 13 * (size_t)dub_cap);
    return b;
}

__device__ inline AsWs as_carve(char* base, int cap, int hsize, int max_nodes, int dub_cap = 0) {
    AsWs w;
    char* p = base;
    auto take = [&](size_t bytes) { char* r = p; p += as_align(bytes); return r; };
    w.nx = (double*)take(sizeof(double) * cap); w.ny = (double*)take(sizeof(double) * cap);
    w.nyaw = (double*)take(sizeof(double) * cap); w.ng = (double*)take(sizeof(double) * cap);
    w.nkey = (long long*)take(sizeof(long long) * cap);
    w.nparent = (int*)take(sizeof(int) * cap); w.nheap = (int*)take(sizeof(int) * cap);
    w.nhpos = (int*)take(sizeof(int) * cap);
    w.nprim = (signed char*)take(cap); w.nsteps = (signed char*)take(cap); w.nstate = (signed char*)take(cap);
    w.hkey = (long long*)take(sizeof(long long) * hsize); w.hval = (int*)take(sizeof(int) * hsize);
    w.hprio = (double*)take(sizeof(double) * cap); w.hslot = (int*)take(sizeof(int) * cap);
    w.corder = (int*)take(sizeof(int) * (max_nodes + 4));
    w.cref = (long long*)take(sizeof(long long) * (max_nodes + 4));
    w.dub = (double*)take(sizeof(double) * 13 * (size_t)dub_cap);
    return w;
}

// ---- grid key (calculate_node_index, :82-89): Python round() = half-to-even = rint
__device__ __forceinline__ bool make_key(double x, double y, double yaw, double res, double yaw_res,
                                         int& ix, int& iy, int& iyaw, long long& key) {
    double fx = rint(xdiv(x, res)), fy = rint(xdiv(y, res)), fw = rint(xdiv(yaw, yaw_res));
    if (!(fabs(fx) < 8388607.0) || !(fabs(fy) < 8388607.0) || !(fabs(fw) < 127.0)) return false;
    ix = (int)fx; iy = (int)fy; iyaw = (int)fw;
    key = ((long long)(ix + 8388608) << 32) | ((long long)(iy + 8388608) << 8) | (long long)(iyaw + 128);
    return true;
}

__device__ __forceinline__ void unpack_key(long long key, int& ix, int& iy, int& iyaw) {
    ix = (int)(key >> 32) - 8388608;
    iy = (int)((key >> 8) & 0xFFFFFF) - 8388608;
    iyaw = (int)(key & 0xFF) - 128;
}

__device__ __forceinline__ unsigned hash_key(long long k) {
    unsigned long long z = (unsigned long long)k * 0x9E3779B97F4A7C15ULL;
    return (unsigned)(z >> 40);
}

// returns slot or -1; *pos = table position where the key is / would be inserted
__device__ __noinline__ int hash_find(const AsWs& w, int hmask, long long key, int* pos) {
    unsigned h = hash_key(key) & hmask;
    while (true) {
        long long k = w.hkey[h];
        if (k == key) { *pos = (int)h; return w.hval[h]; }
        if (k == KEY_EMPTY) { *pos = (int)h; return -1; }
        h = (h + 1) & hmask;
    }
}

// ---- heapdict replay (oracle/heapdict_port.py) on (hprio, hslot) with nheap[] positions
// heapdict moves entries by swaps; here the moving entry is carried in registers and the entries it passes are
// shifted into the hole -- the arrangement after every operation is the one the swaps produce (comparisons look at the
// priority only, strict `<`, left child first), with half the memory operations on the dependent chain.
// The first HS heap positions (the top log2(HS+1) levels, where every sift spends most of its steps) may live in
// SHARED memory (sp / ss): an LDS is ~30 cycles, a workspace load that misses L1 several hundred, and the sifts are a
// serial chain on one lane (K4 spec variant: pop + merge were 25 % of the expander's time on global memory).
template <int HS> struct HeapRef {
    const AsWs& w; double* sp; int* ss;
    __device__ __forceinline__ double prio(int i) const { return (HS > 0 && i < HS) ? sp[i] : w.hprio[i]; }
    __device__ __forceinline__ int slot(int i) const { return (HS > 0 && i < HS) ? ss[i] : w.hslot[i]; }
    __device__ __forceinline__ void put(int i, double p, int s) const {
        if (HS > 0 && i < HS) { sp[i] = p; ss[i] = s; } else { w.hprio[i] = p; w.hslot[i] = s; }
        w.nheap[s] = i;
    }
};

// _decrease_key (or, with `always`, the unconditional bubbling of __delitem__) of the entry (prio, slot) at position i
template <int HS> __device__ __forceinline__ void heap_up_t(const HeapRef<HS>& H, int i, double prio, int slot, bool always) {
    while (i) {
        const int parent = (i - 1) >> 1;
        const double pp = H.prio(parent);
        if (!always && pp < prio) break;
        H.put(i, pp, H.slot(parent));
        i = parent;
    }
    H.put(i, prio, slot);
}

template <int HS> __device__ __forceinline__ int heap_popitem_t(const HeapRef<HS>& H, int& n) {
    const int top = H.slot(0);
    --n;
    if (n > 0) {
        const double prio = H.prio(n);                 // heap[0] = heap.pop(); _min_heapify(0)
        const int slot = H.slot(n);
        int i = 0;
        while (true) {
            const int l = (i << 1) + 1, r = l + 1;
            int low = i;
            double lowp = prio;
            if (l < n) {
                const double pl = H.prio(l);
                const double pr = (r < n) ? H.prio(r) : 0.0;
                if (pl < lowp) { low = l; lowp = pl; }
                if (r < n && pr < lowp) { low = r; lowp = pr; }
            }
            if (low == i) break;
            H.put(i, lowp, H.slot(low));
            i = low;
        }
        H.put(i, prio, slot);
    }
    H.w.nheap[top] = -1;
    return top;
}

template <int HS> __device__ __forceinline__ void heap_set_t(const HeapRef<HS>& H, int& n, int slot, double prio) {
    const int at = H.w.nheap[slot];
    if (at >= 0) {                                     // __setitem__ on an existing key: pop(key) first
        heap_up_t<HS>(H, at, 0.0, slot, true);         // __delitem__: bubble to the root unconditionally
        heap_popitem_t<HS>(H, n);
    }
    heap_up_t<HS>(H, n++, prio, slot, false);
}

// workspace-only heap (one-warp-per-scenario and level-synchronous variants)
__device__ __noinline__ int heap_popitem(const AsWs& w, int& n) {
    const HeapRef<0> H{w, nullptr, nullptr};
    return heap_popitem_t<0>(H, n);
}
__device__ __noinline__ void heap_set(const AsWs& w, int& n, int slot, double prio) {
    const HeapRef<0> H{w, nullptr, nullptr};
    heap_set_t<0>(H, n, slot, prio);
}

// Ternary footprint status of one pose (body only): HL_FREE / HL_HIT / HL_AMBIG(+mask)
__device__ HL_CODE int pose_filter(const EnvDesc& D, const EnvSmem& E, double x, double y, double yaw,
                                           unsigned flags, unsigned* amb) {
    float px = (float)(x - D.origin[0]), py = (float)(y - D.origin[1]);
    if (fabsf(px) > E.reach || fabsf(py) > E.reach) return far_status(flags, E.n_seg);
    if (!(fabs(yaw) < 1e6) || !(px == px) || !(py == py)) { *amb = flags; return HL_AMBIG; }
    float sf, cf;
    sincosf((float)yaw, &sf, &cf);
    return filter_part(E, px, py, cf, sf, E.ext, flags, amb);
}

__device__ __noinline__ bool pose_exact(const EnvBatchDev& eb, const EnvDesc& D, double x, double y, double yaw,
                                           unsigned amb) {
    Pose64 p;
    p.x = x; p.y = y; p.c = m_cos(yaw); p.s = m_sin(yaw);
    return exact_part_check(p, D.body_ext, eb, D, amb);
}

// float32 environment of a warp's scenario into its shared-memory slice (falls back to global pointers)
__device__ __noinline__ void stage_env_warp(const EnvBatchDev& eb, const EnvDesc& D, float* sm, int cap_floats,
                                            EnvSmem& E, int lane) {
    const int n_o = D.n_obs * HL_OBS32_STRIDE, n_f = D.n_field * HL_FIELD32_STRIDE, n_s = D.n_seg * 4;
    E.n_obs = D.n_obs; E.n_field = D.n_field; E.n_seg = D.n_seg; E.all_rect = D.all_rect;
    E.eps = D.eps; E.reach = D.reach;
    for (int k = 0; k < 4; ++k) E.ext[k] = (float)D.body_ext[k];
    const float* g_obs = eb.obs32 + (size_t)HL_OBS32_STRIDE * D.obs_off;
    const float* g_field = eb.field32 + HL_FIELD32_STRIDE * (size_t)D.field_off;
    const float* g_seg = eb.seg32 + 4 * (size_t)D.seg_off;
    if (n_o + n_f + n_s <= cap_floats) {
        float* s_obs = sm;
        float* s_field = s_obs + n_o;
        float* s_seg = s_field + n_f;
        for (int i = lane; i < n_o; i += 32) s_obs[i] = g_obs[i];
        for (int i = lane; i < n_f; i += 32) s_field[i] = g_field[i];
        for (int i = lane; i < n_s; i += 32) s_seg[i] = g_seg[i];
        E.obs = s_obs; E.field = s_field; E.seg = s_seg;
    } else {
        E.obs = g_obs; E.field = g_field; E.seg = g_seg;
    }
    __syncwarp();
}

// calculate_state_cost (reference_line_heuristic.py:131-158) for one pose, one warp.
__device__ __noinline__ double warp_state_cost(const EnvBatchDev& eb, const EnvDesc& D, double x, double y, double yaw, int lane) {
    const double* gx = eb.guide_x + D.guide_off;
    const double* gy = eb.guide_y + D.guide_off;
    const int n = D.n_guide;
    if (n <= 0) return 0.0;
    // pass 1: minimum squared distance (ordering filter only)
    double best = INFINITY;
#pragma unroll 1
    for (int i = lane; i < n; i += 32) {
        double dx = gx[i] - x, dy = gy[i] - y;
        best = fmin(best, dx * dx + dy * dy);
    }
    for (int o = 16; o; o >>= 1) best = fmin(best, __shfl_xor_sync(0xffffffffu, best, o));
    // pass 2: exact hypot on the near-minimal candidates, first minimum wins (np.argmin)
    const double thr = best * (1.0 + 1e-9) + 1e-300;
    double bh = INFINITY;
    int bi = 0x7fffffff;
#pragma unroll 1
    for (int i = lane; i < n; i += 32) {
        double dx = xsub(gx[i], x), dy = xsub(gy[i], y);
        if (dx * dx + dy * dy <= thr) {
            double h = hypot_cr(dx, dy);
            if (h < bh || (h == bh && i < bi)) { bh = h; bi = i; }
        }
    }
    for (int o = 16; o; o >>= 1) {
        double oh = __shfl_xor_sync(0xffffffffu, bh, o);
        int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oh < bh || (oh == bh && oi < bi)) { bh = oh; bi = oi; }
    }
    double dist = xmul(bh, 100.0);
    double yaw_diff = fabs(angle_wrap(xsub(eb.guide_yaw[D.guide_off + bi], yaw)));
    if (dist > 2.0) dist = 100.0;
    double to_goal = xsub(eb.guide_s[D.guide_off + n - 1], eb.guide_s[D.guide_off + bi]);
    return xadd(xadd(dist, xmul(yaw_diff, 0.2)), xmul(to_goal, 5.0));
}

// One step of the kinematic rollout (kinematic_simulation_node, :366-390): yaws[i] of
// np.linspace(init_yaw, init_yaw + yaw_step*(n+1), n+2) after angle_wrap.
__device__ HL_TINY double rollout_yaw(double init_yaw, double stop, double step, double delta, int div, int i) {
    double v;
    if (i == div) v = stop;                                     // y[-1] = stop
    else if (step != 0.0) v = xadd(xmul((double)i, step), init_yaw);
    else v = xadd(xmul(xdiv((double)i, (double)div), delta), init_yaw);
    return angle_wrap(v);
}


// ---- both ends of a search, shared by the three kernels (spec, warp, level)

struct AsStart { int status; long long start_key, goal_key; double prio; };

// Start / goal feasibility (:76-80, :516-519), start node and its priority (:500-510), whole warp.  Node 0 and its
// hash entry are written here; the heap push is the caller's.  The result is valid on lane 0: status -1 = search,
// else HL_STATUS_CAPACITY (a pose outside the grid-key range) or HL_STATUS_START_GOAL_BLOCKED.  Inlined: the spec
// kernel spills more when it is a call.
__device__ __forceinline__ AsStart start_node(const AsWs& W, const AsParams& P, const EnvBatchDev& eb, const EnvDesc& D,
                                           const EnvSmem& E, const double* start, const double* goal, unsigned flags,
                                           int lane) {
    int bad = 0;
    if (lane < 2) {
        const double* q = lane == 0 ? start : goal;
        unsigned amb = flags;
        int r = pose_filter(D, E, q[0], q[1], q[2], flags, &amb);
        bad = (r == HL_HIT) || (r == HL_AMBIG && pose_exact(eb, D, q[0], q[1], q[2], amb));
    }
    bad = __any_sync(FULL, bad);
    const double h = warp_state_cost(eb, D, start[0], start[1], start[2], lane);
    AsStart s;
    s.status = -1; s.start_key = 0; s.goal_key = 0; s.prio = 0.0;
    if (lane == 0) {
        int ix, iy, iw;
        bool ok = make_key(start[0], start[1], start[2], P.res, P.yaw_res, ix, iy, iw, s.start_key);
        ok = make_key(goal[0], goal[1], goal[2], P.res, P.yaw_res, ix, iy, iw, s.goal_key) && ok;
        if (!ok) s.status = HL_STATUS_CAPACITY;
        else if (bad) s.status = HL_STATUS_START_GOAL_BLOCKED;
        else {
            W.nx[0] = start[0]; W.ny[0] = start[1]; W.nyaw[0] = start[2]; W.ng[0] = 0.0;
            W.nkey[0] = s.start_key; W.nparent[0] = 0; W.nprim[0] = -1; W.nsteps[0] = 0; W.nstate[0] = 0;
            W.nheap[0] = -1;
            int pos;
            hash_find(W, P.hash_size - 1, s.start_key, &pos);
            W.hkey[pos] = s.start_key; W.hval[pos] = 0; W.nhpos[0] = pos;
            s.prio = xmul(P.hybrid_cost, h);
            s.prio = (s.prio > 0.0) ? s.prio : 0.0;       // max(start.cost = 0, 50*h)
        }
    }
    return s;
}

struct AsWritten { int status, n_keys; long long keys_off; int path_len; long long path_off; };

// Expanded keys and path (get_path_from_expanded_nodes, :429-454) of a finished search, whole warp.  `end` is the node
// the search ended on.  At arrival == 1 the path ends with the goal extension: the Reeds-Shepp word `plan`, sampled
// here, or with plan == NULL the `dub_rows` rows of the Dubins course kept in W.dub.  A pool that is too small gives
// HL_STATUS_CAPACITY, never a truncated result: no keys when the keys pool overflows, no path when the node chain or
// the path pool does.  The result is the same on every lane.
__device__ __noinline__ AsWritten write_outputs(const AsWs& W, const AsParams& P, const AsOut& O, int status, int n_closed,
                                                int end, int arrival, long long start_key, long long goal_key,
                                                const RsPlan* plan, int dub_rows, int lane) {
    AsWritten w;
    long long koff = 0;
    if (lane == 0 && n_closed > 0) {
        koff = (long long)atomicAdd(O.keys_cursor, (unsigned long long)n_closed);
        if (koff + n_closed > O.keys_capacity) koff = -1;
    }
    koff = __shfl_sync(FULL, koff, 0);
    w.n_keys = n_closed;
    if (koff < 0) { status = HL_STATUS_CAPACITY; w.n_keys = 0; koff = 0; }
    w.keys_off = koff;
    int32_t* ek = O.expanded_keys + (size_t)koff * 3;
    for (int i = lane; i < w.n_keys; i += 32) {
        int ix, iy, iw;
        unpack_key(W.nkey[W.corder[i]], ix, iy, iw);
        ek[3 * i] = ix; ek[3 * i + 1] = iy; ek[3 * i + 2] = iw;
    }
    const int ext_rows = arrival != 1 ? 0 : (plan ? plan->npts : dub_rows);
    int len = 0, path_len = 0;
    long long path_off = 0;
    if (lane == 0 && status == HL_STATUS_OK) {
        // Walk end -> parent -> ... -> start (slot 0 is the only node with the start key).  The chain is kept in
        // hslot[] (the heap is dead once the search is over), goal side first.  closed_set[goal_key] is the goal
        // node, so a goal in the start's own cell makes the reference's `while current_node_index !=
        // start_node_index` loop a no-op: empty path.
        int poses = 0;
        bool ok = true;
        if (goal_key != start_key) {
            for (int node = end; node != 0; node = W.nparent[node]) {
                if (len >= P.cap_nodes) { ok = false; break; }
                W.hslot[len++] = node;
                poses += W.nsteps[node] + 1;
            }
            poses += ext_rows;
        }
        path_len = poses;
        if (!ok || path_len > P.max_path_poses) { status = HL_STATUS_CAPACITY; path_len = 0; }
        else if (path_len > 0) {
            unsigned long long off = atomicAdd(O.path_cursor, (unsigned long long)path_len);
            if ((long long)(off + path_len) > O.path_capacity) { status = HL_STATUS_CAPACITY; path_len = 0; }
            path_off = (long long)off;
        }
    }
    __syncwarp();
    w.status = __shfl_sync(FULL, status, 0);
    w.path_len = __shfl_sync(FULL, path_len, 0);
    w.path_off = __shfl_sync(FULL, path_off, 0);
    len = __shfl_sync(FULL, len, 0);
    if (w.status == HL_STATUS_OK && w.path_len > 0) {
        for (int c = lane; c < len; c += 32) {
            const int node = W.hslot[len - 1 - c];          // c-th node from the start side
            long long off = w.path_off;
            for (int q = 0; q < c; ++q) off += W.nsteps[W.hslot[len - 1 - q]] + 1;
            const int par = W.nparent[node];
            const int p = W.nprim[node], n = W.nsteps[node];
            const double ys = P.yaw_step[p];
            const double init_yaw = angle_wrap(xadd(W.nyaw[par], ys));
            const double stop = xadd(init_yaw, xmul(ys, (double)(n + 1)));
            const double delta = xsub(stop, init_yaw);
            const double step = xdiv(delta, (double)(n + 1));
            double ax = 0.0, ay = 0.0;
            for (int i = 0; i <= n; ++i) {
                const double yw = rollout_yaw(init_yaw, stop, step, delta, n + 1, i);
                const double txv = xmul(xmul(P.res, m_cos(yw)), P.dir[p]);
                const double tyv = xmul(xmul(P.res, m_sin(yw)), P.dir[p]);
                ax = (i == 0) ? txv : xadd(ax, txv);
                ay = (i == 0) ? tyv : xadd(ay, tyv);
                O.path_x[off + i] = xadd(W.nx[par], ax);
                O.path_y[off + i] = xadd(W.ny[par], ay);
                O.path_yaw[off + i] = rollout_yaw(init_yaw, stop, step, delta, n + 1, i + 1);
                O.path_k[off + i] = P.curv[p];
                O.path_dir[off + i] = (int8_t)P.dir[p];
            }
        }
        const long long off = w.path_off + (w.path_len - ext_rows);
        if (arrival == 1 && plan) {
            const double q0[3] = {W.nx[end], W.ny[end], W.nyaw[end]};
            const double cq = m_cos(-q0[2]), sq = m_sin(-q0[2]);
            for (int j = lane; j < ext_rows; j += 32) {
                double lx, ly, lyaw, wx, wy, wyaw;
                int cs, dir;
                rs_sample_local(*plan, j, P.maxc, lx, ly, lyaw, cs, dir);
                rs_to_world(q0, cq, sq, lx, ly, lyaw, wx, wy, wyaw);
                O.path_x[off + j] = wx; O.path_y[off + j] = wy; O.path_yaw[off + j] = wyaw;
                O.path_k[off + j] = cs == 0 ? 0.0 : (cs > 0 ? P.maxc : -P.maxc);
                O.path_dir[off + j] = (int8_t)dir;
            }
        } else if (arrival == 1) {                          // Pawn: the Dubins course rows kept in the scratch
            const double* rx = W.dub + 9 * (size_t)P.dub_cap;
            const double* ry = rx + P.dub_cap; const double* ryaw = ry + P.dub_cap; const double* rk = ryaw + P.dub_cap;
            for (int j = lane; j < ext_rows; j += 32) {
                O.path_x[off + j] = rx[j]; O.path_y[off + j] = ry[j]; O.path_yaw[off + j] = ryaw[j];
                O.path_k[off + j] = rk[j]; O.path_dir[off + j] = (int8_t)1;
            }
        }
    }
    __syncwarp();
    return w;
}

// Result record of a finished search (one lane).  A blocked start or goal reports no pops and no algorithmic pose
// checks; only an analytic-shot arrival reports the word it took.
__device__ __noinline__ void write_record(const AsOut& O, int sc, const AsWritten& w, int arrival, int rs_word,
                                             double goal_cost, int counter, unsigned long long checks,
                                             unsigned long long exact, unsigned long long checks_ref, long long cycles) {
    const bool blocked = w.status == HL_STATUS_START_GOAL_BLOCKED;
    HlPlanResult r;
    r.status = w.status;
    r.counter = blocked ? 0 : counter;
    r.n_expanded = w.n_keys;
    r.arrival = arrival;
    r.path_len = w.path_len;
    r.rs_word = arrival == 1 ? rs_word : -1;
    r.path_offset = w.path_off;
    r.keys_offset = w.keys_off;
    r.goal_cost = goal_cost;
    r.n_pose_checks = (long long)checks;
    r.n_exact = (long long)exact;
    r.n_pose_checks_ref = blocked ? 0 : (long long)checks_ref;
    r.cycles = cycles;
    O.results[sc] = r;
}
