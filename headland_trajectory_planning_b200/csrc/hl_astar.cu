// hl_astar.cu -- K4: batched Hybrid A* warm-start search, ONE WARP PER SCENARIO, phase-aligned CTAs.
//
// Replaces HybridAStarSearch.hybrid_a_star_search (path_planner/hybrid_a_star_search.py:497-607,
// King mode).  Shared pieces (workspace, keys, hash, heapdict replay, filter, heuristic) are in
// hl_astar_common.cuh; the float64/float32 split is described there and in DESIGN.md.
//
// Why a warp and not a CTA per scenario: the first version (one CTA per scenario, removed; profiles/r1b_*) gave a
// scenario 128 threads.  Its profile (profiles/r1b_*) showed 52 % of warp samples waiting at CTA barriers
// for the serial thread, and 73 % of the remaining stalls were INSTRUCTION-FETCH misses: one expansion walks
// ~100 KB of straight-line float64 code exactly once, and four co-resident CTAs in four different phases
// evict each other from the 32 KB instruction cache.  Here every scenario owns one warp (serial sections on
// lane 0, parallel sections on 32 lanes, __syncwarp instead of __syncthreads), a CTA carries AW_WARPS
// scenarios, and two CTA-wide alignment barriers per expansion keep all warps of the SM inside the same
// code region, so an instruction line fetched once serves AW_WARPS scenarios.  Warps pull scenario ids from
// an atomic counter as soon as theirs finishes.
#include <cstdlib>
#include <cstdio>
#include <mutex>
#include "hl_astar_common.cuh"

#ifndef AW_WARPS
#define AW_WARPS 12
#endif
#ifndef AW_MIN_CTAS
#define AW_MIN_CTAS 1
#endif
#ifndef AW_MAX_PLANS
#define AW_MAX_PLANS 6
#endif

struct AwSmem {                          // one per warp
    double start[3], goal[3];
    long long start_key, goal_key;
    int env, scen, state;
    int n_nodes, heap_n, counter, n_closed;
    int status, arrival, rs_word;
    double goal_cost;
    int cur; double cx, cy, cyaw, cg; int cprim; int nsteps;
    // The Reeds-Shepp shot and the primitive expansion of one node never overlap in time (a successful shot
    // ends the search before any primitive is rolled out), so their scratch shares storage.
    union {
        struct {
            double rs_lens[HL_RS_CANDIDATES][HL_RS_MAX_SEGS];
            double rs_L[HL_RS_CANDIDATES], rs_prio[HL_RS_CANDIDATES], rs_Lc[HL_RS_CANDIDATES];
            int rs_acc[HL_RS_CANDIDATES], rs_order[HL_RS_CANDIDATES];
            unsigned char rs_valid[HL_RS_CANDIDATES + 2], rs_accept[HL_RS_CANDIDATES + 2];
            RsPlan plans[AW_MAX_PLANS];
            RsPlan plan_tmp;
        };
        struct {
            double tx[HL_MAX_PRIMS][AS_ROLL], ty[HL_MAX_PRIMS][AS_ROLL], pyaw[HL_MAX_PRIMS][AS_ROLL];
            unsigned char pamb[HL_MAX_PRIMS][AS_ROLL];
            double pg[HL_MAX_PRIMS], pprio[HL_MAX_PRIMS];
            long long pkey[HL_MAX_PRIMS];
            int pkey_ok[HL_MAX_PRIMS], pslot[HL_MAX_PRIMS], ppos[HL_MAX_PRIMS], pneed[HL_MAX_PRIMS];
        };
    };
    RsProblem rs_prob;
    int rs_n, rs_pick;
    int dub_rows;                        // Pawn: rows of the accepted Dubins course (kept in the slot's global scratch)
    int phit[HL_MAX_PRIMS];
    // stats
    unsigned long long n_checks, n_exact, n_ref;
    long long t_last, t_phase[AS_N_PHASES];
    __align__(16) float envf[AS_ENV_FLOATS];
};

static_assert(sizeof(AwSmem) * AW_WARPS <= 227 * 1024, "per-CTA shared memory exceeds 227 KB");
#define TICK(ph) do { if (lane == 0) { long long _n = clock64(); S.t_phase[ph] += _n - S.t_last; S.t_last = _n; } } while (0)

// Results of a finished scenario: expanded keys, path, record; then the used hash positions are reset for the next
// scenario of this warp.  Inlined: as a call of its own around the write-out call, the kernel spills more.
__device__ __forceinline__ void finalize_scenario(AwSmem& S, const AsWs& W, const AsParams& P, const AsOut& O, int lane) {
    const RsPlan* plan = P.pawn ? nullptr : (S.rs_pick >= 0 && S.rs_pick < AW_MAX_PLANS ? &S.plans[S.rs_pick] : &S.plan_tmp);
    const AsWritten w = write_outputs(W, P, O, S.status, S.n_closed, S.cur, S.arrival, S.start_key, S.goal_key, plan,
                                      S.dub_rows, lane);
    if (lane == 0) {
        S.t_phase[PH_OUTPUT] += clock64() - S.t_last;
        long long tot = 0;
        for (int k = 0; k < AS_N_PHASES; ++k) tot += S.t_phase[k];
        write_record(O, S.scen, w, S.arrival, S.rs_word, S.goal_cost, S.counter, S.n_checks, S.n_exact, S.n_ref, tot);
        for (int k = 0; k < AS_N_PHASES; ++k) atomicAdd(O.phase_cycles + k, (unsigned long long)S.t_phase[k]);
    }
    for (int i = lane; i < S.n_nodes; i += 32) W.hkey[W.nhpos[i]] = KEY_EMPTY;
    __syncwarp();
}

__device__ __noinline__ void setup_scenario(AwSmem& S, const AsWs& W, const AsParams& P, const EnvBatchDev& eb,
                                            const EnvDesc& D, const EnvSmem& E, unsigned FLAGS, int lane) {
    const AsStart st = start_node(W, P, eb, D, E, S.start, S.goal, FLAGS, lane);
    if (lane == 0) {
        S.start_key = st.start_key; S.goal_key = st.goal_key; S.status = st.status;
        if (st.status < 0) { S.n_nodes = 1; heap_set(W, S.heap_n, 0, st.prio); }
    }
    __syncwarp();
}

// Pawn goal extension (_get_goal_extension_with_dubins_path, hybrid_a_star_search.py:184-230 with get_dubins_path
// :289-304 and calculate_dubins_path_cost :162-182): shortest Dubins path from the popped node to the goal, sampled at
// plan_resolution, the goal pose appended, cubic-spline course at plan_resolution, yaws wrapped, footprint check of
// every row, length below MIN_LENGTH_TO_GOAL.  One warp; the knots and the rows live in the slot's global scratch.
__device__ __noinline__ void pawn_shot(AwSmem& S, const AsWs& W, const AsParams& P, const EnvBatchDev& eb, const EnvDesc& D,
                                       const EnvSmem& E, unsigned FLAGS, int lane) {
    const int cap = P.dub_cap;
    double* ts = W.dub; double* kx = ts + cap; double* ky = kx + cap; double* ks = ky + cap; double* dx = ks + cap;
    double* dy = dx + cap; double* cp = dy + cap; double* bx = cp + cap; double* by = bx + cap;
    double* rx = by + cap; double* ry = rx + cap; double* ryaw = ry + cap; double* rk = ryaw + cap;
    const double q0[3] = {S.cx, S.cy, S.cyaw};
    DubPath path;
    dub_shortest(q0, S.goal, xdiv(1.0, P.maxc), path);
    if (path.type < 0) { if (lane == 0) S.status = HL_STATUS_RS_ASSERT; __syncwarp(); return; }   // dubins raises
    const long long n_s = dub_n_samples(dub_length(path), P.res);
    if (n_s + 1 > cap) { if (lane == 0) S.status = HL_STATUS_CAPACITY; __syncwarp(); return; }
    const int m = dub_course_knots(path, P.res, true, S.goal, n_s, ts, kx, ky, ks, lane);
    if (m < 2) { if (lane == 0) S.status = HL_STATUS_RS_ASSERT; __syncwarp(); return; }          // scipy raises on < 2 knots
    if (lane == 0) rp_derivs(ks, kx, ky, m, dx, dy, cp, bx, by);
    __syncwarp();
    const long long cnt = rp_count(ks[m - 1], P.res);
    if (cnt > cap) { if (lane == 0) S.status = HL_STATUS_CAPACITY; __syncwarp(); return; }
    for (long long i = lane; i < cnt; i += 32) {
        const double t = xmul((double)i, P.res);
        double x, x1, x2, y, y1, y2;
        rp_eval(ks, kx, dx, m, t, x, x1, x2);
        rp_eval(ks, ky, dy, m, t, y, y1, y2);
        const double q = x1 * x1 + y1 * y1;
        rx[i] = x; ry[i] = y; ryaw[i] = angle_wrap(m_atan2(y1, x1));
        rk[i] = (y2 * x1 - x2 * y1) / (q * sqrt(q));
    }
    __syncwarp();
    if (lane == 0) S.n_ref += (unsigned long long)cnt;
    int infeasible = 0;
    for (long long base = 0; base < cnt && !infeasible; base += 32) {
        const long long i = base + lane;
        int st = HL_FREE;
        unsigned amb = 0;
        if (i < cnt) st = pose_filter(D, E, rx[i], ry[i], ryaw[i], FLAGS, &amb);
        const unsigned livem = __ballot_sync(FULL, i < cnt);
        const unsigned hitm = __ballot_sync(FULL, st == HL_HIT);
        const unsigned ambm = __ballot_sync(FULL, st == HL_AMBIG);
        infeasible = hitm != 0;
        if (!infeasible && ambm) {
            int bad = 0;
            if (st == HL_AMBIG) bad = pose_exact(eb, D, rx[i], ry[i], ryaw[i], amb) ? 1 : 0;
            if (lane == 0) S.n_exact += (unsigned long long)__popc(ambm);
            infeasible = __any_sync(FULL, bad);
        }
        if (lane == 0) S.n_checks += (unsigned long long)__popc(livem);
    }
    if (!infeasible && lane == 0) {
        // calculate_path_length (np.hypot of the diffs, cumsum) and the spread of the curvature column ([Q]: the
        // reference takes path[:, -1] of the 4-column array for its "delta yaw")
        double len = 0.0, kmin = rk[0], kmax = rk[0];
        for (long long i = 0; i + 1 < cnt; ++i) {
            const double dsl = hypot_cr(xsub(rx[i + 1], rx[i]), xsub(ry[i + 1], ry[i]));
            len = (i == 0) ? dsl : xadd(len, dsl);
        }
        for (long long i = 1; i < cnt; ++i) { kmin = fmin(kmin, rk[i]); kmax = fmax(kmax, rk[i]); }
        if (len < P.min_len_goal) {
            S.arrival = 1; S.rs_word = path.type; S.dub_rows = (int)cnt;
            S.goal_cost = xadd(xadd(S.cg, len), xmul(angle_wrap(xsub(kmax, kmin)), P.steer_cost));
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(AW_WARPS * 32, AW_MIN_CTAS)
k_hybrid_astar_w(EnvBatchDev eb, const HlScenario* __restrict__ scen, int n_scen, AsParams P, char* ws_base,
                 size_t ws_stride, unsigned int* work_counter, AsOut O) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    AwSmem& S = reinterpret_cast<AwSmem*>(smem_raw)[wid];
    const AsWs W = as_carve(ws_base + ((size_t)blockIdx.x * AW_WARPS + wid) * ws_stride, P.cap_nodes, P.hash_size,
                            P.max_nodes, P.dub_cap);
    const int hmask = P.hash_size - 1;
    const unsigned FLAGS = HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY | HL_CHECK_LANE;

    // hash table starts empty; afterwards only the used positions are reset
    for (int i = lane; i < P.hash_size; i += 32) W.hkey[i] = KEY_EMPTY;
    if (lane == 0) S.state = ST_IDLE;
    __syncwarp();

    EnvSmem E;
    E.n_obs = E.n_field = E.n_seg = E.all_rect = 0; E.eps = 0.f; E.reach = 0.f; E.obs = E.field = E.seg = nullptr;
    const EnvDesc* Dp = eb.desc;

    while (true) {
        // ---- refill: a warp without a scenario takes the next one from the global queue
        while (S.state == ST_IDLE) {
            int sc = 0;
            if (lane == 0) sc = (int)atomicAdd(work_counter, 1u);
            sc = __shfl_sync(FULL, sc, 0);
            if (sc >= n_scen) { if (lane == 0) S.state = ST_DONE; __syncwarp(); break; }
            if (lane == 0) {
                const HlScenario s = scen[sc];
                S.scen = sc; S.env = s.env_id;
                for (int k = 0; k < 3; ++k) { S.start[k] = s.start[k]; S.goal[k] = s.goal[k]; }
                S.n_nodes = 0; S.heap_n = 0; S.counter = 0; S.n_closed = 0;
                S.status = -1; S.arrival = 0; S.rs_word = -1; S.goal_cost = 0.0; S.rs_pick = -1;
                S.n_checks = 0; S.n_exact = 0; S.n_ref = 0;
                for (int k = 0; k < AS_N_PHASES; ++k) S.t_phase[k] = 0;
                S.t_last = clock64();
            }
            __syncwarp();
            Dp = eb.desc + S.env;
            stage_env_warp(eb, *Dp, S.envf, AS_ENV_FLOATS, E, lane);
            setup_scenario(S, W, P, eb, *Dp, E, FLAGS, lane);
            TICK(PH_SETUP);
            if (S.status >= 0) finalize_scenario(S, W, P, O, lane);        // blocked / capacity: done already
            else if (lane == 0) S.state = ST_SEARCH;
            __syncwarp();
        }
        if (__syncthreads_and(S.state == ST_DONE)) break;                   // alignment point 1
        const bool live = (S.state == ST_SEARCH);
        const EnvDesc& D = *Dp;
        if (live) {
            // ---- pop (:526-545)
            if (lane == 0) {
                if (S.counter > P.max_nodes) S.status = HL_STATUS_MAX_NODES;
                else {
                    S.counter += 1;
                    if (S.heap_n == 0) S.status = HL_STATUS_OPEN_EMPTY;
                    else {
                        int cur = heap_popitem(W, S.heap_n);
                        W.nstate[cur] = 1;
                        W.corder[S.n_closed++] = cur;
                        S.cur = cur; S.cx = W.nx[cur]; S.cy = W.ny[cur]; S.cyaw = W.nyaw[cur]; S.cg = W.ng[cur];
                        S.cprim = W.nprim[cur];
                        S.rs_pick = -1;
                        const double q0n[3] = {S.cx, S.cy, S.cyaw};
                        if (!P.pawn) S.rs_prob = rs_normalise(q0n, S.goal, P.maxc);   // generate_path (:565-572), once per pop
                    }
                }
            }
            __syncwarp();
            TICK(PH_POP);
        }
        if (live && S.status < 0 && P.pawn) {
            pawn_shot(S, W, P, eb, D, E, FLAGS, lane);
            TICK(PH_RS_SAMPLE);
        }
        if (live && S.status < 0 && !P.pawn) {
            // ---- analytic shot: 46 candidate words (:249-258)
            const double q0[3] = {S.cx, S.cy, S.cyaw};
            for (int c = lane; c < HL_RS_CANDIDATES; c += 32) {
                double l[HL_RS_MAX_SEGS] = {0, 0, 0, 0, 0};
                bool ok = rs_candidate(c, S.rs_prob, l);
                S.rs_valid[c] = ok ? 1 : 0;
                for (int k = 0; k < HL_RS_MAX_SEGS; ++k) S.rs_lens[c][k] = l[k];
            }
            __syncwarp();
            TICK(PH_RS_CAND);
            if (lane < RS_N_GROUPS) rs_select_group(lane, S.rs_valid, S.rs_lens, S.rs_accept, S.rs_Lc);
            __syncwarp();
            {
                // accepted rows in evaluation order: ballot + prefix count instead of a serial scan
                const int a0 = S.rs_accept[lane];
                const int a1 = (lane + 32 < HL_RS_CANDIDATES) ? S.rs_accept[lane + 32] : 0;
                const unsigned b0 = __ballot_sync(FULL, a0 == 1), b1 = __ballot_sync(FULL, a1 == 1);
                const unsigned bad = __ballot_sync(FULL, a0 == 2 || a1 == 2);      // `assert path.L >= 0.01`
                const unsigned lt = (1u << lane) - 1u;
                const int n0 = __popc(b0);
                if (a0 == 1) { int k = __popc(b0 & lt); S.rs_acc[k] = lane; S.rs_L[k] = S.rs_Lc[lane]; }
                if (a1 == 1) { int k = n0 + __popc(b1 & lt); S.rs_acc[k] = lane + 32; S.rs_L[k] = S.rs_Lc[lane + 32]; }
                const int m = bad ? 0 : n0 + __popc(b1);
                __syncwarp();
                for (int k = lane; k < m; k += 32)
                    S.rs_prio[k] = rs_path_cost(S.cg, S.rs_acc[k], S.rs_lens[S.rs_acc[k]], P.max_steer,
                                                P.reverse_cost, P.dir_change_cost, P.steer_cost);
                __syncwarp();
                if (lane == 0) {
                    if (bad) S.status = HL_STATUS_RS_ASSERT;
                    S.rs_n = m;
                    if (m > 0) heapdict_order(S.rs_prio, m, S.rs_order);
                }
            }
            __syncwarp();
            TICK(PH_RS_SELECT);
        }
        if (live && S.status < 0) {
            const double q0[3] = {S.cx, S.cy, S.cyaw};
            const int m = P.pawn ? 0 : S.rs_n;
            const double stepn = xmul(P.res, P.maxc);
            const double cq = m_cos(-q0[2]), sq = m_sin(-q0[2]);
            // sampling plans of the first AW_MAX_PLANS words in pop order, one lane each
            if (lane < m && lane < AW_MAX_PLANS) {
                int c = S.rs_acc[S.rs_order[lane]];
                rs_make_plan(c, S.rs_lens[c], P.maxc, stepn, S.plans[lane]);
                rs_plan_world32(S.plans[lane], q0, cq, sq, D.origin);
            }
            __syncwarp();
            TICK(PH_RS_PLAN);
            // sampled poses are float32 for the filter (1 sincosf per pose); their error (~1e-5 m) widens the band
            EnvSmem Ers = E;
            Ers.eps = E.eps + 6e-5f;
            const float inv_maxc = (float)(1.0 / P.maxc);
            for (int r = 0; r < m; ++r) {
                const int k = S.rs_order[r];
                const int c = S.rs_acc[k];
                if (r >= AW_MAX_PLANS) {
                    __syncwarp();
                    if (lane == 0) {
                        rs_make_plan(c, S.rs_lens[c], P.maxc, stepn, S.plan_tmp);
                        rs_plan_world32(S.plan_tmp, q0, cq, sq, D.origin);
                    }
                    __syncwarp();
                }
                const RsPlan& plan = (r < AW_MAX_PLANS) ? S.plans[r] : S.plan_tmp;
                const int npts = plan.npts;
                if (lane == 0) S.n_ref += (unsigned long long)npts;
                int infeasible = 0;
                // Poses are visited with stride `passes` (lane*passes + pass): the first pass already spans the
                // whole word, so an infeasible word is almost always rejected after one 32-pose pass.
                const int passes = (npts + 31) >> 5;
                for (int pass = 0; pass < passes && !infeasible; ++pass) {
                    const int j = lane * passes + pass;
                    int st = HL_FREE;
                    unsigned amb = 0;
                    if (j < npts) {
                        float fx, fy, fc, fs;
                        rs_sample_world32(plan, j, inv_maxc, fx, fy, fc, fs);
                        if (fabsf(fx) > Ers.reach || fabsf(fy) > Ers.reach) st = far_status(FLAGS, Ers.n_seg);
                        else if (!(fx == fx) || !(fy == fy) || !(fc == fc)) { st = HL_AMBIG; amb = FLAGS; }
                        else st = filter_part(Ers, fx, fy, fc, fs, Ers.ext, FLAGS, &amb);
                    }
                    const unsigned livem = __ballot_sync(FULL, j < npts);
                    const unsigned hitm = __ballot_sync(FULL, st == HL_HIT);
                    const unsigned ambm = __ballot_sync(FULL, st == HL_AMBIG);
                    infeasible = hitm != 0;
                    if (!infeasible && ambm) {          // float64 sample + exact predicate, ambiguous poses only
                        int bad = 0;
                        if (st == HL_AMBIG) {
                            double lx, ly, lyaw, wx, wy, wyaw;
                            int cs, dir;
                            rs_sample_local(plan, j, P.maxc, lx, ly, lyaw, cs, dir);
                            rs_to_world(q0, cq, sq, lx, ly, lyaw, wx, wy, wyaw);
                            bad = pose_exact(eb, D, wx, wy, wyaw, amb) ? 1 : 0;
                        }
                        if (lane == 0) S.n_exact += (unsigned long long)__popc(ambm);
                        infeasible = __any_sync(FULL, bad);
                    }
                    if (lane == 0) S.n_checks += (unsigned long long)__popc(livem);
                }
                const bool short_enough = xdiv(S.rs_L[k], P.maxc) < P.min_len_goal;     // path.L < MIN_LENGTH_TO_GOAL
                if (!infeasible && short_enough) {
                    if (lane == 0) { S.rs_pick = r; S.arrival = 1; S.rs_word = c; S.goal_cost = S.rs_prio[k]; }
                    break;
                }
            }
            __syncwarp();
            TICK(PH_RS_SAMPLE);
            // ---- tolerance arrival (:464-495) overrides the shot; else the search length of this node (:368)
            if (lane == 0) {
                double xd = fabs(xsub(S.cx, S.goal[0])), yd = fabs(xsub(S.cy, S.goal[1]));
                double wd = fabs(angle_wrap(xsub(S.cyaw, S.goal[2])));
                if (xd < P.res && yd < P.res && wd < P.yaw_res) { S.arrival = 2; S.goal_cost = S.cg; S.rs_word = -1; }
                if (S.arrival) S.status = HL_STATUS_OK;
                else {
                    int seg = exact_search_segment(eb, D, S.cx, S.cy);
                    double len = seg < 0 ? D.default_len : eb.seg_len[D.seg_off + seg];
                    S.nsteps = (int)rint(xdiv(len, P.res));                    // Python round()
                    if (S.nsteps + 1 > HL_MAX_ROLLOUT || S.nsteps < 1) S.status = HL_STATUS_CAPACITY;
                }
            }
            if (lane < HL_MAX_PRIMS) S.phit[lane] = 0;
            __syncwarp();
            TICK(PH_ARRIVE);
        }
        __syncthreads();                                                    // alignment point 2
        if (live && S.status < 0) {
            // ---- primitive expansion (:558-596)
            const int n = S.nsteps, np1 = n + 1;
            const int total = P.n_prims * np1;
            // phase A: per (p, i) displacement terms  (res*cos(yaws[i]))*dir, i = 0..n
            for (int idx = lane; idx < total; idx += 32) {
                const int p = idx / np1, i = idx - p * np1;
                const double ys = P.yaw_step[p];
                const double init_yaw = angle_wrap(xadd(S.cyaw, ys));
                const double stop = xadd(init_yaw, xmul(ys, (double)(n + 1)));
                const double delta = xsub(stop, init_yaw);
                const double step = xdiv(delta, (double)(n + 1));
                const double yw = rollout_yaw(init_yaw, stop, step, delta, n + 1, i);
                S.tx[p][i] = xmul(xmul(P.res, m_cos(yw)), P.dir[p]);
                S.ty[p][i] = xmul(xmul(P.res, m_sin(yw)), P.dir[p]);
                S.pyaw[p][i] = rollout_yaw(init_yaw, stop, step, delta, n + 1, i + 1);
            }
            __syncwarp();
            // phase B: sequential cumsum per primitive (np.cumsum), then + init
            if (lane < P.n_prims) {
                double ax = 0.0, ay = 0.0;
                for (int i = 0; i < np1; ++i) {
                    ax = (i == 0) ? S.tx[lane][0] : xadd(ax, S.tx[lane][i]);
                    ay = (i == 0) ? S.ty[lane][0] : xadd(ay, S.ty[lane][i]);
                    S.tx[lane][i] = xadd(S.cx, ax);
                    S.ty[lane][i] = xadd(S.cy, ay);
                }
            }
            __syncwarp();
            TICK(PH_ROLLOUT);
            // phase C: float32 filter of every pose
            for (int idx = lane; idx < total; idx += 32) {
                const int p = idx / np1, j = idx - p * np1;
                unsigned amb = 0;
                int st = pose_filter(D, E, S.tx[p][j], S.ty[p][j], S.pyaw[p][j], FLAGS, &amb);
                S.pamb[p][j] = (st == HL_AMBIG) ? (unsigned char)amb : 0;
                if (st == HL_HIT) atomicOr(&S.phit[p], 1);
            }
            if (lane == 0) { S.n_checks += (unsigned long long)total; S.n_ref += (unsigned long long)total; }
            __syncwarp();
            TICK(PH_FILTER);
            // phase D: float64 escalation only where it can still change the answer
            for (int idx = lane; idx < total; idx += 32) {
                const int p = idx / np1, j = idx - p * np1;
                if (S.pamb[p][j] && !S.phit[p]) {
                    atomicAdd(&S.n_exact, 1ULL);
                    if (pose_exact(eb, D, S.tx[p][j], S.ty[p][j], S.pyaw[p][j], S.pamb[p][j])) atomicOr(&S.phit[p], 2);
                }
            }
            __syncwarp();
            TICK(PH_EXACT);
            // phase E: cost and key (lane per primitive), heuristic (whole warp per primitive)
            if (lane < HL_MAX_PRIMS) S.pneed[lane] = 1;
            __syncwarp();
            if (lane < P.n_prims && !S.phit[lane]) {
                const int p = lane;
                double len = 0.0;                                   // calculate_path_length (path_utils.py:5-12)
                for (int i = 0; i + 1 < np1; ++i) {
                    double ds = hypot_cr(xsub(S.tx[p][i + 1], S.tx[p][i]), xsub(S.ty[p][i + 1], S.ty[p][i]));
                    len = (i == 0) ? ds : xadd(len, ds);
                }
                double cost = xadd(S.cg, len);                       // simulated_path_cost (:306-329)
                if (P.dir[p] == -1.0) cost = xadd(cost, P.reverse_cost);
                cost = xadd(cost, xmul(P.steer[p], P.steer_cost));
                const double parent_steer = S.cprim < 0 ? 0.0 : P.steer_eff[S.cprim];
                cost = xadd(cost, xmul(fabs(xsub(P.steer[p], parent_steer)), P.delta_steer_cost));
                const double parent_dir = S.cprim < 0 ? 1.0 : P.dir[S.cprim];
                if (parent_dir != P.dir[p]) cost = xadd(cost, P.dir_change_cost);
                S.pg[p] = cost;
                int ix, iy, iw;
                long long key = 0;
                S.pkey_ok[p] = make_key(S.tx[p][n], S.ty[p][n], S.pyaw[p][n], P.res, P.yaw_res, ix, iy, iw, key) ? 1 : 0;
                S.pkey[p] = key;
                // look the key up now, all primitives in parallel (the table only changes in the merge below)
                int pos = -1;
                const int slot = S.pkey_ok[p] ? hash_find(W, hmask, key, &pos) : -1;
                S.pslot[p] = slot;
                S.ppos[p] = pos;
                // the heuristic is only needed if the merge will insert or improve this cell: a closed cell
                // stays closed and an open cell's g can only drop further during this merge
                if (slot >= 0 && (W.nstate[slot] == 1 || !(cost < W.ng[slot]))) S.pneed[p] = 0;
            }
            __syncwarp();
            for (int p = 0; p < P.n_prims; ++p) {
                if (!S.phit[p] && S.pneed[p]) {
                    double h = warp_state_cost(eb, D, S.tx[p][n], S.ty[p][n], S.pyaw[p][n], lane);
                    if (lane == 0) S.pprio[p] = xmul(P.hybrid_cost, h);
                }
            }
            __syncwarp();
            TICK(PH_COST_HEUR);
            // phase F: merge into the open list in primitive order (:580-596)
            if (lane == 0) {
                for (int p = 0; p < P.n_prims; ++p) {
                    if (S.phit[p]) continue;
                    if (!S.pkey_ok[p]) { S.status = HL_STATUS_CAPACITY; break; }
                    // the prefetched lookup is still valid unless this merge touched its probe position
                    int pos = S.ppos[p];
                    int slot = S.pslot[p];
                    if (slot < 0 ? (W.hkey[pos] != KEY_EMPTY) : false) slot = hash_find(W, hmask, S.pkey[p], &pos);
                    const double g = S.pg[p];
                    const double prio = (S.pprio[p] > g) ? S.pprio[p] : g;      // max(sim.cost, 50*h)
                    if (slot >= 0) {
                        if (W.nstate[slot] == 1) continue;                         // in closed_set
                        if (!(g < W.ng[slot])) continue;                           // not strictly better
                        if (!S.pneed[p]) { S.status = HL_STATUS_CAPACITY; break; } // cannot happen (see above)
                    } else {
                        if (S.n_nodes >= P.cap_nodes) { S.status = HL_STATUS_CAPACITY; break; }
                        slot = S.n_nodes++;
                        W.hkey[pos] = S.pkey[p]; W.hval[pos] = slot; W.nhpos[slot] = pos;
                        W.nkey[slot] = S.pkey[p]; W.nstate[slot] = 0; W.nheap[slot] = -1;
                    }
                    W.nx[slot] = S.tx[p][n]; W.ny[slot] = S.ty[p][n]; W.nyaw[slot] = S.pyaw[p][n];
                    W.ng[slot] = g; W.nparent[slot] = S.cur; W.nprim[slot] = (signed char)p;
                    W.nsteps[slot] = (signed char)n;
                    heap_set(W, S.heap_n, slot, prio);
                }
            }
            __syncwarp();
            TICK(PH_MERGE);
        }
        if (live && S.status >= 0) {
            finalize_scenario(S, W, P, O, lane);
            if (lane == 0) S.state = ST_IDLE;
            __syncwarp();
        }
    }
}

#include "hl_astar_spec.cuh"
#include "hl_astar_level.cuh"

// ------------------------------------------------------------------------------ host side
static void fill_params(const hl_ctx* ctx, const HlSearchParams* h, AsParams& P) {
    memset(&P, 0, sizeof(P));
    P.res = h->plan_resolution; P.yaw_res = h->yaw_resolution; P.maxc = h->maxc;
    P.max_steer = h->max_steer; P.wheel_base = h->wheel_base; P.n_prims = h->n_prims;
    for (int i = 0; i < HL_MAX_PRIMS; ++i) {
        P.steer[i] = h->prim_steer[i]; P.dir[i] = h->prim_dir[i]; P.yaw_step[i] = h->prim_yaw_step[i];
        P.curv[i] = h->prim_curv[i]; P.steer_eff[i] = h->prim_steer_eff[i];
    }
    P.steer_cost = h->steer_cost; P.delta_steer_cost = h->delta_steer_cost;
    P.dir_change_cost = h->direction_change_cost; P.reverse_cost = h->reverse_cost;
    P.hybrid_cost = h->hybrid_cost; P.min_len_goal = h->min_length_to_goal;
    P.max_nodes = h->max_nodes; P.max_path_poses = h->max_path_poses;
    P.cap_nodes = h->n_prims * (h->max_nodes + 1) + 2;
    int hs = 1024;
    while (hs < 2 * P.cap_nodes) hs <<= 1;
    P.hash_size = hs;
    P.pawn = h->motion_type == 1 ? 1 : 0;
    P.dub_cap = P.pawn ? (h->dubins_capacity > 0 ? h->dubins_capacity : 2048) : 0;
}


// ---- level-synchronous variant: per-context state (pools, the iteration graph, its two streams)
struct LsState {
    LsCall* d_call; LsCall* h_call;          // device block + pinned staging copy
    int* h_nact;                             // pinned read-back of the active count
    char* pool; size_t pool_bytes;
    cudaGraph_t graph; cudaGraphExec_t exec;
    cudaStream_t s1, s2;
    cudaEvent_t ev_fork, ev_join;
    int grid;
};

static void ls_state_free(void* p) {
    LsState* L = (LsState*)p;
    if (!L) return;
    if (L->exec) cudaGraphExecDestroy(L->exec);
    if (L->graph) cudaGraphDestroy(L->graph);
    if (L->ev_fork) cudaEventDestroy(L->ev_fork);
    if (L->ev_join) cudaEventDestroy(L->ev_join);
    if (L->s1) cudaStreamDestroy(L->s1);
    if (L->s2) cudaStreamDestroy(L->s2);
    if (L->pool) cudaFree(L->pool);
    if (L->d_call) cudaFree(L->d_call);
    if (L->h_call) cudaFreeHost(L->h_call);
    if (L->h_nact) cudaFreeHost(L->h_nact);
    delete L;
}

// Builds the state into a local object and publishes it in the context only after the graph was instantiated: a
// failure half-way (allocation, capture, instantiate) ends the capture, frees everything and leaves ctx->ls_state NULL,
// so the next call starts over instead of launching a half-built graph.
static int ls_state_build(hl_ctx* ctx, LsState* L, bool* capturing) {
    L->grid = ctx->sm_count * LS_GRID_MULT;
    HL_CUDA_OK(cudaMalloc(&L->d_call, sizeof(LsCall)));
    HL_CUDA_OK(cudaMallocHost(&L->h_call, sizeof(LsCall)));
    HL_CUDA_OK(cudaMallocHost(&L->h_nact, 64));
    HL_CUDA_OK(cudaStreamCreateWithFlags(&L->s1, cudaStreamNonBlocking));
    HL_CUDA_OK(cudaStreamCreateWithFlags(&L->s2, cudaStreamNonBlocking));
    HL_CUDA_OK(cudaEventCreateWithFlags(&L->ev_fork, cudaEventDisableTiming));
    HL_CUDA_OK(cudaEventCreateWithFlags(&L->ev_join, cudaEventDisableTiming));
    // LS_CHUNK iterations; the first one reads the list the initial step(0) filled (parity 1)
    const int g = L->grid;
    HL_CUDA_OK(cudaStreamBeginCapture(L->s1, cudaStreamCaptureModeThreadLocal));
    *capturing = true;
    for (int it = 0; it < LS_CHUNK; ++it) {
        const int parity = (it & 1) ^ 1;
        HL_CUDA_OK(cudaEventRecord(L->ev_fork, L->s1));
        HL_CUDA_OK(cudaStreamWaitEvent(L->s2, L->ev_fork, 0));
        ls_cand<<<g, LS_THREADS, 0, L->s1>>>(L->d_call, parity);
        ls_select<<<g, LS_THREADS, 0, L->s1>>>(L->d_call, parity);
        ls_sample<<<g, LS_THREADS, 0, L->s1>>>(L->d_call);
        ls_rollout<<<g, LS_THREADS, 0, L->s2>>>(L->d_call, parity);
        ls_filter<<<g, LS_THREADS, 0, L->s2>>>(L->d_call, parity);
        ls_cost<<<g, LS_THREADS, 0, L->s2>>>(L->d_call, parity);
        HL_CUDA_OK(cudaEventRecord(L->ev_join, L->s2));
        HL_CUDA_OK(cudaStreamWaitEvent(L->s1, L->ev_join, 0));
        ls_step<<<g, LS_THREADS, 0, L->s1>>>(L->d_call, parity);
    }
    *capturing = false;
    HL_CUDA_OK(cudaStreamEndCapture(L->s1, &L->graph));
    HL_CUDA_OK(cudaGraphInstantiate(&L->exec, L->graph, 0));
    return 0;
}

static int ls_state_get(hl_ctx* ctx, LsState** out) {
    if (ctx->ls_state) { *out = (LsState*)ctx->ls_state; return 0; }
    LsState* L = new LsState();
    memset(L, 0, sizeof(*L));
    bool capturing = false;
    if (ls_state_build(ctx, L, &capturing)) {
        if (capturing) {                               // leave s1 out of capture mode; the partial graph is dropped
            cudaGraph_t g = nullptr;
            cudaStreamEndCapture(L->s1, &g);
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
        }
        ls_state_free(L);
        return 1;
    }
    ctx->ls_state = L; ctx->ls_free = ls_state_free;
    *out = L;
    return 0;
}

static int ls_run(hl_ctx* ctx, const hl_env_batch* envs, const HlScenario* d_scen, int n_scen, const AsParams& P,
                  const AsOut& O, cudaStream_t st) {
    LsState* L = nullptr;
    if (ls_state_get(ctx, &L)) return 1;
    const size_t stride = as_ws_bytes(P.cap_nodes, P.hash_size, P.max_nodes, P.dub_cap);
    const int nb_max = n_scen < LS_MAX_BATCH ? n_scen : LS_MAX_BATCH;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t r = off; off += as_align(bytes); return r; };
    const size_t o_ws = take(stride * (size_t)nb_max);
    const size_t o_scn = take(sizeof(LsScn) * (size_t)nb_max);
    const size_t o_prim = take(sizeof(LsPrim) * (size_t)nb_max * P.n_prims);
    const size_t o_shot = take(sizeof(LsShot) * (size_t)nb_max);
    const size_t o_act0 = take(sizeof(int) * (size_t)nb_max);
    const size_t o_act1 = take(sizeof(int) * (size_t)nb_max);
    const size_t o_cnt = take(sizeof(int) * 8);
    const size_t o_words = take(sizeof(int2) * (size_t)nb_max * HL_RS_CANDIDATES);
    if (off > L->pool_bytes) {
        if (L->pool) cudaFree(L->pool);
        L->pool = nullptr; L->pool_bytes = 0;
        HL_CUDA_OK(cudaMalloc(&L->pool, off));
        L->pool_bytes = off;
    }
    const int max_iters = P.max_nodes + 3;
    for (int base = 0; base < n_scen; base += nb_max) {
        const int nb = (n_scen - base) < nb_max ? (n_scen - base) : nb_max;
        LsCall& H = *L->h_call;
        H.eb = envs->dev; H.scen = d_scen + base; H.n_scen = nb; H.P = P;
        H.ws = L->pool + o_ws; H.ws_stride = stride;
        H.scn = (LsScn*)(L->pool + o_scn); H.prim = (LsPrim*)(L->pool + o_prim); H.shot = (LsShot*)(L->pool + o_shot);
        H.act[0] = (int*)(L->pool + o_act0); H.act[1] = (int*)(L->pool + o_act1);
        H.n_act = (int*)(L->pool + o_cnt); H.n_words = H.n_act + 2;
        H.words = (int2*)(L->pool + o_words);
        H.O = O; H.O.results = O.results + base;
        HL_CUDA_OK(cudaMemcpyAsync(L->d_call, L->h_call, sizeof(LsCall), cudaMemcpyHostToDevice, st));
        HL_CUDA_OK(cudaMemsetAsync(H.n_act, 0, sizeof(int) * 8, st));
        ls_setup<<<L->grid, LS_THREADS, 0, st>>>(L->d_call);
        ls_step<<<L->grid, LS_THREADS, 0, st>>>(L->d_call, 0);
        if (getenv("HL_LS_TIMING")) {
            // debug: the same kernels one by one on the caller's stream with an event pair around each
            const char* names[7] = {"cand", "select", "sample", "rollout", "filter", "cost", "step"};
            double acc[7] = {0, 0, 0, 0, 0, 0, 0};
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            const int g = L->grid;
            int iters = 0;
            for (int it = 0; it < max_iters; ++it, ++iters) {
                const int parity = (it & 1) ^ 1;
                for (int k = 0; k < 7; ++k) {
                    cudaEventRecord(e0, st);
                    switch (k) {
                        case 0: ls_cand<<<g, LS_THREADS, 0, st>>>(L->d_call, parity); break;
                        case 1: ls_select<<<g, LS_THREADS, 0, st>>>(L->d_call, parity); break;
                        case 2: ls_sample<<<g, LS_THREADS, 0, st>>>(L->d_call); break;
                        case 3: ls_rollout<<<g, LS_THREADS, 0, st>>>(L->d_call, parity); break;
                        case 4: ls_filter<<<g, LS_THREADS, 0, st>>>(L->d_call, parity); break;
                        case 5: ls_cost<<<g, LS_THREADS, 0, st>>>(L->d_call, parity); break;
                        default: ls_step<<<g, LS_THREADS, 0, st>>>(L->d_call, parity); break;
                    }
                    cudaEventRecord(e1, st);
                    cudaEventSynchronize(e1);
                    float ms = 0.f;
                    cudaEventElapsedTime(&ms, e0, e1);
                    if (it >= 100) acc[k] += ms;
                }
                cudaMemcpyAsync(L->h_nact, H.n_act + (parity ^ 1), sizeof(int), cudaMemcpyDeviceToHost, st);
                cudaStreamSynchronize(st);
                if (*L->h_nact == 0) break;
            }
            fprintf(stderr, "[ls timing] %d iterations; mean us per kernel over iterations >= 100:", iters);
            for (int k = 0; k < 7; ++k) fprintf(stderr, " %s %.1f", names[k], iters > 100 ? 1000.0 * acc[k] / (iters - 100) : 0.0);
            fprintf(stderr, "\n");
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        } else
        for (int done = 0; done < max_iters; done += LS_CHUNK) {
            HL_CUDA_OK(cudaGraphLaunch(L->exec, st));
            HL_CUDA_OK(cudaMemcpyAsync(L->h_nact, H.n_act + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
            HL_CUDA_OK(cudaStreamSynchronize(st));             // also keeps h_call stable until it was consumed
            if (*L->h_nact == 0) break;
        }
        ls_finalize<<<L->grid, LS_THREADS, 0, st>>>(L->d_call);
        HL_CUDA_OK(cudaGetLastError());
        if (base + nb_max < n_scen) HL_CUDA_OK(cudaStreamSynchronize(st));   // the pinned call block is rewritten next
    }
    return 0;
}

static size_t astar_smem() { return sizeof(AwSmem) * AW_WARPS; }

extern "C" int hl_astar_phase_cycles(hl_ctx* ctx, uint64_t* h_out, int32_t n, int32_t reset) {
    if (!ctx || !h_out || n < 1 || n > AS_N_PHASES) { hl_set_error("hl_astar_phase_cycles: bad arguments"); return 1; }
    if (hl_enter(ctx, nullptr, nullptr, "hl_astar_phase_cycles")) return 1;
    HL_CUDA_OK(cudaMemcpy(h_out, ctx->d_counters + 16, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost));
    if (reset) HL_CUDA_OK(cudaMemset(ctx->d_counters + 16, 0, sizeof(uint64_t) * AS_N_PHASES));
    return 0;
}

extern "C" int64_t hl_hybrid_astar_workspace_bytes(const hl_ctx* ctx, const HlSearchParams* h) {
    if (!ctx || !h) return -1;
    AsParams P;
    fill_params(ctx, h, P);
    return (int64_t)as_ws_bytes(P.cap_nodes, P.hash_size, P.max_nodes, P.dub_cap);
}

extern "C" int hl_hybrid_astar_batch(hl_ctx* ctx, const hl_env_batch* envs, const HlScenario* d_scen,
                                     int32_t n_scen, const HlSearchParams* h_params,
                                     HlPlanResult* d_results, int32_t* d_expanded_keys, int64_t keys_capacity,
                                     unsigned long long* d_keys_cursor, double* d_path_x, double* d_path_y, double* d_path_yaw,
                                     double* d_path_k, int8_t* d_path_dir, int64_t path_capacity,
                                     unsigned long long* d_path_cursor, void* stream) {
    if (ctx && n_scen == 0 && d_path_cursor && d_keys_cursor) {          // empty batch: nothing but the cursors is touched
        if (hl_enter(ctx, envs, d_path_cursor, "hl_hybrid_astar_batch")) return 1;
        HL_CUDA_OK(cudaMemsetAsync(d_path_cursor, 0, sizeof(unsigned long long), (cudaStream_t)stream));
        HL_CUDA_OK(cudaMemsetAsync(d_keys_cursor, 0, sizeof(unsigned long long), (cudaStream_t)stream));
        return 0;
    }
    if (!ctx || !envs || !d_scen || !h_params || !d_results || !d_expanded_keys || !d_path_x || !d_path_y ||
        !d_path_yaw || !d_path_k || !d_path_dir || !d_path_cursor || !d_keys_cursor || n_scen < 0) {
        hl_set_error("hl_hybrid_astar_batch: bad arguments"); return 1;
    }
    if (h_params->n_prims < 1 || h_params->n_prims > HL_MAX_PRIMS || h_params->max_nodes < 0) {
        hl_set_error("hl_hybrid_astar_batch: n_prims/max_nodes out of range"); return 1;
    }
    if (h_params->motion_type != 0 && h_params->motion_type != 1) {
        hl_set_error("hl_hybrid_astar_batch: motion_type must be 0 (King) or 1 (Pawn)"); return 1;
    }
    if (hl_enter(ctx, envs, d_results, "hl_hybrid_astar_batch")) return 1;
    AsParams P;
    fill_params(ctx, h_params, P);
    // The node/hash workspace, the work-queue counter and the level variant's state are PER CONTEXT: the host part
    // runs under the context mutex and the launch waits for the previous search of this context (event recorded
    // below), so searches issued from several threads or streams of one device serialise instead of sharing scratch.
    std::lock_guard<std::recursive_mutex> lock(*(std::recursive_mutex*)ctx->ws_mu);
    // variant: "spec" = two warps per scenario with the analytic shot decoupled (hl_astar_spec.cuh),
    // "warp" = one warp per scenario, "level" = level-synchronous graph (hl_ctx_set_astar_variant / HL_ASTAR_VARIANT
    // at context creation; A/B runs only, the results are identical).
    // Pawn mode (Dubins goal extension) exists in the one-warp-per-scenario kernel only
    const bool level = !P.pawn && ctx->astar_variant == HL_ASTAR_LEVEL;
    const bool spec = !P.pawn && ctx->astar_variant != HL_ASTAR_WARP;
    cudaStream_t st = (cudaStream_t)stream;
    HL_CUDA_OK(cudaStreamWaitEvent(st, (cudaEvent_t)ctx->astar_done, 0));      // no-op until the first record
    AsOut O;
    O.results = d_results; O.expanded_keys = d_expanded_keys;
    O.keys_capacity = (long long)keys_capacity; O.keys_cursor = d_keys_cursor;
    O.path_x = d_path_x; O.path_y = d_path_y; O.path_yaw = d_path_yaw; O.path_k = d_path_k; O.path_dir = d_path_dir;
    O.path_capacity = (long long)path_capacity; O.path_cursor = d_path_cursor;
    O.phase_cycles = (unsigned long long*)(ctx->d_counters + 16);
    O.order = nullptr; O.order_count = nullptr; O.defer_list = nullptr; O.defer_count = nullptr; O.first_only = 0;
    if (level) {
        HL_CUDA_OK(cudaMemsetAsync(d_path_cursor, 0, sizeof(unsigned long long), st));
        HL_CUDA_OK(cudaMemsetAsync(d_keys_cursor, 0, sizeof(unsigned long long), st));
        const int rc = ls_run(ctx, envs, d_scen, n_scen, P, O, st);
        if (rc == 0) HL_CUDA_OK(cudaEventRecord((cudaEvent_t)ctx->astar_done, st));
        return rc;
    }
    const int slots = spec ? AQ_SLOTS : AW_WARPS;
    const int threads = spec ? AQ_SLOTS * AQ_WARPS_PER_SLOT * 32 : AW_WARPS * 32;
    const size_t smem = spec ? sizeof(AqSmem) * AQ_SLOTS : astar_smem();
    if ((int)smem > ctx->max_smem_optin) {
        hl_set_error("hl_hybrid_astar_batch: %zu B of shared memory per CTA exceed the device limit %d", smem, ctx->max_smem_optin);
        return 1;
    }
    int per_sm = 0;
    if (spec) {
        HL_CUDA_OK(cudaFuncSetAttribute(k_hybrid_astar_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HL_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_hybrid_astar_s, threads, smem));
    } else {
        HL_CUDA_OK(cudaFuncSetAttribute(k_hybrid_astar_w, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HL_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_hybrid_astar_w, threads, smem));
    }
    if (per_sm < 1) per_sm = 1;
    long long want = ((long long)n_scen + slots - 1) / slots;
    long long cap = (long long)ctx->sm_count * per_sm;
    const int grid = (int)(want < cap ? want : cap);
    const size_t stride = as_ws_bytes(P.cap_nodes, P.hash_size, P.max_nodes, P.dub_cap);
    const size_t need = stride * (size_t)grid * slots;
    if (need > ctx->astar_ws_bytes) {
        if (ctx->astar_ws) cudaFree(ctx->astar_ws);          // synchronises the device: the previous search is done
        ctx->astar_ws = nullptr; ctx->astar_ws_bytes = 0;
        HL_CUDA_OK(cudaMalloc(&ctx->astar_ws, need));
        ctx->astar_ws_bytes = need;
    }
    HL_CUDA_OK(cudaMemsetAsync(ctx->d_counters, 0, sizeof(unsigned int), st));
    HL_CUDA_OK(cudaMemsetAsync(d_path_cursor, 0, sizeof(unsigned long long), st));
    HL_CUDA_OK(cudaMemsetAsync(d_keys_cursor, 0, sizeof(unsigned long long), st));
    // Two-phase sweep: when the batch is several times larger than the resident scenario slots, a first launch runs
    // only the FIRST analytic shot of every scenario (most headland scenarios end there: 72 % of config 5) and lists
    // the rest; the second launch searches the listed ones, which then all start at once instead of waiting in the
    // work queue behind trivial scenarios (the sweep's tail is the start time of its longest searches).  Results are
    // identical: the second launch redoes a listed scenario from its first pop.
    if (spec && (long long)n_scen > 2LL * grid * slots) {
        if ((size_t)n_scen > ctx->astar_defer_cap) {
            if (ctx->astar_defer) cudaFree(ctx->astar_defer);
            ctx->astar_defer = nullptr; ctx->astar_defer_cap = 0;
            HL_CUDA_OK(cudaMalloc(&ctx->astar_defer, sizeof(int) * (size_t)n_scen));
            ctx->astar_defer_cap = (size_t)n_scen;
        }
        int* defer_count = (int*)(ctx->d_counters + 4);
        HL_CUDA_OK(cudaMemsetAsync(ctx->d_counters + 4, 0, sizeof(unsigned int), st));
        HL_CUDA_OK(cudaMemsetAsync(ctx->d_counters + 8, 0, sizeof(unsigned int), st));
        AsOut O1 = O;
        O1.first_only = 1; O1.defer_list = ctx->astar_defer; O1.defer_count = defer_count;
        k_hybrid_astar_s<<<grid, threads, smem, st>>>(envs->dev, d_scen, n_scen, P, (char*)ctx->astar_ws, stride,
                                                      ctx->d_counters, O1);
        HL_CUDA_OK(cudaGetLastError());
        AsOut O2 = O;
        O2.order = ctx->astar_defer; O2.order_count = defer_count;
        k_hybrid_astar_s<<<grid, threads, smem, st>>>(envs->dev, d_scen, n_scen, P, (char*)ctx->astar_ws, stride,
                                                      ctx->d_counters + 8, O2);
    } else if (spec)
        k_hybrid_astar_s<<<grid, threads, smem, st>>>(envs->dev, d_scen, n_scen, P, (char*)ctx->astar_ws, stride,
                                                      ctx->d_counters, O);
    else
        k_hybrid_astar_w<<<grid, threads, smem, st>>>(envs->dev, d_scen, n_scen, P, (char*)ctx->astar_ws, stride,
                                                      ctx->d_counters, O);
    HL_CUDA_OK(cudaGetLastError());
    HL_CUDA_OK(cudaEventRecord((cudaEvent_t)ctx->astar_done, st));
    return 0;
}
