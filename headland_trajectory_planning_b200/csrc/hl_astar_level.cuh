// hl_astar_level.cuh -- K4 variant D: level-synchronous batch search.
//
// The scenario-per-warp kernels (hl_astar.cu, hl_astar_spec.cuh) are bound by the LATENCY of one hard scenario:
// 401 pops x ~58 us even alone on the GPU (profiles/r1d), because one warp walks a 250 KB instruction stream
// (32 KB instruction cache) with 168 registers and 12 warps per SM.  Here the whole sweep advances one pop per
// iteration and every phase of the reference's loop body (hybrid_a_star_search.py:542-596) is its own small
// kernel over ALL active scenarios:
//
//      step(k)  ->  { cand -> select -> sample }      analytic shot   (:232-287)
//               \-> { rollout -> filter -> cost }     expansion       (:357-427, :306-329, heuristic)
//      step(k+1) = resolve the shot, merge the children (:580-596), pop the next node (:526-560)
//
// The two branches are independent (a failed shot has no side effect) and run on two captured streams; an
// iteration is 4 kernels deep.  The iterations are recorded ONCE per context as a CUDA graph (all per-call
// values live in a device-side LsCall block, so the graph never changes) and replayed in chunks; the host
// reads the number of active scenarios between chunks.  Each kernel has its own register budget and fits the
// instruction cache; items are (scenario, candidate), (scenario, word), (scenario, primitive, pose) ... so the
// lanes are busy even when only a few hundred long scenarios are left.
//
// Results are bit-identical to the other variants: same float64 operation order per item, same heapdict
// replay, same float32 filter + float64 escalation.
#pragma once
#include "hl_astar_common.cuh"

#define LS_ROLL_STRIDE (AS_ROLL + 1)        // yaws[0 .. n+1] of one primitive
#define LS_MAX_BATCH 8192                   // scenarios per pass (bounds the workspace: ~260 KB each)
#define LS_CHUNK 32                         // iterations per graph launch (even)
#define LS_GRID_MULT 4                      // CTAs per SM of the phase kernels (grid-stride loops)
#define LS_THREADS 256

struct LsScn {                              // one per scenario
    double start[3], goal[3];
    long long start_key, goal_key;
    int env, status, arrival, has_cur;
    int n_nodes, heap_n, counter, n_closed;
    int cur, cprim, nsteps, rs_n;
    double cx, cy, cyaw, cg;
    double goal_cost;
    int rs_pick, rs_word, rs_bad, pad0;
    RsProblem rs_prob;
    unsigned long long checks, exact, ref;
};

struct LsPrim {                             // one per (scenario, primitive)
    double dtx[AS_ROLL], dty[AS_ROLL];      // per-step translation (rollout), summed by the filter
    double tx[AS_ROLL], ty[AS_ROLL], pyaw[AS_ROLL];
    double pg, pprio;
    long long pkey;
    int phit, pkey_ok, pslot, ppos, pneed, pad0;
    unsigned char pamb[AS_ROLL + 7];
};

struct LsShot {                             // one per scenario
    double rs_lens[HL_RS_CANDIDATES][HL_RS_MAX_SEGS];
    double rs_L[HL_RS_CANDIDATES], rs_prio[HL_RS_CANDIDATES], rs_Lc[HL_RS_CANDIDATES];
    int rs_acc[HL_RS_CANDIDATES], rs_order[HL_RS_CANDIDATES];
    unsigned char rs_valid[HL_RS_CANDIDATES + 2], rs_accept[HL_RS_CANDIDATES + 2], word_bad[HL_RS_CANDIDATES + 2];
    int word_npts[HL_RS_CANDIDATES + 2];
};

struct LsCall {                             // per-call block in device memory, read by every kernel
    EnvBatchDev eb;
    const HlScenario* scen;
    int n_scen;
    AsParams P;
    char* ws; size_t ws_stride;
    LsScn* scn; LsPrim* prim; LsShot* shot;
    int* act[2];                            // active scenario lists (double buffered by iteration parity)
    int* n_act;                             // [2]
    int2* words;                            // (scenario, rank) of every word to sample this iteration
    int* n_words;
    AsOut O;
};

#define LS_FLAGS (HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY | HL_CHECK_LANE)

__device__ __forceinline__ AsWs ls_ws(const LsCall& C, int sc) {
    return as_carve(C.ws + (size_t)sc * C.ws_stride, C.P.cap_nodes, C.P.hash_size, C.P.max_nodes);
}

// ------------------------------------------------------------------------------------------------ setup
// Start / goal feasibility (:76-80, :516-519), start node and its priority (:500-510).  Warp per scenario.
__global__ void __launch_bounds__(LS_THREADS) ls_setup(const LsCall* __restrict__ Cp) {
    const LsCall& C = *Cp;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const AsParams& P = C.P;
    for (int sc = warp; sc < C.n_scen; sc += n_warps) {
        LsScn& S = C.scn[sc];
        const AsWs W = ls_ws(C, sc);
        for (int i = lane; i < P.hash_size; i += 32) W.hkey[i] = KEY_EMPTY;
        const HlScenario& s = C.scen[sc];
        if (lane == 0) {
            S.env = s.env_id;
            for (int k = 0; k < 3; ++k) { S.start[k] = s.start[k]; S.goal[k] = s.goal[k]; }
            S.n_nodes = 0; S.heap_n = 0; S.counter = 0; S.n_closed = 0;
            S.status = -1; S.arrival = 0; S.has_cur = 0; S.goal_cost = 0.0;
            S.cur = 0; S.cprim = -1; S.nsteps = 0; S.rs_n = 0; S.rs_pick = -1; S.rs_word = -1; S.rs_bad = 0;
            S.cx = S.cy = S.cyaw = S.cg = 0.0;
            S.checks = 0; S.exact = 0; S.ref = 0;
        }
        __syncwarp();
        const EnvDesc& D = C.eb.desc[s.env_id];
        EnvSmem E;
        global_env(C.eb, D, E);
        const AsStart st = start_node(W, P, C.eb, D, E, s.start, s.goal, LS_FLAGS, lane);
        if (lane == 0) {
            S.start_key = st.start_key; S.goal_key = st.goal_key; S.status = st.status;
            if (st.status < 0) {
                S.n_nodes = 1;
                int hn = 0;
                heap_set(W, hn, 0, st.prio);
                S.heap_n = hn;
                C.act[0][atomicAdd(&C.n_act[0], 1)] = sc;
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------- step
// Warp per active scenario: resolve the shot of the current node, merge its children, pop the next node.
__global__ void __launch_bounds__(LS_THREADS) ls_step(const LsCall* __restrict__ Cp, int parity) {
    const LsCall& C = *Cp;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const AsParams& P = C.P;
    const int hmask = P.hash_size - 1;
    const int n_act = C.n_act[parity];
    if (blockIdx.x == 0 && threadIdx.x == 0) *C.n_words = 0;
    const int* act = C.act[parity];
    for (int a = warp; a < n_act; a += n_warps) {
        const int sc = act[a];
        LsScn& S = C.scn[sc];
        const AsWs W = ls_ws(C, sc);
        int status = S.status;
        if (S.has_cur) {
            const LsShot& T = C.shot[sc];
            // ---- the analytic shot of the current node: first free word in heapdict order (:273-285)
            const int m = S.rs_n;
            int first = -1;
            for (int r0 = 0; r0 < m && first < 0; r0 += 32) {
                const int r = r0 + lane;
                const unsigned free_m = __ballot_sync(FULL, r < m && T.word_bad[r] == 0);
                if (free_m) first = r0 + __ffs(free_m) - 1;
            }
            if (lane == 0) {
                const int tried = first >= 0 ? first + 1 : m;
                unsigned long long ref = 0;
                for (int r = 0; r < tried; ++r) ref += (unsigned long long)T.word_npts[r];
                S.ref += ref;
                if (S.rs_bad) { status = HL_STATUS_RS_ASSERT; S.arrival = 0; }      // the reference would raise here
                else if (first >= 0) {
                    const int k = T.rs_order[first];
                    S.rs_pick = first; S.rs_word = T.rs_acc[k]; S.goal_cost = T.rs_prio[k];
                    S.arrival = 1; status = HL_STATUS_OK;
                } else {
                    // ---- merge the children (:580-596), in primitive order
                    const int n = S.nsteps;
                    S.ref += (unsigned long long)(P.n_prims * (n + 1));
                    int n_nodes = S.n_nodes, heap_n = S.heap_n;
                    for (int p = 0; p < P.n_prims; ++p) {
                        const LsPrim& R = C.prim[(size_t)sc * P.n_prims + p];
                        if (R.phit) continue;
                        if (!R.pkey_ok) { status = HL_STATUS_CAPACITY; break; }
                        int pos = R.ppos;
                        int slot2 = R.pslot;
                        if (slot2 < 0 ? (W.hkey[pos] != KEY_EMPTY) : false) slot2 = hash_find(W, hmask, R.pkey, &pos);
                        const double g = R.pg;
                        const double prio = (R.pprio > g) ? R.pprio : g;
                        if (slot2 >= 0) {
                            if (W.nstate[slot2] == 1) continue;
                            if (!(g < W.ng[slot2])) continue;
                            if (!R.pneed) { status = HL_STATUS_CAPACITY; break; }
                        } else {
                            if (n_nodes >= P.cap_nodes) { status = HL_STATUS_CAPACITY; break; }
                            slot2 = n_nodes++;
                            W.hkey[pos] = R.pkey; W.hval[pos] = slot2; W.nhpos[slot2] = pos;
                            W.nkey[slot2] = R.pkey; W.nstate[slot2] = 0; W.nheap[slot2] = -1;
                        }
                        W.nx[slot2] = R.tx[n]; W.ny[slot2] = R.ty[n]; W.nyaw[slot2] = R.pyaw[n];
                        W.ng[slot2] = g; W.nparent[slot2] = S.cur; W.nprim[slot2] = (signed char)p;
                        W.nsteps[slot2] = (signed char)n;
                        heap_set(W, heap_n, slot2, prio);
                    }
                    S.n_nodes = n_nodes; S.heap_n = heap_n;
                }
                S.has_cur = 0;
            }
        }
        if (lane == 0 && status < 0) {
            // ---- next pop (:526-560)
            if (S.counter > P.max_nodes) status = HL_STATUS_MAX_NODES;
            else {
                S.counter += 1;
                int heap_n = S.heap_n;
                if (heap_n == 0) status = HL_STATUS_OPEN_EMPTY;
                else {
                    const int cur = heap_popitem(W, heap_n);
                    S.heap_n = heap_n;
                    W.nstate[cur] = 1;
                    W.corder[S.n_closed] = cur;
                    S.n_closed += 1;
                    const double cx = W.nx[cur], cy = W.ny[cur], cyaw = W.nyaw[cur];
                    S.cur = cur; S.cx = cx; S.cy = cy; S.cyaw = cyaw; S.cg = W.ng[cur];
                    S.cprim = W.nprim[cur];
                    // tolerance arrival (:464-495)
                    const double xd = fabs(xsub(cx, S.goal[0])), yd = fabs(xsub(cy, S.goal[1]));
                    const double wd = fabs(angle_wrap(xsub(cyaw, S.goal[2])));
                    if (xd < P.res && yd < P.res && wd < P.yaw_res) {
                        S.arrival = 2; S.goal_cost = S.cg; status = HL_STATUS_OK;
                    } else {
                        const EnvDesc& D = C.eb.desc[S.env];
                        const int seg = exact_search_segment(C.eb, D, cx, cy);
                        const double len = seg < 0 ? D.default_len : C.eb.seg_len[D.seg_off + seg];
                        const int nsteps = (int)rint(xdiv(len, P.res));
                        S.nsteps = nsteps;
                        if (nsteps + 1 > HL_MAX_ROLLOUT || nsteps < 1) status = HL_STATUS_CAPACITY;
                        else {
                            const double q0[3] = {cx, cy, cyaw};
                            S.rs_prob = rs_normalise(q0, S.goal, P.maxc);
                            S.has_cur = 1;
                        }
                    }
                }
            }
        }
        if (lane == 0) {
            S.status = status;
            if (status < 0) C.act[parity ^ 1][atomicAdd(&C.n_act[parity ^ 1], 1)] = sc;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------- shot: cand
// Thread per (active scenario, candidate row): the 46 word solvers (reeds_shepp.py, table in hl_rs.cuh).
__global__ void __launch_bounds__(LS_THREADS) ls_cand(const LsCall* __restrict__ Cp, int parity) {
    const LsCall& C = *Cp;
    const int n_items = C.n_act[parity] * HL_RS_CANDIDATES;
    const int* act = C.act[parity];
    for (int it = blockIdx.x * blockDim.x + threadIdx.x; it < n_items; it += gridDim.x * blockDim.x) {
        const int a = it / HL_RS_CANDIDATES, c = it - a * HL_RS_CANDIDATES;
        const int sc = act[a];
        const RsProblem prob = C.scn[sc].rs_prob;
        LsShot& T = C.shot[sc];
        double l[HL_RS_MAX_SEGS] = {0, 0, 0, 0, 0};
        const bool ok = rs_candidate(c, prob, l);
        T.rs_valid[c] = ok ? 1 : 0;
        for (int k = 0; k < HL_RS_MAX_SEGS; ++k) T.rs_lens[c][k] = l[k];
    }
}

// ----------------------------------------------------------------------------------------- shot: select
// Warp per active scenario: set_path dedup by word group, costs, heapdict order; emits the word work list.
__global__ void __launch_bounds__(LS_THREADS) ls_select(const LsCall* __restrict__ Cp, int parity) {
    const LsCall& C = *Cp;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const AsParams& P = C.P;
    const int n_act = C.n_act[parity];
    const int* act = C.act[parity];
    for (int a = warp; a < n_act; a += n_warps) {
        const int sc = act[a];
        LsScn& S = C.scn[sc];
        LsShot& T = C.shot[sc];
        if (lane < RS_N_GROUPS) rs_select_group(lane, T.rs_valid, T.rs_lens, T.rs_accept, T.rs_Lc);
        __syncwarp();
        const int a0 = T.rs_accept[lane];
        const int a1 = (lane + 32 < HL_RS_CANDIDATES) ? T.rs_accept[lane + 32] : 0;
        const unsigned b0 = __ballot_sync(FULL, a0 == 1), b1 = __ballot_sync(FULL, a1 == 1);
        const unsigned bad = __ballot_sync(FULL, a0 == 2 || a1 == 2);
        const unsigned lt = (1u << lane) - 1u;
        const int n0 = __popc(b0);
        if (a0 == 1) { int k = __popc(b0 & lt); T.rs_acc[k] = lane; T.rs_L[k] = T.rs_Lc[lane]; }
        if (a1 == 1) { int k = n0 + __popc(b1 & lt); T.rs_acc[k] = lane + 32; T.rs_L[k] = T.rs_Lc[lane + 32]; }
        const int m = bad ? 0 : n0 + __popc(b1);
        __syncwarp();
        const double sg = S.cg;
        for (int k = lane; k < m; k += 32)
            T.rs_prio[k] = rs_path_cost(sg, T.rs_acc[k], T.rs_lens[T.rs_acc[k]], P.max_steer, P.reverse_cost,
                                        P.dir_change_cost, P.steer_cost);
        __syncwarp();
        int base = 0;
        if (lane == 0) {
            S.rs_n = m; S.rs_bad = bad ? 1 : 0;
            if (m > 0) {
                double prio[HL_RS_CANDIDATES];
                int order[HL_RS_CANDIDATES];
                for (int k = 0; k < m; ++k) prio[k] = T.rs_prio[k];
                heapdict_order(prio, m, order);
                for (int k = 0; k < m; ++k) T.rs_order[k] = order[k];
                base = atomicAdd(C.n_words, m);
            }
        }
        base = __shfl_sync(FULL, base, 0);
        for (int r = lane; r < m; r += 32) { C.words[base + r] = make_int2(sc, r); T.word_bad[r] = 1; }
        __syncwarp();
    }
}

// ----------------------------------------------------------------------------------------- shot: sample
// Warp per (scenario, word): sample the word (generate_local_course, :471-562) and collision-check its poses.
__global__ void __launch_bounds__(LS_THREADS) ls_sample(const LsCall* __restrict__ Cp) {
    __shared__ RsPlan s_plan[LS_THREADS / 32];
    const LsCall& C = *Cp;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const AsParams& P = C.P;
    const int n_words = *C.n_words;
    const float inv_maxc = (float)(1.0 / P.maxc);
    const double stepn = xmul(P.res, P.maxc);
    RsPlan& plan = s_plan[wib];
    for (int w = warp; w < n_words; w += n_warps) {
        const int2 item = C.words[w];
        const int sc = item.x, r = item.y;
        LsScn& S = C.scn[sc];
        LsShot& T = C.shot[sc];
        const EnvDesc& D = C.eb.desc[S.env];
        EnvSmem E;
        global_env(C.eb, D, E);
        E.eps += 6e-5f;                                   // float32 sampling error of rs_sample_world32
        const int k = T.rs_order[r];
        const int c = T.rs_acc[k];
        const double q0[3] = {S.cx, S.cy, S.cyaw};
        const double cq = m_cos(-q0[2]), sq = m_sin(-q0[2]);
        __syncwarp();
        if (lane == 0) {
            rs_make_plan(c, T.rs_lens[c], P.maxc, stepn, plan);
            rs_plan_world32(plan, q0, cq, sq, D.origin);
        }
        __syncwarp();
        const int npts = plan.npts;
        int infeasible = 0;
        const int passes = (npts + 31) >> 5;
        unsigned long long checks = 0, exact = 0;
        for (int pass = 0; pass < passes && !infeasible; ++pass) {
            const int j = lane * passes + pass;
            int st2 = HL_FREE;
            unsigned amb = 0;
            if (j < npts) {
                float fx, fy, fc, fs;
                rs_sample_world32(plan, j, inv_maxc, fx, fy, fc, fs);
                if (fabsf(fx) > E.reach || fabsf(fy) > E.reach) st2 = far_status(LS_FLAGS, E.n_seg);
                else if (!(fx == fx) || !(fy == fy) || !(fc == fc)) { st2 = HL_AMBIG; amb = LS_FLAGS; }
                else st2 = filter_part(E, fx, fy, fc, fs, E.ext, LS_FLAGS, &amb);
            }
            const unsigned livem = __ballot_sync(FULL, j < npts);
            const unsigned hitm = __ballot_sync(FULL, st2 == HL_HIT);
            const unsigned ambm = __ballot_sync(FULL, st2 == HL_AMBIG);
            infeasible = hitm != 0;
            if (!infeasible && ambm) {
                int bad2 = 0;
                if (st2 == HL_AMBIG) {
                    double lx, ly, lyaw, wx, wy, wyaw;
                    int cs, dir;
                    rs_sample_local(plan, j, P.maxc, lx, ly, lyaw, cs, dir);
                    rs_to_world(q0, cq, sq, lx, ly, lyaw, wx, wy, wyaw);
                    bad2 = pose_exact(C.eb, D, wx, wy, wyaw, amb) ? 1 : 0;
                }
                exact += (unsigned long long)__popc(ambm);
                infeasible = __any_sync(FULL, bad2);
            }
            checks += (unsigned long long)__popc(livem);
        }
        if (lane == 0) {
            T.word_npts[r] = npts;
            T.word_bad[r] = infeasible ? 1 : 0;
            atomicAdd(&S.checks, checks);
            if (exact) atomicAdd(&S.exact, exact);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------- expand: rollout
// Thread per (scenario, primitive, yaw index): kinematic_simulation_node (:357-410) yaws and step vectors.
__global__ void __launch_bounds__(LS_THREADS) ls_rollout(const LsCall* __restrict__ Cp, int parity) {
    const LsCall& C = *Cp;
    const AsParams& P = C.P;
    const int per_scn = P.n_prims * LS_ROLL_STRIDE;
    const int n_items = C.n_act[parity] * per_scn;
    const int* act = C.act[parity];
    if (blockIdx.x == 0 && threadIdx.x == 0) C.n_act[parity ^ 1] = 0;      // the list the next step() fills
    for (int it = blockIdx.x * blockDim.x + threadIdx.x; it < n_items; it += gridDim.x * blockDim.x) {
        const int a = it / per_scn, rem = it - a * per_scn;
        const int p = rem / LS_ROLL_STRIDE, i = rem - p * LS_ROLL_STRIDE;
        const int sc = act[a];
        const LsScn& S = C.scn[sc];
        const int n = S.nsteps, np1 = n + 1;
        if (i > np1) continue;
        LsPrim& R = C.prim[(size_t)sc * P.n_prims + p];
        const double ys = P.yaw_step[p];
        const double init_yaw = angle_wrap(xadd(S.cyaw, ys));
        const double stop = xadd(init_yaw, xmul(ys, (double)(n + 1)));
        const double delta = xsub(stop, init_yaw);
        const double step = xdiv(delta, (double)(n + 1));
        const double yw = rollout_yaw(init_yaw, stop, step, delta, n + 1, i);
        if (i >= 1) R.pyaw[i - 1] = yw;
        if (i <= n) {
            double sn, cs;
            m_sincos(yw, &sn, &cs);
            R.dtx[i] = xmul(xmul(P.res, cs), P.dir[p]);
            R.dty[i] = xmul(xmul(P.res, sn), P.dir[p]);
        }
        if (i == 0) { R.phit = 0; R.pneed = 1; }
    }
}

// -------------------------------------------------------------------------------------- expand: filter
// Thread per (scenario, primitive, pose): np.cumsum of the step vectors in sequence, float32 footprint filter.
__global__ void __launch_bounds__(LS_THREADS) ls_filter(const LsCall* __restrict__ Cp, int parity) {
    const LsCall& C = *Cp;
    const AsParams& P = C.P;
    const int per_scn = P.n_prims * AS_ROLL;
    const int n_items = C.n_act[parity] * per_scn;
    const int* act = C.act[parity];
    for (int it = blockIdx.x * blockDim.x + threadIdx.x; it < n_items; it += gridDim.x * blockDim.x) {
        const int a = it / per_scn, rem = it - a * per_scn;
        const int p = rem / AS_ROLL, j = rem - p * AS_ROLL;
        const int sc = act[a];
        LsScn& S = C.scn[sc];
        const int np1 = S.nsteps + 1;
        if (j >= np1) continue;
        LsPrim& R = C.prim[(size_t)sc * P.n_prims + p];
        double ax = R.dtx[0], ay = R.dty[0];
        for (int i = 1; i <= j; ++i) { ax = xadd(ax, R.dtx[i]); ay = xadd(ay, R.dty[i]); }
        const double x = xadd(S.cx, ax), y = xadd(S.cy, ay);
        R.tx[j] = x; R.ty[j] = y;
        const EnvDesc& D = C.eb.desc[S.env];
        EnvSmem E;
        global_env(C.eb, D, E);
        unsigned amb = 0;
        const int st = pose_filter(D, E, x, y, R.pyaw[j], LS_FLAGS, &amb);
        R.pamb[j] = (st == HL_AMBIG) ? (unsigned char)amb : 0;
        if (st == HL_HIT) atomicOr(&R.phit, 1);
        if (j == 0 && p == 0) atomicAdd(&S.checks, (unsigned long long)(P.n_prims * np1));
    }
}

// ---------------------------------------------------------------------------------------- expand: cost
// Warp per (scenario, primitive): float64 escalation of the ambiguous poses, g-cost (:306-329), grid key and
// closed/open lookup, guide-line heuristic (reference_line_heuristic.py:131-158) of the end pose.
__global__ void __launch_bounds__(LS_THREADS) ls_cost(const LsCall* __restrict__ Cp, int parity) {
    const LsCall& C = *Cp;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const AsParams& P = C.P;
    const int hmask = P.hash_size - 1;
    const int n_items = C.n_act[parity] * P.n_prims;
    const int* act = C.act[parity];
    for (int it = warp; it < n_items; it += n_warps) {
        const int a = it / P.n_prims, p = it - a * P.n_prims;
        const int sc = act[a];
        LsScn& S = C.scn[sc];
        LsPrim& R = C.prim[(size_t)sc * P.n_prims + p];
        const EnvDesc& D = C.eb.desc[S.env];
        const int n = S.nsteps, np1 = n + 1;
        int hit = R.phit;
        if (!hit) {
            int bad = 0;
            const int am = lane < np1 ? R.pamb[lane] : 0;
            if (am) bad = pose_exact(C.eb, D, R.tx[lane], R.ty[lane], R.pyaw[lane], am) ? 1 : 0;
            const unsigned ambm = __ballot_sync(FULL, am != 0);
            if (ambm && lane == 0) atomicAdd(&S.exact, (unsigned long long)__popc(ambm));
            if (__any_sync(FULL, bad)) hit = 2;
        }
        if (hit) { if (lane == 0) R.phit = hit; __syncwarp(); continue; }
        double ds = 0.0;
        if (lane < n) ds = hypot_cr(xsub(R.tx[lane + 1], R.tx[lane]), xsub(R.ty[lane + 1], R.ty[lane]));
        double len = __shfl_sync(FULL, ds, 0);
        for (int i = 1; i < n; ++i) len = xadd(len, __shfl_sync(FULL, ds, i));
        if (n < 1) len = 0.0;
        int need = 1, key_ok = 0;
        if (lane == 0) {
            const AsWs W = ls_ws(C, sc);
            double cost = xadd(S.cg, len);
            if (P.dir[p] == -1.0) cost = xadd(cost, P.reverse_cost);
            cost = xadd(cost, xmul(P.steer[p], P.steer_cost));
            const int cprim = S.cprim;
            const double parent_steer = cprim < 0 ? 0.0 : P.steer_eff[cprim];
            cost = xadd(cost, xmul(fabs(xsub(P.steer[p], parent_steer)), P.delta_steer_cost));
            const double parent_dir = cprim < 0 ? 1.0 : P.dir[cprim];
            if (parent_dir != P.dir[p]) cost = xadd(cost, P.dir_change_cost);
            R.pg = cost;
            int ix, iy, iw;
            long long key = 0;
            key_ok = make_key(R.tx[n], R.ty[n], R.pyaw[n], P.res, P.yaw_res, ix, iy, iw, key) ? 1 : 0;
            R.pkey_ok = key_ok;
            R.pkey = key;
            int pos = -1;
            const int slot2 = key_ok ? hash_find(W, hmask, key, &pos) : -1;
            R.pslot = slot2;
            R.ppos = pos;
            if (slot2 >= 0 && (W.nstate[slot2] == 1 || !(cost < W.ng[slot2]))) need = 0;
            R.pneed = need;
            R.phit = 0;
        }
        need = __shfl_sync(FULL, need, 0);
        key_ok = __shfl_sync(FULL, key_ok, 0);
        if (need && key_ok) {
            const double h = warp_state_cost(C.eb, D, R.tx[n], R.ty[n], R.pyaw[n], lane);
            if (lane == 0) R.pprio = xmul(P.hybrid_cost, h);
        }
        __syncwarp();
    }
}

// --------------------------------------------------------------------------------------------- finalize
// Warp per scenario: expanded keys, path (get_path_from_expanded_nodes, :429-454), result record.
__global__ void __launch_bounds__(LS_THREADS) ls_finalize(const LsCall* __restrict__ Cp) {
    __shared__ RsPlan s_plan[LS_THREADS / 32];
    const LsCall& C = *Cp;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const AsParams& P = C.P;
    RsPlan& plan = s_plan[wib];
    for (int sc = warp; sc < C.n_scen; sc += n_warps) {
        const LsScn& S = C.scn[sc];
        const AsWs W = ls_ws(C, sc);
        const int status = S.status < 0 ? HL_STATUS_CAPACITY : S.status;   // iteration budget exhausted (cannot happen)
        if (lane == 0 && S.arrival == 1)                                   // the goal extension: the winning word
            rs_make_plan(S.rs_word, C.shot[sc].rs_lens[S.rs_word], P.maxc, xmul(P.res, P.maxc), plan);
        __syncwarp();
        const int end = (S.n_closed > 0) ? W.corder[S.n_closed - 1] : 0;   // the node the search ended on
        const AsWritten w = write_outputs(W, P, C.O, status, S.n_closed, end, S.arrival, S.start_key, S.goal_key, &plan,
                                          0, lane);
        if (lane == 0)
            write_record(C.O, sc, w, S.arrival, S.rs_word, S.goal_cost, S.counter, S.checks, S.exact, S.ref, 0);
        __syncwarp();
    }
}
