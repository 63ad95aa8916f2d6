// hl_astar_spec.cuh -- K4 (default): an expander team and a shooter warp per scenario, speculative decoupling of
// the analytic shot.
//
// In the reference every popped node first gets a Reeds-Shepp shot and is expanded only if the shot fails
// (hybrid_a_star_search.py:542-596).  A FAILED shot has no side effect, and a successful one ends the search
// with a result that depends only on nodes closed up to that pop (closed nodes are immutable).  So the two
// halves of an expansion can run concurrently and even out of step:
//   * the EXPANDER warp pops, tests the tolerance arrival, rolls out / checks / costs / merges the
//     primitives and keeps going, assuming shots fail (true for 400 of 401 pops of a hard scenario);
//   * the SHOOTER warp walks the closed list in pop order and evaluates the shot of each node;
//   * if the shooter finds a free word at pop i the search ends THERE: the record is truncated to the first
//     i+1 closed nodes, exactly what the reference returns; the expander's extra work is discarded.
// The critical path per pop becomes max(shot, expansion) instead of their sum.
// The expander is a TEAM of AQ_EXPANDERS warps (warp 0 owns the open list; the helper shares rollout, filter,
// escalation and heuristics); same-role warps of a CTA are kept in step by named barriers so that they share
// instruction-cache fills -- a pop is bound by the ~86 KB of distinct code it walks, see DESIGN.md section 5.
#pragma once
#include "hl_astar_common.cuh"

#define AQ_EXPANDERS 2                 // expander warps per scenario: warp 0 + a helper that shares the rollout / filter / heuristic
#ifndef AQ_SLOTS
#define AQ_SLOTS 5                     // scenarios per CTA (5 x 3 warps at 128 registers)
#endif
#define AQ_MAX_PLANS 6
// one shooter warp per scenario (shots of different pops are independent, but 2-3 shooters measured slower: the
// expander is the critical path)
#define AQ_WARPS_PER_SLOT (AQ_EXPANDERS + 1)
#ifndef AQ_HEAP_SM
#define AQ_HEAP_SM 1023                // open-list entries kept in shared memory (top 10 levels of the heap)
#endif
static_assert(AQ_HEAP_SM > 0, "the search keeps the top of its open list in shared memory");
#ifndef AQ_GUIDE_CAP
#define AQ_GUIDE_CAP 192               // guide polyline points staged in shared memory (longer polylines are read from HBM / L2)
#endif
#ifndef AQ_GD_UNROLL
#define AQ_GD_UNROLL 4                // unroll factor of the guide-distance loop (team_state_costs)
#endif
#define AQ_PRAGMA_(x) _Pragma(#x)
#define AQ_PRAGMA_UNROLL(n) AQ_PRAGMA_(unroll n)
#define AQ_SUB (AQ_TEAM / 16)          // lanes per primitive in the batched guide-distance pass
#ifndef AQ_FAR
#define AQ_FAR 4                       // poses per primitive (farthest first) in the first filter round
#endif
#define AQ_TEAM (32 * AQ_EXPANDERS)
#define AQ_NO_HIT 0x7fffffff
#define AQ_STATUS_DEFER 100              // internal: first shot failed in a first-shot-only launch -> second launch
#ifndef AQ_TIMERS
#define AQ_TIMERS 1                    // per-role phase timers (hl_astar_phase_cycles); 0 removes ~26 hot timing sites
#endif
#if AQ_TIMERS
#define ETICK(ph) do { if (lane == 0) { long long _n = clock64(); S.te[ph] += _n - S.te_last; S.te_last = _n; } } while (0)
#define STICK(ph) do { if (lane == 0) { long long _n = clock64(); S.ts[ph] += _n - S.ts_last; S.ts_last = _n; } } while (0)
#else
#define ETICK(ph) do { } while (0)
#define STICK(ph) do { } while (0)
#endif

struct AqShot {                          // scratch of one shooter warp
    int s_cur; double sx, sy, syaw, sg;
    double rs_lens[HL_RS_CANDIDATES][HL_RS_MAX_SEGS];
    double rs_L[HL_RS_CANDIDATES], rs_prio[HL_RS_CANDIDATES], rs_Lc[HL_RS_CANDIDATES];
    int rs_acc[HL_RS_CANDIDATES], rs_order[HL_RS_CANDIDATES];
    unsigned char rs_valid[HL_RS_CANDIDATES + 2], rs_accept[HL_RS_CANDIDATES + 2];
    RsProblem rs_prob;
    int rs_npts[HL_RS_CANDIDATES];       // sample count of every word planned so far (evaluation order)
    int rs_n, rs_word, rs_assert;
    double rs_goal_cost;
    RsPlan plans[AQ_MAX_PLANS];
    RsPlan plan_tmp;                     // single words; at a successful shot the winning word (the goal extension)
    unsigned long long s_checks, s_exact, s_ref;
    volatile int done_epoch;             // this shooter finished the epoch
};

struct AqSmem {                          // one per scenario slot, shared by its two warps
    double start[3], goal[3];
    long long start_key, goal_key;
    int env, scen;
    volatile int state;                  // ST_IDLE / ST_SEARCH / ST_DONE (written by the expander)
    volatile int epoch;                  // bumped by the expander when a scenario is ready for the shooter
    volatile int popped;                 // closed nodes published to the shooter
    volatile int ew_done;                // expander stopped; shots needed for nodes < shot_limit
    volatile int shot_limit;
    volatile int x_expanding, x_finished;   // expander warp 0 -> helper warp(s)
    int shot_best;                       // smallest pop index with a free word (atomicMin), AQ_NO_HIT if none
    // expander state
    int n_nodes, heap_n, counter, n_closed, ew_status, ew_arrival2;
    int cur; double cx, cy, cyaw, cg; int cprim; int nsteps;
    // the shooter warp's scratch: an array of one, read through `win` (always 0) where the result is assembled.
    // Folding that index away changes the kernel's generated code, so it is left to a change measured on its own.
    AqShot sh[1];
    // expander scratch
    double tx[HL_MAX_PRIMS][AS_ROLL], ty[HL_MAX_PRIMS][AS_ROLL], pyaw[HL_MAX_PRIMS][AS_ROLL];
    unsigned char pamb[HL_MAX_PRIMS][AS_ROLL];
    int phit[HL_MAX_PRIMS];
    double pg[HL_MAX_PRIMS], pprio[HL_MAX_PRIMS];
    long long pkey[HL_MAX_PRIMS];
    int pkey_ok[HL_MAX_PRIMS], pslot[HL_MAX_PRIMS], ppos[HL_MAX_PRIMS], pneed[HL_MAX_PRIMS];
    // stats (per role)
    unsigned long long e_checks, e_exact, e_ref;
    long long t0;
    long long te_last, te[AS_N_PHASES];      // expander phase timers (lane 0 cycles)
    long long ts_last, ts[AS_N_PHASES];      // shooter phase timers
    // result assembly
    int status, arrival, fin_closed, fin_counter, win;
    double goal_cost;
    __align__(16) float envf[AS_ENV_FLOATS];
    double gx[AQ_GUIDE_CAP], gy[AQ_GUIDE_CAP];       // guide polyline of the scenario (calculate_state_cost's argmin)
    double gyaw[AQ_GUIDE_CAP], gs[AQ_GUIDE_CAP];     // ... its headings and arc lengths
    double pds[HL_MAX_PRIMS][AS_ROLL];               // step lengths of the rolled-out primitives (g-cost)
    int guide_staged, need_seg;
    double hp_prio[AQ_HEAP_SM];                     // top of the open-list heap (HeapRef)
    int hp_slot[AQ_HEAP_SM];
};
static_assert(sizeof(AqSmem) * AQ_SLOTS <= 227 * 1024, "per-CTA shared memory exceeds 227 KB");

// Alignment of the AQ_SLOTS warps of one role (named barrier `id`, all threads of those warps) with an AND
// reduction: keeps the role's warps inside the same code region (instruction cache) and tells them when
// every one of them is finished.  Every iteration of either role passes it (measured, DESIGN.md section 5: without it
// the kernel is 2x slower, at every second iteration only 25.7 instead of 21.2 ms per sweep).
__device__ __forceinline__ bool role_barrier_all(int id, int nthreads, bool pred) {
    int r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.s32 p, %1, 0;\n\tbarrier.red.and.pred q, %2, %3, p;\n\tselp.s32 %0, 1, 0, q;\n\t}"
                 : "=r"(r) : "r"((int)pred), "r"(id), "r"(nthreads) : "memory");
    return r != 0;
}

// the warps of one scenario's expander team (named barrier 3 + slot)
__device__ __forceinline__ void team_sync(int slot) {
    asm volatile("bar.sync %0, %1;" :: "r"(3 + slot), "r"(AQ_TEAM) : "memory");
}

__device__ __forceinline__ int warp_read(volatile int* p, int lane) {
    int v = 0;
    if (lane == 0) v = *p;
    return __shfl_sync(FULL, v, 0);
}

__device__ __noinline__ int aq_heap_pop(AqSmem& S, const AsWs& w, int& n) {
    const HeapRef<AQ_HEAP_SM> H{w, S.hp_prio, S.hp_slot};
    return heap_popitem_t<AQ_HEAP_SM>(H, n);
}
__device__ __noinline__ void aq_heap_set(AqSmem& S, const AsWs& w, int& n, int slot, double prio) {
    const HeapRef<AQ_HEAP_SM> H{w, S.hp_prio, S.hp_slot};
    heap_set_t<AQ_HEAP_SM>(H, n, slot, prio);
}

// Open-list insertion of a NEW key by a whole warp (heapdict.__setitem__ -> append + _decrease_key): lane L looks at
// the L-th ancestor of the insertion position, a ballot finds the first ancestor that stays (strictly smaller
// priority), the ancestors below it move down one level in parallel and the new entry takes the freed position --
// the arrangement the sequential swaps produce, in one step instead of up to 13 dependent ones.
__device__ __forceinline__ void aq_heap_push_warp(AqSmem& S, const AsWs& w, int slot, double prio, int lane) {
    const HeapRef<AQ_HEAP_SM> H{w, S.hp_prio, S.hp_slot};
    const int i = S.heap_n;
    const int depth = 31 - __clz(i + 1);                 // the root is the depth-th ancestor
    const bool mine = lane >= 1 && lane <= depth;
    const int a = ((i + 1) >> lane) - 1;
    double ap = 0.0;
    int as = 0;
    if (mine) { ap = H.prio(a); as = H.slot(a); }
    const unsigned stopm = __ballot_sync(FULL, mine && ap < prio);
    const int stop = stopm ? (__ffs(stopm) - 1) : depth + 1;
    __syncwarp();
    if (mine && lane < stop) H.put(((i + 1) >> (lane - 1)) - 1, ap, as);
    if (lane == 0) { H.put(((i + 1) >> (stop - 1)) - 1, prio, slot); S.heap_n = i + 1; }
    __syncwarp();
}

// calculate_state_cost (reference_line_heuristic.py:131-158) of EVERY primitive that needs one, the whole expander
// team at once: AQ_SUB lanes per primitive walk the guide polyline (shared memory) with stride AQ_SUB -- one pass for
// the minimum squared distance (ordering filter), one for the exact hypot of the near-minimal points (first minimum
// wins, np.argmin) -- and one lane per primitive finishes the cost.  Same arithmetic as warp_state_cost; the serial
// part (7 calls per warp, 5-step 64-bit shuffle reductions, the fmod tail) is what it replaces.
__device__ __noinline__ void team_state_costs(AqSmem& S, const EnvBatchDev& eb, const EnvDesc& D, const AsParams& P,
                                              int nst, int tl, int lane) {
    const unsigned needm = __ballot_sync(FULL, lane < P.n_prims && !S.phit[lane] && S.pneed[lane]);
    const int slot = tl / AQ_SUB, sub = tl - slot * AQ_SUB;
    const int p = slot < __popc(needm) ? (int)__fns(needm, 0, slot + 1) : -1;
    const int n = D.n_guide;
    const double* gx = S.gx;                             // shared memory (LDS): the caller takes the per-primitive
    const double* gy = S.gy;                             // warp_state_cost path when the polyline was too long to stage
    const double x = p >= 0 ? S.tx[p][nst] : 0.0, y = p >= 0 ? S.ty[p][nst] : 0.0;
    double best = INFINITY;
AQ_PRAGMA_UNROLL(AQ_GD_UNROLL)
    for (int i = sub; i < n; i += AQ_SUB) {
        const double dx = gx[i] - x, dy = gy[i] - y;
        const double d2 = dx * dx + dy * dy;
        best = d2 < best ? d2 : best;                    // = fmin (a NaN never replaces best) without its NaN fix-up code
    }
#pragma unroll
    for (int o = AQ_SUB / 2; o; o >>= 1) best = fmin(best, __shfl_xor_sync(FULL, best, o));
    const double thr = best * (1.0 + 1e-9) + 1e-300;
    double bh = INFINITY;
    int bi = 0x7fffffff;
#pragma unroll 1
    for (int i = sub; i < n; i += AQ_SUB) {
        const double dx = xsub(gx[i], x), dy = xsub(gy[i], y);
        if (dx * dx + dy * dy <= thr) {
            const double h = hypot_cr(dx, dy);
            if (h < bh || (h == bh && i < bi)) { bh = h; bi = i; }
        }
    }
#pragma unroll
    for (int o = AQ_SUB / 2; o; o >>= 1) {
        const double oh = __shfl_xor_sync(FULL, bh, o);
        const int oi = __shfl_xor_sync(FULL, bi, o);
        if (oh < bh || (oh == bh && oi < bi)) { bh = oh; bi = oi; }
    }
    if (p >= 0 && sub == 0) {
        double h = 0.0;
        if (n > 0) {
            double dist = xmul(bh, 100.0);
            const double yaw_diff = fabs(angle_wrap(xsub(S.gyaw[bi], S.pyaw[p][nst])));
            if (dist > 2.0) dist = 100.0;
            const double to_goal = xsub(S.gs[n - 1], S.gs[bi]);
            h = xadd(xadd(dist, xmul(yaw_diff, 0.2)), xmul(to_goal, 5.0));
        }
        S.pprio[p] = xmul(P.hybrid_cost, h);
    }
}

// Footprint check of ONE planned Reeds-Shepp word by a whole warp: 32 poses per pass, lane-strided, float32 filter first
// and the float64 predicate only for the poses inside the band when no other pose of the pass decided the word.
// Returns true when the word collides.
__device__ __noinline__ bool aq_word_collides(const EnvSmem& Ers, const EnvBatchDev& eb, const EnvDesc& D, const RsPlan& plan,
                                              const double* q0, double cq, double sq, double maxc, float inv_maxc,
                                              unsigned FLAGS, AqShot& T, int lane) {
    const int npts = plan.npts;
    int infeasible = 0;
    const int passes = (npts + 31) >> 5;
#pragma unroll 1
    for (int pass = 0; pass < passes && !infeasible; ++pass) {
        const int j = lane * passes + pass;
        int st2 = HL_FREE;
        unsigned amb = 0;
        if (j < npts) {
            float fx, fy, fc, fs;
            rs_sample_world32(plan, j, inv_maxc, fx, fy, fc, fs);
            if (fabsf(fx) > Ers.reach || fabsf(fy) > Ers.reach) st2 = far_status(FLAGS, Ers.n_seg);
            else if (!(fx == fx) || !(fy == fy) || !(fc == fc)) { st2 = HL_AMBIG; amb = FLAGS; }
            else st2 = filter_part(Ers, fx, fy, fc, fs, Ers.ext, FLAGS, &amb);
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
                rs_sample_local(plan, j, maxc, lx, ly, lyaw, cs, dir);
                rs_to_world(q0, cq, sq, lx, ly, lyaw, wx, wy, wyaw);
                bad2 = pose_exact(eb, D, wx, wy, wyaw, amb) ? 1 : 0;
            }
            if (lane == 0) T.s_exact += (unsigned long long)__popc(ambm);
            infeasible = __any_sync(FULL, bad2);
        }
        if (lane == 0) T.s_checks += (unsigned long long)__popc(livem);
    }
    return infeasible != 0;
}

// Result record + path of a finished scenario (expander warp, after the shooter reported).  Inlined: as a call of its
// own around the write-out call, the kernel spills more.
__device__ __forceinline__ void finalize_spec(AqSmem& S, const AsWs& W, const AsParams& P, const AsOut& O, int lane) {
    const int n_closed = S.fin_closed;
    const int end = (n_closed > 0) ? W.corder[n_closed - 1] : 0;       // the node the search ended on
    const AqShot& T = S.sh[S.win];
    const AsWritten w = write_outputs(W, P, O, S.status, n_closed, end, S.arrival, S.start_key, S.goal_key, &T.plan_tmp,
                                      0, lane);
    if (lane == 0) {
        unsigned long long checks = S.e_checks + S.sh[0].s_checks, exact = S.e_exact + S.sh[0].s_exact, ref = S.sh[0].s_ref;
        // algorithmic count: shots of pops <= the final one (the shooter stops there) + the expansions of the
        // pops BEFORE a successful shot (the expander may have run ahead; that work is not the reference's)
        const bool shot_won = (S.arrival == 1) || (w.status == HL_STATUS_RS_ASSERT);
        ref += (shot_won && n_closed > 0) ? (unsigned long long)W.cref[n_closed - 1] : S.e_ref;
        write_record(O, S.scen, w, S.arrival, T.rs_word, S.goal_cost, S.fin_counter, checks, exact, ref, clock64() - S.t0);
        for (int k = 0; k < AS_N_PHASES; ++k) {
            const long long v = S.te[k] + S.ts[k];
            if (v) atomicAdd(O.phase_cycles + k, (unsigned long long)v);
        }
    }
    for (int i = lane; i < S.n_nodes; i += 32) W.hkey[W.nhpos[i]] = KEY_EMPTY;
    __syncwarp();
}

__global__ void __launch_bounds__(AQ_SLOTS * AQ_WARPS_PER_SLOT * 32, 1)
k_hybrid_astar_s(EnvBatchDev eb, const HlScenario* __restrict__ scen, int n_scen, AsParams P, char* ws_base,
                 size_t ws_stride, unsigned int* work_counter, AsOut O) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int slot = wid / AQ_WARPS_PER_SLOT;
    const int wrole = wid % AQ_WARPS_PER_SLOT;          // 0 .. AQ_EXPANDERS-1 = expander team, then the shooter
    const int ew = wrole;                               // index inside the expander team
    const bool shooter = wrole >= AQ_EXPANDERS;
    const int tl = ew * 32 + lane;                      // lane inside the expander team
    AqSmem& S = reinterpret_cast<AqSmem*>(smem_raw)[slot];
    const AsWs W = as_carve(ws_base + ((size_t)blockIdx.x * AQ_SLOTS + slot) * ws_stride, P.cap_nodes, P.hash_size,
                            P.max_nodes);
    const int hmask = P.hash_size - 1;
    const unsigned FLAGS = HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY | HL_CHECK_LANE;
    if (ew == 0) {
#pragma unroll 1
        for (int i = lane; i < P.hash_size; i += 32) W.hkey[i] = KEY_EMPTY;
        if (lane == 0) {
            S.x_expanding = 0; S.x_finished = 0; S.need_seg = 0;
            S.state = ST_IDLE; S.epoch = 0; S.popped = 0; S.ew_done = 0; S.shot_best = AQ_NO_HIT;
            S.sh[0].done_epoch = 0;
        }
    }
    __syncthreads();

    EnvSmem E;
    E.n_obs = E.n_field = E.n_seg = E.all_rect = 0; E.eps = 0.f; E.reach = 0.f; E.obs = E.field = E.seg = nullptr;

    if (shooter) {
        // =========================================== SHOOTER ===========================================
        AqShot& T = S.sh[0];
        int my_epoch = 0;
        int i = 0;
        bool active = false;            // a scenario is attached and its shots are not finished
        bool finished = false;          // queue drained
        const EnvDesc* Dp = eb.desc;
        EnvSmem Ers = E;
        const float inv_maxc = (float)(1.0 / P.maxc);
        const double stepn = xmul(P.res, P.maxc);
        while (true) {
            if (role_barrier_all(1, AQ_SLOTS * 32, finished)) break;   // alignment point of the shooters
            bool shooting = false, success = false;
            int m = 0;
            double q0[3] = {0.0, 0.0, 0.0}, cq = 1.0, sq = 0.0;
            do {
            if (finished) break;
            if (active) STICK(PH_OUTPUT);     // shooter time in the alignment barrier / waiting for pops
            if (!active) {
                const int st = warp_read(&S.state, lane);
                const int ep = warp_read(&S.epoch, lane);
                if (ep != my_epoch) {
                    my_epoch = ep;
                    __threadfence_block();
                    Dp = eb.desc + S.env;
                    const EnvDesc& D0 = *Dp;
                    // same float32 environment the expander staged in this slot
                    const int n_o = D0.n_obs * HL_OBS32_STRIDE, n_f = D0.n_field * HL_FIELD32_STRIDE, n_s = D0.n_seg * 4;
                    E.n_obs = D0.n_obs; E.n_field = D0.n_field; E.n_seg = D0.n_seg; E.all_rect = D0.all_rect;
                    E.eps = D0.eps; E.reach = D0.reach;
                    for (int k = 0; k < 4; ++k) E.ext[k] = (float)D0.body_ext[k];
                    if (n_o + n_f + n_s <= AS_ENV_FLOATS) { E.obs = S.envf; E.field = S.envf + n_o; E.seg = S.envf + n_o + n_f; }
                    else {
                        E.obs = eb.obs32 + (size_t)HL_OBS32_STRIDE * D0.obs_off;
                        E.field = eb.field32 + HL_FIELD32_STRIDE * (size_t)D0.field_off;
                        E.seg = eb.seg32 + 4 * (size_t)D0.seg_off;
                    }
                    Ers = E;
                    Ers.eps = E.eps + 6e-5f;
                    if (lane == 0) { T.s_checks = 0; T.s_exact = 0; T.s_ref = 0; T.rs_assert = 0; }
                    __syncwarp();
                    i = 0;
                    active = true;
                } else if (st == ST_DONE) { finished = true; break; }
                else { __nanosleep(200); break; }
            }
            {
                // is pop i available, has the expander stopped short of it, or did an EARLIER pop already succeed?
                const int done = warp_read(&S.ew_done, lane);
                __threadfence_block();
                const int popped = warp_read(&S.popped, lane);
                const int best = warp_read((volatile int*)&S.shot_best, lane);
                bool stop = false, have = false;
                if (best < i) stop = true;                         // the search ends before this pop
                else if (done) { if (i >= warp_read(&S.shot_limit, lane)) stop = true; else have = true; }   // limit <= popped
                else if (popped > i) have = true;
                if (stop) {
                    if (lane == 0) { __threadfence_block(); T.done_epoch = my_epoch; }
                    __syncwarp();
                    active = false;
                    break;
                }
                if (!have) { __nanosleep(100); break; }
                __threadfence_block();
                if (lane == 0) {
                    const int cur = W.corder[i];
                    T.s_cur = cur; T.sx = W.nx[cur]; T.sy = W.ny[cur]; T.syaw = W.nyaw[cur]; T.sg = W.ng[cur];
                }
                __syncwarp();
                q0[0] = T.sx; q0[1] = T.sy; q0[2] = T.syaw;
                {
                    // generate_path's normalisation (reeds_shepp.py:565-572, rs_normalise): the sine / cosine of the
                    // node heading and of the heading difference are ONE sincos each, on two lanes at the same time
                    // (sincos == sin, cos and sin odd / cos even bit for bit: tools/sincos_check.cu); the node
                    // heading's pair also gives cq / sq = cos(-yaw), sin(-yaw) of the local -> world rotation.
                    const double phi = xsub(S.goal[2], q0[2]);
                    double sn, cs;
                    m_sincos(lane == 1 ? phi : q0[2], &sn, &cs);
                    const double c0 = __shfl_sync(FULL, cs, 0), s0 = __shfl_sync(FULL, sn, 0);
                    const double cp = __shfl_sync(FULL, cs, 1), sp = __shfl_sync(FULL, sn, 1);
                    cq = c0; sq = -s0;
                    if (lane == 0) {
                        RsProblem Pr;
                        const double dx = xsub(S.goal[0], q0[0]), dy = xsub(S.goal[1], q0[1]);
                        Pr.phi = phi;
                        Pr.x = xmul(xadd(xmul(c0, dx), xmul(s0, dy)), P.maxc);
                        Pr.y = xmul(xadd(xmul(-s0, dx), xmul(c0, dy)), P.maxc);
                        Pr.sp = sp; Pr.cp = cp;
                        Pr.xb = xadd(xmul(Pr.x, cp), xmul(Pr.y, sp));
                        Pr.yb = xsub(xmul(Pr.x, sp), xmul(Pr.y, cp));
                        T.rs_prob = Pr;
                    }
                    __syncwarp();
                }
                rs_candidates_warp(T.rs_prob, T.rs_valid, T.rs_lens, lane);
                STICK(PH_RS_CAND);
                if (lane < RS_N_GROUPS) rs_select_group(lane, T.rs_valid, T.rs_lens, T.rs_accept, T.rs_Lc);
                __syncwarp();
                {
                    const int a0 = T.rs_accept[lane];
                    const int a1 = (lane + 32 < HL_RS_CANDIDATES) ? T.rs_accept[lane + 32] : 0;
                    const unsigned b0 = __ballot_sync(FULL, a0 == 1), b1 = __ballot_sync(FULL, a1 == 1);
                    const unsigned bad = __ballot_sync(FULL, a0 == 2 || a1 == 2);
                    const unsigned lt = (1u << lane) - 1u;
                    const int n0 = __popc(b0);
                    if (a0 == 1) { int k = __popc(b0 & lt); T.rs_acc[k] = lane; T.rs_L[k] = T.rs_Lc[lane]; }
                    if (a1 == 1) { int k = n0 + __popc(b1 & lt); T.rs_acc[k] = lane + 32; T.rs_L[k] = T.rs_Lc[lane + 32]; }
                    m = bad ? 0 : n0 + __popc(b1);
                    __syncwarp();
                    if (lane == 0) { if (bad) T.rs_assert = 1; T.rs_n = m; }
                    __syncwarp();
                    if (bad) success = true;     // the reference would raise here: report it as the end of the search
                }
                STICK(PH_RS_SELECT);
                // The words are planned and refuted in EVALUATION order: a failing shot (every pop but the last one of
                // a scenario) must refute every word whatever the order, so the cost queue (rs_path_cost + heapdict
                // replay, hybrid_a_star_search.py:265-271) is only built when some word turns out to be free.
                shooting = true;
            }
            } while (0);
            if (!shooting) continue;
            const EnvDesc& D = *Dp;
            {
                // Words in batches of AQ_MAX_PLANS: plan the batch (one warp-wide call), probe all its words coarsely --
                // almost every word of a failing shot collides somewhere and ONE hit kills a word: 32 / nw evenly spaced
                // poses each, only definite float32 HITs count -- then the survivors get their own 32-pose passes.
                int first_free = -1;
                unsigned long long ref_all = 0;              // poses of the words refuted so far (lane 0's tally)
#pragma unroll 1
                for (int k0 = 0; k0 < m && first_free < 0; k0 += AQ_MAX_PLANS) {
                    const int nw = (m - k0) < AQ_MAX_PLANS ? (m - k0) : AQ_MAX_PLANS;
                    rs_make_plans_warp(T.rs_acc, T.rs_lens, T.rs_npts, k0, nw, T.plans, q0, cq, sq, D.origin, P.maxc, stepn, lane);
                    STICK(PH_RS_PLAN);
                    unsigned dead = 0;
                    if (nw >= 2) {
                        const int per = 32 / nw;
                        const int r = lane / per, q = lane - r * per;
                        int st2 = HL_FREE;
                        if (r < nw) {
                            const RsPlan& plan = T.plans[r];
                            const int npts = plan.npts;
                            const int j = (int)(((long long)(2 * q + 1) * npts) / (2 * per));
                            if (j < npts) {
                                float fx, fy, fc, fs;
                                unsigned amb = 0;
                                rs_sample_world32(plan, j, inv_maxc, fx, fy, fc, fs);
                                if (fabsf(fx) > Ers.reach || fabsf(fy) > Ers.reach) st2 = far_status(FLAGS, Ers.n_seg);
                                else if (!(fx == fx) || !(fy == fy) || !(fc == fc)) st2 = HL_AMBIG;
                                else st2 = filter_part(Ers, fx, fy, fc, fs, Ers.ext, FLAGS, &amb);
                            }
                        }
                        const unsigned hitm = __ballot_sync(FULL, st2 == HL_HIT);
                        const unsigned livem = __ballot_sync(FULL, r < nw);
                        for (int w = 0; w < nw; ++w)
                            if (hitm & (((per >= 32) ? 0xffffffffu : ((1u << per) - 1u)) << (w * per))) dead |= 1u << w;
                        if (lane == 0) T.s_checks += (unsigned long long)__popc(livem);
                    }
#pragma unroll 1
                    for (int w = 0; w < nw; ++w) {
                        const RsPlan& plan = T.plans[w];
                        ref_all += (unsigned long long)plan.npts;
                        if (dead & (1u << w)) continue;
                        const bool hit = aq_word_collides(Ers, eb, D, plan, q0, cq, sq, P.maxc, inv_maxc, FLAGS, T, lane);
                        if (!hit && xdiv(T.rs_L[k0 + w], P.maxc) < P.min_len_goal) { first_free = k0 + w; break; }
                    }
                    STICK(PH_RS_SAMPLE);
                }
                if (first_free < 0) {
                    if (lane == 0) T.s_ref += ref_all;       // every word tried and refuted (:272-287 falls through)
                } else {
                    // Some word is free: the reference returns the FIRST free word in the pop order of its cost queue.
                    // Words before `first_free` in evaluation order are refuted, the ones after it are examined here
                    // only as far as the pop order reaches them.
                    __syncwarp();
#pragma unroll 1
                    for (int k = lane; k < m; k += 32)
                        T.rs_prio[k] = rs_path_cost(T.sg, T.rs_acc[k], T.rs_lens[T.rs_acc[k]], P.max_steer,
                                                    P.reverse_cost, P.dir_change_cost, P.steer_cost);
                    __syncwarp();
                    if (lane == 0) heapdict_order(T.rs_prio, m, T.rs_order);
                    __syncwarp();
                    unsigned long long tally = 0;
                    int winner = -1;
#pragma unroll 1
                    for (int r = 0; r < m && winner < 0; ++r) {
                        const int k = T.rs_order[r];
                        if (k < first_free) { tally += (unsigned long long)T.rs_npts[k]; continue; }
                        if (k == first_free) { tally += (unsigned long long)T.rs_npts[k]; winner = k; break; }
                        rs_make_plans_warp(T.rs_acc, T.rs_lens, T.rs_npts, k, 1, &T.plan_tmp, q0, cq, sq, D.origin, P.maxc, stepn, lane);
                        const RsPlan& plan = T.plan_tmp;
                        tally += (unsigned long long)plan.npts;
                        const bool hit = aq_word_collides(Ers, eb, D, plan, q0, cq, sq, P.maxc, inv_maxc, FLAGS, T, lane);
                        if (!hit && xdiv(T.rs_L[k], P.maxc) < P.min_len_goal) winner = k;
                    }
                    __syncwarp();
                    rs_make_plans_warp(T.rs_acc, T.rs_lens, T.rs_npts, winner, 1, &T.plan_tmp, q0, cq, sq, D.origin, P.maxc, stepn, lane);   // the result path's plan
                    if (lane == 0) {
                        T.s_ref += tally;
                        T.rs_word = T.rs_acc[winner]; T.rs_goal_cost = T.rs_prio[winner];
                    }
                    success = true;
                }
                __syncwarp();
                STICK(PH_RS_SAMPLE);
            }
            if (success) {
                if (lane == 0) { __threadfence_block(); atomicMin(&S.shot_best, i); __threadfence_block(); T.done_epoch = my_epoch; }
                __syncwarp();
                active = false;
            } else ++i;
        }
        return;
    }

    // ============================================ EXPANDER ============================================
    // One alignment barrier per loop iteration (role barrier 2): an iteration is either "attach a scenario",
    // "expand one node" or "wait for the shooter / write the result".
    int mode = 0;                       // 0 need a scenario, 1 expanding, 2 waiting for the shooter
    bool finished = false;
    int my_epoch = 0;
    const EnvDesc* Dp = eb.desc;
    int helper_epoch = 0;
    while (true) {
        if (role_barrier_all(2, AQ_SLOTS * AQ_TEAM, finished)) break;
        bool expanding = false;
        if (ew == 0) {
        do {
        if (finished) break;
        ETICK(PH_SETUP);                 // time spent in the alignment barrier (+ attach / wait modes)
        if (mode == 0) {
        // ---- next scenario
        int sc = 0;
        if (lane == 0) {
            sc = (int)atomicAdd(work_counter, 1u);
            const int n_eff = O.order_count ? *O.order_count : n_scen;
            sc = sc < n_eff ? (O.order ? O.order[sc] : sc) : -1;
        }
        sc = __shfl_sync(FULL, sc, 0);
        if (sc < 0) { if (lane == 0) { __threadfence_block(); S.state = ST_DONE; } finished = true; break; }
        if (lane == 0) {
            const HlScenario s = scen[sc];
            S.scen = sc; S.env = s.env_id;
            for (int k = 0; k < 3; ++k) { S.start[k] = s.start[k]; S.goal[k] = s.goal[k]; }
            S.n_nodes = 0; S.heap_n = 0; S.counter = 0; S.n_closed = 0;
            S.status = -1; S.arrival = 0; S.goal_cost = 0.0; S.ew_status = -1; S.ew_arrival2 = 0;
            S.e_checks = 0; S.e_exact = 0; S.e_ref = 0; S.win = 0;
            S.sh[0].s_checks = 0; S.sh[0].s_exact = 0; S.sh[0].s_ref = 0; S.sh[0].rs_assert = 0;
            S.fin_closed = 0; S.fin_counter = 0;
            S.popped = 0; S.ew_done = 0; S.shot_limit = 0; S.shot_best = AQ_NO_HIT;
            S.t0 = clock64();
            for (int k = 0; k < AS_N_PHASES; ++k) { S.te[k] = 0; S.ts[k] = 0; }
            S.te_last = S.t0; S.ts_last = S.t0;
        }
        __syncwarp();
        Dp = eb.desc + S.env;
        const EnvDesc& D = *Dp;
        stage_env_warp(eb, D, S.envf, AS_ENV_FLOATS, E, lane);
        if (D.n_guide <= AQ_GUIDE_CAP) {
            for (int i = lane; i < D.n_guide; i += 32) {
                S.gx[i] = eb.guide_x[D.guide_off + i]; S.gy[i] = eb.guide_y[D.guide_off + i];
                S.gyaw[i] = eb.guide_yaw[D.guide_off + i]; S.gs[i] = eb.guide_s[D.guide_off + i];
            }
        }
        if (lane == 0) S.guide_staged = D.n_guide <= AQ_GUIDE_CAP ? 1 : 0;
        {
            const AsStart st = start_node(W, P, eb, D, E, S.start, S.goal, FLAGS, lane);
            if (lane == 0) {
                S.start_key = st.start_key; S.goal_key = st.goal_key; S.ew_status = st.status;
                if (st.status < 0) { S.n_nodes = 1; aq_heap_set(S, W, S.heap_n, 0, st.prio); }
            }
            __syncwarp();
        }
        if (S.ew_status >= 0) {                       // blocked / capacity: no shooter involved
            if (lane == 0) { S.status = S.ew_status; S.fin_closed = 0; S.fin_counter = 0; }
            __syncwarp();
            finalize_spec(S, W, P, O, lane);
            break;
        }
        // hand the scenario to the shooter
        if (lane == 0) { __threadfence_block(); S.state = ST_SEARCH; S.epoch = S.epoch + 1; }
        __syncwarp();
        my_epoch = warp_read(&S.epoch, lane);

            mode = 1;
            break;
        }
        if (mode == 1) {
            const EnvDesc& D = *Dp;
            if (lane == 0) {
                if (*(volatile int*)&S.shot_best != AQ_NO_HIT) S.ew_status = HL_STATUS_OK;   // a shooter ended the search
                else if (S.counter > P.max_nodes) S.ew_status = HL_STATUS_MAX_NODES;
                else {
                    S.counter += 1;
                    if (S.heap_n == 0) S.ew_status = HL_STATUS_OPEN_EMPTY;
                    else {
                        int cur = aq_heap_pop(S, W, S.heap_n);
                        W.nstate[cur] = 1;
                        W.cref[S.n_closed] = (long long)S.e_ref;
                        W.corder[S.n_closed++] = cur;
                        S.cur = cur; S.cx = W.nx[cur]; S.cy = W.ny[cur]; S.cyaw = W.nyaw[cur]; S.cg = W.ng[cur];
                        S.cprim = W.nprim[cur];
                        __threadfence_block();
                        S.popped = S.n_closed;                                   // publish to the shooter
                        // tolerance arrival (:464-495) ends the search at this pop (if no earlier shot succeeds)
                        double xd = fabs(xsub(S.cx, S.goal[0])), yd = fabs(xsub(S.cy, S.goal[1]));
                        double wd = fabs(angle_wrap(xsub(S.cyaw, S.goal[2])));
                        if (xd < P.res && yd < P.res && wd < P.yaw_res) { S.ew_arrival2 = 1; S.ew_status = HL_STATUS_OK; }
                        else S.need_seg = 1;
                    }
                }
            }
            __syncwarp();
            const int need_seg = S.need_seg;
            __syncwarp();
            if (need_seg) {
                // search length of this node (reference_line_heuristic.py:120-129: LAST capsule whose interior holds
                // the point), one capsule per lane
                bool in = false;
                if (lane < D.n_seg)
                    in = exact_point_in_capsule(eb.seg64 + 4 * (size_t)(D.seg_off + lane),
                                                eb.seg_poly + 2 * HL_CAPSULE_VERTS * (size_t)(D.seg_off + lane), S.cx, S.cy, true);
                const unsigned inm = __ballot_sync(FULL, in);
                if (lane == 0) {
                    const int seg = inm ? 31 - __clz(inm) : -1;
                    const double len = seg < 0 ? D.default_len : eb.seg_len[D.seg_off + seg];
                    S.nsteps = (int)rint(xdiv(len, P.res));
                    if (S.nsteps + 1 > HL_MAX_ROLLOUT || S.nsteps < 1) S.ew_status = HL_STATUS_CAPACITY;
                    S.need_seg = 0;
                }
            }
            if (lane < HL_MAX_PRIMS) { S.phit[lane] = 0; S.pneed[lane] = 1; }
            __syncwarp();
            if (O.first_only && S.ew_status < 0) {           // first-shot-only launch: the shooter decides this scenario's fate
                if (lane == 0) S.ew_status = AQ_STATUS_DEFER;
                __syncwarp();
            }
            ETICK(PH_POP);
            if (S.ew_status >= 0) mode = 2; else expanding = true;
        }
        } while (0);
        }
        if (ew == 0 && lane == 0) { S.x_expanding = expanding ? 1 : 0; S.x_finished = finished ? 1 : 0; }
        team_sync(slot);
        if (ew != 0) {                                       // the helper follows warp 0's decisions
            expanding = S.x_expanding != 0; finished = S.x_finished != 0;
            const int ep = S.epoch;
            if (expanding && ep != helper_epoch) {           // new scenario: the float32 environment warp 0 staged
                helper_epoch = ep;
                Dp = eb.desc + S.env;
                const EnvDesc& D0 = *Dp;
                const int n_o = D0.n_obs * HL_OBS32_STRIDE, n_f = D0.n_field * HL_FIELD32_STRIDE, n_s = D0.n_seg * 4;
                E.n_obs = D0.n_obs; E.n_field = D0.n_field; E.n_seg = D0.n_seg; E.all_rect = D0.all_rect;
                E.eps = D0.eps; E.reach = D0.reach;
                for (int k = 0; k < 4; ++k) E.ext[k] = (float)D0.body_ext[k];
                if (n_o + n_f + n_s <= AS_ENV_FLOATS) { E.obs = S.envf; E.field = S.envf + n_o; E.seg = S.envf + n_o + n_f; }
                else {
                    E.obs = eb.obs32 + (size_t)HL_OBS32_STRIDE * D0.obs_off;
                    E.field = eb.field32 + HL_FIELD32_STRIDE * (size_t)D0.field_off;
                    E.seg = eb.seg32 + 4 * (size_t)D0.seg_off;
                }
            }
        }
        const EnvDesc& D = *Dp;
        if (expanding) {
            {
            const int n = S.nsteps, np1 = n + 1;
            const int total = P.n_prims * np1;
            // yaws[0..n+1] of every primitive once (the pose yaw of step i is yaws[i+1]), one sincos each
#pragma unroll 1
            for (int idx = tl; idx < P.n_prims * (np1 + 1); idx += AQ_TEAM) {
                const int p = idx / (np1 + 1), i = idx - p * (np1 + 1);
                const double ys = P.yaw_step[p];
                const double init_yaw = angle_wrap(xadd(S.cyaw, ys));
                const double stop = xadd(init_yaw, xmul(ys, (double)(n + 1)));
                const double delta = xsub(stop, init_yaw);
                const double step = xdiv(delta, (double)(n + 1));
                const double yw = rollout_yaw(init_yaw, stop, step, delta, n + 1, i);
                if (i >= 1) S.pyaw[p][i - 1] = yw;
                if (i <= n) {
                    double sn, cs;
                    m_sincos(yw, &sn, &cs);
                    S.tx[p][i] = xmul(xmul(P.res, cs), P.dir[p]);
                    S.ty[p][i] = xmul(xmul(P.res, sn), P.dir[p]);
                }
            }
            team_sync(slot);
            if (tl < P.n_prims) {
                double ax = 0.0, ay = 0.0;
#pragma unroll 1
                for (int i = 0; i < np1; ++i) {
                    ax = (i == 0) ? S.tx[lane][0] : xadd(ax, S.tx[lane][i]);
                    ay = (i == 0) ? S.ty[lane][0] : xadd(ay, S.ty[lane][i]);
                    S.tx[lane][i] = xadd(S.cx, ax);
                    S.ty[lane][i] = xadd(S.cy, ay);
                }
            }
            team_sync(slot);
            if (ew == 0) ETICK(PH_ROLLOUT);
            // One hit kills a primitive, and a primitive that collides does so far from the (feasible) node it starts
            // at: test the two farthest poses of every primitive first, then only the live primitives' other poses.
            {
                const int far_cnt = np1 < AQ_FAR ? np1 : AQ_FAR;
#pragma unroll 1
                for (int idx = tl; idx < P.n_prims * far_cnt; idx += AQ_TEAM) {
                    const int p = idx / far_cnt, j = n - (idx - p * far_cnt);
                    unsigned amb = 0;
                    int st = pose_filter(D, E, S.tx[p][j], S.ty[p][j], S.pyaw[p][j], FLAGS, &amb);
                    S.pamb[p][j] = (st == HL_AMBIG) ? (unsigned char)amb : 0;
                    if (st == HL_HIT) atomicOr(&S.phit[p], 1);
                }
                team_sync(slot);
                const unsigned live = __ballot_sync(FULL, lane < P.n_prims && S.phit[lane] == 0);
                const int rem = np1 - far_cnt;
                const int total2 = __popc(live) * rem;
#pragma unroll 1
                for (int idx = tl; idx < total2; idx += AQ_TEAM) {
                    const int q = idx / rem, j = idx - q * rem;
                    const int p = __fns(live, 0, q + 1);
                    unsigned amb = 0;
                    int st = pose_filter(D, E, S.tx[p][j], S.ty[p][j], S.pyaw[p][j], FLAGS, &amb);
                    S.pamb[p][j] = (st == HL_AMBIG) ? (unsigned char)amb : 0;
                    if (st == HL_HIT) atomicOr(&S.phit[p], 1);
                }
                if (tl == 0) { S.e_checks += (unsigned long long)(P.n_prims * far_cnt + total2); S.e_ref += (unsigned long long)total; }
            }
            team_sync(slot);
            if (ew == 0) ETICK(PH_FILTER);
#pragma unroll 1
            for (int idx = tl; idx < total; idx += AQ_TEAM) {
                const int p = idx / np1, j = idx - p * np1;
                if (S.pamb[p][j] && !S.phit[p]) {
                    atomicAdd(&S.e_exact, 1ULL);
                    if (pose_exact(eb, D, S.tx[p][j], S.ty[p][j], S.pyaw[p][j], S.pamb[p][j])) atomicOr(&S.phit[p], 2);
                }
            }
            team_sync(slot);
            if (ew == 0) ETICK(PH_EXACT);
            }
        }
        if (expanding) {
            {
            const int n = S.nsteps, np1 = n + 1;
            // step lengths of calculate_path_length (np.hypot of np.diff), one lane per (primitive, step)
#pragma unroll 1
            for (int idx = tl; idx < P.n_prims * n; idx += AQ_TEAM) {
                const int p = idx / n, i = idx - p * n;
                if (!S.phit[p]) S.pds[p][i] = hypot_cr(xsub(S.tx[p][i + 1], S.tx[p][i]), xsub(S.ty[p][i + 1], S.ty[p][i]));
            }
            team_sync(slot);
            if (tl < P.n_prims && !S.phit[lane]) {
                const int p = lane;
                double len = 0.0;
#pragma unroll 1
                for (int i = 0; i + 1 < np1; ++i) len = (i == 0) ? S.pds[p][0] : xadd(len, S.pds[p][i]);
                double cost = xadd(S.cg, len);
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
                int pos = -1;
                const int slot2 = S.pkey_ok[p] ? hash_find(W, hmask, key, &pos) : -1;
                S.pslot[p] = slot2;
                S.ppos[p] = pos;
                if (slot2 >= 0 && (W.nstate[slot2] == 1 || !(cost < W.ng[slot2]))) S.pneed[p] = 0;
            }
            team_sync(slot);
            if (ew == 0) ETICK(PH_ARRIVE);                   // (timer slot reused: g-cost + key + hash probe)
            if (S.guide_staged) team_state_costs(S, eb, D, P, n, tl, lane);
            else {                                           // polyline longer than AQ_GUIDE_CAP: one warp call per primitive
                int q = 0;
#pragma unroll 1
                for (int p = 0; p < P.n_prims; ++p) {
                    if (!S.phit[p] && S.pneed[p]) {
                        if ((q % AQ_EXPANDERS) == ew) {
                            const double h = warp_state_cost(eb, D, S.tx[p][n], S.ty[p][n], S.pyaw[p][n], lane);
                            if (lane == 0) S.pprio[p] = xmul(P.hybrid_cost, h);
                        }
                        ++q;
                    }
                }
            }
            team_sync(slot);
            if (ew == 0) ETICK(PH_COST_HEUR);
            if (ew == 0) {
                // merge into the open list (:580-596).  What the cost phase looked up (hash position, existing node,
                // "not needed") stays valid unless two children of THIS expansion meet in the hash table -- the same
                // empty position or the same node.  Without such a meeting (the rule) every child is written by its own
                // lane -- new node ids by a prefix count over the primitives, in order -- and only the open-list
                // insertions are serialised (warp-wide pushes, primitive order).  Otherwise (rare) the ordered
                // re-probing loop below does everything.
                const bool live = lane < P.n_prims && !S.phit[lane];
                const int my_pos = live ? S.ppos[lane] : -1, my_slot = live ? S.pslot[lane] : -1;
                bool meet = live && !S.pkey_ok[lane];
                if (live) {
#pragma unroll 1
                    for (int q = 0; q < lane; ++q) {
                        if (S.phit[q]) continue;
                        if (my_slot < 0 ? (S.pslot[q] < 0 && S.ppos[q] == my_pos) : (S.pslot[q] == my_slot)) meet = true;
                    }
                }
                const unsigned newm = __ballot_sync(FULL, live && my_slot < 0);
                const bool slow = __any_sync(FULL, meet) || S.n_nodes + __popc(newm) > P.cap_nodes;
                unsigned todo = __ballot_sync(FULL, live);
                if (!slow) {
                    const unsigned pushm = __ballot_sync(FULL, live && (my_slot < 0 || S.pneed[lane]));
                    const int base = S.n_nodes;
                    __syncwarp();
                    if (live && (my_slot < 0 || S.pneed[lane])) {
                        const int p = lane;
                        int slot2 = my_slot;
                        if (slot2 < 0) {
                            slot2 = base + __popc(newm & ((1u << lane) - 1u));
                            W.hkey[my_pos] = S.pkey[p]; W.hval[my_pos] = slot2; W.nhpos[slot2] = my_pos;
                            W.nkey[slot2] = S.pkey[p]; W.nstate[slot2] = 0; W.nheap[slot2] = -1;
                            S.pslot[p] = -1 - slot2;             // new node: id handed to the push loop
                        }
                        W.nx[slot2] = S.tx[p][n]; W.ny[slot2] = S.ty[p][n]; W.nyaw[slot2] = S.pyaw[p][n];
                        W.ng[slot2] = S.pg[p]; W.nparent[slot2] = S.cur; W.nprim[slot2] = (signed char)p;
                        W.nsteps[slot2] = (signed char)n;
                    }
                    if (lane == 0) S.n_nodes = base + __popc(newm);
                    __syncwarp();
                    unsigned push = pushm;
#pragma unroll 1
                    while (push) {
                        const int p = __ffs(push) - 1;
                        push &= push - 1;
                        const double g = S.pg[p];
                        const double prio = (S.pprio[p] > g) ? S.pprio[p] : g;
                        const int ps = S.pslot[p];
                        if (ps < 0) aq_heap_push_warp(S, W, -1 - ps, prio, lane);
                        else {                                   // an open node got cheaper: heapdict re-keys it
                            if (lane == 0) aq_heap_set(S, W, S.heap_n, ps, prio);
                            __syncwarp();
                        }
                    }
                    todo = 0;
                }
#pragma unroll 1
                while (todo) {
                    const int p = __ffs(todo) - 1;
                    todo &= todo - 1;
                    if (!S.pkey_ok[p]) { if (lane == 0) S.ew_status = HL_STATUS_CAPACITY; break; }
                    int pos = S.ppos[p];
                    int slot2 = S.pslot[p];
                    if (slot2 < 0 ? (W.hkey[pos] != KEY_EMPTY) : false) slot2 = hash_find(W, hmask, S.pkey[p], &pos);
                    const double g = S.pg[p];
                    const double prio = (S.pprio[p] > g) ? S.pprio[p] : g;
                    int at = -1;                                 // position of an existing OPEN entry of this key
                    if (slot2 >= 0) {
                        if (W.nstate[slot2] == 1) continue;
                        if (!(g < W.ng[slot2])) continue;
                        if (!S.pneed[p]) { if (lane == 0) S.ew_status = HL_STATUS_CAPACITY; break; }
                        at = W.nheap[slot2];
                    } else {
                        const int nn = S.n_nodes;
                        if (nn >= P.cap_nodes) { if (lane == 0) S.ew_status = HL_STATUS_CAPACITY; break; }
                        slot2 = nn;
                        __syncwarp();
                        if (lane == 0) {
                            S.n_nodes = nn + 1;
                            W.hkey[pos] = S.pkey[p]; W.hval[pos] = slot2; W.nhpos[slot2] = pos;
                            W.nkey[slot2] = S.pkey[p]; W.nstate[slot2] = 0; W.nheap[slot2] = -1;
                        }
                    }
                    if (lane == 0) {
                        W.nx[slot2] = S.tx[p][n]; W.ny[slot2] = S.ty[p][n]; W.nyaw[slot2] = S.pyaw[p][n];
                        W.ng[slot2] = g; W.nparent[slot2] = S.cur; W.nprim[slot2] = (signed char)p;
                        W.nsteps[slot2] = (signed char)n;
                    }
                    __syncwarp();
                    if (at >= 0) {                               // re-keying an open node: heapdict pops it first (rare)
                        if (lane == 0) aq_heap_set(S, W, S.heap_n, slot2, prio);
                        __syncwarp();
                    } else aq_heap_push_warp(S, W, slot2, prio, lane);
                }
            }
            __syncwarp();
            }
            if (ew == 0) { ETICK(PH_MERGE); if (S.ew_status >= 0) mode = 2; }
        }
        if (ew != 0) continue;                               // the bookkeeping below is warp 0's
        if (finished) continue;
        if (mode == 2 && !S.ew_done) {
        // ---- tell the shooter how far its shots are needed, wait for it, assemble the result
        if (lane == 0) {
            // every popped node gets its shot, as in the reference (:542-545); at a tolerance arrival the shot of
            // that pop is still evaluated (and counted) but the arrival overrides its result
            S.shot_limit = S.n_closed;
            __threadfence_block();
            S.ew_done = 1;
        }
        __syncwarp();
        }
        if (mode == 2) {
            if (warp_read(&S.sh[0].done_epoch, lane) != my_epoch) { __nanosleep(100); continue; }
        __threadfence_block();
        if (lane == 0) {
            const int best = *(volatile int*)&S.shot_best;
            const int hit = (best == AQ_NO_HIT) ? -1 : best;
            if (hit >= 0) S.win = 0;
            if (hit >= 0 && S.sh[S.win].rs_assert && !(S.ew_arrival2 && hit >= S.n_closed - 1)) {
                S.status = HL_STATUS_RS_ASSERT; S.fin_closed = hit + 1; S.fin_counter = hit + 1; S.arrival = 0;
            } else if (hit >= 0 && !(S.ew_arrival2 && hit >= S.n_closed - 1)) {     // first free word at pop `hit`
                // (a shot raced at the tolerance-arrival pop itself does not count: the arrival overrides it)
                S.status = HL_STATUS_OK; S.arrival = 1; S.fin_closed = hit + 1; S.fin_counter = hit + 1;
                S.goal_cost = S.sh[S.win].rs_goal_cost;
            } else if (S.ew_arrival2) {
                S.status = HL_STATUS_OK; S.arrival = 2; S.fin_closed = S.n_closed; S.fin_counter = S.counter;
                S.goal_cost = S.cg;
            } else {
                S.status = S.ew_status; S.arrival = 0; S.fin_closed = S.n_closed; S.fin_counter = S.counter;
            }
        }
        __syncwarp();
        if (S.status == AQ_STATUS_DEFER) {                   // not decided by its first shot: hand it to the second launch
            if (lane == 0) O.defer_list[atomicAdd(O.defer_count, 1)] = S.scen;
            for (int i = lane; i < S.n_nodes; i += 32) W.hkey[W.nhpos[i]] = KEY_EMPTY;
            __syncwarp();
        } else finalize_spec(S, W, P, O, lane);
            mode = 0;
        }
    }
}
