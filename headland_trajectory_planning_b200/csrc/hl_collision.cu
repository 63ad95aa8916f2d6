// hl_collision.cu -- K1: per-pose footprint collision check.
//
// Replaces OrchardGeometryEnvironment.check_path_feasibility
// (orchard_geometry_environment.py:423-458) + CarModel.get_path_poly
// (car_model.py:39-73) and ReferenceLineHeuristic.check_path_feasibility
// (reference_line_heuristic.py:105-118), decomposed per pose (SURVEY.md 8a-10).
//
// Round-2 structure (DESIGN.md section 5, K1):
//   * a CTA of 8 warps walks 1024-pose tiles; the tile's poses (24 KB, contiguous) arrive by ONE cp.async.bulk
//     (TMA, 1-D) on the CTA's mbarrier, and the copy of the NEXT tile is issued as soon as the current one has been
//     converted to the float32 frame, so HBM latency hides behind the filter stages;
//   * the environment's float32 records are staged by three bulk copies and read with LDS.128 (broadcast);
//   * the float32 filter runs as STAGES over the tile, cheapest and most decisive first -- lane centre test,
//     obstacles (box-box SAT), field-edge pass, nearby field edges, lane corners.  Between stages the CTA COMPACTS
//     the poses that are still undecided into a shared list (ballot + popc + one shared atomic per warp), so every
//     stage runs on dense warps instead of dragging 32 unrelated poses through every section, and the 8 warps of
//     a CTA execute the same stage at the same time: a stage's code is fetched into the 32 KB instruction cache
//     once per 1024 poses (the first cut with per-warp lists ran at 72-88 % instruction-cache hit rate and 68 %
//     lane occupancy, profiles/r2b-r2d);
//   * poses inside the float32 error band are resolved by a whole warp with the float64 predicates (hl_geom.cuh).
// Tiles that cannot use this path (environment larger than the staging area, several environments in one tile,
// non-rectangular obstacle quads) take the monolithic per-pose filter on global memory (k1_slow_slice).
// Roofline: FP32 ALU (24 B of HBM traffic per ~2.5 kflop check).
#include "hl_geom.cuh"

#ifndef K1_WARPS
#define K1_WARPS 8
#endif
#define K1_THREADS (K1_WARPS * 32)
#define K1_TILE (K1_WARPS * 128)          // poses per CTA tile
#define K1_PER_THREAD (K1_TILE / K1_THREADS)
#define K1_SLICE (K1_TILE / K1_WARPS)     // poses per warp in the per-pose fallback
#define K1_ENV_FLOATS 1024                // staged float32 records (canonical environment: 432 floats)
#define K1_PAIR_CAP 2048                  // (pose, nearby edge) pairs per tile; poses beyond it go to the float64 predicate
#define K1_QBITS 11                       // bits of the pose index inside a pair (K1_TILE <= 2048, edges < 32)
#ifndef K1_MIN_CTAS
#define K1_MIN_CTAS 4
#endif
#ifndef K1_UNROLL_OBS
#define K1_UNROLL_OBS 2
#endif
#ifndef K1_UNROLL_FLD
#define K1_UNROLL_FLD 2
#endif
#define K1_PRAGMA(x) _Pragma(#x)
#define K1_UNROLL(n) K1_PRAGMA(unroll n)

// ------------------------------------------------------------------ PTX: mbarrier + 1-D bulk copy (TMA)
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
// generic-proxy reads of a buffer must be ordered before the async proxy overwrites it
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// 16-byte load of a staged record.  The pointers below all derive from the kernel's `extern __shared__` block, so
// the compiler proves the address space and emits LDS.128 (checked in the SASS, profiles/r2_k1_sass.txt).
__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// ------------------------------------------------------------------ shared-memory layout
// A pose inside the float32 band needs the float64 predicates: a whole warp for ~25 us while the 7 other warps of the
// CTA wait at the next barrier (2e-4 of the poses, but 12 % of the kernel's stall samples).  Such poses are QUEUED
// instead; the float32 pipeline goes on as if the ambiguous test had passed (a later verdict can only add "hit"), and
// when the CTA has no tile left its warps resolve the queue, one entry per warp at a time, all in parallel.
#define K1_DEFER_CAP 48
// Draining between tiles measured slower (16.86 vs 17.43 G checks/s, 16 Mi random poses): tiles are assigned by a fixed
// stride, so a CTA that stops to drain simply finishes that much later.
struct K1Defer { long long i; int env; unsigned amb; int rect; int pad; };
struct __align__(16) K1Cta {
    double raw[K1_TILE * 3];              // TMA landing zone: x, y, yaw of the tile                        24 KB
    float px[K1_TILE], py[K1_TILE];       // pose relative to the environment origin                         8 KB
    float yr[K1_TILE];                    // heading reduced to [-pi, pi]                                    4 KB
    unsigned short pairs[K1_PAIR_CAP];    // (pose, nearby field edge) pairs of the tile: q | edge << K1_QBITS       4 KB
    unsigned short la[K1_TILE], lb[K1_TILE], lc[K1_TILE];      // compacted pose lists                       6 KB
    unsigned char st[K1_TILE];            // K1S_* bits
    unsigned char amb[K1_TILE];           // HL_CHECK_* bits inside the float32 band
    float env[K1_ENV_FLOATS];             // obstacle records | field-edge records | lane segments           4 KB
    float4 segd[HL_MAX_SEGS];             // per lane segment: ex, ey, 1/len^2, 1/len (derived once per staging)
    float4 fld[32][3];                    // per field edge, first pass: (Ax, Ay, Ex, Ey) with the endpoints
                                          // ordered so that Ey >= 0, (nx, ny, c, By), (tmin, tmax, -, -) -- see k1_field1
    unsigned long long bar_env, bar_raw;  // mbarriers of the two kinds of bulk copy
    int cnt[8];                           // list counters: la, lb, lc, pending, pairs
    float aabb[8];                        // field polygon: xmin, xmax, ymin, ymax; all obstacles: xmin, xmax, ymin, ymax
    K1Defer dq[K1_DEFER_CAP];             // poses waiting for the float64 predicates (drained when the CTA has no tile left)
    int dq_cnt;
};
enum { K1S_HIT = 1, K1S_INSIDE = 2, K1S_NOTCLEAR = 4, K1S_CORNERS = 8, K1S_DONE = 16, K1S_FAR = 32, K1S_OFF = 64, K1S_CUT = 128 };

struct K1Env {                            // staged environment (shared memory, uniform per CTA)
    const float* obs_a; const float* field_a; const float* seg_a; const float* segd_a; const float* fld_a;
    int n_obs, n_field, n_seg;
    float eps;
};

// Ambiguous poses of a warp are resolved one at a time by the WHOLE warp (warp_exact_part_check): the pose
// is broadcast with shuffles and the exact float64 predicate runs on 32 lanes.
__device__ __noinline__ void warp_resolve(bool need, double x, double y, double yaw, int env, const double* ext,
                                             unsigned amb, bool& bad, const EnvBatchDev& eb,
                                             unsigned long long* n_exact, int lane) {
    unsigned m = __ballot_sync(0xffffffffu, need);
    if (m && n_exact && lane == 0) atomicAdd(n_exact, (unsigned long long)__popc(m));
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        Pose64 p;
        p.x = __shfl_sync(0xffffffffu, x, src);
        p.y = __shfl_sync(0xffffffffu, y, src);
        const double byaw = __shfl_sync(0xffffffffu, yaw, src);
        p.c = cos(byaw); p.s = sin(byaw);
        double e4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) e4[k] = __shfl_sync(0xffffffffu, ext[k], src);
        const int be = __shfl_sync(0xffffffffu, env, src);
        const unsigned ba = __shfl_sync(0xffffffffu, amb, src);
        const bool res = warp_exact_part_check(p, e4, eb, eb.desc[be], ba, lane);
        if (lane == src) bad = res;
    }
}

// shared-memory fetch-and-add as ONE instruction (ATOMS.ADD): `atomicAdd` makes the compiler wrap its own warp
// aggregation (vote / popc / shuffle, ~15 instructions) around an atomic that one elected lane already issues alone
__device__ __forceinline__ int atoms_add(int* p, int v) {
    int old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(p)), "r"(v) : "memory");
    return old;
}

// appends q to the CTA list for every lane with `pred`: one shared atomic per warp
__device__ __forceinline__ void cta_append(unsigned short* list, int* cnt, bool pred, int q, int lane) {
    const unsigned m = __ballot_sync(0xffffffffu, pred);
    int base = 0;
    if (lane == 0 && m) base = atoms_add(cnt, __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (pred) list[base + __popc(m & ((1u << lane) - 1u))] = (unsigned short)q;
}

// pose of list entry q: px, py, cos, sin (the hardware sine / cosine of the reduced heading: abs. error 2^-21.4 in
// [-pi, pi], < 2e-6 m on a footprint corner, far inside the band eps)
__device__ __forceinline__ float4 k1_pose(const K1Cta& S, int q) {
    const float yr = S.yr[q];
    return make_float4(S.px[q], S.py[q], __cosf(yr), __sinf(yr));
}

// ------------------------------------------------------------------ filter stages (float32, staged environment)
// Same formulations and the same conservative band as filt_stage1 / filt_field2 / filt_lane (hl_geom.cuh), split so
// that every stage is a short uniform loop over shared-memory records.
struct K1Rect { float hx, hy, mx, my, x0, x1, y0, y1; };
__device__ __forceinline__ K1Rect k1_rect(const float* ext) {
    K1Rect R;
    R.hx = 0.5f * (ext[1] - ext[0]); R.hy = 0.5f * (ext[3] - ext[2]);
    R.mx = 0.5f * (ext[1] + ext[0]); R.my = 0.5f * (ext[3] + ext[2]);
    R.x0 = ext[0]; R.x1 = ext[1]; R.y0 = ext[2]; R.y1 = ext[3];
    return R;
}

// Stage A: rectangle centre against every capsule axis.  0 = the whole rectangle is inside one capsule,
// 1 = every point of it is outside every capsule (HIT), 2 = the corners decide.
__device__ __forceinline__ int k1_lane_centre(const K1Env& E, const K1Rect& R, float4 P, float rho) {
    const float Cx = fmaf(P.z, R.mx, fmaf(-P.w, R.my, P.x)), Cy = fmaf(P.w, R.mx, fmaf(P.z, R.my, P.y));
    const float rin = (float)HL_LANE_RIN - E.eps, rout = (float)HL_LANE_R + E.eps;
    bool accepted = false, need = false;
#pragma unroll 1
    for (int i = 0; i < E.n_seg; ++i) {
        const float4 sg = lds4(E.seg_a + 4 * i), sd = lds4(E.segd_a + 4 * i);
        const float qx = Cx - sg.x, qy = Cy - sg.y;
        const float t = fminf(fmaxf(fmaf(qx, sd.x, qy * sd.y) * sd.z, 0.f), 1.f);
        const float ddx = fmaf(-t, sd.x, qx), ddy = fmaf(-t, sd.y, qy);
        const float d = f_sqrt(fmaf(ddx, ddx, ddy * ddy));
        accepted |= d + rho <= rin;
        need |= d - rho <= rout;
    }
    return accepted ? 0 : (need ? 2 : 1);
}

// Stage B: rectangular obstacles, 4-axis box-box separating test on (centre, axis, half extents).
__device__ __forceinline__ void k1_obstacles(const K1Env& E, const K1Rect& R, float4 P, bool& hit, bool& amb) {
    const float c = P.z, s = P.w;
    const float Cx = fmaf(c, R.mx, fmaf(-s, R.my, P.x)), Cy = fmaf(s, R.mx, fmaf(c, R.my, P.y));
    hit = false; amb = false;
    K1_UNROLL(K1_UNROLL_OBS)
    for (int k = 0; k < E.n_obs; ++k) {
        const float4 b0 = lds4(E.obs_a + HL_OBS32_STRIDE * k + 20);      // flag, cx, cy, ax
        const float4 b1 = lds4(E.obs_a + HL_OBS32_STRIDE * k + 24);      // ay, ha, hb, pad
        const float dx = b0.y - Cx, dy = b0.z - Cy;
        const float ax = b0.w, ay = b1.x, ha = b1.y, hb = b1.z;
        const float p = fabsf(fmaf(ax, c, ay * s)), q = fabsf(fmaf(ay, c, -ax * s));
        const float du = fabsf(fmaf(dx, c, dy * s)), dv = fabsf(fmaf(dy, c, -dx * s));
        const float da = fabsf(fmaf(dx, ax, dy * ay)), db = fabsf(fmaf(dy, ax, -dx * ay));
        const float sep = fmaxf(fmaxf(du - fmaf(ha, p, fmaf(hb, q, R.hx)), dv - fmaf(ha, q, fmaf(hb, p, R.hy))),
                                fmaxf(da - fmaf(R.hx, p, fmaf(R.hy, q, ha)), db - fmaf(R.hx, q, fmaf(R.hy, p, hb))));
        hit |= sep < -E.eps;
        amb |= fabsf(sep) <= E.eps;
    }
}

// Stage C: one pass over the field edges -- crossing parity of the centre + mask of the edges whose LINE passes
// within the circumradius of the rectangle (the support-radius refinement of those few edges is stage D's first
// test).  Branch-free: 2 LDS.128 + ~17 ALU instructions per edge.  The derived records have the endpoints ordered
// by y (Ey >= 0), so the crossing rule is one comparison; the straddle test uses the very same float values for a
// vertex in both of its edges, which keeps the half-open rule consistent.
__device__ __forceinline__ void k1_field1(const K1Env& E, const K1Rect& R, float4 P, float rho_eps,
                                          unsigned& near_mask, bool& inside) {
    const float c = P.z, s = P.w;
    const float Cx = fmaf(c, R.mx, fmaf(-s, R.my, P.x)), Cy = fmaf(s, R.mx, fmaf(c, R.my, P.y));
    unsigned nm = 0, par = 0;
    K1_UNROLL(K1_UNROLL_FLD)
    for (int i = 0; i < E.n_field; ++i) {
        const float4 f0 = lds4(E.fld_a + 12 * i);         // Ax, Ay, Ex, Ey   (Ay <= By)
        const float4 f1 = lds4(E.fld_a + 12 * i + 4);     // nx, ny, c, By
        const float2 f2 = *reinterpret_cast<const float2*>(E.fld_a + 12 * i + 8);   // extent of the edge along its direction
        const float lhs = (Cx - f0.x) * f0.w, rhs = f0.z * (Cy - f0.y);
        par ^= (unsigned)(!(f0.y > Cy) && (f1.w > Cy) && (lhs < rhs));
        const float sd = fmaf(f1.x, Cx, fmaf(f1.y, Cy, -f1.z));
        const float ct = fmaf(-f1.y, Cx, f1.x * Cy);
        // near = the circumcircle of the rectangle reaches the edge's line AND overlaps the edge's extent along it (a
        // field boundary is mostly runs of collinear edges: the line test alone flags the whole run)
        nm |= (unsigned)(!(fabsf(sd) > rho_eps) && !(ct - rho_eps > f2.y) && !(ct + rho_eps < f2.x)) << i;
    }
    near_mask = nm; inside = par != 0;
}

// Stage D: the nearby edges of one pose (support radius along the normal, extent along the edge, Liang-Barsky
// against the shrunken rectangle), then the field verdict.  Returns HL_HIT / HL_FREE / HL_AMBIG.
__device__ __forceinline__ int k1_field2(const K1Env& E, const K1Rect& R, float4 P, unsigned near_mask, bool inside) {
    const float eps = E.eps;
    const float px = P.x, py = P.y, c = P.z, s = P.w;
    const float Cx = fmaf(c, R.mx, fmaf(-s, R.my, px)), Cy = fmaf(s, R.mx, fmaf(c, R.my, py));
    bool all_clear = true, cut = false;
#pragma unroll 1
    while (near_mask) {
        const int i = __ffs(near_mask) - 1;
        near_mask &= near_mask - 1;
        const float4 r0 = lds4(E.field_a + HL_FIELD32_STRIDE * i);        // Ax, Ay, Ex, Ey
        const float4 r1 = lds4(E.field_a + HL_FIELD32_STRIDE * i + 4);    // nx, ny, c, By
        const float4 r2 = lds4(E.field_a + HL_FIELD32_STRIDE * i + 8);    // t.A, t.B
        const float Ax = r0.x, Ay = r0.y, Bx = Ax + r0.z, By = r1.w, nx = r1.x, ny = r1.y;
        const float nu = fmaf(nx, c, ny * s), nv = fmaf(ny, c, -nx * s);
        const float sd = fmaf(nx, Cx, fmaf(ny, Cy, -r1.z));                  // signed distance of the centre to the line
        if (fabsf(sd) > fmaf(R.hx, fabsf(nu), R.hy * fabsf(nv)) + eps) continue;   // clear by the support radius along n
        const float ct = fmaf(-ny, Cx, nx * Cy);
        const float rt = fmaf(R.hx, fabsf(nv), R.hy * fabsf(nu));
        if (ct - rt > fmaxf(r2.x, r2.y) + eps || ct + rt < fminf(r2.x, r2.y) - eps) continue;
        const float dxa = Ax - px, dya = Ay - py, dxb = Bx - px, dyb = By - py;
        const float ua = fmaf(c, dxa, s * dya), wa = fmaf(c, dya, -s * dxa);
        const float ub = fmaf(c, dxb, s * dyb), wb = fmaf(c, dyb, -s * dxb);
        if ((fminf(ua, ub) > R.x1 + eps) || (fmaxf(ua, ub) < R.x0 - eps) ||
            (fminf(wa, wb) > R.y1 + eps) || (fmaxf(wa, wb) < R.y0 - eps)) continue;
        all_clear = false;
        float t0 = 0.f, t1 = 1.f;
        bool dead = false;
        const float a2[2] = {ua, wa}, d2v[2] = {ub - ua, wb - wa};
        const float lo2[2] = {R.x0 + eps, R.y0 + eps}, hi2[2] = {R.x1 - eps, R.y1 - eps};
#pragma unroll
        for (int ax = 0; ax < 2; ++ax) {
            if (fabsf(d2v[ax]) < 1e-12f) {
                if (a2[ax] <= lo2[ax] || a2[ax] >= hi2[ax]) dead = true;
            } else {
                const float inv = f_rcp(d2v[ax]);
                const float tl = (lo2[ax] - a2[ax]) * inv, th = (hi2[ax] - a2[ax]) * inv;
                t0 = fmaxf(t0, fminf(tl, th));
                t1 = fminf(t1, fmaxf(tl, th));
            }
        }
        if (!dead && (t1 - t0) * f_sqrt(fmaf(d2v[0], d2v[0], d2v[1] * d2v[1])) > 8.0f * eps) { cut = true; break; }
    }
    if (cut) return HL_HIT;
    if (all_clear) return inside ? HL_FREE : HL_HIT;
    return HL_AMBIG;
}

// Stage D, pair form: ONE nearby edge of one pose (the body of k1_field2's loop).  0 = the edge is clear of the rectangle,
// 1 = not certified clear, 2 = the edge definitely cuts the rectangle.
__device__ __forceinline__ int k1_field_pair(const K1Env& E, const K1Rect& R, float4 P, int i) {
    const float eps = E.eps;
    const float px = P.x, py = P.y, c = P.z, s = P.w;
    const float Cx = fmaf(c, R.mx, fmaf(-s, R.my, px)), Cy = fmaf(s, R.mx, fmaf(c, R.my, py));
    const float4 r0 = lds4(E.field_a + HL_FIELD32_STRIDE * i);        // Ax, Ay, Ex, Ey
    const float4 r1 = lds4(E.field_a + HL_FIELD32_STRIDE * i + 4);    // nx, ny, c, By
    const float4 r2 = lds4(E.field_a + HL_FIELD32_STRIDE * i + 8);    // t.A, t.B
    const float Ax = r0.x, Ay = r0.y, Bx = Ax + r0.z, By = r1.w, nx = r1.x, ny = r1.y;
    const float nu = fmaf(nx, c, ny * s), nv = fmaf(ny, c, -nx * s);
    const float sd = fmaf(nx, Cx, fmaf(ny, Cy, -r1.z));
    if (fabsf(sd) > fmaf(R.hx, fabsf(nu), R.hy * fabsf(nv)) + eps) return 0;
    const float ct = fmaf(-ny, Cx, nx * Cy);
    const float rt = fmaf(R.hx, fabsf(nv), R.hy * fabsf(nu));
    if (ct - rt > fmaxf(r2.x, r2.y) + eps || ct + rt < fminf(r2.x, r2.y) - eps) return 0;
    const float dxa = Ax - px, dya = Ay - py, dxb = Bx - px, dyb = By - py;
    const float ua = fmaf(c, dxa, s * dya), wa = fmaf(c, dya, -s * dxa);
    const float ub = fmaf(c, dxb, s * dyb), wb = fmaf(c, dyb, -s * dxb);
    if ((fminf(ua, ub) > R.x1 + eps) || (fmaxf(ua, ub) < R.x0 - eps) ||
        (fminf(wa, wb) > R.y1 + eps) || (fmaxf(wa, wb) < R.y0 - eps)) return 0;
    float t0 = 0.f, t1 = 1.f;
    bool dead = false;
    const float a2[2] = {ua, wa}, d2v[2] = {ub - ua, wb - wa};
    const float lo2[2] = {R.x0 + eps, R.y0 + eps}, hi2[2] = {R.x1 - eps, R.y1 - eps};
#pragma unroll
    for (int ax = 0; ax < 2; ++ax) {
        if (fabsf(d2v[ax]) < 1e-12f) {
            if (a2[ax] <= lo2[ax] || a2[ax] >= hi2[ax]) dead = true;
        } else {
            const float inv = f_rcp(d2v[ax]);
            const float tl = (lo2[ax] - a2[ax]) * inv, th = (hi2[ax] - a2[ax]) * inv;
            t0 = fmaxf(t0, fminf(tl, th));
            t1 = fminf(t1, fmaxf(tl, th));
        }
    }
    if (!dead && (t1 - t0) * f_sqrt(fmaf(d2v[0], d2v[0], d2v[1] * d2v[1])) > 8.0f * eps) return 2;
    return 1;
}

// corner_in_capsule (hl_geom.cuh) on the staged segment + its derived record
__device__ __forceinline__ int k1_corner_in_capsule(float4 sg, float4 sd, float wx, float wy, float eps) {
    const float ex = sd.x, ey = sd.y;
    const float qx = wx - sg.x, qy = wy - sg.y;
    const float tt = fmaf(qx, ex, qy * ey) * sd.z;
    const float t = fminf(fmaxf(tt, 0.f), 1.f);
    const float ddx = fmaf(-t, ex, qx), ddy = fmaf(-t, ey, qy);
    const float d2 = fmaf(ddx, ddx, ddy * ddy);
    const float rin = (float)HL_LANE_RIN - eps, rout = (float)HL_LANE_R + eps;
    if (d2 <= rin * rin) return 1;
    if (d2 > rout * rout) return 0;
    float g = f_sqrt(d2);
    if (tt < 0.f || tt > 1.f) {                                 // cap: chord fan of the GEOS buffer polygon
        const float il = sd.w;
        const float along = fabsf(fmaf(ddx, ex, ddy * ey)) * il, across = fabsf(fmaf(ddy, ex, -ddx * ey)) * il;
        const float phi = atan2f(across, along);
        const float q = 1.5707963267948966f - phi;
        const float step = 0.09817477042468103f;                // pi/32
        const float k = floorf(q / step);
        const float delta = fabsf(q - (k + 0.5f) * step);
        g = g * cosf(delta) * 1.0012061467251643f;              // / cos(pi/64)
    }
    if (g <= (float)HL_LANE_R - eps) return 1;
    if (g > (float)HL_LANE_R + eps) return 0;
    return 2;
}

// Stage E: the four corners against every capsule polygon, then the piecewise cover certificate.
// Returns HL_HIT, HL_FREE, or HL_AMBIG (cover not certified in float32).
__device__ __forceinline__ int k1_lane_corners(const K1Env& E, const K1Rect& R, float4 P) {
    const float eps = E.eps;
    const float px = P.x, py = P.y, c = P.z, s = P.w;
    const float rin = (float)HL_LANE_RIN - eps;
    float rx[4], ry[4];
    const float lx[4] = {R.x0, R.x0, R.x1, R.x1};
    const float ly[4] = {R.y1, R.y0, R.y0, R.y1};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        rx[j] = fmaf(c, lx[j], fmaf(-s, ly[j], px));
        ry[j] = fmaf(s, lx[j], fmaf(c, ly[j], py));
    }
    bool one_holds_all = false;
    unsigned maybe = 0;
#pragma unroll 1
    for (int i = 0; i < E.n_seg; ++i) {
        const float4 sg = lds4(E.seg_a + 4 * i), sd = lds4(E.segd_a + 4 * i);
        bool all_in = true;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int st = k1_corner_in_capsule(sg, sd, rx[j], ry[j], eps);
            all_in = all_in && (st == 1);
            if (st != 0) maybe |= 1u << j;
        }
        if (all_in) one_holds_all = true;
    }
    if (one_holds_all) return HL_FREE;
    if (maybe != 0xFu) return HL_HIT;
    unsigned prev = 0;
    bool covered = true;
#pragma unroll 1
    for (int q = 0; q <= 4 && covered; ++q) {
        const float lxq = R.x0 + 0.25f * (float)q * (R.x1 - R.x0);
        unsigned m = 0xFFFFu;
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const float lyq = side ? R.y1 : R.y0;
            const float wx = fmaf(c, lxq, fmaf(-s, lyq, px)), wy = fmaf(s, lxq, fmaf(c, lyq, py));
            unsigned in = 0;
            for (int i = 0; i < E.n_seg; ++i) {
                const float4 sg = lds4(E.seg_a + 4 * i), sd = lds4(E.segd_a + 4 * i);
                const float qx = wx - sg.x, qy = wy - sg.y;
                const float t = fminf(fmaxf(fmaf(qx, sd.x, qy * sd.y) * sd.z, 0.f), 1.f);
                const float ddx = fmaf(-t, sd.x, qx), ddy = fmaf(-t, sd.y, qy);
                if (fmaf(ddx, ddx, ddy * ddy) <= rin * rin) in |= 1u << i;
            }
            m &= in;
        }
        if (q > 0 && (prev & m) == 0) covered = false;
        prev = m;
    }
    return covered ? HL_FREE : HL_AMBIG;
}

// Monolithic per-pose filter on global memory for slices the staged pipeline cannot take.
__device__ __noinline__ void k1_slow_slice(const EnvBatchDev& eb, const int32_t* env_id, const double* poses,
                                           const int32_t* pose_idx, long long n, long long base, unsigned flags,
                                           uint8_t* out, unsigned long long* n_exact, int lane) {
    for (int j = 0; j < (K1_SLICE / 32); ++j) {
        const long long i = base + j * 32 + lane;
        const bool active = i < n;
        const int e = active ? (env_id ? env_id[i] : 0) : 0;
        const EnvDesc& D = eb.desc[e];
        EnvSmem E;
        global_env(eb, D, E);
        double x = 0.0, y = 0.0, yaw = 0.0;
        if (active) { x = poses[3 * i]; y = poses[3 * i + 1]; yaw = poses[3 * i + 2]; }
        const bool with_aux = active && (pose_idx ? ((pose_idx[i] & 1) == 0) : true);
        const float px = (float)(x - D.origin[0]), py = (float)(y - D.origin[1]);
        const bool beyond = fabsf(px) > E.reach || fabsf(py) > E.reach;
        const bool far = !beyond && (!(fabs(yaw) < 1e6) || !(px == px) || !(py == py));
        float sf, cf;
        sincosf((float)yaw, &sf, &cf);
        bool bad = false;
        unsigned amb = flags;
        int r = HL_FREE;
        if (active) r = beyond ? far_status(flags, E.n_seg) : (far ? HL_AMBIG : filter_part(E, px, py, cf, sf, E.ext, flags, &amb));
        if (r == HL_HIT) bad = true;
        warp_resolve(r == HL_AMBIG, x, y, yaw, e, D.body_ext, amb, bad, eb, n_exact, lane);
        if (flags & HL_CHECK_AUX) {
            const unsigned aflags = flags & (HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY);
            const int na = (active && with_aux && !beyond) ? D.n_aux : 0;
            int na_max = na;
            for (int o = 16; o; o >>= 1) na_max = max(na_max, __shfl_xor_sync(0xffffffffu, na_max, o));
            for (int a = 0; a < na_max; ++a) {
                const bool mine = a < na && !bad;
                const double* ext64 = eb.aux64 + 4 * (size_t)(D.aux_off + (a < D.n_aux ? a : 0));
                unsigned amb2 = aflags;
                int r2 = HL_FREE;
                if (mine) {
                    float ext32[4] = {(float)ext64[0], (float)ext64[1], (float)ext64[2], (float)ext64[3]};
                    r2 = far ? HL_AMBIG : filter_part(E, px, py, cf, sf, ext32, aflags, &amb2);
                    if (r2 == HL_HIT) bad = true;
                }
                bool bad2 = false;
                warp_resolve(r2 == HL_AMBIG, x, y, yaw, e, D.n_aux > 0 ? ext64 : D.body_ext, amb2, bad2, eb, n_exact, lane);
                bad = bad || bad2;
            }
        }
        if (active) out[i] = bad ? 1 : 0;
    }
}

__global__ void __launch_bounds__(K1_THREADS, K1_MIN_CTAS)
k_collision(EnvBatchDev eb, const int32_t* __restrict__ env_id, const double* __restrict__ poses,
            const int32_t* __restrict__ pose_idx, long long n, unsigned flags,
            uint8_t* __restrict__ out, unsigned long long* n_exact, int use_tma) {
    extern __shared__ __align__(16) unsigned char k1_smem[];
    K1Cta& S = *reinterpret_cast<K1Cta*>(k1_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned rbar = smem_u32(&S.bar_raw), ebar = smem_u32(&S.bar_env);
    const long long n_tiles = (n + K1_TILE - 1) / K1_TILE;
    if (tid == 0) { mbar_init(rbar, 1); mbar_init(ebar, 1); S.dq_cnt = 0; }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    unsigned rphase = 0, ephase = 0;
    int staged_env = -1;
    bool env_ok = false;                               // staged environment usable by the pipeline
    K1Env E;
    E.obs_a = E.field_a = E.seg_a = S.env; E.segd_a = reinterpret_cast<const float*>(S.segd);
    E.fld_a = reinterpret_cast<const float*>(S.fld);
    E.n_obs = E.n_field = E.n_seg = 0; E.eps = 0.f;

    // does `tile` arrive by TMA?  (full tile, 16-byte aligned source)
    auto tile_tma = [&](long long tile) -> bool { return use_tma && tile < n_tiles && (tile + 1) * K1_TILE <= n; };
    auto issue_tile = [&](long long tile) {
        if (tid == 0 && tile_tma(tile)) {
            mbar_expect_tx(rbar, K1_TILE * 24);
            bulk_g2s(smem_u32(S.raw), poses + 3 * tile * K1_TILE, K1_TILE * 24, rbar);
        }
    };
    // The queued float64 resolutions, one entry per warp at a time.  Called by all threads of the CTA (between two
    // tiles: after the verdict store of the tile that queued the entries, so a drained "hit" lands on top of it).
    auto drain_queue = [&]() {
        const int nq = min(S.dq_cnt, K1_DEFER_CAP);
#pragma unroll 1
        for (int e = warp; e < nq; e += K1_WARPS) {
            const K1Defer d = S.dq[e];
            const EnvDesc& D = eb.desc[d.env];
            const double* ext64 = d.rect == 0 ? D.body_ext : eb.aux64 + 4 * (size_t)(D.aux_off + d.rect - 1);
            Pose64 p;
            p.x = poses[3 * d.i]; p.y = poses[3 * d.i + 1];
            const double yaw = poses[3 * d.i + 2];
            p.c = cos(yaw); p.s = sin(yaw);
            double e4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) e4[k] = ext64[k];
            const bool res = warp_exact_part_check(p, e4, eb, D, d.amb, lane);
            if (lane == 0) {
                if (res) out[d.i] = 1;
                if (n_exact) atomicAdd(n_exact, 1ULL);
            }
        }
    };
    issue_tile(blockIdx.x);

    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = tile * K1_TILE;
        // ---- environment of the tile (CTA-uniform): staged by bulk copies when it changes
        const int e0 = env_id ? env_id[base] : 0;
        if (e0 != staged_env) {
            __syncthreads();                           // nobody still reads the previous environment
            const EnvDesc& D0 = eb.desc[e0];
            const int n_o = D0.n_obs * HL_OBS32_STRIDE, n_f = D0.n_field * HL_FIELD32_STRIDE, n_s = D0.n_seg * 4;
            env_ok = (n_o + n_f + n_s <= K1_ENV_FLOATS) && D0.all_rect && D0.n_seg <= HL_MAX_SEGS && D0.n_field <= 32;
            if (env_ok) {
                if (tid == 0) {
                    fence_proxy_async();
                    const unsigned bytes = 4u * (unsigned)(n_o + n_f + n_s);
                    if (bytes) {
                        mbar_expect_tx(ebar, bytes);
                        if (n_o) bulk_g2s(smem_u32(S.env), eb.obs32 + (size_t)HL_OBS32_STRIDE * D0.obs_off, 4u * n_o, ebar);
                        if (n_f) bulk_g2s(smem_u32(S.env + n_o), eb.field32 + (size_t)HL_FIELD32_STRIDE * D0.field_off, 4u * n_f, ebar);
                        if (n_s) bulk_g2s(smem_u32(S.env + n_o + n_f), eb.seg32 + 4 * (size_t)D0.seg_off, 4u * n_s, ebar);
                    }
                }
                if (n_o + n_f + n_s) { mbar_wait(ebar, ephase); ephase ^= 1u; }
                if (tid < D0.n_seg) {                  // derived per-segment record: ex, ey, 1/len^2, 1/len
                    const float* sg = S.env + n_o + n_f + 4 * tid;
                    const float ex = sg[2] - sg[0], ey = sg[3] - sg[1];
                    const float len2 = fmaf(ex, ex, ey * ey);
                    S.segd[tid] = make_float4(ex, ey, f_rcp(len2), rsqrtf(len2));
                }
                if (tid >= 32 && tid < 32 + D0.n_field) {     // first-pass field records, endpoints ordered by y
                    const int i = tid - 32;
                    const float* e = S.env + n_o + HL_FIELD32_STRIDE * i;
                    const bool up = !(e[1] > e[7]);                    // Ay <= By
                    S.fld[i][0] = up ? make_float4(e[0], e[1], e[2], e[3]) : make_float4(e[0] + e[2], e[7], -e[2], -e[3]);
                    S.fld[i][1] = make_float4(e[4], e[5], e[6], up ? e[7] : e[1]);
                    S.fld[i][2] = make_float4(fminf(e[8], e[9]), fmaxf(e[8], e[9]), 0.f, 0.f);
                }
                if (warp == 2) {                       // bounding boxes of the field polygon and of all obstacles
                    float lo_x = INFINITY, hi_x = -INFINITY, lo_y = INFINITY, hi_y = -INFINITY;
                    for (int i = lane; i < D0.n_field; i += 32) {
                        const float* e = S.env + n_o + HL_FIELD32_STRIDE * i;
                        lo_x = fminf(lo_x, e[0]); hi_x = fmaxf(hi_x, e[0]); lo_y = fminf(lo_y, e[1]); hi_y = fmaxf(hi_y, e[1]);
                    }
                    float olo_x = INFINITY, ohi_x = -INFINITY, olo_y = INFINITY, ohi_y = -INFINITY;
                    for (int i = lane; i < 4 * D0.n_obs; i += 32) {
                        const float* v = S.env + HL_OBS32_STRIDE * (i >> 2) + 2 * (i & 3);
                        olo_x = fminf(olo_x, v[0]); ohi_x = fmaxf(ohi_x, v[0]); olo_y = fminf(olo_y, v[1]); ohi_y = fmaxf(ohi_y, v[1]);
                    }
#pragma unroll
                    for (int o = 16; o; o >>= 1) {
                        lo_x = fminf(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, o)); hi_x = fmaxf(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, o));
                        lo_y = fminf(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, o)); hi_y = fmaxf(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, o));
                        olo_x = fminf(olo_x, __shfl_xor_sync(0xffffffffu, olo_x, o)); ohi_x = fmaxf(ohi_x, __shfl_xor_sync(0xffffffffu, ohi_x, o));
                        olo_y = fminf(olo_y, __shfl_xor_sync(0xffffffffu, olo_y, o)); ohi_y = fmaxf(ohi_y, __shfl_xor_sync(0xffffffffu, ohi_y, o));
                    }
                    if (lane == 0) {
                        S.aabb[0] = lo_x; S.aabb[1] = hi_x; S.aabb[2] = lo_y; S.aabb[3] = hi_y;
                        S.aabb[4] = olo_x; S.aabb[5] = ohi_x; S.aabb[6] = olo_y; S.aabb[7] = ohi_y;
                    }
                }
                E.obs_a = S.env; E.field_a = S.env + n_o; E.seg_a = S.env + n_o + n_f;
                E.n_obs = D0.n_obs; E.n_field = D0.n_field; E.n_seg = D0.n_seg; E.eps = D0.eps;
            }
            staged_env = e0;
        }
        const EnvDesc& D = eb.desc[e0];
        const bool tma = tile_tma(tile);
        if (tid < 8) S.cnt[tid] = 0;
        if (tma) { mbar_wait(rbar, rphase); rphase ^= 1u; }
        // ---- stage 0: poses -> float32 frame; is the whole tile in the staged environment?
        bool same_env = env_ok;
        {
            const double ox = D.origin[0], oy = D.origin[1];
            const float reach = D.reach;
#pragma unroll 1
            for (int j = 0; j < K1_PER_THREAD; ++j) {
                const int q = j * K1_THREADS + tid;
                const long long i = base + q;
                const bool active = i < n;
                double x = 0.0, y = 0.0, yaw = 0.0;
                if (active) {
                    if (tma) { x = S.raw[3 * q]; y = S.raw[3 * q + 1]; yaw = S.raw[3 * q + 2]; }
                    else { x = poses[3 * i]; y = poses[3 * i + 1]; yaw = poses[3 * i + 2]; }
                    if (env_id && env_id[i] != e0) same_env = false;
                }
                const float px = (float)(x - ox), py = (float)(y - oy);
                const bool beyond = fabsf(px) > reach || fabsf(py) > reach;
                const bool far = !beyond && (!(fabs(yaw) < 1e6) || !(px == px) || !(py == py));
                // the heading is reduced to [-pi, pi] in float64 (exact enough for any |yaw| < 1e6)
                const double kk = rint(yaw * 0.15915494309189535);
                S.px[q] = px; S.py[q] = py; S.yr[q] = (float)fma(-kk, 6.283185307179586, yaw);
                unsigned char st = 0;
                if (!active) st = K1S_OFF | K1S_DONE;
                else if (beyond) st = K1S_DONE | (far_status(flags, D.n_seg) == HL_HIT ? K1S_HIT : 0) | K1S_OFF;   // no aux test either
                else if (far) st = K1S_FAR;
                S.st[q] = st;
                S.amb[q] = 0;
            }
        }
        same_env = __syncthreads_and(same_env);        // also: every read of the landing zone is done
        if (tid == 0) fence_proxy_async();
        issue_tile(tile + gridDim.x);                  // fetch the next tile behind the filter stages
        if (!same_env) {
            k1_slow_slice(eb, env_id, poses, pose_idx, n, base + (long long)warp * K1_SLICE, flags, out, n_exact, lane);
            continue;
        }
        // ---- rectangles of the footprint: 0 = body (obstacles, field, lane), 1.. = implement rectangles (obstacles +
        // field polygon, never the lane, poses 0,2,4,.. of a path: orchard_geometry_environment.py:439-456,
        // car_model.py:58).  ONE instance of the stage code serves all of them.
        const int n_rect = ((flags & HL_CHECK_AUX) ? D.n_aux : 0) + 1;
#pragma unroll 1
        for (int rect = 0; rect < n_rect; ++rect) {
            const double* ext64 = rect == 0 ? D.body_ext : eb.aux64 + 4 * (size_t)(D.aux_off + rect - 1);
            float ext[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) ext[k] = (float)ext64[k];
            const K1Rect R = k1_rect(ext);
            const unsigned rflags = rect == 0 ? flags : (flags & (HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY));
            const bool do_lane = rect == 0 && (flags & HL_CHECK_LANE) && E.n_seg > 0;
            const float rho = sqrtf(fmaf(R.hx, R.hx, R.hy * R.hy));
            const float rho_eps = rho + E.eps;
            // ---- stage A: input lists.  Two bounding-box culls on the rectangle centre come first: a centre outside the
            // box of the field polygon is outside the polygon (HIT, 4 comparisons instead of lane + obstacle + field
            // stages); a centre farther than the circumradius from the box of all obstacles cannot touch any of them and
            // goes straight to the obstacle stage's OUTPUT list.  Body: then the lane centre test (decides every pose far
            // from the guide).  Implement: live poses at even path indices.
            const bool cull_f = (rflags & HL_CHECK_BOUNDARY) && E.n_field > 0, cull_o = (rflags & HL_CHECK_OBSTACLES) != 0;
            const float fx0 = S.aabb[0] - E.eps, fx1 = S.aabb[1] + E.eps, fy0 = S.aabb[2] - E.eps, fy1 = S.aabb[3] + E.eps;
            const float ox0 = S.aabb[4] - rho_eps, ox1 = S.aabb[5] + rho_eps, oy0 = S.aabb[6] - rho_eps, oy1 = S.aabb[7] + rho_eps;
#pragma unroll 1
            for (int j = 0; j < K1_PER_THREAD; ++j) {
                const int q = j * K1_THREADS + tid;
                unsigned char st = S.st[q];
                bool live = !(st & (K1S_DONE | K1S_FAR));
                if (rect > 0) {
                    const bool with_aux = !(st & (K1S_DONE | K1S_OFF)) && (pose_idx ? ((pose_idx[base + q] & 1) == 0) : true);
                    live = live && with_aux;
                    S.amb[q] = (with_aux && (st & K1S_FAR)) ? (unsigned char)rflags : (unsigned char)0;
                }
                bool skip_obs = false;
                if (live) {
                    const float4 P = k1_pose(S, q);
                    const float Cx = fmaf(P.z, R.mx, fmaf(-P.w, R.my, P.x)), Cy = fmaf(P.w, R.mx, fmaf(P.z, R.my, P.y));
                    if (cull_f && (Cx < fx0 || Cx > fx1 || Cy < fy0 || Cy > fy1)) { st |= K1S_HIT; live = false; }
                    else {
                        skip_obs = cull_o && (Cx < ox0 || Cx > ox1 || Cy < oy0 || Cy > oy1);
                        if (do_lane) {
                            const int r = k1_lane_centre(E, R, P, rho);
                            if (r == 1) { st |= K1S_HIT; live = false; }
                            else if (r == 2) st |= K1S_CORNERS;
                        }
                    }
                    S.st[q] = st;
                }
                cta_append(S.la, &S.cnt[0], live && !skip_obs, q, lane);
                if (cull_o) cta_append(S.lb, &S.cnt[1], live && skip_obs, q, lane);
            }
            __syncthreads();
            const int n_a = S.cnt[0];
            // ---- stage B: obstacles (la -> lb)
            int n_b = n_a;
            const unsigned short* lb = S.la;
            if (rflags & HL_CHECK_OBSTACLES) {
#pragma unroll 1
                for (int k = warp * 32; k < n_a; k += K1_THREADS) {
                    const int idx = k + lane;
                    const bool v = idx < n_a;
                    const int q = v ? S.la[idx] : 0;
                    bool hit = false, amb = false;
                    if (v) {
                        k1_obstacles(E, R, k1_pose(S, q), hit, amb);
                        if (hit) S.st[q] |= K1S_HIT;
                        else if (amb) S.amb[q] |= HL_CHECK_OBSTACLES;
                    }
                    cta_append(S.lb, &S.cnt[1], v && !hit, q, lane);
                }
                __syncthreads();
                n_b = S.cnt[1];
                lb = S.lb;
            }
            // ---- stages C + D: field polygon.  C: one pass over the edges per pose (crossing parity + mask of the edges
            // whose line passes nearby); poses without nearby edges are decided, the others go to `pend` and emit one
            // (pose, edge) PAIR per nearby edge.  D: the pairs, one per lane -- dense warps and one short uniform body
            // instead of a divergent per-pose loop over 1..8 edges (it was 17 % of the kernel's instructions).
            int n_c = n_b, n_d = 0;
            const unsigned short* lc = lb;
            const unsigned short* pend = nullptr;
            if (rflags & HL_CHECK_BOUNDARY) {
                unsigned short* pendw = (lb == S.la) ? S.lb : S.la;
#pragma unroll 1
                for (int k = warp * 32; k < n_b; k += K1_THREADS) {
                    const int idx = k + lane;
                    const bool v = idx < n_b;
                    const int q = v ? lb[idx] : 0;
                    bool keep = false, need2 = false;
                    unsigned nm = 0;
                    if (v) {
                        bool inside;
                        k1_field1(E, R, k1_pose(S, q), rho_eps, nm, inside);
                        if (nm == 0) {                            // every edge clear: the parity of the centre decides
                            if (inside) keep = true; else S.st[q] |= K1S_HIT;
                        } else {
                            need2 = true;
                            S.st[q] = (unsigned char)((S.st[q] & ~(K1S_INSIDE | K1S_NOTCLEAR | K1S_CUT)) | (inside ? K1S_INSIDE : 0));
                        }
                    }
                    cta_append(S.lc, &S.cnt[2], keep, q, lane);
                    cta_append(pendw, &S.cnt[3], need2, q, lane);
                    // pairs: warp prefix sum of the edge counts, one shared atomic per warp
                    const int c = __popc(nm);
                    int incl = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
                    const int total = __shfl_sync(0xffffffffu, incl, 31);
                    if (total) {
                        int base = 0;
                        if (lane == 0) base = atoms_add(&S.cnt[4], total);
                        base = __shfl_sync(0xffffffffu, base, 0) + incl - c;
                        if (c) {
                            if (base + c > K1_PAIR_CAP) {             // list full: this pose goes to the float64 predicate
                                S.st[q] |= K1S_NOTCLEAR;
                            } else {
                                unsigned m = nm;
#pragma unroll 1
                                while (m) {
                                    const int i = __ffs(m) - 1;
                                    m &= m - 1;
                                    S.pairs[base++] = (unsigned short)(q | (i << K1_QBITS));
                                }
                            }
                        }
                    }
                }
                __syncthreads();
                n_d = S.cnt[3];
                const int n_p = min(S.cnt[4], K1_PAIR_CAP);
                unsigned* st32 = reinterpret_cast<unsigned*>(S.st);
#pragma unroll 1
                for (int k = warp * 32; k < n_p; k += K1_THREADS) {
                    const int idx = k + lane;
                    if (idx < n_p) {
                        const unsigned e = S.pairs[idx];
                        const int q = e & ((1u << K1_QBITS) - 1u), i = e >> K1_QBITS;
                        const int r = k1_field_pair(E, R, k1_pose(S, q), i);
                        if (r) atomicOr(st32 + (q >> 2), (unsigned)(r == 2 ? (K1S_CUT | K1S_NOTCLEAR) : K1S_NOTCLEAR) << (8 * (q & 3)));
                    }
                }
                __syncthreads();
                n_c = S.cnt[2];
                lc = S.lc;
                pend = pendw;
            }
            // ---- stage E: verdict of the pending poses (field), then the lane corners of the body survivors that need them
            {
                const int n_e = n_c + n_d;
#pragma unroll 1
                for (int k = warp * 32; k < n_e; k += K1_THREADS) {
                    const int idx = k + lane;
                    if (idx < n_e) {
                        const int q = idx < n_c ? lc[idx] : pend[idx - n_c];
                        unsigned char st = S.st[q];
                        if (idx >= n_c) {                         // field verdict: cut -> HIT; all clear -> parity; else band
                            if (st & K1S_CUT) st |= K1S_HIT;
                            else if (!(st & K1S_NOTCLEAR)) { if (!(st & K1S_INSIDE)) st |= K1S_HIT; }
                            else S.amb[q] |= HL_CHECK_BOUNDARY;
                            S.st[q] = st;
                        }
                        if (do_lane && !(st & K1S_HIT) && (st & K1S_CORNERS)) {
                            const int r = k1_lane_corners(E, R, k1_pose(S, q));
                            if (r == HL_HIT) S.st[q] |= K1S_HIT;
                            else if (r == HL_AMBIG) S.amb[q] |= HL_CHECK_LANE;
                        }
                    }
                }
            }
            __syncthreads();                               // every list and counter of this rectangle has been consumed
            if (tid < 8) S.cnt[tid] = 0;
            // ---- float64 resolution of this rectangle; then "infeasible" becomes K1S_DONE | K1S_HIT
#pragma unroll 1
            for (int j = 0; j < K1_PER_THREAD; ++j) {
                const int q = j * K1_THREADS + tid;
                unsigned char st = S.st[q];
                const unsigned amb = (rect == 0 && (st & K1S_FAR)) ? rflags : (unsigned)S.amb[q];
                bool need = !(st & (K1S_HIT | K1S_DONE)) && amb != 0;
                if (need) {                                  // queue it; resolved after the CTA's last tile
                    const int slot = atomicAdd(&S.dq_cnt, 1);
                    if (slot < K1_DEFER_CAP) {
                        K1Defer d;
                        d.i = base + q; d.env = e0; d.amb = amb; d.rect = rect; d.pad = 0;
                        S.dq[slot] = d;
                        need = false;
                    }
                }
                if (__any_sync(0xffffffffu, need)) {        // queue full (rare): resolve in place
                    const long long i = base + q;
                    double x = 0.0, y = 0.0, yaw = 0.0;
                    if (need) { x = poses[3 * i]; y = poses[3 * i + 1]; yaw = poses[3 * i + 2]; }
                    bool b2 = false;
                    warp_resolve(need, x, y, yaw, e0, ext64, amb, b2, eb, n_exact, lane);
                    if (b2) st |= K1S_HIT;
                }
                if (st & K1S_HIT) st |= K1S_DONE;
                S.st[q] = st;
                S.amb[q] = 0;
            }
            __syncthreads();
        }
        // ---- verdicts: 4 consecutive poses per thread, one 32-bit store when the output is aligned
        if (base + K1_TILE <= n && ((reinterpret_cast<uintptr_t>(out) & 3) == 0)) {
            const uchar4 s4 = *reinterpret_cast<const uchar4*>(&S.st[4 * tid]);
            uchar4 o4;
            o4.x = s4.x & K1S_HIT; o4.y = s4.y & K1S_HIT; o4.z = s4.z & K1S_HIT; o4.w = s4.w & K1S_HIT;
            *reinterpret_cast<uchar4*>(out + base + 4 * tid) = o4;
        } else {
#pragma unroll 1
            for (int j = 0; j < K1_PER_THREAD; ++j) {
                const long long i = base + j * K1_THREADS + tid;
                if (i < n) out[i] = (S.st[j * K1_THREADS + tid] & K1S_HIT) ? 1 : 0;
            }
        }
        __syncthreads();                                   // S.st / lists are rewritten by the next tile
    }
    // ---- what is still queued: one entry per warp at a time, every warp busy
    drain_queue();
}

__global__ void k_path_reduce(const uint8_t* __restrict__ pose_bad, const long long* __restrict__ path_start,
                              long long n_paths, uint8_t* __restrict__ path_bad) {
    // one warp per path: OR over its pose flags
    long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (warp >= n_paths) return;
    long long a = path_start[warp], b = path_start[warp + 1];
    int any = 0;
    for (long long i = a + lane; i < b; i += 32) any |= pose_bad[i];
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) path_bad[warp] = any ? 1 : 0;
}

extern "C" int hl_collision_check(hl_ctx* ctx, const hl_env_batch* envs, const int32_t* d_env_id,
                                  const double* d_poses, const int32_t* d_pose_idx, int64_t n,
                                  uint32_t flags, uint8_t* d_out, unsigned long long* d_n_exact,
                                  void* stream) {
    if (!ctx || !envs || !d_poses || !d_out || n < 0) { hl_set_error("hl_collision_check: bad arguments"); return 1; }
    if (n == 0) return 0;
    if (hl_enter(ctx, envs, d_out, "hl_collision_check")) return 1;
    const int smem_bytes = (int)sizeof(K1Cta);
    static_assert(sizeof(K1Cta) * K1_MIN_CTAS + 1024 * K1_MIN_CTAS <= 227 * 1024, "K1 shared memory exceeds the SM");
    HL_CUDA_OK(cudaFuncSetAttribute(k_collision, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    const long long tiles = (n + K1_TILE - 1) / K1_TILE;
#ifndef K1_GRID_MULT
#define K1_GRID_MULT 1                    // CTAs in the grid per resident CTA
#endif
    const long long cap = (long long)ctx->sm_count * K1_MIN_CTAS * K1_GRID_MULT;
    const int grid = (int)(tiles < cap ? tiles : cap);
    const int use_tma = (((uintptr_t)d_poses) & 15) == 0 ? 1 : 0;     // cp.async.bulk needs a 16-byte aligned source
    k_collision<<<grid, K1_THREADS, smem_bytes, (cudaStream_t)stream>>>(
        envs->dev, d_env_id, d_poses, d_pose_idx, (long long)n, flags, d_out, d_n_exact, use_tma);
    HL_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int hl_path_reduce(hl_ctx* ctx, const uint8_t* d_pose_bad, const int64_t* d_path_start,
                              int64_t n_paths, uint8_t* d_path_bad, void* stream) {
    if (!ctx || !d_pose_bad || !d_path_start || !d_path_bad || n_paths < 0) { hl_set_error("hl_path_reduce: bad arguments"); return 1; }
    if (n_paths == 0) return 0;
    if (hl_enter(ctx, nullptr, d_path_bad, "hl_path_reduce")) return 1;
    long long threads = n_paths * 32;
    int grid = (int)((threads + 255) / 256);
    k_path_reduce<<<grid, 256, 0, (cudaStream_t)stream>>>(d_pose_bad, (const long long*)d_path_start, n_paths, d_path_bad);
    HL_CUDA_OK(cudaGetLastError());
    return 0;
}
