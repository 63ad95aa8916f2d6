// hl_geom.cuh -- footprint predicates (device).
//
// Two tiers per predicate (DESIGN.md "Exactness"):
//   * float32 filter with a conservative band `eps`: answers FREE / HIT when the
//     separating margin is clear of the band, AMBIG otherwise;
//   * float64 exact predicate evaluated with one rounding per operation, the same
//     expression order as oracle/geometry.py -- the boolean the reference's GEOS
//     calls would give (orchard_geometry_environment.py:423-458,
//     reference_line_heuristic.py:105-118) restated for rectangles.
#pragma once
#include "hl_common.cuh"

enum { HL_FREE = 0, HL_HIT = 1, HL_AMBIG = 2 };

// A pose whose reference point is farther than EnvDesc.reach from the centre of the environment's bounding
// box (reach = half diagonal of all geometry + lane radius + footprint reach + margin, hl_env_upload) cannot
// touch an obstacle and lies wholly outside the field polygon and every lane capsule: no test needed.
// Long Reeds-Shepp words (hundreds of metres) produce thousands of such poses.
__device__ __forceinline__ int far_status(unsigned flags, int n_seg) {
    return ((flags & HL_CHECK_BOUNDARY) || ((flags & HL_CHECK_LANE) && n_seg > 0)) ? HL_HIT : HL_FREE;
}

#define HL_LANE_R 6.0
// 6*m_cos(pi/64): radius of the circle inscribed in the 16-segments-per-quadrant cap
#define HL_LANE_RIN 5.992771509254837
#define HL_BAND_IN (HL_LANE_RIN - 1e-6)
#define HL_BAND_OUT (HL_LANE_R + 1e-6)

struct Pose64 {
    double x, y, c, s;     // c, s = cos/m_sin(yaw) in float64
};

// ------------------------------------------------------------------- float64
__device__ __forceinline__ void exact_corners(const Pose64& p, const double* ext, double* cx, double* cy) {
    // vertex order (x0,y1),(x0,y0),(x1,y0),(x1,y1) -- car_model.py:102-119
    const double lx[4] = {ext[0], ext[0], ext[1], ext[1]};
    const double ly[4] = {ext[3], ext[2], ext[2], ext[3]};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        cx[k] = xadd(xsub(xmul(p.c, lx[k]), xmul(p.s, ly[k])), p.x);
        cy[k] = xadd(xadd(xmul(p.s, lx[k]), xmul(p.c, ly[k])), p.y);
    }
}

__device__ __forceinline__ void exact_local(const Pose64& p, double vx, double vy, double& u, double& w) {
    double dx = xsub(vx, p.x), dy = xsub(vy, p.y);
    u = xadd(xmul(p.c, dx), xmul(p.s, dy));
    w = xsub(xmul(p.c, dy), xmul(p.s, dx));
}

// closed rectangle meets closed convex quad (CCW), strict separation test
static __device__ bool exact_rect_hits_quad(const Pose64& p, const double* ext, const double* cx,
                                     const double* cy, const double* V) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int j = (i + 1) & 3;
        double ex = xsub(V[2 * j], V[2 * i]), ey = xsub(V[2 * j + 1], V[2 * i + 1]);
        double nx = ey, ny = -ex;
        double m = INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double d = xadd(xmul(nx, xsub(cx[k], V[2 * i])), xmul(ny, xsub(cy[k], V[2 * i + 1])));
            m = fmin(m, d);
        }
        if (m > 0.0) return false;
    }
    double umin = INFINITY, umax = -INFINITY, wmin = INFINITY, wmax = -INFINITY;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        double u, w;
        exact_local(p, V[2 * v], V[2 * v + 1], u, w);
        umin = fmin(umin, u); umax = fmax(umax, u);
        wmin = fmin(wmin, w); wmax = fmax(wmax, w);
    }
    if (umin > ext[1] || umax < ext[0] || wmin > ext[3] || wmax < ext[2]) return false;
    return true;
}

static __device__ bool exact_point_in_closed_polygon(double px, double py, const double* poly, int n) {
    bool inside = false;
    for (int i = 0; i < n; ++i) {
        int j = (i + 1 == n) ? 0 : i + 1;
        double ax = poly[2 * i], ay = poly[2 * i + 1], bx = poly[2 * j], by = poly[2 * j + 1];
        double cross = xsub(xmul(xsub(bx, ax), xsub(py, ay)), xmul(xsub(by, ay), xsub(px, ax)));
        if (cross == 0.0 && px >= fmin(ax, bx) && px <= fmax(ax, bx) && py >= fmin(ay, by) &&
            py <= fmax(ay, by))
            return true;
        if ((ay > py) != (by > py)) {
            double xint = xadd(xdiv(xmul(xsub(bx, ax), xsub(py, ay)), xsub(by, ay)), ax);
            if (px < xint) inside = !inside;
        }
    }
    return inside;
}

// Liang-Barsky with strict inequalities: segment meets the OPEN rectangle ext
__device__ __forceinline__ bool exact_seg_meets_open_rect(double ua, double wa, double ub, double wb,
                                                          const double* ext) {
    double t0 = 0.0, t1 = 1.0;
    double a[2] = {ua, wa}, d[2] = {xsub(ub, ua), xsub(wb, wa)};
    double lo[2] = {ext[0], ext[2]}, hi[2] = {ext[1], ext[3]};
#pragma unroll
    for (int ax = 0; ax < 2; ++ax) {
        if (d[ax] == 0.0) {
            if (a[ax] <= lo[ax] || a[ax] >= hi[ax]) return false;
        } else {
            double tlo = xdiv(xsub(lo[ax], a[ax]), d[ax]);
            double thi = xdiv(xsub(hi[ax], a[ax]), d[ax]);
            if (d[ax] > 0.0) { t0 = fmax(t0, tlo); t1 = fmin(t1, thi); }
            else             { t0 = fmax(t0, thi); t1 = fmin(t1, tlo); }
        }
    }
    return t0 < t1;
}

// rectangle inside the closed simple polygon (GEOS contains)
static __device__ bool exact_rect_in_polygon(const Pose64& p, const double* ext, const double* cx,
                                      const double* cy, const double* poly, int n) {
    for (int k = 0; k < 4; ++k)
        if (!exact_point_in_closed_polygon(cx[k], cy[k], poly, n)) return false;
    double ua, wa;
    exact_local(p, poly[0], poly[1], ua, wa);
    double u0 = ua, w0 = wa;
    for (int i = 0; i < n; ++i) {
        double ub, wb;
        if (i + 1 == n) { ub = u0; wb = w0; }
        else exact_local(p, poly[2 * (i + 1)], poly[2 * (i + 1) + 1], ub, wb);
        if (exact_seg_meets_open_rect(ua, wa, ub, wb, ext)) return false;
        ua = ub; wa = wb;
    }
    return true;
}

// ---- lane: union of 66-vertex capsule polygons ------------------------------
__device__ __forceinline__ double seg_dist64(const double* s, double px, double py) {
    double ex = s[2] - s[0], ey = s[3] - s[1];
    double t = ((px - s[0]) * ex + (py - s[1]) * ey) / (ex * ex + ey * ey);
    t = fmin(fmax(t, 0.0), 1.0);
    double qx = s[0] + t * ex, qy = s[1] + t * ey;
    double ddx = px - qx, ddy = py - qy;
    return sqrt(ddx * ddx + ddy * ddy);
}

// g_j = nx_j*(px - vx_j) + ny_j*(py - vy_j), n_j = (e_y, -e_x) of the CCW ring
__device__ __forceinline__ double capsule_halfplane(const double* poly, int j, double px, double py) {
    int k = (j + 1 == HL_CAPSULE_VERTS) ? 0 : j + 1;
    double vx = poly[2 * j], vy = poly[2 * j + 1];
    double nx = xsub(poly[2 * k + 1], vy), ny = -xsub(poly[2 * k], vx);
    return xadd(xmul(nx, xsub(px, vx)), xmul(ny, xsub(py, vy)));
}

static __device__ bool exact_point_in_capsule(const double* seg, const double* poly, double px, double py,
                                       bool strict) {
    double d = seg_dist64(seg, px, py);
    if (d <= HL_BAND_IN) return true;
    if (d > HL_BAND_OUT) return false;
    for (int j = 0; j < HL_CAPSULE_VERTS; ++j) {
        double g = capsule_halfplane(poly, j, px, py);
        if (strict ? !(g < 0.0) : !(g <= 0.0)) return false;
    }
    return true;
}

// rectangle inside the union of capsule polygons -- oracle/geometry.py Lane.rects_inside
static __device__ bool exact_rect_in_lane(const Pose64& p, const double* ext, const double* cx, const double* cy,
                                   const EnvBatchDev& eb, const EnvDesc& e) {
    const int S = e.n_seg;
    const double* segs = eb.seg64 + 4 * (size_t)e.seg_off;
    const double* polys = eb.seg_poly + 2 * HL_CAPSULE_VERTS * (size_t)e.seg_off;
    unsigned covered = 0;                       // corner k covered by some capsule
    for (int i = 0; i < S; ++i) {
        unsigned in = 0;
        for (int k = 0; k < 4; ++k)
            if (exact_point_in_capsule(segs + 4 * i, polys + 2 * HL_CAPSULE_VERTS * i, cx[k], cy[k], false))
                in |= 1u << k;
        if (in == 0xFu) return true;            // step 0: one convex capsule holds all 4 corners
        covered |= in;
    }
    if (covered != 0xFu) return false;          // step 1
    for (int k = 0; k < 4; ++k) {               // step 2: every rectangle edge covered
        int k2 = (k + 1) & 3;
        double lo_s[HL_MAX_SEGS], hi_s[HL_MAX_SEGS];
        int ni = 0;
        for (int i = 0; i < S; ++i) {
            const double* poly = polys + 2 * HL_CAPSULE_VERTS * i;
            double lo = 0.0, hi = 1.0;
            bool ok = true;
            for (int j = 0; j < HL_CAPSULE_VERTS; ++j) {
                double g0 = capsule_halfplane(poly, j, cx[k], cy[k]);
                double g1 = capsule_halfplane(poly, j, cx[k2], cy[k2]);
                if (g0 <= 0.0 && g1 <= 0.0) continue;
                if (g0 > 0.0 && g1 > 0.0) { ok = false; break; }
                double tc = xdiv(g0, xsub(g0, g1));
                if (g0 > 0.0) lo = fmax(lo, tc); else hi = fmin(hi, tc);
            }
            if (ok && lo <= hi) {
                int q = ni++;                    // insertion sort by (lo, hi)
                while (q > 0 && (lo_s[q - 1] > lo || (lo_s[q - 1] == lo && hi_s[q - 1] > hi))) {
                    lo_s[q] = lo_s[q - 1]; hi_s[q] = hi_s[q - 1]; --q;
                }
                lo_s[q] = lo; hi_s[q] = hi;
            }
        }
        double cover = 0.0;
        for (int q = 0; q < ni; ++q) {
            if (lo_s[q] > cover) return false;
            cover = fmax(cover, hi_s[q]);
        }
        if (cover < 1.0) return false;
    }
    const double* crit = eb.crit64 + 2 * (size_t)e.crit_off;   // step 3
    for (int q = 0; q < e.n_crit; ++q) {
        double u, w;
        exact_local(p, crit[2 * q], crit[2 * q + 1], u, w);
        if (u > ext[0] && u < ext[1] && w > ext[2] && w < ext[3]) return false;
    }
    return true;
}

// reference_line_heuristic.py:120-129: LAST capsule whose interior holds the point
static __device__ int exact_search_segment(const EnvBatchDev& eb, const EnvDesc& e, double px, double py) {
    int last = -1;
    for (int i = 0; i < e.n_seg; ++i)
        if (exact_point_in_capsule(eb.seg64 + 4 * (size_t)(e.seg_off + i),
                                   eb.seg_poly + 2 * HL_CAPSULE_VERTS * (size_t)(e.seg_off + i), px, py, true))
            last = i;
    return last;
}

// Full exact check of one footprint rectangle at one pose.  Returns true = infeasible.
static __device__ __noinline__ bool exact_part_check(const Pose64& p, const double* ext, const EnvBatchDev& eb,
                                 const EnvDesc& e, unsigned flags) {
    double cx[4], cy[4];
    exact_corners(p, ext, cx, cy);
    if (flags & HL_CHECK_OBSTACLES) {
        const double* V = eb.obs64 + 8 * (size_t)e.obs_off;
        for (int k = 0; k < e.n_obs; ++k)
            if (exact_rect_hits_quad(p, ext, cx, cy, V + 8 * k)) return true;
    }
    if (flags & HL_CHECK_BOUNDARY)
        if (!exact_rect_in_polygon(p, ext, cx, cy, eb.field64 + 2 * (size_t)e.field_off, e.n_field)) return true;
    if ((flags & HL_CHECK_LANE) && e.n_seg > 0)
        if (!exact_rect_in_lane(p, ext, cx, cy, eb, e)) return true;
    return false;
}

// ---- warp-cooperative exact predicates ------------------------------------------------------------
// Same float64 expressions as the single-thread versions above, evaluated by all 32 lanes of a warp for ONE
// pose (every lane passes the same arguments): obstacles / polygon edges / capsule half-planes are spread
// over the lanes and combined with ballots and shuffles.  A single lane needs ~50k instructions for an
// ambiguous lane-union case; the warp needs ~1.5k.
__device__ __forceinline__ double warp_max(double v) {
    for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
    for (int o = 16; o; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

static __device__ __noinline__ bool warp_exact_rect_in_lane(const Pose64& p, const double* ext, const double* cx,
                                                            const double* cy, const EnvBatchDev& eb, const EnvDesc& e,
                                                            int lane) {
    const int S = e.n_seg;
    const double* segs = eb.seg64 + 4 * (size_t)e.seg_off;
    const double* polys = eb.seg_poly + 2 * HL_CAPSULE_VERTS * (size_t)e.seg_off;
    // steps 0/1: corner k in capsule i, one (i, k) pair per lane (S <= 16 -> two rounds of 32)
    unsigned covered = 0;
    bool one_holds_all = false;
    for (int base = 0; base < 4 * S; base += 32) {
        const int q = base + lane;
        bool in = false;
        if (q < 4 * S) {
            const int i = q >> 2, k = q & 3;
            in = exact_point_in_capsule(segs + 4 * i, polys + 2 * HL_CAPSULE_VERTS * i, cx[k], cy[k], false);
        }
        const unsigned m = __ballot_sync(0xffffffffu, in);
        for (int i = 0; i < 8; ++i) {
            const unsigned four = (m >> (4 * i)) & 0xFu;
            if (four == 0xFu) one_holds_all = true;
            covered |= four;
        }
    }
    if (one_holds_all) return true;
    if (covered != 0xFu) return false;
    // step 2: every rectangle edge covered by the union of clip intervals; the 66 half-planes of a capsule
    // are spread over the lanes (j = lane, lane+32, lane+64)
    for (int k = 0; k < 4; ++k) {
        const int k2 = (k + 1) & 3;
        double lo_s[HL_MAX_SEGS], hi_s[HL_MAX_SEGS];
        int ni = 0;
        for (int i = 0; i < S; ++i) {
            const double* poly = polys + 2 * HL_CAPSULE_VERTS * i;
            double lo = 0.0, hi = 1.0;
            int dead = 0;
            for (int j = lane; j < HL_CAPSULE_VERTS; j += 32) {
                const double g0 = capsule_halfplane(poly, j, cx[k], cy[k]);
                const double g1 = capsule_halfplane(poly, j, cx[k2], cy[k2]);
                if (g0 <= 0.0 && g1 <= 0.0) continue;
                if (g0 > 0.0 && g1 > 0.0) { dead = 1; continue; }
                const double tc = xdiv(g0, xsub(g0, g1));
                if (g0 > 0.0) lo = fmax(lo, tc); else hi = fmin(hi, tc);
            }
            dead = __any_sync(0xffffffffu, dead);
            lo = warp_max(lo);
            hi = warp_min(hi);
            if (!dead && lo <= hi) {
                int q = ni++;                    // insertion sort by (lo, hi), identical on every lane
                while (q > 0 && (lo_s[q - 1] > lo || (lo_s[q - 1] == lo && hi_s[q - 1] > hi))) {
                    lo_s[q] = lo_s[q - 1]; hi_s[q] = hi_s[q - 1]; --q;
                }
                lo_s[q] = lo; hi_s[q] = hi;
            }
        }
        double cover = 0.0;
        for (int q = 0; q < ni; ++q) {
            if (lo_s[q] > cover) return false;
            cover = fmax(cover, hi_s[q]);
        }
        if (cover < 1.0) return false;
    }
    // step 3: vertices of the union boundary strictly inside the rectangle
    const double* crit = eb.crit64 + 2 * (size_t)e.crit_off;
    int inside = 0;
    for (int q = lane; q < e.n_crit; q += 32) {
        double u, w;
        exact_local(p, crit[2 * q], crit[2 * q + 1], u, w);
        if (u > ext[0] && u < ext[1] && w > ext[2] && w < ext[3]) inside = 1;
    }
    return !__any_sync(0xffffffffu, inside);
}

// Full exact check of one rectangle at one pose, by the whole warp.  Returns true = infeasible (uniform).
static __device__ __noinline__ bool warp_exact_part_check(const Pose64& p, const double* ext, const EnvBatchDev& eb,
                                                          const EnvDesc& e, unsigned flags, int lane) {
    double cx[4], cy[4];
    exact_corners(p, ext, cx, cy);
    if (flags & HL_CHECK_OBSTACLES) {
        const double* V = eb.obs64 + 8 * (size_t)e.obs_off;
        int hit = 0;
        for (int k = lane; k < e.n_obs; k += 32)
            if (exact_rect_hits_quad(p, ext, cx, cy, V + 8 * k)) hit = 1;
        if (__any_sync(0xffffffffu, hit)) return true;
    }
    if (flags & HL_CHECK_BOUNDARY) {
        // one polygon edge per lane: crossing parity and on-edge test of the 4 corners, edge vs open rectangle
        const double* poly = eb.field64 + 2 * (size_t)e.field_off;
        const int n = e.n_field;
        unsigned par = 0, on = 0;
        int cut = 0;
        for (int i = lane; i < n; i += 32) {
            const int j = (i + 1 == n) ? 0 : i + 1;
            const double ax = poly[2 * i], ay = poly[2 * i + 1], bx = poly[2 * j], by = poly[2 * j + 1];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double px = cx[k], py = cy[k];
                const double cross = xsub(xmul(xsub(bx, ax), xsub(py, ay)), xmul(xsub(by, ay), xsub(px, ax)));
                if (cross == 0.0 && px >= fmin(ax, bx) && px <= fmax(ax, bx) && py >= fmin(ay, by) && py <= fmax(ay, by))
                    on |= 1u << k;
                if ((ay > py) != (by > py)) {
                    const double xint = xadd(xdiv(xmul(xsub(bx, ax), xsub(py, ay)), xsub(by, ay)), ax);
                    if (px < xint) par ^= 1u << k;
                }
            }
            double ua, wa, ub, wb;
            exact_local(p, ax, ay, ua, wa);
            exact_local(p, bx, by, ub, wb);
            if (exact_seg_meets_open_rect(ua, wa, ub, wb, ext)) cut = 1;
        }
        for (int o = 16; o; o >>= 1) { par ^= __shfl_xor_sync(0xffffffffu, par, o); on |= __shfl_xor_sync(0xffffffffu, on, o); }
        if (((par | on) & 0xFu) != 0xFu) return true;            // some corner outside the closed polygon
        if (__any_sync(0xffffffffu, cut)) return true;
    }
    if ((flags & HL_CHECK_LANE) && e.n_seg > 0)
        if (!warp_exact_rect_in_lane(p, ext, cx, cy, eb, e, lane)) return true;
    return false;
}

// ------------------------------------------------------------------- float32
// Environment staged in shared memory for the float32 filter.
struct EnvSmem {
    int n_obs, n_field, n_seg, all_rect;
    float eps, reach;
    float ext[4];               // body rectangle
    const float* obs;           // [n_obs][HL_OBS32_STRIDE]
    const float* field;         // [n_field][HL_FIELD32_STRIDE]
    const float* seg;           // [n_seg][4]
};

// Membership of a point in capsule POLYGON i (float32).  The polygon is the true capsule of radius 6
// except in the two round caps, where it is the 32-chord fan with vertices at angle_normal + k*pi/32
// (geometry_host.capsule_polygon): a cap point at range rho and angular offset delta from the nearest
// chord midpoint is inside iff rho*m_cos(delta) <= 6*m_cos(pi/64).  Returns 1 inside, 0 outside, 2 when
// the margin is within the float32 band.
// The filter only has to be RIGHT when it is sure: its divisions and square roots feed comparisons that carry a
// margin of eps (~2e-4 m), so the 2-ulp hardware approximations (MUFU.RCP / MUFU.RSQ) are used instead of the
// IEEE-rounded sequences (~8 instructions + slow path each; 15 % of K1's instructions before this change).
__device__ __forceinline__ float f_rcp(float x) { return __fdividef(1.0f, x); }
__device__ __forceinline__ float f_sqrt(float x) { return x > 0.0f ? x * rsqrtf(x) : 0.0f; }

static __device__ HL_CODE int corner_in_capsule(const float* sg, float wx, float wy, float eps) {
    const float ex = sg[2] - sg[0], ey = sg[3] - sg[1];
    const float len2 = fmaf(ex, ex, ey * ey);
    const float qx = wx - sg[0], qy = wy - sg[1];
    const float tt = fmaf(qx, ex, qy * ey) * f_rcp(len2);
    const float t = fminf(fmaxf(tt, 0.f), 1.f);
    const float ddx = fmaf(-t, ex, qx), ddy = fmaf(-t, ey, qy);
    const float d2 = fmaf(ddx, ddx, ddy * ddy);
    const float rin = (float)HL_LANE_RIN - eps, rout = (float)HL_LANE_R + eps;
    if (d2 <= rin * rin) return 1;
    if (d2 > rout * rout) return 0;
    float g = f_sqrt(d2);                                       // straight part: distance to the axis
    if (tt < 0.f || tt > 1.f) {                                 // cap: chord fan
        const float il = rsqrtf(len2);
        const float along = fabsf(fmaf(ddx, ex, ddy * ey)) * il, across = fabsf(fmaf(ddy, ex, -ddx * ey)) * il;
        const float phi = atan2f(across, along);                // 0 .. pi/2 from the segment direction
        const float q = 1.5707963267948966f - phi;              // angle from the first vertex (the normal)
        const float step = 0.09817477042468103f;                // pi/32
        const float k = floorf(q / step);
        const float delta = fabsf(q - (k + 0.5f) * step);
        g = g * cosf(delta) * 1.0012061467251643f;              // / m_cos(pi/64)
    }
    if (g <= (float)HL_LANE_R - eps) return 1;
    if (g > (float)HL_LANE_R + eps) return 0;
    return 2;
}

// One rectangle `ext` at pose (px,py,c,s) [float32, relative to env origin].
// Returns HL_FREE / HL_HIT / HL_AMBIG per enabled test, combined:
//   any HIT -> HIT; else any AMBIG -> AMBIG; else FREE.
// Formulation: the rectangle is (centre C, unit axes u=(c,s), v=(-s,c), half extents hx,hy).
//   * obstacles that are rectangles (tree rows, squares) use the 4-axis box-box separating test on
//     (centre, axis, half extents) -- ~30 flop instead of the 8-axis vertex form; other convex quads
//     keep the generic vertex form;
//   * field polygon: per edge the signed distance of C to the edge's line against the support radius
//     of the rectangle along the edge normal decides "clear" for most edges in ~12 flop; an edge whose
//     line the rectangle straddles is checked along the edge direction and in the pose frame; the
//     crossing parity of C decides inside/outside when every edge is clear;
//   * lane: one centre-to-segment distance accepts / rejects against (r_in - rho) / (r_out + rho)
//     before the four corner distances are needed.
// ---- the filter in three stages (K1 runs them as separate, compacted passes; filter_part chains them) ----
struct FiltState {                 // what stage 1 leaves for the later stages
    unsigned near_mask;            // field edges whose line the rectangle may touch
    unsigned amb;                  // HL_CHECK_* bits that are inside the float32 band so far
    bool hit, inside, overflow;
};

// Stage 1: obstacles + first pass over the field edges (crossing parity of the centre, nearby-edge mask).
static __device__ __forceinline__ void filt_stage1(const EnvSmem& E, float px, float py, float c, float s,
                                                   const float* ext, unsigned flags, FiltState& F) {
    const float eps = E.eps;
    const float hx = 0.5f * (ext[1] - ext[0]), hy = 0.5f * (ext[3] - ext[2]);
    const float mx = 0.5f * (ext[1] + ext[0]), my = 0.5f * (ext[3] + ext[2]);
    const float Cx = fmaf(c, mx, fmaf(-s, my, px)), Cy = fmaf(s, mx, fmaf(c, my, py));
    unsigned amb = 0;
    // Branch-light on purpose: the lanes of a warp hold unrelated poses, so every data-dependent
    // branch is paid by the whole warp.  Obstacles and field edges are evaluated for all lanes and
    // folded into hit / ambiguous flags; the rare second-stage edge tests are a separate stage.
    bool hit = false;
    if (flags & HL_CHECK_OBSTACLES) {
        bool a_obs = false;
        if (E.all_rect) {
            HL_LOOP
            for (int k = 0; k < E.n_obs; ++k) {
                const float* o = E.obs + HL_OBS32_STRIDE * k;
                const float4 b0 = *reinterpret_cast<const float4*>(o + 20);      // flag, cx, cy, ax
                const float4 b1 = *reinterpret_cast<const float4*>(o + 24);      // ay, ha, hb, pad
                const float dx = b0.y - Cx, dy = b0.z - Cy;
                const float ax = b0.w, ay = b1.x, ha = b1.y, hb = b1.z;
                const float p = fabsf(fmaf(ax, c, ay * s)), q = fabsf(fmaf(ay, c, -ax * s));
                const float du = fabsf(fmaf(dx, c, dy * s)), dv = fabsf(fmaf(dy, c, -dx * s));
                const float da = fabsf(fmaf(dx, ax, dy * ay)), db = fabsf(fmaf(dy, ax, -dx * ay));
                const float sep = fmaxf(fmaxf(du - fmaf(ha, p, fmaf(hb, q, hx)), dv - fmaf(ha, q, fmaf(hb, p, hy))),
                                        fmaxf(da - fmaf(hx, p, fmaf(hy, q, ha)), db - fmaf(hx, q, fmaf(hy, p, hb))));
                hit |= sep < -eps;
                a_obs |= fabsf(sep) <= eps;
            }
        } else {
            float rx[4], ry[4];
            const float lx[4] = {ext[0], ext[0], ext[1], ext[1]};
            const float ly[4] = {ext[3], ext[2], ext[2], ext[3]};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                rx[j] = fmaf(c, lx[j], fmaf(-s, ly[j], px));
                ry[j] = fmaf(s, lx[j], fmaf(c, ly[j], py));
            }
            HL_LOOP
            for (int k = 0; k < E.n_obs; ++k) {                  // generic convex quads: 8 axes on vertices
                const float* o = E.obs + HL_OBS32_STRIDE * k;
                float sep = -INFINITY;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float nx = o[8 + 3 * i], ny = o[9 + 3 * i], cc = o[10 + 3 * i];
                    float m = fminf(fminf(fmaf(nx, rx[0], ny * ry[0]), fmaf(nx, rx[1], ny * ry[1])),
                                    fminf(fmaf(nx, rx[2], ny * ry[2]), fmaf(nx, rx[3], ny * ry[3])));
                    sep = fmaxf(sep, m - cc);
                }
                float umin = INFINITY, umax = -INFINITY, wmin = INFINITY, wmax = -INFINITY;
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    float dx = o[2 * v] - px, dy = o[2 * v + 1] - py;
                    float u = fmaf(c, dx, s * dy), w = fmaf(c, dy, -s * dx);
                    umin = fminf(umin, u); umax = fmaxf(umax, u);
                    wmin = fminf(wmin, w); wmax = fmaxf(wmax, w);
                }
                sep = fmaxf(sep, fmaxf(fmaxf(umin - ext[1], ext[0] - umax), fmaxf(wmin - ext[3], ext[2] - wmax)));
                hit |= sep < -eps;
                a_obs |= fabsf(sep) <= eps;
            }
        }
        if (a_obs) amb |= HL_CHECK_OBSTACLES;
    }
    bool inside = false, overflow = false;
    unsigned near_mask = 0;                           // edges whose LINE the rectangle may touch (n <= 32 here)
    if (flags & HL_CHECK_BOUNDARY) {
        const int n = E.n_field;
        const float rho_eps = sqrtf(fmaf(hx, hx, hy * hy)) + eps;
        HL_LOOP
        for (int i = 0; i < n; ++i) {
            const float* e = E.field + HL_FIELD32_STRIDE * i;
            const float4 r0 = *reinterpret_cast<const float4*>(e);               // Ax, Ay, Ex, Ey
            const float4 r1 = *reinterpret_cast<const float4*>(e + 4);           // nx, ny, c, By
            // crossing parity of the rectangle centre, division-free: Cx < Ax + Ex*(Cy-Ay)/Ey
            // By is bit-identical to the next edge's Ay, so the half-open rule stays consistent at vertices
            const float dyc = Cy - r0.y;
            const bool straddle = (r0.y > Cy) != (r1.w > Cy);
            const float lhs = (Cx - r0.x) * r0.w, rhs = r0.z * dyc;
            inside ^= straddle && ((r0.w > 0.0f) ? (lhs < rhs) : (lhs > rhs));
            const float sd = fmaf(r1.x, Cx, fmaf(r1.y, Cy, -r1.z));                      // signed distance to the line
            if (!(fabsf(sd) > rho_eps)) {                     // within the circumradius: use the exact support radius
                const float nu = fmaf(r1.x, c, r1.y * s), nv = fmaf(r1.y, c, -r1.x * s);  // n.u, n.v
                const float rn = fmaf(hx, fabsf(nu), hy * fabsf(nv));                    // support radius along n
                if (!(fabsf(sd) > rn + eps)) { if (i < 32) near_mask |= 1u << i; else overflow = true; }
            }
        }
    }
    F.near_mask = near_mask; F.amb = amb; F.hit = hit; F.inside = inside; F.overflow = overflow;
}

// Stage 2: the few nearby field edges of this pose (Liang-Barsky against the shrunken rectangle), then the
// field verdict.  Needs only F.near_mask / inside / overflow; updates F.hit / F.amb.
static __device__ __forceinline__ void filt_field2(const EnvSmem& E, float px, float py, float c, float s,
                                                   const float* ext, FiltState& F) {
    const float eps = E.eps;
    const float hx = 0.5f * (ext[1] - ext[0]), hy = 0.5f * (ext[3] - ext[2]);
    const float mx = 0.5f * (ext[1] + ext[0]), my = 0.5f * (ext[3] + ext[2]);
    const float Cx = fmaf(c, mx, fmaf(-s, my, px)), Cy = fmaf(s, mx, fmaf(c, my, py));
    unsigned near_mask = F.near_mask;
    bool all_clear = !F.overflow, cut = false;
    while (near_mask) {                           // second stage, only for the few nearby edges of this lane
        const int i = __ffs(near_mask) - 1;
        near_mask &= near_mask - 1;
        const float* e = E.field + HL_FIELD32_STRIDE * i;
        const float Ax = e[0], Ay = e[1], Bx = Ax + e[2], By = e[7], nx = e[4], ny = e[5];
        const float nu = fmaf(nx, c, ny * s), nv = fmaf(ny, c, -nx * s);
        // along the edge direction t = (-ny, nx):  t.u = -n.v,  t.v = n.u
        const float ct = fmaf(-ny, Cx, nx * Cy);
        const float rt = fmaf(hx, fabsf(nv), hy * fabsf(nu));
        if (ct - rt > fmaxf(e[8], e[9]) + eps || ct + rt < fminf(e[8], e[9]) - eps) continue;
        float dxa = Ax - px, dya = Ay - py, dxb = Bx - px, dyb = By - py;
        float ua = fmaf(c, dxa, s * dya), wa = fmaf(c, dya, -s * dxa);
        float ub = fmaf(c, dxb, s * dyb), wb = fmaf(c, dyb, -s * dxb);
        if ((fminf(ua, ub) > ext[1] + eps) || (fmaxf(ua, ub) < ext[0] - eps) ||
            (fminf(wa, wb) > ext[3] + eps) || (fmaxf(wa, wb) < ext[2] - eps)) continue;
        all_clear = false;
        // definite cut: Liang-Barsky against the rectangle shrunk by eps
        float t0 = 0.f, t1 = 1.f;
        bool dead = false;
        const float a2[2] = {ua, wa}, d2v[2] = {ub - ua, wb - wa};
        const float lo2[2] = {ext[0] + eps, ext[2] + eps}, hi2[2] = {ext[1] - eps, ext[3] - eps};
#pragma unroll
        for (int ax = 0; ax < 2; ++ax) {
            if (fabsf(d2v[ax]) < 1e-12f) {
                if (a2[ax] <= lo2[ax] || a2[ax] >= hi2[ax]) dead = true;
            } else {
                float inv = f_rcp(d2v[ax]);
                float tl = (lo2[ax] - a2[ax]) * inv, th = (hi2[ax] - a2[ax]) * inv;
                t0 = fmaxf(t0, fminf(tl, th));
                t1 = fminf(t1, fmaxf(tl, th));
            }
        }
        // the chord inside the shrunken rectangle must be clearly longer than the band
        if (!dead && (t1 - t0) * f_sqrt(fmaf(d2v[0], d2v[0], d2v[1] * d2v[1])) > 8.0f * eps) { cut = true; break; }
    }
    if (cut) F.hit = true;
    else if (all_clear) { if (!F.inside) F.hit = true; }
    else F.amb |= HL_CHECK_BOUNDARY;
}

// Stage 3: the guide lane (union of capsule polygons).  Returns HL_HIT, or HL_FREE with *lane_amb set when the
// cover could not be certified in float32.
static __device__ __forceinline__ int filt_lane(const EnvSmem& E, float px, float py, float c, float s,
                                                const float* ext, bool* lane_amb) {
    const float eps = E.eps;
    const float hx = 0.5f * (ext[1] - ext[0]), hy = 0.5f * (ext[3] - ext[2]);
    const float mx = 0.5f * (ext[1] + ext[0]), my = 0.5f * (ext[3] + ext[2]);
    const float Cx = fmaf(c, mx, fmaf(-s, my, px)), Cy = fmaf(s, mx, fmaf(c, my, py));
    *lane_amb = false;
    const float rho = sqrtf(fmaf(hx, hx, hy * hy));
    const float rin = (float)HL_LANE_RIN - eps, rout = (float)HL_LANE_R + eps;
    bool accepted = false, need_corners = false;
    HL_LOOP
    for (int i = 0; i < E.n_seg && !accepted; ++i) {
        const float* sg = E.seg + 4 * i;
        float ex = sg[2] - sg[0], ey = sg[3] - sg[1];
        float inv = f_rcp(fmaf(ex, ex, ey * ey));
        float qx = Cx - sg[0], qy = Cy - sg[1];
        float t = fminf(fmaxf(fmaf(qx, ex, qy * ey) * inv, 0.f), 1.f);
        float ddx = fmaf(-t, ex, qx), ddy = fmaf(-t, ey, qy);
        float d = f_sqrt(fmaf(ddx, ddx, ddy * ddy));
        if (d + rho <= rin) accepted = true;                 // whole rectangle inside capsule i
        else if (d - rho <= rout) need_corners = true;       // capsule i may hold some corner
    }
    if (accepted) return HL_FREE;
    if (!need_corners) return HL_HIT;                        // every point is outside every capsule
    float rx[4], ry[4];
    const float lx[4] = {ext[0], ext[0], ext[1], ext[1]};
    const float ly[4] = {ext[3], ext[2], ext[2], ext[3]};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        rx[j] = fmaf(c, lx[j], fmaf(-s, ly[j], px));
        ry[j] = fmaf(s, lx[j], fmaf(c, ly[j], py));
    }
    bool one_holds_all = false;
    unsigned maybe = 0;                    // corner j is inside (or within the band of) some capsule
    HL_LOOP
    for (int i = 0; i < E.n_seg; ++i) {
        const float* sg = E.seg + 4 * i;
        bool all_in = true;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int st = corner_in_capsule(sg, rx[j], ry[j], eps);
            all_in = all_in && (st == 1);
            if (st != 0) maybe |= 1u << j;
        }
        if (all_in) one_holds_all = true;
    }
    if (one_holds_all) return HL_FREE;
    if (maybe != 0xFu) return HL_HIT;
    // The corners sit in different capsules.  Certify the union cover piecewise: cut the
    // rectangle into 4 slices along its long side; a slice whose 4 corners are clearly inside
    // ONE (convex) capsule is inside the lane.  Only what this cannot certify is ambiguous.
    unsigned prev = 0;
    bool covered = true;
#pragma unroll 1
    for (int q = 0; q <= 4 && covered; ++q) {
        const float lxq = ext[0] + 0.25f * (float)q * (ext[1] - ext[0]);
        unsigned m = 0xFFFFu;                 // capsules holding BOTH points of this cross-section
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const float lyq = side ? ext[3] : ext[2];
            const float wx = fmaf(c, lxq, fmaf(-s, lyq, px)), wy = fmaf(s, lxq, fmaf(c, lyq, py));
            unsigned in = 0;
            HL_LOOP
            for (int i = 0; i < E.n_seg; ++i) {
                const float* sg = E.seg + 4 * i;
                float ex = sg[2] - sg[0], ey = sg[3] - sg[1];
                float inv = f_rcp(fmaf(ex, ex, ey * ey));
                float qx = wx - sg[0], qy = wy - sg[1];
                float t = fminf(fmaxf(fmaf(qx, ex, qy * ey) * inv, 0.f), 1.f);
                float ddx = fmaf(-t, ex, qx), ddy = fmaf(-t, ey, qy);
                if (fmaf(ddx, ddx, ddy * ddy) <= rin * rin) in |= 1u << i;
            }
            m &= in;
        }
        if (q > 0 && (prev & m) == 0) covered = false;
        prev = m;
    }
    if (!covered) *lane_amb = true;
    return HL_FREE;
}

static __device__ HL_CODE int filter_part(const EnvSmem& E, float px, float py, float c, float s,
                                           const float* ext, unsigned flags, unsigned* which_ambig) {
    FiltState F;
    filt_stage1(E, px, py, c, s, ext, flags, F);
    if (flags & HL_CHECK_BOUNDARY) filt_field2(E, px, py, c, s, ext, F);
    if (F.hit) return HL_HIT;
    unsigned amb = F.amb;
    if ((flags & HL_CHECK_LANE) && E.n_seg > 0) {
        bool lane_amb;
        if (filt_lane(E, px, py, c, s, ext, &lane_amb) == HL_HIT) return HL_HIT;
        if (lane_amb) amb |= HL_CHECK_LANE;
    }
    if (amb) { if (which_ambig) *which_ambig = amb; return HL_AMBIG; }
    return HL_FREE;
}

// Resolve one pose against its environment.  Shared by K1 and the search kernels.
static __device__ bool pose_infeasible(const EnvBatchDev& eb, const EnvDesc& D, const EnvSmem& E,
                                double x, double y, double yaw, bool with_aux, unsigned flags,
                                unsigned long long* n_exact) {
    float px = (float)(x - D.origin[0]), py = (float)(y - D.origin[1]);
    if (fabsf(px) > E.reach || fabsf(py) > E.reach) return far_status(flags, E.n_seg) == HL_HIT;
    bool far = !(fabs(yaw) < 1e6) || !(px == px) || !(py == py);       // NaN / absurd input: exact path decides
    float sf, cf;
    sincosf((float)yaw, &sf, &cf);
    unsigned amb = flags;
    int r = far ? HL_AMBIG : filter_part(E, px, py, cf, sf, E.ext, flags, &amb);
    if (r == HL_HIT) return true;
    bool bad = false;
    Pose64 p;
    bool have64 = false;
    if (r == HL_AMBIG) {
        p.x = x; p.y = y; p.c = m_cos(yaw); p.s = m_sin(yaw);
        have64 = true;
        if (n_exact) atomicAdd(n_exact, 1ULL);
        bad = exact_part_check(p, D.body_ext, eb, D, amb);
        if (bad) return true;
    }
    if (with_aux && (flags & HL_CHECK_AUX)) {
        // implement rectangles: obstacles + field polygon, never the lane
        // (orchard_geometry_environment.py:439-456; reference_line_heuristic.py:105-108)
        unsigned aflags = flags & (HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY);
        for (int a = 0; a < D.n_aux; ++a) {
            const double* ext64 = eb.aux64 + 4 * (size_t)(D.aux_off + a);
            float ext32[4] = {(float)ext64[0], (float)ext64[1], (float)ext64[2], (float)ext64[3]};
            unsigned amb2 = aflags;
            int r2 = far ? HL_AMBIG : filter_part(E, px, py, cf, sf, ext32, aflags, &amb2);
            if (r2 == HL_HIT) return true;
            if (r2 == HL_AMBIG) {
                if (!have64) { p.x = x; p.y = y; p.c = m_cos(yaw); p.s = m_sin(yaw); have64 = true; }
                if (n_exact) atomicAdd(n_exact, 1ULL);
                if (exact_part_check(p, ext64, eb, D, amb2)) return true;
            }
        }
    }
    return false;
}

__device__ __forceinline__ void global_env(const EnvBatchDev& eb, const EnvDesc& D, EnvSmem& E) {
    E.n_obs = D.n_obs; E.n_field = D.n_field; E.n_seg = D.n_seg; E.all_rect = D.all_rect;
    E.eps = D.eps; E.reach = D.reach;
    for (int k = 0; k < 4; ++k) E.ext[k] = (float)D.body_ext[k];
    E.obs = eb.obs32 + (size_t)HL_OBS32_STRIDE * D.obs_off;
    E.field = eb.field32 + HL_FIELD32_STRIDE * (size_t)D.field_off;
    E.seg = eb.seg32 + 4 * (size_t)D.seg_off;
}

