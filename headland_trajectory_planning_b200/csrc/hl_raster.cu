// hl_raster.cu -- K12: occupancy grids from environment geometry (hl_env_rasterize).
//
// Cell (i, j) of a grid is the closed square with the float64 edges fl((i0+i)*res) .. fl((i0+i+1)*res) by
// fl((j0+j)*res) .. fl((j0+j+1)*res), K7's cells.  It is occupied when K1's float64 predicates, applied to that
// square at the identity pose, find it meeting an obstacle quad (HL_CHECK_OBSTACLES) or not contained in the field
// polygon (HL_CHECK_BOUNDARY).  No reference implementation exists (the reference's grid path is commented out,
// orchard_geometry_environment.py:8,35-43,460-461): parity is unpinned and the closed-set rule is the definition.
//
// One CTA per RT_TI x RT_TJ tile of one grid; every decision below is either exact or K1's filter model:
//   * obstacles are culled per tile by their float64 bounding boxes.  Under the identity pose the last test of
//     exact_rect_hits_quad IS the closed bounding-box test, so a culled obstacle gives false for every cell exactly;
//   * a tile whose cells all lie more than the environment's band eps (L-inf) from every field edge is wholly inside or
//     wholly outside the field: one float64 point-in-polygon of the tile centre decides all its cells;
//   * every other cell runs K1's float32 filter (filt_stage1 / filt_field2 on the cell's square, relative to the
//     environment's origin) and goes to the float64 predicates only inside the band (counted in d_n_exact).  Cells
//     reaching beyond EnvDesc.reach (only with cells far larger than the footprints K1 sizes its band for) skip the
//     filter and go to the float64 predicates directly.
// Stores: one byte per thread, a warp writes 32 consecutive bytes of a grid row; no atomics on the output.
#include <climits>
#include <cstring>
#include <algorithm>
#include <vector>
#include "hl_geom.cuh"

#define RT_TI 16                // tile rows (i)
#define RT_TJ 64                // tile columns (j, contiguous in memory)
#define RT_THREADS 256
#define RT_OBS_CAP 64           // culled obstacles staged per tile; more fall back to the environment's global records
#define RT_FIELD_CAP 128        // field edges staged per tile; more are read from global memory

struct RtGrid {
    long long out_offset;
    long long tile_base;        // first tile of this grid in the launch's tile numbering
    int env, w, h, i0, j0, tiles_j;
};

__device__ __forceinline__ int rt_grid_of(const RtGrid* __restrict__ gs, int n, long long t) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (gs[mid].tile_base <= t) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(RT_THREADS)
k_env_rasterize(EnvBatchDev eb, const RtGrid* __restrict__ grids, int n_grids, double res, unsigned flags,
                uint8_t* __restrict__ out, unsigned long long* __restrict__ n_exact) {
    __shared__ __align__(16) float s_obs[RT_OBS_CAP * HL_OBS32_STRIDE];
    __shared__ __align__(16) float s_field[RT_FIELD_CAP * HL_FIELD32_STRIDE];
    __shared__ int s_idx[RT_OBS_CAP];
    __shared__ int s_n_obs, s_near, s_inside, s_rect;
    __shared__ unsigned long long s_exact;
    const int tid = threadIdx.x;
    const long long t = blockIdx.x;
    const RtGrid G = grids[rt_grid_of(grids, n_grids, t)];
    const EnvDesc D = eb.desc[G.env];
    const long long tile = t - G.tile_base;
    const int ti = (int)(tile / G.tiles_j), tj = (int)(tile % G.tiles_j);
    const int li0 = ti * RT_TI, lj0 = tj * RT_TJ;
    const int ni = min(RT_TI, G.w - li0), nj = min(RT_TJ, G.h - lj0);
    // the tile's closed bounding box: the outer edges of its first and last cells
    const long long gi_a = (long long)G.i0 + li0, gj_a = (long long)G.j0 + lj0;
    const double X0 = (double)gi_a * res, X1 = ((double)gi_a + ni) * res;
    const double Y0 = (double)gj_a * res, Y1 = ((double)gj_a + nj) * res;
    const double* obs64 = eb.obs64 + 8 * (size_t)D.obs_off;
    const double* fld64 = eb.field64 + 2 * (size_t)D.field_off;
    if (tid == 0) { s_n_obs = 0; s_near = 0; s_inside = 0; s_rect = 1; s_exact = 0; }
    __syncthreads();
    if (flags & HL_CHECK_OBSTACLES) {
        for (int k = tid; k < D.n_obs; k += RT_THREADS) {
            const double* V = obs64 + 8 * k;
            const double xa = fmin(fmin(V[0], V[2]), fmin(V[4], V[6])), xb = fmax(fmax(V[0], V[2]), fmax(V[4], V[6]));
            const double ya = fmin(fmin(V[1], V[3]), fmin(V[5], V[7])), yb = fmax(fmax(V[1], V[3]), fmax(V[5], V[7]));
            if (xa <= X1 && xb >= X0 && ya <= Y1 && yb >= Y0) {
                const int slot = atomicAdd(&s_n_obs, 1);
                if (slot < RT_OBS_CAP) s_idx[slot] = k;
            }
        }
    }
    const double eps = (double)D.eps;
    if (flags & HL_CHECK_BOUNDARY) {
        const int n = D.n_field;
        int near = 0;
        for (int i = tid; i < n; i += RT_THREADS) {
            const int j = (i + 1 == n) ? 0 : i + 1;
            const double ax = fld64[2 * i], ay = fld64[2 * i + 1], bx = fld64[2 * j], by = fld64[2 * j + 1];
            if (fmin(ax, bx) <= X1 + eps && fmax(ax, bx) >= X0 - eps && fmin(ay, by) <= Y1 + eps && fmax(ay, by) >= Y0 - eps)
                near = 1;
        }
        if (__syncthreads_or(near)) {
            if (tid == 0) s_near = 1;
            if (n <= RT_FIELD_CAP) {
                const float* src = eb.field32 + HL_FIELD32_STRIDE * (size_t)D.field_off;
                for (int k = tid; k < n * HL_FIELD32_STRIDE; k += RT_THREADS) s_field[k] = src[k];
            }
        } else if (tid == 0) {
            // every cell of the tile is farther than eps from the ring: all inside or all outside
            s_inside = exact_point_in_closed_polygon(xadd(xmul(0.5, X0), xmul(0.5, X1)), xadd(xmul(0.5, Y0), xmul(0.5, Y1)),
                                                     fld64, n);
        }
    }
    __syncthreads();
    const int n_cand = s_n_obs;
    const bool obs_global = n_cand > RT_OBS_CAP;      // too many to stage: test every obstacle of the environment
    if (!obs_global) {
        for (int k = tid; k < n_cand * HL_OBS32_STRIDE; k += RT_THREADS) {
            const int o = k / HL_OBS32_STRIDE, f = k % HL_OBS32_STRIDE;
            const float v = eb.obs32[HL_OBS32_STRIDE * (size_t)(D.obs_off + s_idx[o]) + f];
            s_obs[k] = v;
            if (f == 20 && v == 0.0f) s_rect = 0;
        }
    }
    __syncthreads();
    EnvSmem E;
    E.n_obs = obs_global ? D.n_obs : n_cand;
    E.obs = obs_global ? eb.obs32 + HL_OBS32_STRIDE * (size_t)D.obs_off : s_obs;
    E.all_rect = obs_global ? D.all_rect : s_rect;
    E.n_field = D.n_field;
    E.field = D.n_field <= RT_FIELD_CAP ? s_field : eb.field32 + HL_FIELD32_STRIDE * (size_t)D.field_off;
    E.n_seg = 0; E.seg = nullptr;
    E.eps = D.eps; E.reach = D.reach;
    E.ext[0] = E.ext[1] = E.ext[2] = E.ext[3] = 0.0f;
    const bool near = s_near != 0;
    const bool out_all = (flags & HL_CHECK_BOUNDARY) && !near && !s_inside;
    unsigned filt = 0;                                 // tests the float32 filter has to run in this tile
    if ((flags & HL_CHECK_OBSTACLES) && n_cand > 0) filt |= HL_CHECK_OBSTACLES;
    if ((flags & HL_CHECK_BOUNDARY) && near) filt |= HL_CHECK_BOUNDARY;
    uint8_t* __restrict__ dst = out + G.out_offset;
    unsigned my_exact = 0;
    const int lj = tid % RT_TJ;
    for (int li = tid / RT_TJ; li < ni; li += RT_THREADS / RT_TJ) {
        if (lj >= nj) break;
        const long long gi = gi_a + li, gj = gj_a + lj;
        const double x0 = (double)gi * res, x1 = ((double)gi + 1.0) * res;
        const double y0 = (double)gj * res, y1 = ((double)gj + 1.0) * res;
        bool occ = out_all;
        if (!occ && filt) {
            // the cell's square in the float32 frame: centre relative to the origin, half extents
            const double xc = xsub(xadd(xmul(0.5, x0), xmul(0.5, x1)), D.origin[0]);
            const double yc = xsub(xadd(xmul(0.5, y0), xmul(0.5, y1)), D.origin[1]);
            const double hx = xmul(0.5, xsub(x1, x0)), hy = xmul(0.5, xsub(y1, y0));
            unsigned amb = filt;
            if (fabs(xc) + hx <= (double)D.reach && fabs(yc) + hy <= (double)D.reach) {
                const float ext[4] = {-(float)hx, (float)hx, -(float)hy, (float)hy};
                FiltState F;
                filt_stage1(E, (float)xc, (float)yc, 1.0f, 0.0f, ext, filt, F);
                if (filt & HL_CHECK_BOUNDARY) filt_field2(E, (float)xc, (float)yc, 1.0f, 0.0f, ext, F);
                occ = F.hit;
                amb = F.hit ? 0u : F.amb;
            }
            if (amb) {
                // K1's float64 predicates at the identity pose: corners and pose-frame coordinates are the edges
                const Pose64 p = {0.0, 0.0, 1.0, 0.0};
                const double e64[4] = {x0, x1, y0, y1};
                double cx[4], cy[4];
                exact_corners(p, e64, cx, cy);
                ++my_exact;
                if (amb & HL_CHECK_OBSTACLES) {
                    const int m = obs_global ? D.n_obs : n_cand;
                    for (int k = 0; k < m && !occ; ++k)
                        occ = exact_rect_hits_quad(p, e64, cx, cy, obs64 + 8 * (obs_global ? k : s_idx[k]));
                }
                if (!occ && (amb & HL_CHECK_BOUNDARY)) occ = !exact_rect_in_polygon(p, e64, cx, cy, fld64, D.n_field);
            }
        }
        dst[(long long)(li0 + li) * G.h + (lj0 + lj)] = occ ? 1 : 0;
    }
    if (n_exact) {
        if (my_exact) atomicAdd(&s_exact, (unsigned long long)my_exact);
        __syncthreads();
        if (tid == 0 && s_exact) atomicAdd(n_exact, s_exact);
    }
}

extern "C" int hl_env_rasterize(hl_ctx* ctx, const hl_env_batch* envs, const HlRasterGrid* h_grids, int32_t n_grids,
                                double res, uint32_t flags, uint8_t* d_out, int64_t out_elems,
                                unsigned long long* d_n_exact, void* stream) {
    const char* what = "hl_env_rasterize";
    if (!ctx || !envs || n_grids < 0 || out_elems < 0 || (n_grids > 0 && (!h_grids || !d_out))) {
        hl_set_error("%s: bad arguments", what); return 1;
    }
    if (!(res > 0) || !isfinite(res)) { hl_set_error("%s: res must be finite and positive, got %g", what, res); return 1; }
    if (flags == 0 || (flags & ~(HL_CHECK_OBSTACLES | HL_CHECK_BOUNDARY))) {
        hl_set_error("%s: flags must be HL_CHECK_OBSTACLES and / or HL_CHECK_BOUNDARY, got %u", what, flags); return 1;
    }
    const int n_env = envs->dev.n_env;
    std::vector<RtGrid> tab(n_grids);
    long long n_tiles = 0;
    for (int k = 0; k < n_grids; ++k) {
        const HlRasterGrid& g = h_grids[k];
        if (g.env_id < 0 || g.env_id >= n_env) {
            hl_set_error("%s: grid %d: env_id %d outside the batch of %d environments", what, k, g.env_id, n_env); return 1;
        }
        if (g.w < 1 || g.h < 1) { hl_set_error("%s: grid %d: a %dx%d grid (w and h must be at least 1)", what, k, g.w, g.h); return 1; }
        if ((long long)g.i0 + g.w > INT_MAX || (long long)g.j0 + g.h > INT_MAX) {
            hl_set_error("%s: grid %d: a %dx%d grid at (%d, %d) overflows the int32 cell index", what, k, g.w, g.h, g.i0, g.j0);
            return 1;
        }
        if (!isfinite((double)g.i0 * res) || !isfinite((double)(g.i0 + g.w) * res) || !isfinite((double)g.j0 * res) ||
            !isfinite((double)(g.j0 + g.h) * res)) {
            hl_set_error("%s: grid %d: cell edges are not finite at res = %g", what, k, res); return 1;
        }
        const long long cells = (long long)g.w * g.h;
        if (g.out_offset < 0 || g.out_offset > out_elems - cells) {
            hl_set_error("%s: grid %d: output slice [%lld, %lld) outside the %lld bytes of d_out", what, k,
                         (long long)g.out_offset, (long long)g.out_offset + cells, (long long)out_elems); return 1;
        }
        RtGrid& r = tab[k];
        r.out_offset = g.out_offset; r.env = g.env_id; r.w = g.w; r.h = g.h; r.i0 = g.i0; r.j0 = g.j0;
        r.tiles_j = (g.h + RT_TJ - 1) / RT_TJ;
        r.tile_base = n_tiles;
        n_tiles += (long long)((g.w + RT_TI - 1) / RT_TI) * r.tiles_j;
    }
    // sorted by start, two slices overlap only if some pair of neighbours does
    std::vector<int> order(n_grids);
    for (int k = 0; k < n_grids; ++k) order[k] = k;
    std::sort(order.begin(), order.end(), [&](int a, int b) {
        return h_grids[a].out_offset != h_grids[b].out_offset ? h_grids[a].out_offset < h_grids[b].out_offset : a < b;
    });
    for (int k = 1; k < n_grids; ++k) {
        const HlRasterGrid& a = h_grids[order[k - 1]];
        if (h_grids[order[k]].out_offset < a.out_offset + (long long)a.w * a.h) {
            hl_set_error("%s: grids %d and %d: output slices overlap", what, std::min(order[k - 1], order[k]),
                         std::max(order[k - 1], order[k]));
            return 1;
        }
    }
    if (n_tiles > INT_MAX) { hl_set_error("%s: %lld tiles exceed the %d of one launch", what, n_tiles, INT_MAX); return 1; }
    if (hl_enter(ctx, envs, n_grids ? d_out : nullptr, what)) return 1;
    if (n_grids == 0) return 0;
    const cudaStream_t st = (cudaStream_t)stream;
    RtGrid* d_tab = nullptr;
    HL_CUDA_OK(cudaMallocAsync((void**)&d_tab, sizeof(RtGrid) * (size_t)n_grids, st));
    cudaError_t e = cudaMemcpyAsync(d_tab, tab.data(), sizeof(RtGrid) * (size_t)n_grids, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        k_env_rasterize<<<(unsigned)n_tiles, RT_THREADS, 0, st>>>(envs->dev, d_tab, n_grids, res, flags, d_out, d_n_exact);
        e = cudaGetLastError();
    }
    cudaFreeAsync(d_tab, st);
    if (e != cudaSuccess) { hl_set_error("%s: CUDA error: %s", what, cudaGetErrorString(e)); return 1; }
    return 0;
}
