// hl_grid.cu -- K6: holonomic grid distance field; K7: occupancy-grid footprint check.
//
// K6 replaces holonomic_costs_with_obstacles (path_planner/utils/a_star_utils.py:75-142).
// The reference runs a binary-heap Dijkstra from the goal cell with edge costs 1 and
// hypot(1,1) accumulated as sequential float64 sums.  Because fl(d + w) is monotone in d,
// its result is the least fixed point of D(v) = min_m fl(D(v - m) + w(m)), which ANY
// relaxation order reaches bit-exactly in float64 -- so the GPU runs a tiled wavefront:
// a CTA pulls a DF_TILE x DF_TILE tile (16 x 16, +1 halo) into shared memory, relaxes it to its local fixed
// point there, writes it back and flags the neighbouring tiles whose halo changed.  Only
// flagged tiles do work in the next launch (the frontier), so the traffic per launch is
// the frontier's, not the map's.  Roofline: nominally HBM, really launch/dependency
// depth (DESIGN.md).
//
// K7 is the grid-based footprint check the reference left commented out
// (orchard_geometry_environment.py:8,35-43,460-461) on the grid layout of
// occupancy_grid_utils.py:70-101; parity unpinned (no reference implementation).
#include <algorithm>
#include <climits>
#include <cstring>
#include <vector>
#include "hl_common.cuh"

#ifndef DF_TILE
#define DF_TILE 16                      // tile edge: 16 -> 310 launches of 13 us for the 4096 x 4096 field (4.03 ms), 32 -> 157 of 27 us
#endif                                   // (4.26 ms), 64 -> 79 of 80 us (6.37 ms): short visits and a long frontier list win
#define DF_THREADS 256

struct DfMoves { int n; int di[8]; int dj[8]; double w[8]; };

// One grid of a batch: a map, or the (2W-1) x (2H-1) extended grid of an open-border map (see k_df_ext_init).  Every K6
// kernel walks a table of these; the first 32 bytes are what a relaxation CTA reads for a tile.
struct __align__(16) DfField {
    const uint8_t* occ;           // [w][h], non-zero = occupied
    double* D;                    // [w][h] costs
    int w, h;
    int tiles_j, tile_base;       // tiles per row; first tile of this grid in the wavefront's global tile numbering
    long long cell_base;          // first cell of this grid in its table's global cell numbering (elementwise kernels)
    int gi, gj;                   // goal cell
};

// entry of global cell c in a table whose cell_base increase (every grid has at least one cell)
__device__ __forceinline__ int df_field_of(const DfField* __restrict__ fs, int n, long long c) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (fs[mid].cell_base <= c) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// a map whose goal lies strictly inside a grid of at least 3 x 3 is relaxed in place unless a border cell is free
__host__ __device__ inline bool df_goal_inside(const DfField& f) {
    return f.w >= 3 && f.h >= 3 && f.gi > 0 && f.gj > 0 && f.gi < f.w - 1 && f.gj < f.h - 1;
}

// the goal's 3 x 3 tile neighbourhood of grid fi joins the first frontier.  List entries are (grid, tile of that grid).
__device__ void df_seed(const DfField& f, int fi, int2* __restrict__ list, int* __restrict__ count) {
    const int tiles_i = (f.w + DF_TILE - 1) / DF_TILE, ti = f.gi / DF_TILE, tj = f.gj / DF_TILE;
    for (int a = -1; a <= 1; ++a)
        for (int b = -1; b <= 1; ++b) {
            const int x = ti + a, y = tj + b;
            if (x >= 0 && y >= 0 && x < tiles_i && y < f.tiles_j) list[atomicAdd(count, 1)] = make_int2(fi, x * f.tiles_j + y);
        }
}

// +inf everywhere and 0 at the goal of every map; open[f] = 1 when a border cell of map f is free (aliases reachable).
// Maps with their goal inside are seeded on the table's own tiling, which is the wavefront's when no border is open.
__global__ void k_df_init(const DfField* __restrict__ fs, int n, long long cells, int* __restrict__ open,
                          int2* __restrict__ list, int* __restrict__ count) {
    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const int fi = df_field_of(fs, n, c);
    const DfField f = fs[fi];
    const long long idx = c - f.cell_base;
    const int i = (int)(idx / f.h), j = (int)(idx % f.h);
    f.D[idx] = (i == f.gi && j == f.gj) ? 0.0 : INFINITY;
    if ((i == 0 || j == 0 || i == f.w - 1 || j == f.h - 1) && !f.occ[idx]) open[fi] = 1;
    if (i == f.gi && j == f.gj && df_goal_inside(f)) df_seed(f, fi, list, count);
}

__global__ void k_df_seed(const DfField* __restrict__ fs, int n, int2* __restrict__ list, int* __restrict__ count) {
    const int fi = blockIdx.x * blockDim.x + threadIdx.x;
    if (fi < n) df_seed(fs[fi], fi, list, count);
}

// DF_CPT vertically adjacent cells per thread of a DF_TILE x DF_TILE tile (DF_TILE^2 / DF_CPT threads), the move set a
// template parameter: the 8 (King) or 5 (Pawn) predecessors are compile-time offsets into the shared tile.  Only the
// neighbours that read an improved border cell in their halo are flagged for the next launch.  How each step of this
// design was measured on the 4096 x 4096 King field: DESIGN.md section 5, "K6 relaxation".
#ifndef DF_CPT
#define DF_CPT 2
#endif
#define DF_RELAX_THREADS (DF_TILE * DF_TILE / DF_CPT)
// min of two costs.  Costs are +0, positive or +inf, never NaN, so the minimum is a compare + two selects (DSETP.LT, 3
// instructions, one on the FP64 pipe) instead of fmin's DSETP.MIN + NaN fix-up + moves (7).  The relaxation kernel is
// issue-bound (ncu: issue-active 74 %), instructions are time.
__device__ __forceinline__ double df_min(double a, double b) { return (b < a) ? b : a; }
// non-negative doubles order like their bit patterns
__device__ __forceinline__ bool df_less(double a, double b) { return __double_as_longlong(a) < __double_as_longlong(b); }
#ifndef DF_MIN_CTAS
#define DF_MIN_CTAS 2                    // launch bound (with 32 x 32 tiles: 64 registers = two 512-thread CTAs per SM, 66 would leave one)
#endif
// ONE: the wavefront has a single grid, passed by value (`one`) instead of read from the table per tile: its fields are
// then kernel constants, as in the single-map kernel before batching, and take no registers across the relaxation loop
// (measured on the 4096 x 4096 King field: reading the table per tile costs 1.7 %)
template <bool KING, bool ONE>
__global__ void __launch_bounds__(DF_RELAX_THREADS, DF_MIN_CTAS)
k_df_relax(const DfField* __restrict__ fields, const DfField one, const int2* __restrict__ list_cur, const int* __restrict__ count_cur,
           int2* __restrict__ list_next, int* __restrict__ count_next, int* __restrict__ mark_next, int* __restrict__ mark_cur,
           int* __restrict__ count_clear, int* __restrict__ any_next) {
    // the frontier is a LIST of tiles walked by a small grid with a stride (instead of one CTA per tile of the map, 16 k
    // CTAs of which a few hundred have work).  No memset between launches: a tile clears its own mark when it is
    // processed, and the counter the launch after next appends to is zeroed here (three counters rotate).  The tiles of
    // all grids of a batch share the list; marks are indexed by the global tile id (tile_base + tile).
    // programmatic dependent launch: this grid was scheduled while the previous relaxation launch was still running;
    // nothing that launch wrote is read before it has completed, and the NEXT launch may be scheduled from here on
    // (its CTAs wait at the same point), so the ~2 us between two dependent launches overlap with the work
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (blockIdx.x == 0 && threadIdx.x == 0) *count_clear = 0;
    __shared__ double sd[DF_TILE + 2][DF_TILE + 3];
    __shared__ unsigned char so[DF_TILE + 2][DF_TILE + 2];
    __shared__ int s_border_changed;
    __shared__ int s_rowchg[2][DF_TILE + 2];            // rows that changed in the previous / this iteration
    const double W1 = 1.0, W2 = 1.4142135623730951;       // hypot(1, 0), hypot(1, 1) as the host's libm gives them
    const int n_cur = *count_cur;
    const int tid = threadIdx.x;
    const int a0 = 1 + DF_CPT * (tid / DF_TILE), b = 1 + (tid % DF_TILE);   // cell q of this thread: row a0 + q, column b
    for (int li = blockIdx.x; li < n_cur; li += gridDim.x) {
        const int2 entry = list_cur[li];
        const DfField f = ONE ? one : fields[entry.x];
        // the grid pointers come from memory, so without this they are generic: LD / ST instead of LDG / STG, occupancy
        // without the read-only path, and every access ordered against the shared tile (measured: +10 % per launch)
        __builtin_assume(__isGlobal(f.occ));
        __builtin_assume(__isGlobal(f.D));
        const uint8_t* __restrict__ occ = f.occ;
        double* __restrict__ D = f.D;
        const int W = f.w, H = f.h, tiles_j = f.tiles_j, tile_base = f.tile_base;
        const int tile = entry.y;
        const int ti = tile / tiles_j, tj = tile % tiles_j;
        const int i0 = ti * DF_TILE - 1, j0 = tj * DF_TILE - 1;
        if (tid == 0) { s_border_changed = 0; mark_cur[tile_base + tile] = 0; }
        if (tid < DF_TILE + 2) { s_rowchg[0][tid] = 1; s_rowchg[1][tid] = 0; }      // first iteration: every row counts as changed
        int it = 0;
        for (int k = tid; k < (DF_TILE + 2) * (DF_TILE + 2); k += DF_RELAX_THREADS) {
            const int x = k / (DF_TILE + 2), y = k % (DF_TILE + 2);
            const int i = i0 + x, j = j0 + y;
            const bool in = i >= 0 && j >= 0 && i < W && j < H;
            sd[x][y] = in ? D[(long long)i * H + j] : INFINITY;
            so[x][y] = in ? __ldg(occ + (long long)i * H + j) : 1;
        }
        __syncthreads();
        double init[DF_CPT], cur[DF_CPT];
        bool enter[DF_CPT];
#pragma unroll
        for (int q = 0; q < DF_CPT; ++q) {
            const int a = a0 + q;
            init[q] = cur[q] = sd[a][b];
            // occupied cells are never entered (the goal cell itself is exempt: it starts closed at 0)
            enter[q] = !so[a][b] && i0 + a < W && j0 + b < H;
        }
        while (true) {
            double best[DF_CPT];
            // a cell can only change if a cell of rows a0 - 1 .. a0 + DF_CPT changed in the previous iteration: the warp
            // (one group of DF_CPT rows) sits the iteration out otherwise (the wave crosses a tile as a band)
            int seen = 0;
#pragma unroll
            for (int r = 0; r < DF_CPT + 2; ++r) seen |= s_rowchg[it & 1][a0 - 1 + r];
            if (!seen) {
#pragma unroll
                for (int q = 0; q < DF_CPT; ++q) best[q] = cur[q];
            } else {
                // columns b - 1, b, b + 1 of rows a0 - 1 .. a0 + DF_CPT; the thread's own cells (column b) are in
                // registers, and a cell sees the value its upper neighbour in the same thread was just given (any
                // relaxation order reaches the same fixed point)
                double L[DF_CPT + 2], M[DF_CPT + 2], R[DF_CPT + 2];
#pragma unroll
                for (int r = 0; r < DF_CPT + 2; ++r) {
                    L[r] = sd[a0 - 1 + r][b - 1];
                    R[r] = KING ? sd[a0 - 1 + r][b + 1] : 0.0;
                }
                M[0] = sd[a0 - 1][b]; M[DF_CPT + 1] = sd[a0 + DF_CPT][b];
#pragma unroll
                for (int q = 0; q < DF_CPT; ++q) M[q + 1] = cur[q];
                // fl(x + w) is monotone in x, so min(fl(x + w), fl(y + w)) == fl(min(x, y) + w) bit for bit: ONE addition
                // per weight and cell (the minimum of the straight predecessors + 1, of the diagonal ones + sqrt 2)
                // instead of eight, and the minimum of a row's left and right cell serves the cell between them
                // (straight) and the two cells above / below it (diagonal).  Pawn moves only come from column b - 1.
                double hr[DF_CPT + 2];
#pragma unroll
                for (int r = 0; r < DF_CPT + 2; ++r) hr[r] = KING ? df_min(L[r], R[r]) : L[r];
#pragma unroll
                for (int q = 0; q < DF_CPT; ++q) {
                    const int r = q + 1;
                    double v = cur[q];
                    if (enter[q]) {
                        const double m1 = df_min(df_min(M[r - 1], M[r + 1]), hr[r]);
                        const double m2 = df_min(hr[r - 1], hr[r + 1]);
                        v = df_min(v, df_min(__dadd_rn(m1, W1), __dadd_rn(m2, W2)));
                    }
                    best[q] = v;
                    M[r] = v;
                }
            }
            __syncthreads();
            bool ch = false;
#pragma unroll
            for (int q = 0; q < DF_CPT; ++q)
                if (df_less(best[q], cur[q])) {
                    sd[a0 + q][b] = best[q]; cur[q] = best[q]; ch = true;
                    s_rowchg[(it + 1) & 1][a0 + q] = 1;
                }
            if (tid < DF_TILE + 2) s_rowchg[it & 1][tid] = 0;      // read before the barrier above, written again in iteration it + 2
            ++it;
            if (!__syncthreads_or(ch)) break;
        }
#pragma unroll
        for (int q = 0; q < DF_CPT; ++q) {
            const int a = a0 + q;
            const int i = i0 + a, j = j0 + b;
            if (cur[q] < init[q] && i < W && j < H) {
                D[(long long)i * H + j] = cur[q];
                // which neighbouring tiles read this cell in their halo: bit 3 * (x + 1) + (y + 1) for neighbour (x, y)
                // (a side cell is read by that side's neighbour only, a corner cell also by the diagonal neighbour)
                const int x = (a == 1) ? -1 : (a == DF_TILE ? 1 : 0), y = (b == 1) ? -1 : (b == DF_TILE ? 1 : 0);
                if (x || y) {
                    unsigned m = 0;
                    if (x) m |= 1u << (3 * (x + 1) + 1);
                    if (y) m |= 1u << (3 + (y + 1));
                    if (x && y) m |= 1u << (3 * (x + 1) + (y + 1));
                    atomicOr(&s_border_changed, (int)m);
                }
            }
        }
        __syncthreads();
        if (tid < 9 && tid != 4 && (s_border_changed >> tid) & 1) {
            const int tx = ti + tid / 3 - 1, ty = tj + tid % 3 - 1;     // flags stay inside the tile's own grid
            const int tiles_i = (W + DF_TILE - 1) / DF_TILE;
            if (tx >= 0 && ty >= 0 && tx < tiles_i && ty < tiles_j && atomicExch(&mark_next[tile_base + tx * tiles_j + ty], 1) == 0)
                list_next[atomicAdd(count_next, 1)] = make_int2(entry.x, tx * tiles_j + ty);
            *any_next = 1;
        }
        __syncthreads();                                   // the shared tile is reused by the next list entry
    }
}

// ---- the reference's index wrap-around (a_star_utils.py:49-64) --------------------------------------------
// Validity is `abs(index) < dim` and obstacles[i][j] is read with Python's negative indexing, so the reference
// really searches the EXTENDED grid of nodes (i, j), -W < i < W, -H < j < H, whose occupancy is the map's at
// (i mod W, j mod H); every closed node writes holonomicCost[i][j] (again with negative indexing) in closing order,
// so a map cell ends up with the cost of its LAST-closed alias.  Nodes close in the order of their heap entries
// (priority at push time, index tuple) -- there is no decrease-key (:131), so the priority of a node is the cost
// offered by its FIRST-closed neighbour, not its final cost.  All of it has a relaxation-order-free form:
//   C = least fixed point of the cost relaxation on the extended grid            (k_df_relax, as for closed maps)
//   P(v) = C(u*) + w(u* -> v),  u* = the neighbour of v with the smallest (P(u), i_u, j_u)      (fixed point, k_df_prio)
//   out[cell] = C(alias of the cell with the largest (P, i, j))                                   (k_df_fold)
// oracle/distance_field.py (pinned bit-for-bit on the reference) agrees on every tested grid
// (tests/test_grid_gpu.py::test_wrap_around_quirk_matches_reference).
// The extended grids of a batch are packed in one workspace: entry k of `ex` (grid of map `mx[k]`) owns cells
// ex[k].cell_base .. + EW * EH of eocc, C (= ex[k].D) and the two priority buffers.  This pass builds the extended
// occupancy and initialises C (+inf, 0 at the goal).
__global__ void k_df_ext_init(const DfField* __restrict__ mx, const DfField* __restrict__ ex, int n, long long cells,
                              uint8_t* __restrict__ eocc) {
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= cells) return;
    const int k = df_field_of(ex, n, g);
    const DfField e = ex[k];
    const int W = mx[k].w, H = mx[k].h;
    const long long idx = g - e.cell_base;
    const int a = (int)(idx / e.h), b = (int)(idx % e.h);
    const int i = a - (W - 1), j = b - (H - 1);
    eocc[g] = mx[k].occ[(long long)(i < 0 ? i + W : i) * H + (j < 0 ? j + H : j)];
    e.D[idx] = (a == e.gi && b == e.gj) ? 0.0 : INFINITY;
}

__global__ void k_df_prio(const DfField* __restrict__ ex, int n, long long cells, const double* __restrict__ Pin_all,
                          double* __restrict__ Pout_all, DfMoves mv, int* __restrict__ changed) {
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= cells) return;
    const DfField e = ex[df_field_of(ex, n, g)];
    const double* __restrict__ C = e.D;
    const double* __restrict__ Pin = Pin_all + e.cell_base;
    const int EW = e.w, EH = e.h, ga = e.gi, gb = e.gj;
    const long long idx = g - e.cell_base;
    const int a = (int)(idx / EH), b = (int)(idx % EH);
    double np_ = INFINITY;
    if (a == ga && b == gb) np_ = 0.0;
    else if (C[idx] < INFINITY) {
        double bp = INFINITY; int ba = 0x7fffffff, bb = 0x7fffffff;
        for (int m = 0; m < mv.n; ++m) {
            const int ua = a - mv.di[m], ub = b - mv.dj[m];
            if (ua < 0 || ub < 0 || ua >= EW || ub >= EH) continue;
            const long long u = (long long)ua * EH + ub;
            const double cu = C[u];
            if (!(cu < INFINITY)) continue;
            const double pu = Pin[u];
            if (pu < bp || (pu == bp && (ua < ba || (ua == ba && ub < bb)))) { bp = pu; ba = ua; bb = ub; np_ = __dadd_rn(cu, mv.w[m]); }
        }
    }
    if (np_ != Pin[idx]) *changed = 1;
    Pout_all[g] = np_;
}

// each cell of map mx[k] takes the cost of its alias with the largest (P, i, j) on the extended grid ex[k]
__global__ void k_df_fold(const DfField* __restrict__ mx, const DfField* __restrict__ ex, int n, long long cells,
                          const double* __restrict__ P_all) {
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= cells) return;
    const int k = df_field_of(mx, n, g);
    const DfField m = mx[k];
    const double* __restrict__ C = ex[k].D;
    const double* __restrict__ P = P_all + ex[k].cell_base;
    const int W = m.w, H = m.h;
    const long long idx = g - m.cell_base;
    const int ci = (int)(idx / H), cj = (int)(idx % H);
    const int EH = 2 * H - 1;
    double best_c = INFINITY, best_p = -INFINITY;
    int best_i = -0x7fffffff, best_j = -0x7fffffff;
    for (int ai = 0; ai < 2; ++ai) {
        if (ai == 1 && ci < 1) continue;
        const int i = ai == 0 ? ci : ci - W;
        for (int aj = 0; aj < 2; ++aj) {
            if (aj == 1 && cj < 1) continue;
            const int j = aj == 0 ? cj : cj - H;
            const long long v = (long long)(i + W - 1) * EH + (j + H - 1);
            const double c = C[v];
            if (!(c < INFINITY)) continue;
            const double p = P[v];
            if (p > best_p || (p == best_p && (i > best_i || (i == best_i && j > best_j)))) { best_p = p; best_i = i; best_j = j; best_c = c; }
        }
    }
    m.D[idx] = best_c;
}

// Launches are queued DF_BATCH at a time with one host look per batch (launches behind the first empty frontier do
// nothing and cost ~2 us each).  The wavefront needs about one launch per tile it crosses, so the first look comes
// after (tiles_i + tiles_j) / 2 launches of the deepest grid, the later ones every 32: 2 host looks for the
// 4096 x 4096 field (157 launches) instead of 10 -- every look is a stream synchronisation, i.e. an idle GPU for as
// long as the host thread takes to come back.
enum { DF_BATCH_MAX = 128, DF_BATCH_NEXT = 32 };

// ints of a wavefront workspace: list[2][n_tiles] (int2) | mark[2][n_tiles] | count[4] | flags[1 + DF_BATCH_MAX]
static size_t df_ws_ints(long long n_tiles) { return 6 * (size_t)n_tiles + 4 + 1 + DF_BATCH_MAX; }

// Tiled wavefront to the fixed point of every grid of the table `rel` (device copy d_rel; cells outside a grid count as
// occupied).  The grids' tiles share one global numbering (tile_base), so a relaxation launch walks the frontier of all
// of them and a batch costs about the depth of its deepest grid.  The caller initialises the costs and hands over the
// workspace `ws` zeroed, with the first frontier in list[0] / count[0].
static int df_wavefront(const char* what, const std::vector<DfField>& rel, const DfField* d_rel, int* ws, int n_tiles,
                        const DfMoves& mv, cudaStream_t st, int* sweeps_out) {
    int depth = 0;                           // the largest tiles_i + tiles_j of the batch
    for (const DfField& f : rel) depth = std::max(depth, (f.w + DF_TILE - 1) / DF_TILE + f.tiles_j);
    int DF_BATCH = depth / 2 < 16 ? 16 : (depth / 2 > DF_BATCH_MAX ? DF_BATCH_MAX : depth / 2);
    int2* list[2] = {(int2*)ws, (int2*)ws + n_tiles};
    int* mark[2] = {ws + 4 * (size_t)n_tiles, ws + 5 * (size_t)n_tiles};
    int* count = ws + 6 * (size_t)n_tiles;
    int* flags = count + 4;                  // count[0..2]: three rotating frontier counters
    int rc = 0, sweeps = 0;
    int sm = 148;
    { int dev_id = 0; cudaGetDevice(&dev_id); cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev_id); }
    // CTAs per SM in the grid: MORE than are resident.  The frontier list is walked with a grid
    // stride, so with a grid of exactly the resident CTAs a CTA that drew a slow tile keeps its second tile waiting; with
    // twice as many the block scheduler hands the next list entry to whichever SM frees a slot first
    // (4096 x 4096 King, 32 x 32 tiles of 512 threads: 2 per SM 4.87 ms, 4 per SM 4.26 ms; 16 x 16 tiles of 128 threads:
    // 16 or 32 per SM 4.03 ms).
#ifndef DF_GRID_PER_SM
#define DF_GRID_PER_SM 16
#endif
    const int per_sm = DF_GRID_PER_SM;
    const int grid = n_tiles < sm * per_sm ? n_tiles : sm * per_sm;
    const bool one = rel.size() == 1;
    auto relax = mv.n == 8 ? (one ? k_df_relax<true, true> : k_df_relax<true, false>)
                           : (one ? k_df_relax<false, true> : k_df_relax<false, false>);
    do {
        int host_flags[1 + DF_BATCH_MAX] = {0};
        int cur = 0;                            // launch number: lists / marks alternate (cur & 1), counters rotate (cur % 3)
        const int max_sweeps = 8 * depth * DF_TILE + 64;
        bool converged = false;
        while (!converged && sweeps < max_sweeps) {
            cudaMemsetAsync(flags + 1, 0, DF_BATCH * sizeof(int), st);
            for (int k = 0; k < DF_BATCH; ++k) {
                const int lc = cur & 1, ln = lc ^ 1;
                int* c_cur = count + cur % 3; int* c_nxt = count + (cur + 1) % 3; int* c_clr = count + (cur + 2) % 3;
                cudaLaunchConfig_t cfg;
                memset(&cfg, 0, sizeof(cfg));
                cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(DF_RELAX_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = st;
                cudaLaunchAttribute attr[1];
                attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                attr[0].val.programmaticStreamSerializationAllowed = 1;
                cfg.attrs = attr; cfg.numAttrs = 1;
                const int2* a_lc = list[lc]; const int* a_cc = c_cur;
                int* a_fl = flags + 1 + k;
                if (cudaLaunchKernelEx(&cfg, relax, d_rel, rel[0], a_lc, a_cc, list[ln], c_nxt, mark[ln], mark[lc], c_clr, a_fl) != cudaSuccess) {
                    rc = 1; break;                              // a launch that did not happen would read as "frontier empty"
                }
                ++cur;
            }
            if (rc) { cudaStreamSynchronize(st); break; }
            if (cudaMemcpyAsync(host_flags + 1, flags + 1, DF_BATCH * sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) { rc = 1; break; }
            for (int k = 0; k < DF_BATCH && !converged; ++k) {   // launches after the first empty frontier did nothing
                ++sweeps;
                if (!host_flags[1 + k]) converged = true;
            }
            DF_BATCH = DF_BATCH_NEXT;
        }
        if (rc == 0 && !converged) { hl_set_error("%s: no convergence after %d launches", what, sweeps); rc = 2; }
    } while (0);
    if (rc == 1) hl_set_error("%s: CUDA error: %s", what, cudaGetErrorString(cudaGetLastError()));
    if (sweeps_out) *sweeps_out += sweeps;
    return rc;
}

// move set of a_star_utils.py:8-21 (motion_type 0, King) or :24-34 (1, Pawn); false for any other motion_type
static bool df_moves(int motion_type, DfMoves* mv) {
    static const int king[8][2] = {{-1, 0}, {-1, 1}, {0, 1}, {1, 1}, {1, 0}, {1, -1}, {0, -1}, {-1, -1}};
    static const int pawn[5][2] = {{-1, 0}, {0, 1}, {-1, 1}, {1, 1}, {1, 0}};
    memset(mv, 0, sizeof(*mv));
    if (motion_type != 0 && motion_type != 1) return false;
    const int (*k)[2] = motion_type == 0 ? king : pawn;
    mv->n = motion_type == 0 ? 8 : 5;
    for (int m = 0; m < mv->n; ++m) { mv->di[m] = k[m][0]; mv->dj[m] = k[m][1]; mv->w[m] = hypot((double)k[m][0], (double)k[m][1]); }
    return true;
}

// Distance fields of n validated maps in one wavefront.  A map whose border is occupied and whose goal lies strictly
// inside is the whole search space and is relaxed in place; any other map takes part as its extended grid (the
// reference's index wrap-around) and is folded into its output slice afterwards.  When every map is of the first kind
// (the common case) the call is one allocation, the init pass that also seeds the frontier, one synchronisation to read
// the open-border flags, and the wavefront.
static int df_run(const char* what, const uint8_t* d_occ, const HlGridField* hf, int n, const DfMoves& mv, double* d_out,
                  int32_t* h_sweeps, cudaStream_t st) {
    std::vector<DfField> map(n);
    long long cells = 0, n_tiles = 0;
    for (int k = 0; k < n; ++k) {
        DfField& f = map[k];
        memset(&f, 0, sizeof(f));
        f.occ = d_occ + hf[k].occ_offset; f.D = d_out + hf[k].out_offset;
        f.w = hf[k].w; f.h = hf[k].h; f.gi = hf[k].gi; f.gj = hf[k].gj;
        f.tiles_j = (f.h + DF_TILE - 1) / DF_TILE;
        f.tile_base = (int)std::min(n_tiles, (long long)INT_MAX);
        n_tiles += (long long)((f.w + DF_TILE - 1) / DF_TILE) * f.tiles_j;
        f.cell_base = cells; cells += (long long)f.w * f.h;
    }
    const long long max_tiles = INT_MAX / 6;
    if (n_tiles > max_tiles) { hl_set_error("%s: %lld tiles exceed the %lld of one wavefront", what, n_tiles, max_tiles); return 1; }
    // map[n] | mx[n] | wavefront workspace for the maps' own tiling | open[n] | changed
    char* d_tab = nullptr;
    const size_t tab_bytes = 2 * (size_t)n * sizeof(DfField) + (df_ws_ints(n_tiles) + n + 1) * sizeof(int);
    if (cudaMalloc(&d_tab, tab_bytes) != cudaSuccess) {
        cudaGetLastError();
        hl_set_error("%s: cudaMalloc of %zu bytes for the field tables and the wavefront failed", what, tab_bytes);
        return 1;
    }
    DfField* d_map = (DfField*)d_tab; DfField* d_mx = d_map + n;
    int* ws = (int*)(d_mx + n);
    int* d_open = ws + df_ws_ints(n_tiles);
    int* d_changed = d_open + n;
    char* d_ext = nullptr;                   // rel[n] | C | P0 | P1 of all extended grids | their wavefront workspace | eocc
    int rc = 0, sweeps = 0;
    do {
        std::vector<int> open(n, 0);
        if (cudaMemsetAsync(d_tab, 0, tab_bytes, st) != cudaSuccess ||
            cudaMemcpyAsync(d_map, map.data(), n * sizeof(DfField), cudaMemcpyHostToDevice, st) != cudaSuccess) { rc = 2; break; }
        k_df_init<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(d_map, n, cells, d_open, (int2*)ws, ws + 6 * n_tiles);
        if (cudaMemcpyAsync(open.data(), d_open, n * sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) { rc = 2; break; }
        std::vector<DfField> rel, ext, mx;
        long long ecells = 0, mcells = 0;
        for (int k = 0; k < n; ++k) {
            const DfField& f = map[k];
            if (df_goal_inside(f) && !open[k]) { rel.push_back(f); continue; }
            DfField m = f;
            m.cell_base = mcells; mcells += (long long)f.w * f.h;
            mx.push_back(m);
            DfField e;
            memset(&e, 0, sizeof(e));
            e.w = 2 * f.w - 1; e.h = 2 * f.h - 1; e.gi = f.gi + f.w - 1; e.gj = f.gj + f.h - 1;
            e.tiles_j = (e.h + DF_TILE - 1) / DF_TILE;
            e.cell_base = ecells; ecells += (long long)e.w * e.h;
            ext.push_back(e);
        }
        const int n_ext = (int)ext.size();
        const DfField* d_rel = d_map;        // no extended grid: the wavefront runs on the map table as seeded
        const DfField* d_ex = nullptr;
        if (n_ext) {
            // the closed maps and the extended grids get a tiling of their own, a workspace for it and a new first frontier
            n_tiles = 0;
            rel.insert(rel.end(), ext.begin(), ext.end());
            for (DfField& f : rel) { f.tile_base = (int)std::min(n_tiles, (long long)INT_MAX); n_tiles += (long long)((f.w + DF_TILE - 1) / DF_TILE) * f.tiles_j; }
            if (n_tiles > max_tiles) { hl_set_error("%s: %lld tiles exceed the %lld of one wavefront", what, n_tiles, max_tiles); rc = 1; break; }
            const size_t ext_bytes = (size_t)n * sizeof(DfField) + 3 * sizeof(double) * (size_t)ecells + df_ws_ints(n_tiles) * sizeof(int) + (size_t)ecells;
            if (cudaMalloc(&d_ext, ext_bytes) != cudaSuccess) {
                cudaGetLastError();
                hl_set_error("%s: the extended grids of %d maps with a free border cell or a border goal need %zu bytes, "
                             "cudaMalloc failed", what, n_ext, ext_bytes);
                rc = 1; break;
            }
            DfField* d_rel2 = (DfField*)d_ext;
            double* C = (double*)(d_rel2 + n);
            ws = (int*)(C + 3 * ecells);
            uint8_t* eocc = (uint8_t*)(ws + df_ws_ints(n_tiles));
            const int n_rel = (int)rel.size();
            for (int k = n_rel - n_ext; k < n_rel; ++k) { rel[k].occ = eocc + rel[k].cell_base; rel[k].D = C + rel[k].cell_base; }
            d_rel = d_rel2;
            d_ex = d_rel2 + (n_rel - n_ext);
            if (cudaMemsetAsync(ws, 0, df_ws_ints(n_tiles) * sizeof(int), st) != cudaSuccess ||
                cudaMemcpyAsync(d_rel2, rel.data(), n_rel * sizeof(DfField), cudaMemcpyHostToDevice, st) != cudaSuccess ||
                cudaMemcpyAsync(d_mx, mx.data(), n_ext * sizeof(DfField), cudaMemcpyHostToDevice, st) != cudaSuccess) { rc = 2; break; }
            k_df_ext_init<<<(unsigned)((ecells + 255) / 256), 256, 0, st>>>(d_mx, d_ex, n_ext, ecells, eocc);
            k_df_seed<<<(unsigned)((n_rel + 127) / 128), 128, 0, st>>>(d_rel2, n_rel, (int2*)ws, ws + 6 * n_tiles);
        }
        if (df_wavefront(what, n_ext ? rel : map, d_rel, ws, (int)n_tiles, mv, st, &sweeps)) { rc = 1; break; }
        if (!n_ext) break;
        // closing-order priorities of all extended grids to their fixed point, then the fold into the maps
        double* C = (double*)((DfField*)d_ext + n);
        double* P0 = C + ecells; double* P1 = C + 2 * ecells;
        if (cudaMemcpyAsync(P0, C, sizeof(double) * (size_t)ecells, cudaMemcpyDeviceToDevice, st) != cudaSuccess) { rc = 2; break; }
        const unsigned eblocks = (unsigned)((ecells + 255) / 256);
        int max_it = 0;
        for (const DfField& e : ext) max_it = std::max(max_it, 4 * (e.w + e.h));
        int it = 0, h_changed = 1;
        while (h_changed && it < max_it) {
            cudaMemsetAsync(d_changed, 0, sizeof(int), st);
            k_df_prio<<<eblocks, 256, 0, st>>>(d_ex, n_ext, ecells, P0, P1, mv, d_changed);
            if (cudaMemcpyAsync(&h_changed, d_changed, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) { rc = 2; break; }
            double* t = P0; P0 = P1; P1 = t;
            ++it; ++sweeps;
        }
        if (rc) break;
        if (h_changed) { hl_set_error("%s: closing-order priorities did not converge", what); rc = 1; break; }
        k_df_fold<<<(unsigned)((mcells + 255) / 256), 256, 0, st>>>(d_mx, d_ex, n_ext, mcells, P0);
        if (cudaStreamSynchronize(st) != cudaSuccess) { rc = 2; break; }
    } while (0);
    if (rc == 2) hl_set_error("%s: CUDA error: %s", what, cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_tab);
    if (d_ext) cudaFree(d_ext);
    if (h_sweeps) *h_sweeps = sweeps;
    return rc ? 1 : 0;
}

extern "C" int hl_distance_field(hl_ctx* ctx, const uint8_t* d_occ, int32_t w, int32_t h, int32_t gi,
                                 int32_t gj, int32_t motion_type, double* d_out, int32_t* h_sweeps,
                                 void* stream) {
    if (!ctx || !d_occ || !d_out || w < 1 || h < 1) { hl_set_error("hl_distance_field: bad arguments"); return 1; }
    if (gi < 0 || gj < 0 || gi >= w || gj >= h) { hl_set_error("hl_distance_field: goal (%d,%d) outside the %dx%d grid", gi, gj, w, h); return 1; }
    if (hl_enter(ctx, nullptr, d_out, "hl_distance_field")) return 1;
    DfMoves mv;
    if (!df_moves(motion_type, &mv)) { hl_set_error("hl_distance_field: motion_type must be 0 (King) or 1 (Pawn)"); return 1; }
    const HlGridField f = {0, 0, w, h, gi, gj};
    return df_run("hl_distance_field", d_occ, &f, 1, mv, d_out, h_sweeps, (cudaStream_t)stream);
}

extern "C" int hl_distance_field_batch(hl_ctx* ctx, const uint8_t* d_occ, int64_t occ_bytes, const HlGridField* h_fields,
                                       int32_t n_fields, int32_t motion_type, double* d_out, int64_t out_elems,
                                       int32_t* h_sweeps, void* stream) {
    const char* what = "hl_distance_field_batch";
    if (h_sweeps) *h_sweeps = 0;
    if (!ctx || n_fields < 0 || occ_bytes < 0 || out_elems < 0 || (n_fields > 0 && (!h_fields || !d_occ || !d_out))) {
        hl_set_error("%s: bad arguments", what); return 1;
    }
    DfMoves mv;
    if (!df_moves(motion_type, &mv)) { hl_set_error("%s: motion_type must be 0 (King) or 1 (Pawn), got %d", what, motion_type); return 1; }
    for (int k = 0; k < n_fields; ++k) {
        const HlGridField& f = h_fields[k];
        if (f.w < 1 || f.h < 1) { hl_set_error("%s: field %d: a %dx%d grid (w and h must be at least 1)", what, k, f.w, f.h); return 1; }
        if (f.gi < 0 || f.gj < 0 || f.gi >= f.w || f.gj >= f.h) {
            hl_set_error("%s: field %d: goal (%d,%d) outside the %dx%d grid", what, k, f.gi, f.gj, f.w, f.h); return 1;
        }
        const long long cells = (long long)f.w * f.h;
        if (f.occ_offset < 0 || f.occ_offset > occ_bytes - cells) {
            hl_set_error("%s: field %d: grid bytes [%lld, %lld) outside the %lld bytes of d_occ", what, k,
                         (long long)f.occ_offset, (long long)f.occ_offset + cells, (long long)occ_bytes); return 1;
        }
        if (f.out_offset < 0 || f.out_offset > out_elems - cells) {
            hl_set_error("%s: field %d: output slice [%lld, %lld) outside the %lld elements of d_out", what, k,
                         (long long)f.out_offset, (long long)f.out_offset + cells, (long long)out_elems); return 1;
        }
    }
    // sorted by start, two slices overlap only if some pair of neighbours does
    std::vector<int> order(n_fields);
    for (int k = 0; k < n_fields; ++k) order[k] = k;
    std::sort(order.begin(), order.end(), [&](int a, int b) {
        return h_fields[a].out_offset != h_fields[b].out_offset ? h_fields[a].out_offset < h_fields[b].out_offset : a < b;
    });
    for (int k = 1; k < n_fields; ++k) {
        const HlGridField& a = h_fields[order[k - 1]];
        if (h_fields[order[k]].out_offset < a.out_offset + (long long)a.w * a.h) {
            hl_set_error("%s: fields %d and %d: output slices overlap", what, std::min(order[k - 1], order[k]),
                         std::max(order[k - 1], order[k]));
            return 1;
        }
    }
    if (n_fields == 0) return 0;
    if (hl_enter(ctx, nullptr, d_occ, what) || hl_enter(ctx, nullptr, d_out, what)) return 1;
    return df_run(what, d_occ, h_fields, n_fields, mv, d_out, h_sweeps, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------- K7
__global__ void k_grid_pack(const uint8_t* __restrict__ occ, long long cells, uint32_t* __restrict__ bits) {
    long long wd = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long n_words = (cells + 31) / 32;
    if (wd >= n_words) return;
    uint32_t v = 0;
    for (int b = 0; b < 32; ++b) {
        long long c = wd * 32 + b;
        if (c < cells && occ[c]) v |= 1u << b;
    }
    bits[wd] = v;
}

extern "C" int hl_grid_pack(hl_ctx* ctx, const uint8_t* d_occ, int32_t w, int32_t h, uint32_t* d_bits, void* stream) {
    if (!ctx || !d_occ || !d_bits || w <= 0 || h <= 0) { hl_set_error("hl_grid_pack: bad arguments"); return 1; }
    if (hl_enter(ctx, nullptr, d_bits, "hl_grid_pack")) return 1;
    long long cells = (long long)w * h, n_words = (cells + 31) / 32;
    k_grid_pack<<<(unsigned)((n_words + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_occ, cells, d_bits);
    HL_CUDA_OK(cudaGetLastError());
    return 0;
}

// any occupied bit among cells (i, j0..j1) of the bit-packed grid
__device__ __forceinline__ bool row_any(const uint32_t* __restrict__ bits, long long base, int j0, int j1) {
    long long a = base + j0, b = base + j1;
    long long wa = a >> 5, wb = b >> 5;
    for (long long wd = wa; wd <= wb; ++wd) {
        uint32_t m = 0xFFFFFFFFu;
        if (wd == wa) m &= 0xFFFFFFFFu << (a & 31);
        if (wd == wb) m &= 0xFFFFFFFFu >> (31 - (b & 31));
        if (__ldg(bits + wd) & m) return true;
    }
    return false;
}

// Cells [lo, hi] (global indices, clamped to [g0, g0+n-1]) whose closed interval [fl(i*res), fl((i+1)*res)] meets
// [vmin, vmax].  fl(i*res) is monotone in i, so the candidates are contiguous: start from the floor() estimate (clamped
// to [g0-1, g0+n] before the conversion, so huge coordinates cannot overflow) and step it by the edge comparisons
// themselves.  floor(v/res) alone is off by one where fl(i*res)/res rounds below i (an edge touching from below) or an
// edge one ulp below fl(i*res) still divides to i (an overlap of one ulp).  Indices are 64-bit here so that g0 - 1 and
// g0 + n + 1 stay representable; (double)i + 1.0 is exactly (double)(i + 1) for every int32 i.
__device__ __forceinline__ void cell_range(double vmin, double vmax, double res, int g0, int n, long long& lo, long long& hi) {
    const long long a = (long long)g0 - 1, b = (long long)g0 + n;
    lo = (long long)fmin(fmax(floor(vmin / res), (double)a), (double)b);
    while (lo > a && (double)lo * res >= vmin) --lo;             // cell lo-1 ends at fl(lo*res) >= vmin
    while (lo < b && ((double)lo + 1.0) * res < vmin) ++lo;      // cell lo ends before vmin
    hi = (long long)fmin(fmax(floor(vmax / res), (double)a), (double)b);
    while (hi < b && ((double)hi + 1.0) * res <= vmax) ++hi;     // cell hi+1 starts at or before vmax
    while (hi > a && (double)hi * res > vmax) --hi;              // cell hi starts after vmax
    lo = max(lo, (long long)g0); hi = min(hi, b - 1);
}

// (gi0, gj0): global index of the grid's cell (0, 0); bits are indexed by the local cell (i - gi0) * H + (j - gj0)
__global__ void __launch_bounds__(256)
k_grid_footprint(const uint32_t* __restrict__ bits, int W, int H, int gi0, int gj0, double res, const double* __restrict__ poses,
                 long long n, double x0, double x1, double y0, double y1, uint8_t* __restrict__ out) {
    long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const double px = poses[3 * idx], py = poses[3 * idx + 1], yaw = poses[3 * idx + 2];
    // a pose that is not finite can never be certified free (fmin / fmax below would drop NaN corners)
    if (!isfinite(px) || !isfinite(py) || !isfinite(yaw)) { out[idx] = 1; return; }
    const double c = cos(yaw), s = sin(yaw);
    const double lx[4] = {x0, x0, x1, x1}, ly[4] = {y1, y0, y0, y1};
    double cx[4], cy[4];
    double xmin = INFINITY, xmax = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        cx[k] = xadd(xsub(xmul(c, lx[k]), xmul(s, ly[k])), px);
        cy[k] = xadd(xadd(xmul(s, lx[k]), xmul(c, ly[k])), py);
        xmin = fmin(xmin, cx[k]); xmax = fmax(xmax, cx[k]);
    }
    // closed sets: a rectangle touching a cell edge meets the cells on both sides of it
    long long ia, ib;
    cell_range(xmin, xmax, res, gi0, W, ia, ib);
    bool hit = false;
    for (long long i = ia; i <= ib && !hit; ++i) {
        const double a = (double)i * res, b = ((double)i + 1.0) * res;
        double ymin = INFINITY, ymax = -INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (cx[k] >= a && cx[k] <= b) { ymin = fmin(ymin, cy[k]); ymax = fmax(ymax, cy[k]); }
            const int k2 = (k + 1) & 3;
            const double ex = cx[k2] - cx[k];
            if (ex != 0.0) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double X = e ? b : a;
                    if ((cx[k] - X) * (cx[k2] - X) < 0.0) {
                        double y = cy[k] + (X - cx[k]) * (cy[k2] - cy[k]) / ex;
                        ymin = fmin(ymin, y); ymax = fmax(ymax, y);
                    }
                }
            }
        }
        if (ymin > ymax) continue;
        long long ja, jb;
        cell_range(ymin, ymax, res, gj0, H, ja, jb);
        if (ja <= jb) hit = row_any(bits, (i - gi0) * H, (int)(ja - gj0), (int)(jb - gj0));
    }
    out[idx] = hit ? 1 : 0;
}

static int grid_footprint_launch(hl_ctx* ctx, const uint32_t* d_occ_bits, int32_t w, int32_t h, int32_t i0, int32_t j0,
                                 double res, const double* d_poses, int64_t n, const double body_ext[4], uint8_t* d_out,
                                 void* stream, const char* what) {
    if (n == 0) return 0;
    if (hl_enter(ctx, nullptr, d_out, what)) return 1;
    k_grid_footprint<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_occ_bits, w, h, i0, j0, res, d_poses, (long long)n, body_ext[0], body_ext[1], body_ext[2], body_ext[3], d_out);
    HL_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int hl_grid_footprint_check(hl_ctx* ctx, const uint32_t* d_occ_bits, int32_t w, int32_t h,
                                       double res, const double* d_poses, int64_t n,
                                       const double body_ext[4], uint8_t* d_out, void* stream) {
    if (!ctx || !d_occ_bits || !d_poses || !d_out || !body_ext || n < 0 || w <= 0 || h <= 0 || !(res > 0)) {
        hl_set_error("hl_grid_footprint_check: bad arguments"); return 1;
    }
    return grid_footprint_launch(ctx, d_occ_bits, w, h, 0, 0, res, d_poses, n, body_ext, d_out, stream, "hl_grid_footprint_check");
}

extern "C" int hl_grid_footprint_check_at(hl_ctx* ctx, const uint32_t* d_occ_bits, int32_t w, int32_t h, int32_t i0,
                                          int32_t j0, double res, const double* d_poses, int64_t n,
                                          const double body_ext[4], uint8_t* d_out, void* stream) {
    const char* what = "hl_grid_footprint_check_at";
    if (!ctx || !d_occ_bits || !d_poses || !d_out || !body_ext || n < 0 || w <= 0 || h <= 0 || !(res > 0) || !isfinite(res)) {
        hl_set_error("%s: bad arguments", what); return 1;
    }
    if ((long long)i0 + w > INT_MAX || (long long)j0 + h > INT_MAX) {
        hl_set_error("%s: a %dx%d grid at (%d, %d) overflows the int32 cell index", what, w, h, i0, j0); return 1;
    }
    if (!isfinite((double)i0 * res) || !isfinite((double)(i0 + w) * res) || !isfinite((double)j0 * res) ||
        !isfinite((double)(j0 + h) * res)) {
        hl_set_error("%s: the grid's cell edges are not finite at res = %g", what, res); return 1;
    }
    return grid_footprint_launch(ctx, d_occ_bits, w, h, i0, j0, res, d_poses, n, body_ext, d_out, stream, what);
}
