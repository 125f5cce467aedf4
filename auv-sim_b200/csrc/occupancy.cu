// occupancy.cu -- SharkOccupancyGrid.convert (/root/reference/path_planning/sharkOccupancyGrid.py:47-71):
// shark tracks -> per-time-bin AUV-detection probability grids, the [T][C] input of the path cost.
// SURVEY.md section 8(f) row N2: the data format on the producer side of the hot path.
//
//   k_occ_hist  one thread per track point: first time bin containing t (:253-258), first cell (in
//               cell_list order) that contains the point, boundary included (`point.within(cell) or
//               cell.touches(point)`, :232; exact orientation predicate), searched among the candidates of
//               the point's bucket (auvrrt_occ_create) -> integer histogram; also createBinList's T
//   k_occ_norm  occupancy of (bin, shark, square): 0.01 for squares that hold a cell, +1 per point
//               (added one by one, as the reference does), / (points + 0.01 * cells)   (:217-241)
//   k_occ_auv   disc sum of radius ceil(range / cell) around every cell, in the reference's window
//               order (:189-201)
//   k_occ_avg   mean over sharks, in dict order                                           (:160-171)
//   k_occ_to_env  a world's probs[b][c] = grid[b][cellToIndex(c)] (createSharkGrid's layout), fp64 and fp32
// All of them run from an auvrrt_occ handle, asynchronously on the caller's stream, with no allocation.
// fp64 with separately rounded operations: bit-identical to the reference (tests/golden/occupancy.npz).
#include <math.h>
#include <string.h>
#include <algorithm>
#include <cmath>
#include <memory>
#include <vector>
#include "launch.h"

namespace auv {

// +1 strictly inside, 0 on the boundary, -1 outside; ragged polygon, exact.  Not inlined: k_occ_hist then keeps
// no live registers across the exact-orientation fallback call, and spills nothing.
__device__ __noinline__ int poly_locate(const double *xy, int n, double px, double py) {
    bool inside = false, boundary = false;
    for (int i = 0; i < n; i++) {
        const int j = i + 1 == n ? 0 : i + 1;
        const double ax = xy[2 * i], ay = xy[2 * i + 1], bx = xy[2 * j], by = xy[2 * j + 1];
        if (px == ax && py == ay) boundary = true;
        if (ay == py && by == py) {
            if (fmin(ax, bx) <= px && px <= fmax(ax, bx)) boundary = true;
            continue;
        }
        if ((ay > py) != (by > py)) {
            const int s = orient2d(ax, ay, bx, by, px, py);
            if (s == 0) boundary = true;
            if ((s > 0) == (by > ay)) inside = !inside;
        }
    }
    return boundary ? 0 : (inside ? 1 : -1);
}

// the bucket grid of the candidate-cell index (auvrrt_occ_create): buckets of side `side` from (x0, y0), nx * ny of
// them, over the union [x0, x1] x [y0, y1] of the cells' bounding boxes
struct OccIndex { double x0, y0, x1, y1, side; int nx, ny; };

__global__ void __launch_bounds__(256) k_occ_hist(const double *cell_xy, const long long *cell_off, const double *cell_bb,
                                                  const int *cell_sq, const int *bkt_off, const int *bkt_cell, OccIndex ix,
                                                  const double *trk, const long long *trk_off, long long n, int T, int S,
                                                  int RC, double bin_interval, int *counts, int *npts, int *t_occ) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n) return;
    int lo = 0, hi = S - 1;                                  // shark of point k: the last s with trk_off[s] <= k
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (trk_off[mid] <= k) lo = mid; else hi = mid - 1;
    }
    const int s = lo;
    if (!(trk_off[s] <= k && k < trk_off[s + 1])) return;    // a point of no track
    const double x = trk[3 * k], y = trk[3 * k + 1], t = trk[3 * k + 2];
    // createBinList's T = floor(longest / bin_interval), longest = max(0, last stamp of every track) (:307-314)
    if (t_occ && k == trk_off[s + 1] - 1 && t > 0.0) atomicMax(t_occ, (int)floor(__ddiv_rn(t, bin_interval)));
    int tb = -1;
    for (int b = 0; b < T; b++)
        if (t >= __dmul_rn((double)b, bin_interval) && t <= __dmul_rn((double)(b + 1), bin_interval)) { tb = b; break; }
    if (tb < 0) return;
    atomicAdd(&npts[tb * S + s], 1);
    // the bucket's list holds, in cell_list order, every cell whose bounding box can contain the point, so the first
    // match below is the first match of a scan over all cells
    if (ix.nx <= 0 || !(x >= ix.x0 && x <= ix.x1 && y >= ix.y0 && y <= ix.y1)) return;
    const int bx = min(max((int)floor(__ddiv_rn(__dsub_rn(x, ix.x0), ix.side)), 0), ix.nx - 1);
    const int by = min(max((int)floor(__ddiv_rn(__dsub_rn(y, ix.y0), ix.side)), 0), ix.ny - 1);
    const int bk = by * ix.nx + bx;
    for (int q = bkt_off[bk]; q < bkt_off[bk + 1]; q++) {
        const int c = bkt_cell[q];
        const double *bb = cell_bb + 4 * c;
        if (x < bb[0] || x > bb[2] || y < bb[1] || y > bb[3]) continue;       // outside the cell's bounding box
        if (poly_locate(cell_xy + 2 * cell_off[c], (int)(cell_off[c + 1] - cell_off[c]), x, y) >= 0) {
            atomicAdd(&counts[((size_t)tb * S + s) * RC + cell_sq[c]], 1);
            break;
        }
    }
}

__global__ void __launch_bounds__(256) k_occ_norm(const int *counts, const int *npts, const unsigned char *is_cell, int T,
                                                  int S, int RC, int C, double *occ) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= (long long)T * S * RC) return;
    const int sq = (int)(i % RC);
    const long long bs = i / RC;
    double v = is_cell[sq] ? 0.01 : 0.0;
    const int cnt = counts[i];
    for (int k = 0; k < cnt; k++) v = __dadd_rn(v, 1.0);                        // `grid[row][col] += 1` per point
    const double nor = __dadd_rn((double)npts[bs], __dmul_rn((double)C, 0.01));
    occ[i] = __ddiv_rn(v, nor);
}

__global__ void __launch_bounds__(256) k_occ_auv(const double *occ, const int *sq_off, int T, int S,
                                                 int rows, int cols, int count, double *auv) {
    const int RC = rows * cols;
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= (long long)T * S * RC) return;
    const int sq = (int)(i % RC), row = sq / cols, col = sq % cols;
    const double *o = occ + (i - sq);
    double acc = 0.0;
    for (int cc = sq_off[sq]; cc < sq_off[sq + 1]; cc++) {        // one pass per cell mapped to this square (:190)
        for (int a = 0; a < 4 * count; a++) {
            const int rt = row - 2 * count + a;
            for (int b = 0; b < 4 * count; b++) {
                const int ct = col - 2 * count + b;
                if (rt >= 0 && rt < rows && ct >= 0 && ct < cols) {
                    const int dr = rt - row, dc = ct - col;
                    if (dr * dr + dc * dc <= count * count) acc = __dadd_rn(acc, o[rt * cols + ct]);
                }
            }
        }
    }
    auv[i] = acc;
}

__global__ void __launch_bounds__(256) k_occ_avg(const double *auv, int T, int S, int RC, double *grid) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= (long long)T * RC) return;
    const int sq = (int)(i % RC);
    const int b = (int)(i / RC);
    double acc = 0.0;
    for (int s = 0; s < S; s++) acc = __dadd_rn(acc, auv[((size_t)b * S + s) * RC + sq]);
    grid[i] = __ddiv_rn(acc, (double)S);
}

// probs[b][c] of both precisions' world blobs: grid[b][cell_sq[c]] of an occupancy grid [T][RC], or (cell_sq NULL) a
// probs[T][C] table.  __double2float_rn is the round-to-nearest host cast of build_blob.
__global__ void __launch_bounds__(256) k_occ_to_env(const double *src, const int *cell_sq, int T, int C, int RC, double *p64,
                                                    float *p32) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= (long long)T * C) return;
    const int c = (int)(i % C);
    const long long b = i / C;
    const double v = cell_sq ? src[b * RC + cell_sq[c]] : src[i];
    p64[i] = v;
    p32[i] = __double2float_rn(v);
}

int launch_probs_to_env(auvrrt_env *env, const double *src, const int *cell_sq, int RC, cudaStream_t s) {
    const long long n = (long long)env->T * env->C;
    if (n == 0) return AUVRRT_OK;
    k_occ_to_env<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, cell_sq, env->T, env->C, RC,
                                                             (double *)(env->blob64 + env->h64.off_probs),
                                                             (float *)(env->blob32 + env->h32.off_probs));
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

}  // namespace auv

using namespace auv;

// One SharkOccupancyGrid with fixed cells, bounds, cell size, bins and detection range.  Everything that does not
// depend on the tracks lives in one device allocation made at creation: the cell tables, the candidate-cell index and
// the per-call workspace (sized for n_bins x max_sharks).
struct auvrrt_occ {
    int device, C, rows, cols, RC, n_bins, max_sharks, count;
    int64_t max_points;
    double bin_interval;
    OccIndex ix;
    void *arena;
    const double *d_xy, *d_bb;
    const long long *d_off;
    const int *d_csq, *d_sqo, *d_boff, *d_bcell;
    const unsigned char *d_isc;
    int *d_cnt, *d_np;
    double *d_occ, *d_auv, *d_grid;
};

static int occ_shape(const double bounds[4], double cell_size, int *rows, int *cols) {
    *cols = (int)(ceil(bounds[2] - bounds[0]) / cell_size) + 1;
    *rows = (int)(ceil(bounds[3] - bounds[1]) / cell_size) + 1;
    return AUVRRT_OK;
}

extern "C" int auvrrt_occupancy_dims(const double bounds[4], double cell_size, double bin_interval, const double *tracks,
                                     const int64_t *track_off, int S, int *T, int *rows, int *cols) {
    if (!bounds || !track_off || !T || !rows || !cols || !(cell_size > 0) || !(bin_interval > 0))
        return set_err(AUVRRT_ERR_ARG, "occupancy_dims: bad argument");
    double longest = 0;                                                                  // createBinList :307-314
    for (int s = 0; s < S; s++)
        if (track_off[s + 1] > track_off[s] && tracks[3 * (track_off[s + 1] - 1) + 2] > longest)
            longest = tracks[3 * (track_off[s + 1] - 1) + 2];
    *T = (int)floor(longest / bin_interval);
    return occ_shape(bounds, cell_size, rows, cols);
}

extern "C" void auvrrt_occ_destroy(auvrrt_occ_t *o) {
    if (!o) return;
    if (o->arena) { cudaSetDevice(o->device); cudaFree(o->arena); }
    delete o;
}

extern "C" int auvrrt_occ_create(const double *cell_xy, const int64_t *cell_off, int C, const double bounds[4], double cell_size,
                                 double bin_interval, double detect_range, int n_bins, int max_sharks, int64_t max_points,
                                 int device, auvrrt_occ_t **out) {
    if (!out) return set_err(AUVRRT_ERR_ARG, "occ_create: out is NULL");
    *out = nullptr;
    if (C < 0 || (C > 0 && (!cell_xy || !cell_off)) || !bounds || !(cell_size > 0) || !(bin_interval > 0) || n_bins < 1 ||
        max_sharks < 1 || max_points < 0)
        return set_err(AUVRRT_ERR_ARG, "occ_create: bad argument");
    int rows, cols;
    occ_shape(bounds, cell_size, &rows, &cols);
    if (rows < 1 || cols < 1 || (int64_t)rows * cols > INT32_MAX) return set_err(AUVRRT_ERR_ARG, "occ_create: bad grid shape %d x %d", rows, cols);
    const int RC = rows * cols;
    // host-side flattening: bounding boxes, square index of every cell (cellToIndex :294-299), cells per square
    std::vector<double> bb(4 * (size_t)std::max(C, 1));
    std::vector<int> csq(std::max(C, 1)), sq_off(RC + 1, 0);
    std::vector<unsigned char> is_cell(RC, 0);
    double ux0 = INFINITY, uy0 = INFINITY, ux1 = -INFINITY, uy1 = -INFINITY;
    for (int c = 0; c < C; c++) {
        double x0 = INFINITY, y0 = INFINITY, x1 = -INFINITY, y1 = -INFINITY;
        for (int64_t k = cell_off[c]; k < cell_off[c + 1]; k++) {
            x0 = fmin(x0, cell_xy[2 * k]); x1 = fmax(x1, cell_xy[2 * k]); y0 = fmin(y0, cell_xy[2 * k + 1]); y1 = fmax(y1, cell_xy[2 * k + 1]);
        }
        bb[4 * c] = x0; bb[4 * c + 1] = y0; bb[4 * c + 2] = x1; bb[4 * c + 3] = y1;
        ux0 = fmin(ux0, x0); uy0 = fmin(uy0, y0); ux1 = fmax(ux1, x1); uy1 = fmax(uy1, y1);
        const int col = (int)((x0 - bounds[0]) / cell_size), row = (int)((y0 - bounds[1]) / cell_size);
        if (row < 0 || row >= rows || col < 0 || col >= cols) return set_err(AUVRRT_ERR_ARG, "occupancy_grid: cell %d lies outside the boundary's grid (IndexError in the reference)", c);
        csq[c] = row * cols + col; is_cell[csq[c]] = 1; sq_off[csq[c] + 1]++;
    }
    for (int i = 0; i < RC; i++) sq_off[i + 1] += sq_off[i];
    // candidate-cell index: a bucket grid of side cell_size (doubled until there are at most 2^22 buckets) over the
    // union of the cells' bounding boxes.  Bucket (bx, by) lists, in cell_list order, the cells whose closed bounding
    // box grown by `margin` meets it.  The margin is far above the rounding error of the device's bucket index
    // floor((x - x0) / side), and both sides compute it with the same separately rounded fp64 operations, so the bucket
    // a point is filed under lists every cell whose bounding box holds the point.
    OccIndex ix;
    ix.x0 = ux0; ix.y0 = uy0; ix.x1 = ux1; ix.y1 = uy1; ix.side = cell_size; ix.nx = ix.ny = 0;
    std::vector<int> boff(1, 0), bcell;
    const bool finite_box = C > 0 && std::isfinite(ux0) && std::isfinite(uy0) && std::isfinite(ux1) && std::isfinite(uy1);
    if (finite_box) {
        const double margin = 1e-9 * std::max({1.0, fabs(ux0), fabs(uy0), fabs(ux1), fabs(uy1), ux1 - ux0, uy1 - uy0});
        for (;;) {
            const double nx = floor((ux1 - ux0) / ix.side) + 1, ny = floor((uy1 - uy0) / ix.side) + 1;
            if (nx * ny <= 4194304.0) { ix.nx = (int)nx; ix.ny = (int)ny; break; }
            ix.side *= 2;
        }
        const int NBK = ix.nx * ix.ny;
        auto range = [&](double lo, double hi, double o, int n, int &i0, int &i1) {
            i0 = std::min(std::max((int)floor((lo - margin - o) / ix.side), 0), n - 1);
            i1 = std::min(std::max((int)floor((hi + margin - o) / ix.side), 0), n - 1);
        };
        std::vector<int64_t> cnt(NBK + 1, 0);
        for (int pass = 0; pass < 2; pass++) {
            std::vector<int64_t> fill;
            if (pass == 1) {
                for (int b = 0; b < NBK; b++) cnt[b + 1] += cnt[b];
                if (cnt[NBK] > INT32_MAX) return set_err(AUVRRT_ERR_UNSUPPORTED, "occ_create: the cell index would hold more than 2^31 entries");
                fill.assign(cnt.begin(), cnt.end() - 1);
                bcell.resize(std::max<int64_t>(cnt[NBK], 1));
            }
            for (int c = 0; c < C; c++) {
                int i0, i1, j0, j1;
                range(bb[4 * c], bb[4 * c + 2], ux0, ix.nx, i0, i1);
                range(bb[4 * c + 1], bb[4 * c + 3], uy0, ix.ny, j0, j1);
                for (int j = j0; j <= j1; j++)
                    for (int i = i0; i <= i1; i++) {
                        if (pass == 0) cnt[(size_t)j * ix.nx + i + 1]++;
                        else bcell[fill[(size_t)j * ix.nx + i]++] = c;
                    }
            }
        }
        boff.resize(NBK + 1);
        for (int b = 0; b <= NBK; b++) boff[b] = (int)cnt[b];
    }
    if (bcell.empty()) bcell.push_back(0);
    AUV_TRY(need_device(device));
    // one allocation: the tables (uploaded once), then the workspace
    const size_t nv = C > 0 ? (size_t)cell_off[C] : 0, ws = (size_t)n_bins * max_sharks * RC;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 255) & ~(size_t)255; return r; };
    const size_t o_xy = take(16 * nv), o_off = take(8 * (size_t)(C + 1)), o_bb = take(32 * (size_t)C), o_csq = take(4 * (size_t)C),
                 o_isc = take((size_t)RC), o_sqo = take(4 * (size_t)(RC + 1)), o_boff = take(4 * boff.size()),
                 o_bcell = take(4 * bcell.size());
    const size_t tables = o;
    const size_t o_cnt = take(4 * ws), o_np = take(4 * (size_t)n_bins * max_sharks), o_occ = take(8 * ws), o_auv = take(8 * ws),
                 o_grid = take(8 * (size_t)n_bins * RC);
    std::vector<unsigned char> h(tables, 0);
    if (nv) memcpy(h.data() + o_xy, cell_xy, 16 * nv);
    if (C > 0) {
        memcpy(h.data() + o_off, cell_off, 8 * (size_t)(C + 1));
        memcpy(h.data() + o_bb, bb.data(), 32 * (size_t)C);
        memcpy(h.data() + o_csq, csq.data(), 4 * (size_t)C);
    }
    memcpy(h.data() + o_isc, is_cell.data(), (size_t)RC);
    memcpy(h.data() + o_sqo, sq_off.data(), 4 * (size_t)(RC + 1));
    memcpy(h.data() + o_boff, boff.data(), 4 * boff.size());
    memcpy(h.data() + o_bcell, bcell.data(), 4 * bcell.size());
    auvrrt_occ *q = new auvrrt_occ();
    memset(q, 0, sizeof(*q));
    q->device = device; q->C = C; q->rows = rows; q->cols = cols; q->RC = RC; q->n_bins = n_bins; q->max_sharks = max_sharks;
    q->max_points = max_points; q->bin_interval = bin_interval; q->ix = ix;
    q->count = (int)ceil(detect_range / cell_size);
    cudaError_t er = cudaMalloc(&q->arena, o);
    if (er == cudaSuccess) er = cudaMemcpy(q->arena, h.data(), tables, cudaMemcpyHostToDevice);
    if (er != cudaSuccess) {
        auvrrt_occ_destroy(q);
        return set_err(AUVRRT_ERR_CUDA, "occ_create: %s", cudaGetErrorString(er));
    }
    unsigned char *a = (unsigned char *)q->arena;
    q->d_xy = (const double *)(a + o_xy); q->d_off = (const long long *)(a + o_off); q->d_bb = (const double *)(a + o_bb);
    q->d_csq = (const int *)(a + o_csq); q->d_isc = a + o_isc; q->d_sqo = (const int *)(a + o_sqo);
    q->d_boff = (const int *)(a + o_boff); q->d_bcell = (const int *)(a + o_bcell);
    q->d_cnt = (int *)(a + o_cnt); q->d_np = (int *)(a + o_np); q->d_occ = (double *)(a + o_occ); q->d_auv = (double *)(a + o_auv);
    q->d_grid = (double *)(a + o_grid);
    *out = q;
    return AUVRRT_OK;
}

extern "C" int auvrrt_occ_shape(const auvrrt_occ_t *o, int *T, int *rows, int *cols) {
    if (!o) return set_err(AUVRRT_ERR_ARG, "occ_shape: NULL handle");
    if (T) *T = o->n_bins;
    if (rows) *rows = o->rows;
    if (cols) *cols = o->cols;
    return AUVRRT_OK;
}

extern "C" int auvrrt_occ_grid_dev(auvrrt_occ_t *o, const double *d_tracks, const int64_t *d_track_off, int S, int64_t n_points,
                                   double *d_grid, auvrrt_env_t *env, int32_t *d_t_occ, void *stream) {
    if (!o || !d_track_off || (n_points > 0 && !d_tracks)) return set_err(AUVRRT_ERR_ARG, "occ_grid_dev: NULL argument");
    if (S < 1 || S > o->max_sharks) return set_err(AUVRRT_ERR_ARG, "occ_grid_dev: %d sharks, the handle takes 1 to %d", S, o->max_sharks);
    if (n_points < 0 || n_points > o->max_points)
        return set_err(AUVRRT_ERR_ARG, "occ_grid_dev: %lld points, the handle takes at most %lld", (long long)n_points, (long long)o->max_points);
    if (env) {
        if (env->device != o->device) return set_err(AUVRRT_ERR_ARG, "occ_grid_dev: the world is on device %d, the grid on %d", env->device, o->device);
        if (env->C != o->C || env->T != o->n_bins)
            return set_err(AUVRRT_ERR_ARG, "occ_grid_dev: the world has %d bins x %d cells, the grid %d x %d", env->T, env->C, o->n_bins, o->C);
        for (int b = 0; b < env->T; b++)
            if (!(env->h_bins[2 * b] == (double)b * o->bin_interval && env->h_bins[2 * b + 1] == (double)(b + 1) * o->bin_interval))
                return set_err(AUVRRT_ERR_ARG, "occ_grid_dev: bin %d of the world is (%.17g, %.17g), not (%d, %d) x %.17g (createBinList)",
                               b, env->h_bins[2 * b], env->h_bins[2 * b + 1], b, b + 1, o->bin_interval);
    }
    AUV_CUDA(cudaSetDevice(o->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int T = o->n_bins, RC = o->RC;
    const long long tot = (long long)T * S * RC;
    double *grid = d_grid ? d_grid : o->d_grid;
    AUV_CUDA(cudaMemsetAsync(o->d_cnt, 0, 4 * (size_t)tot, s));
    AUV_CUDA(cudaMemsetAsync(o->d_np, 0, 4 * (size_t)T * S, s));
    if (d_t_occ) AUV_CUDA(cudaMemsetAsync(d_t_occ, 0, 4, s));
    if (n_points > 0) {
        k_occ_hist<<<(unsigned)((n_points + 255) / 256), 256, 0, s>>>(o->d_xy, o->d_off, o->d_bb, o->d_csq, o->d_boff, o->d_bcell, o->ix,
                                                                      d_tracks, (const long long *)d_track_off, n_points, T, S, RC,
                                                                      o->bin_interval, o->d_cnt, o->d_np, d_t_occ);
        AUV_LAUNCH_CHECK();
    }
    k_occ_norm<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(o->d_cnt, o->d_np, o->d_isc, T, S, RC, o->C, o->d_occ);
    AUV_LAUNCH_CHECK();
    k_occ_auv<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(o->d_occ, o->d_sqo, T, S, o->rows, o->cols, o->count, o->d_auv);
    AUV_LAUNCH_CHECK();
    k_occ_avg<<<(unsigned)(((long long)T * RC + 255) / 256), 256, 0, s>>>(o->d_auv, T, S, RC, grid);
    AUV_LAUNCH_CHECK();
    if (env) return launch_probs_to_env(env, grid, o->d_csq, RC, s);
    return AUVRRT_OK;
}

// The one-shot host-buffer form: a handle for exactly these tracks' bins, sharks and points.
extern "C" int auvrrt_occupancy_grid(const double *cell_xy, const int64_t *cell_off, int C, const double bounds[4],
                                     double cell_size, double bin_interval, double detect_range, const double *tracks,
                                     const int64_t *track_off, int S, int device, double *out_grid, int64_t out_cap) {
    int T, rows, cols;
    int rc = auvrrt_occupancy_dims(bounds, cell_size, bin_interval, tracks, track_off, S, &T, &rows, &cols);
    if (rc) return rc;
    if (C < 0 || S <= 0 || !out_grid) return set_err(AUVRRT_ERR_ARG, "occupancy_grid: bad argument");
    const int RC = rows * cols;
    if ((int64_t)T * RC > out_cap) return set_err(AUVRRT_ERR_ARG, "occupancy_grid: output holds %lld values, %lld needed", (long long)out_cap, (long long)T * RC);
    if (T == 0) return AUVRRT_OK;
    AUV_TRY(need_device(device));
    const int64_t n = track_off[S];
    auvrrt_occ_t *o = nullptr;
    if ((rc = auvrrt_occ_create(cell_xy, cell_off, C, bounds, cell_size, bin_interval, detect_range, T, S, n, device, &o))) return rc;
    std::unique_ptr<auvrrt_occ_t, void (*)(auvrrt_occ_t *)> own(o, auvrrt_occ_destroy);
    const size_t trk_bytes = (24 * (size_t)n + 255) & ~(size_t)255;
    DBuf trk;
    AUV_TRY(trk.alloc(trk_bytes + 8 * (size_t)(S + 1)));
    double *d_trk = trk.as<double>();
    int64_t *d_toff = (int64_t *)((unsigned char *)trk.p + trk_bytes);
    if (n > 0) AUV_CUDA(cudaMemcpy(d_trk, tracks, 24 * (size_t)n, cudaMemcpyHostToDevice));
    AUV_CUDA(cudaMemcpy(d_toff, track_off, 8 * (size_t)(S + 1), cudaMemcpyHostToDevice));
    if ((rc = auvrrt_occ_grid_dev(o, d_trk, d_toff, S, n, nullptr, nullptr, nullptr, 0))) return rc;
    AUV_CUDA(cudaMemcpy(out_grid, o->d_grid, 8 * (size_t)T * RC, cudaMemcpyDeviceToHost));
    return AUVRRT_OK;
}
