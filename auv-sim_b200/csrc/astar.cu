// astar.cu -- the fixed-length lattice A* with the shark-occupancy cost,
// /root/reference/path_planning/astar_fixLenSOG.py (class astar, :114-657).  SURVEY.md 8(f) N4.
//
// One WARP per query.  The reference's open list is a Python list scanned for the first strict
// minimum of f and popped; relative order of the survivors never changes, so an append-only node
// array with an "alive" bit per node and a lowest-index tie-break selects the same node.  Per
// expansion the warp does
//   1. argmin of f over the alive nodes: lanes stride over the node array (coalesced fp64 loads),
//      then a 5-step shuffle reduction on (f, index);
//   2. the 8 neighbours, four lanes each: triangle-fan bounds test around the boundary centroid,
//      per-obstacle circle test, path length, time stamp -> time bin, cell lookup through a bucket
//      grid whose candidates are tested with the reference's own predicate in dict order, g, top-n
//      heuristic from per-bin prefix sums of the sorted probabilities, visited bitmap;
//   3. ordered append (ballot + popcount) so the open list has the reference's order.
// Everything is fp64 with separately rounded operations (no FMA contraction): the search is discrete,
// any rounding difference could change the expansion order, and the reference uses IEEE add / mul /
// sqrt only -- so the result is bit-identical (tests/golden/astar.npz).
#include <math.h>
#include <algorithm>
#include <new>
#include <vector>
#include "launch.h"

struct auvrrt_astar_env {
    int device;
    int K, E, H, T, C;
    double cx, cy;
    double *d_f64;          // circles | boundary | habitats | bins | cells_r | probs | topn
    int *d_i32;             // bucket offsets | bucket cells
    size_t off_circ, off_bnd, off_hab, off_bins, off_cells, off_probs, off_topn;
    double gx0, gy0, inv_bs;
    int gnx, gny;
    size_t n_boff;
    void *d_ws;
    size_t ws_bytes;
    cudaStream_t stream;
};

namespace auv {

typedef Ar<double, true> AD;

struct AstarDev {
    int K, E, H, T, C;
    const double *circles, *boundary, *habitats, *bins, *cells_r, *probs, *topn;
    double cx, cy;
    double gx0, gy0, inv_bs;
    int gnx, gny;
    const int *boff, *bcells;
};

#define ASTAR_VIS_WORDS 11264            /* 600 * 600 bits = 11250 words, padded */
#define ASTAR_WARPS 4

__host__ __device__ inline size_t astar_ws_per_query(int cap) {
    return (((size_t)cap * (5 * 8 + 2 * 4)) + 255 & ~(size_t)255) + (size_t)ASTAR_VIS_WORDS * 4;
}

// same_side (:178-186): np.cross of 2-vectors is a0*b1 - a1*b0, np.dot of the two scalars their product
__device__ __forceinline__ bool astar_same_side(double p1x, double p1y, double p2x, double p2y, double ax, double ay,
                                                double bx, double by) {
    const double ux = AD::sub(bx, ax), uy = AD::sub(by, ay);
    const double cp1 = AD::sub(AD::mul(ux, AD::sub(p1y, ay)), AD::mul(uy, AD::sub(p1x, ax)));
    const double cp2 = AD::sub(AD::mul(ux, AD::sub(p2y, ay)), AD::mul(uy, AD::sub(p2x, ax)));
    return AD::mul(cp1, cp2) >= 0.0;
}
// within_bounds (:188-203): inside any triangle (corner i, corner i+1, centroid); triangles i = part, part + parts, ...
__device__ __forceinline__ bool astar_within_bounds(const AstarDev &e, double px, double py, int part = 0, int parts = 1) {
    bool in = false;
    for (int i = part; i < e.E; i += parts) {
        const int j = i + 1 == e.E ? 0 : i + 1;
        const double ax = e.boundary[2 * i], ay = e.boundary[2 * i + 1], bx = e.boundary[2 * j], by = e.boundary[2 * j + 1];
        in |= astar_same_side(px, py, ax, ay, bx, by, e.cx, e.cy) && astar_same_side(px, py, bx, by, ax, ay, e.cx, e.cy) &&
              astar_same_side(px, py, e.cx, e.cy, ax, ay, bx, by);
    }
    return in;
}
// collision_free (:205-221).  The reference tests sqrt(dx^2 + dy^2) <= size; sqrt is monotone and correctly
// rounded, so that is exactly  dx^2 + dy^2 <= thr  with thr = the largest double whose rounded root is <= size
// (computed on the host, sqrt_le_threshold): no fp64 square root in the loop.  circles rows are x, y, thr.
// `part`/`parts`: the circles k = part, part + parts, ... (lanes of one neighbour split the list).
__device__ __forceinline__ bool astar_hits(const AstarDev &e, double px, double py, int part, int parts) {
    bool hit = false;
    for (int k = part; k < e.K; k += parts) {
        const double dx = AD::sub(px, e.circles[3 * k]), dy = AD::sub(py, e.circles[3 * k + 1]);
        hit |= AD::sq2(dx, dy) <= e.circles[3 * k + 2];
    }
    return hit;
}
__device__ __forceinline__ bool astar_collision_free(const AstarDev &e, double px, double py) { return !astar_hits(e, px, py, 0, 1); }
// get_cell_prob's key search (:486-505): the reference's predicate on the bucket's candidates, dict order
__device__ __forceinline__ int astar_find_cell(const AstarDev &e, double px, double py) {
    const double fx = floor(AD::mul(AD::sub(px, e.gx0), e.inv_bs)), fy = floor(AD::mul(AD::sub(py, e.gy0), e.inv_bs));
    if (!(fx >= 0.0 && fy >= 0.0 && fx < (double)e.gnx && fy < (double)e.gny)) return -1;
    const int b = (int)fy * e.gnx + (int)fx;
    for (int i = e.boff[b]; i < e.boff[b + 1]; i++) {
        const int c = e.bcells[i];
        const double b0 = e.cells_r[4 * c], b1 = e.cells_r[4 * c + 1], b2 = e.cells_r[4 * c + 2], b3 = e.cells_r[4 * c + 3];
        const double dx = fabs(AD::sub(b0, b2)), dy = fabs(AD::sub(b1, b3));
        if (fabs(AD::sub(px, b0)) <= dx && fabs(AD::sub(px, b2)) <= dx && fabs(AD::sub(py, b1)) <= dy &&
            fabs(AD::sub(py, b3)) <= dy)
            return c;
    }
    return -1;
}
__device__ __forceinline__ double astar_euclid(double ax, double ay, double bx, double by) {   // module-level :18-29
    const double dx = fabs(AD::sub(ax, bx)), dy = fabs(AD::sub(ay, by));
    return AD::sqrt(AD::add(AD::mul(dx, dx), AD::mul(dy, dy)));
}
// Walkable (:223-246); -1: the loop cannot terminate (both steps 0)
__device__ int astar_walkable(const AstarDev &e, double cx, double cy, double px, double py) {
    double sx = cx, sy = cy;
    const double stepx = (double)(long long)AD::div(fabs(AD::sub(px, cx)), 5.0), stepy = (double)(long long)AD::div(fabs(AD::sub(py, cy)), 5.0);
    for (int guard = 0; sx <= px && sy <= py; guard++) {
        const double ix = sx, iy = sy;
        sx = AD::add(sx, stepx); sy = AD::add(sy, stepy);
        if (!astar_collision_free(e, ix, iy)) return 0;
        if (guard > 100000) return -1;
    }
    return 1;
}

#ifndef AUV_ASTAR_MINB
#define AUV_ASTAR_MINB 8      // 64 registers, 32 warps per SM: the serial expansion loop is latency-bound (measured +26 % over 6 CTAs / 80 registers)
#endif
__global__ void __launch_bounds__(32 * ASTAR_WARPS, AUV_ASTAR_MINB) k_astar(AstarDev e, const auvrrt_astar_query_t *queries, long long Q, int cap,
                                                            int path_cap, unsigned char *ws, auvrrt_astar_record_t *recs, double *paths,
                                                            uint8_t *keep, int *expand_order, double *node_xy) {
    __shared__ unsigned s_alive[ASTAR_WARPS][128];            // cap <= 4096 nodes
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long q = (long long)blockIdx.x * ASTAR_WARPS + warp;
    if (q >= Q) return;
    unsigned *alive = s_alive[warp];
    for (int i = lane; i < 128; i += 32) alive[i] = 0u;
    unsigned char *base = ws + (size_t)q * astar_ws_per_query(cap);
    double *nf = (double *)base, *ncost = nf + cap, *nlen = ncost + cap, *nx = nlen + cap, *ny = nx + cap;
    int *nts = (int *)(ny + cap), *npar = nts + cap;
    unsigned *visited = (unsigned *)(base + (((size_t)cap * 48) + 255 & ~(size_t)255));
    for (int i = lane; i < ASTAR_VIS_WORDS; i += 32) visited[i] = 0u;
    const auvrrt_astar_query_t qu = queries[q];
    const double limit = qu.path_len_limit, w2 = qu.weights[1], w3 = qu.weights[2], w4 = qu.weights[3], vel = qu.velocity;
    if (lane == 0) {
        nx[0] = qu.start[0]; ny[0] = qu.start[1]; nlen[0] = 0.0; nf[0] = 0.0; ncost[0] = 0.0; nts[0] = 0; npar[0] = -1;
        alive[0] = 1u;
    }
    __syncwarp();
    int n = 1, n_exp = 0, status = AUVRRT_ST_NO_PATH, goal = -1, lo_word = 0;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    for (;;) {
        // 1. first strict minimum of f among the alive nodes (:577-583)
        double bf = INF; int bi = 0x7fffffff;
        while (lo_word < ((n - 1) >> 5) && alive[lo_word] == 0u) lo_word++;      // leading blocks of expanded nodes stay dead
        for (int i0 = lo_word << 5; i0 < n; i0 += 32) {
            const unsigned aw = alive[i0 >> 5];
            if (aw == 0u) continue;
            const int i = i0 + lane;
            const bool a = (aw >> lane) & 1u;
            if (a && i < n) { const double f = nf[i]; if (bi == 0x7fffffff || f < bf) { bf = f; bi = i; } }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const double of = __shfl_xor_sync(0xffffffffu, bf, d);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, d);
            if (oi != 0x7fffffff && (bi == 0x7fffffff || of < bf || (of == bf && oi < bi))) { bf = of; bi = oi; }
        }
        if (bi == 0x7fffffff) break;                              // open list empty
        const int cur = bi;
        if (lane == 0) { alive[cur >> 5] &= ~(1u << (cur & 31)); if (expand_order) expand_order[(size_t)q * cap + n_exp] = cur; }
        n_exp++;
        __syncwarp();
        const double cx = nx[cur], cy = ny[cur], clen = nlen[cur], ccost = ncost[cur];
        if (fabs(AD::sub(clen, limit)) <= 10.0) { goal = cur; status = AUVRRT_ST_OK; break; }     // :588
        // 2. the 8 neighbours (:255: (0,-10) (0,10) (-10,0) (10,0) (-10,-10) (-10,10) (10,-10) (10,10))
        int err = 0; bool add = false;
        double px = 0, py = 0, plen = 0, g = 0, f = 0; int ts = 0; unsigned vword = 0, vbit = 0;
        {
            // four lanes per neighbour: they split the boundary triangles and the obstacle list, OR their verdicts,
            // then lane 0 of the four carries the neighbour through the cost terms
            const int d = lane >> 2, part = lane & 3;
            const double ddx = d < 2 ? 0.0 : ((d == 2 || d == 4 || d == 5) ? -10.0 : 10.0);
            const double ddy = (d == 0 || d == 4 || d == 6) ? -10.0 : ((d == 2 || d == 3) ? 0.0 : 10.0);
            px = AD::add(cx, ddx); py = AD::add(cy, ddy);
            unsigned in = astar_within_bounds(e, px, py, part, 4) ? 1u : 0u, hit = astar_hits(e, px, py, part, 4) ? 1u : 0u;
            in |= __shfl_xor_sync(0xffffffffu, in, 1); hit |= __shfl_xor_sync(0xffffffffu, hit, 1);
            in |= __shfl_xor_sync(0xffffffffu, in, 2); hit |= __shfl_xor_sync(0xffffffffu, hit, 2);
            if (part == 0 && in && !hit) {
                plen = AD::add(clen, astar_euclid(cx, cy, px, py));                                 // :636
                const double dist_left = fabs(AD::sub(limit, plen));
                const long long tsl = (long long)AD::div(plen, vel);                                // int()
                ts = (int)tsl;
                int tb = -1;
                for (int t = 0; t < e.T; t++)
                    if ((double)tsl <= e.bins[2 * t + 1] && (double)tsl >= e.bins[2 * t]) { tb = t; break; }
                const int cell = tb >= 0 ? astar_find_cell(e, px, py) : -1;
                const long long nn = (long long)dist_left;
                if (tb < 0 || cell < 0 || nn > e.C) err = AUVRRT_ST_KEY_ERROR;
                else {
                    g = AD::sub(ccost, AD::mul(w4, e.probs[(size_t)tb * e.C + cell]));              // :641
                    const double h = AD::sub(AD::sub(AD::mul(-w2, dist_left), AD::mul(w3, (double)e.H)),
                                             AD::mul(w4, e.topn[(size_t)tb * (e.C + 1) + nn]));   // :644
                    f = AD::add(g, h);
                    long long xi = (long long)AD::add(px, 500.0), yi = (long long)AD::add(py, 200.0);   // get_indices
                    if (xi < 0) xi += 600;
                    if (yi < 0) yi += 600;
                    if (xi < 0 || xi >= 600 || yi < 0 || yi >= 600) err = AUVRRT_ST_KEY_ERROR;
                    else {
                        const int bitpos = (int)(xi * 600 + yi);
                        vword = (unsigned)bitpos >> 5; vbit = 1u << (bitpos & 31);
                        add = !(visited[vword] & vbit);
                    }
                }
            }
        }
        // the reference handles the neighbours in order and raises at the first one that fails: the ones before it
        // have already been put on the open list
        const unsigned errm = __ballot_sync(0xffffffffu, err != 0);
        const unsigned before = errm ? ((1u << (__ffs(errm) - 1)) - 1u) : 0xffffffffu;
        // 3. ordered append
        const unsigned addm = __ballot_sync(0xffffffffu, add) & before;
        const int n_add = __popc(addm);
        if (n + n_add > cap) { status = AUVRRT_ST_OVERFLOW; break; }
        if (add && ((addm >> lane) & 1u)) {
            const int slot = n + __popc(addm & ((1u << lane) - 1u));
            nx[slot] = px; ny[slot] = py; nlen[slot] = plen; nf[slot] = f; ncost[slot] = g; nts[slot] = ts; npar[slot] = cur;
            atomicOr(&alive[slot >> 5], 1u << (slot & 31));
            atomicOr(&visited[vword], vbit);
        }
        if (errm) { n += n_add; status = AUVRRT_ST_KEY_ERROR; break; }
        n += n_add;
        __syncwarp();
    }
    __syncwarp();
    // result (:590-617) on lane 0
    if (lane == 0) {
        auvrrt_astar_record_t r;
        r.status = status; r.n_expanded = n_exp; r.n_nodes = n; r.n_path = 0; r.n_smooth = 0; r.reserved = 0; r.cost = 0.0; r.path_len = 0.0;
        if (status == AUVRRT_ST_OK) {
            int np_ = 0;
            for (int j = goal; j >= 0; j = npar[j]) np_++;
            r.n_path = np_; r.cost = ncost[goal]; r.path_len = nlen[goal];
            if (np_ < 2) r.status = AUVRRT_ST_KEY_ERROR;                    // smoothPath: trajectory[1] IndexError (:419)
            else if (paths && keep) {
                if (np_ > path_cap) r.status = AUVRRT_ST_OVERFLOW;
                else {
                    double *P = paths + (size_t)q * path_cap * 6;
                    uint8_t *kp = keep + (size_t)q * path_cap;
                    int i = np_ - 1;
                    for (int j = goal; j >= 0; j = npar[j], i--) {
                        double *row = P + 6 * i;
                        row[0] = nx[j]; row[1] = ny[j]; row[2] = nlen[j]; row[3] = (double)nts[j]; row[4] = ncost[j]; row[5] = nf[j];
                        kp[i] = 1;
                    }
                    // smoothPath (:416-452)
                    int index = 1, check = 0, curp = 1;
                    while (index < np_ - 1) {
                        const int wk = astar_walkable(e, P[6 * check], P[6 * check + 1], P[6 * curp], P[6 * curp + 1]);
                        if (wk < 0) { r.status = AUVRRT_ST_KEY_ERROR; break; }
                        if (wk) {
                            bool inside = false;
                            for (int h = 0; h < e.H && !inside; h++)
                                inside = astar_euclid(e.habitats[3 * h], e.habitats[3 * h + 1], P[6 * curp], P[6 * curp + 1]) <= e.habitats[3 * h + 2];
                            if (!inside) kp[curp] = 0;
                            index++; curp = index;
                        } else {
                            check = curp; index++; curp = index;
                        }
                    }
                    int ns = 0;
                    for (int k = 0; k < np_; k++) ns += kp[k];
                    r.n_smooth = ns;
                }
            }
        }
        recs[q] = r;
    }
    if (node_xy)
        for (int i = lane; i < n; i += 32) { node_xy[((size_t)q * cap + i) * 2] = nx[i]; node_xy[((size_t)q * cap + i) * 2 + 1] = ny[i]; }
}

static AstarDev astar_dev(const auvrrt_astar_env *e) {
    AstarDev d;
    d.K = e->K; d.E = e->E; d.H = e->H; d.T = e->T; d.C = e->C;
    d.circles = e->d_f64 + e->off_circ; d.boundary = e->d_f64 + e->off_bnd; d.habitats = e->d_f64 + e->off_hab;
    d.bins = e->d_f64 + e->off_bins; d.cells_r = e->d_f64 + e->off_cells; d.probs = e->d_f64 + e->off_probs; d.topn = e->d_f64 + e->off_topn;
    d.cx = e->cx; d.cy = e->cy; d.gx0 = e->gx0; d.gy0 = e->gy0; d.inv_bs = e->inv_bs; d.gnx = e->gnx; d.gny = e->gny;
    d.boff = e->d_i32; d.bcells = e->d_i32 + e->n_boff;
    return d;
}

}  // namespace auv

using namespace auv;

// the largest double t with sqrt(t), correctly rounded, <= r; -1 when no non-negative t qualifies
static double sqrt_le_threshold(double r) {
    if (!(r >= 0.0)) return -1.0;
    if (std::isinf(r)) return r;
    double t = r * r;
    if (std::isinf(t)) t = 1.7976931348623157e308;
    while (sqrt(t) > r) t = nextafter(t, -INFINITY);
    for (;;) {
        const double u = nextafter(t, INFINITY);
        if (std::isinf(u) || sqrt(u) > r) break;
        t = u;
    }
    return t;
}

extern "C" int auvrrt_astar_env_create(const double *circles, int K, const double *boundary, int E, const double centroid[2],
                                       const double *habitats, int H, const double *bins, int T, const double *cells_rounded,
                                       int C, const double *probs, int device, auvrrt_astar_env_t **out) {
    if (!out || K < 0 || E < 3 || H < 0 || T < 0 || C < 0 || !boundary || !centroid || (K && !circles) || (H && !habitats) ||
        (T && !bins) || (C && !cells_rounded) || (T && C && !probs))
        return set_err(AUVRRT_ERR_ARG, "astar_env_create: bad arguments (the boundary needs at least 3 corners)");
    AUV_TRY(need_device(device));
    auvrrt_astar_env *e = new (std::nothrow) auvrrt_astar_env();
    if (!e) return set_err(AUVRRT_ERR_ARG, "astar_env_create: out of memory");
    e->device = device; e->K = K; e->E = E; e->H = H; e->T = T; e->C = C; e->cx = centroid[0]; e->cy = centroid[1];
    e->d_f64 = nullptr; e->d_i32 = nullptr; e->d_ws = nullptr; e->ws_bytes = 0; e->stream = nullptr;
    // get_top_n_prob (:520-536) for every n: probabilities sorted descending, added one by one
    std::vector<double> topn((size_t)T * (C + 1) + 1, 0.0), tmp((size_t)C);
    for (int t = 0; t < T; t++) {
        std::copy(probs + (size_t)t * C, probs + (size_t)(t + 1) * C, tmp.begin());
        std::sort(tmp.begin(), tmp.end(), [](double a, double b) { return a > b; });
        double total = 0.0;
        for (int i = 0; i < C; i++) { total += tmp[i]; topn[(size_t)t * (C + 1) + i + 1] = total; }
    }
    // bucket grid over the cells: a cell is listed in every bucket its box (grown by 1e-6) touches, in
    // ascending (= dict) order, so the first candidate passing the reference's predicate is the first
    // cell passing it.  The bucket coordinate is a monotone function of x evaluated identically here
    // and in the kernel, hence a point the predicate accepts always finds its cell listed.
    double lox = 0, loy = 0, hix = 1, hiy = 1, mean = 0;
    for (int c = 0; c < C; c++) {
        const double *b = cells_rounded + 4 * c;
        const double x0 = std::min(b[0], b[2]), x1 = std::max(b[0], b[2]), y0 = std::min(b[1], b[3]), y1 = std::max(b[1], b[3]);
        if (c == 0) { lox = x0; hix = x1; loy = y0; hiy = y1; }
        lox = std::min(lox, x0); hix = std::max(hix, x1); loy = std::min(loy, y0); hiy = std::max(hiy, y1);
        mean += (x1 - x0) + (y1 - y0);
    }
    double bs = C > 0 ? mean / (2.0 * C) : 1.0;
    if (!(bs > 1e-3)) bs = 1.0;
    e->gx0 = lox - 1.0; e->gy0 = loy - 1.0; e->inv_bs = 1.0 / bs;
    auto bucket = [&](double v, double g0) { return floor((v - g0) * e->inv_bs); };
    e->gnx = (int)std::min(4096.0, bucket(hix + 1.0, e->gx0) + 1.0); e->gny = (int)std::min(4096.0, bucket(hiy + 1.0, e->gy0) + 1.0);
    if (C == 0) { e->gnx = e->gny = 1; }
    if (bucket(hix + 1.0, e->gx0) + 1.0 > 4096.0 || bucket(hiy + 1.0, e->gy0) + 1.0 > 4096.0) { delete e; return set_err(AUVRRT_ERR_UNSUPPORTED, "astar_env_create: cell extent / cell size too large for the bucket grid"); }
    const size_t nb = (size_t)e->gnx * e->gny;
    std::vector<int> boff(nb + 1, 0), bcells;
    for (int pass = 0; pass < 2; pass++) {
        std::vector<int> fill(boff.begin(), boff.end() - 1);
        for (int c = 0; c < C; c++) {
            const double *b = cells_rounded + 4 * c;
            const double x0 = std::min(b[0], b[2]) - 1e-6, x1 = std::max(b[0], b[2]) + 1e-6, y0 = std::min(b[1], b[3]) - 1e-6, y1 = std::max(b[1], b[3]) + 1e-6;
            const int bx0 = (int)std::max(0.0, bucket(x0, e->gx0)), bx1 = (int)std::min((double)e->gnx - 1, bucket(x1, e->gx0));
            const int by0 = (int)std::max(0.0, bucket(y0, e->gy0)), by1 = (int)std::min((double)e->gny - 1, bucket(y1, e->gy0));
            for (int by = by0; by <= by1; by++)
                for (int bx = bx0; bx <= bx1; bx++) {
                    const size_t bi = (size_t)by * e->gnx + bx;
                    if (pass == 0) boff[bi + 1]++; else bcells[fill[bi]++] = c;
                }
        }
        if (pass == 0) { for (size_t i = 0; i < nb; i++) boff[i + 1] += boff[i]; bcells.assign((size_t)boff[nb] + 1, 0); }
    }
    e->n_boff = nb + 1;
    // circles as x, y, thr with  sqrt_rn(s) <= size  <=>  s <= thr  (see astar_hits)
    std::vector<double> circ_thr((size_t)3 * (K > 0 ? K : 1), 0.0);
    for (int k = 0; k < K; k++) {
        circ_thr[3 * k] = circles[3 * k]; circ_thr[3 * k + 1] = circles[3 * k + 1];
        circ_thr[3 * k + 2] = sqrt_le_threshold(circles[3 * k + 2]);
    }
    circles = circ_thr.data();
    // flatten
    std::vector<double> f64;
    auto push = [&](const double *p, size_t n) { size_t o = f64.size(); if (n) f64.insert(f64.end(), p, p + n); else f64.push_back(0.0); return o; };
    e->off_circ = push(circles, (size_t)3 * K); e->off_bnd = push(boundary, (size_t)2 * E); e->off_hab = push(habitats, (size_t)3 * H);
    e->off_bins = push(bins, (size_t)2 * T); e->off_cells = push(cells_rounded, (size_t)4 * C); e->off_probs = push(probs, (size_t)T * C);
    e->off_topn = push(topn.data(), (size_t)T * (C + 1));
    std::vector<int> i32(boff);
    i32.insert(i32.end(), bcells.begin(), bcells.end());
    cudaError_t er = cudaMalloc((void **)&e->d_f64, 8 * f64.size());
    if (er == cudaSuccess) er = cudaMalloc((void **)&e->d_i32, 4 * i32.size());
    if (er == cudaSuccess) er = cudaMemcpy(e->d_f64, f64.data(), 8 * f64.size(), cudaMemcpyHostToDevice);
    if (er == cudaSuccess) er = cudaMemcpy(e->d_i32, i32.data(), 4 * i32.size(), cudaMemcpyHostToDevice);
    if (er == cudaSuccess) er = cudaStreamCreate(&e->stream);
    if (er != cudaSuccess) { auvrrt_astar_env_destroy(e); return set_err(AUVRRT_ERR_CUDA, "astar_env_create: %s", cudaGetErrorString(er)); }
    *out = e;
    return AUVRRT_OK;
}

extern "C" void auvrrt_astar_env_destroy(auvrrt_astar_env_t *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) { cudaStreamSynchronize(e->stream); cudaStreamDestroy(e->stream); }
    cudaFree(e->d_f64); cudaFree(e->d_i32); cudaFree(e->d_ws);
    delete e;
}

extern "C" int64_t auvrrt_astar_workspace_bytes(int64_t Q, int32_t node_cap) {
    if (Q <= 0 || node_cap <= 0) return 0;
    return (int64_t)((size_t)Q * astar_ws_per_query(node_cap));
}

extern "C" int auvrrt_astar_batch_dev(auvrrt_astar_env_t *env, const auvrrt_astar_query_t *d_queries, int64_t Q, int32_t node_cap,
                                      int32_t path_cap, void *d_workspace, int64_t workspace_bytes, auvrrt_astar_record_t *d_records,
                                      double *d_paths, uint8_t *d_keep, int32_t *d_expand_order, double *d_node_xy, void *stream) {
    if (!env || !d_queries || !d_records || Q <= 0) return set_err(AUVRRT_ERR_ARG, "astar_batch: bad arguments");
    if (node_cap < 2 || node_cap > 4096) return set_err(AUVRRT_ERR_ARG, "astar_batch: node_cap must be in [2, 4096]");
    if ((d_paths == nullptr) != (d_keep == nullptr) || (d_paths && path_cap < 2)) return set_err(AUVRRT_ERR_ARG, "astar_batch: paths and keep go together, path_cap >= 2");
    if (!d_workspace || workspace_bytes < auvrrt_astar_workspace_bytes(Q, node_cap)) return set_err(AUVRRT_ERR_ARG, "astar_batch: workspace too small");
    AUV_CUDA(cudaSetDevice(env->device));
    k_astar<<<(unsigned)((Q + ASTAR_WARPS - 1) / ASTAR_WARPS), 32 * ASTAR_WARPS, 0, (cudaStream_t)stream>>>(
        astar_dev(env), d_queries, (long long)Q, node_cap, path_cap, (unsigned char *)d_workspace, d_records, d_paths, d_keep,
        d_expand_order, d_node_xy);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

extern "C" int auvrrt_astar_batch(auvrrt_astar_env_t *env, const auvrrt_astar_query_t *queries, int64_t Q, int32_t node_cap,
                                  int32_t path_cap, auvrrt_astar_record_t *records, double *paths, uint8_t *keep,
                                  int32_t *expand_order, double *node_xy) {
    if (!env || !queries || !records || Q <= 0) return set_err(AUVRRT_ERR_ARG, "astar_batch: bad arguments");
    AUV_CUDA(cudaSetDevice(env->device));
    const size_t need = (size_t)auvrrt_astar_workspace_bytes(Q, node_cap);
    if (need > env->ws_bytes) {
        cudaFree(env->d_ws); env->d_ws = nullptr; env->ws_bytes = 0;
        AUV_CUDA(cudaMalloc(&env->d_ws, need));
        env->ws_bytes = need;
    }
    DBuf dq, dr, dp, dk, de, dn;
    const size_t q = (size_t)Q;
    AUV_TRY(dq.alloc(sizeof(auvrrt_astar_query_t) * q));
    AUV_TRY(dr.alloc(sizeof(auvrrt_astar_record_t) * q));
    // path_cap 0 leaves the device path buffers NULL: the batch then writes records only
    if (paths && path_cap != 0) { AUV_TRY(dp.alloc(48 * q * (size_t)path_cap)); AUV_TRY(dk.alloc(q * (size_t)path_cap)); }
    if (expand_order) AUV_TRY(de.alloc(4 * q * (size_t)node_cap));
    if (node_xy) AUV_TRY(dn.alloc(16 * q * (size_t)node_cap));
    AUV_CUDA(cudaMemcpyAsync(dq.p, queries, sizeof(auvrrt_astar_query_t) * q, cudaMemcpyHostToDevice, env->stream));
    if (paths) {     // rows past a query's path read as zeros
        AUV_CUDA(cudaMemsetAsync(dk.p, 0, q * (size_t)path_cap, env->stream));
        AUV_CUDA(cudaMemsetAsync(dp.p, 0, 48 * q * (size_t)path_cap, env->stream));
    }
    int rc = auvrrt_astar_batch_dev(env, (const auvrrt_astar_query_t *)dq.p, Q, node_cap, path_cap, env->d_ws, (int64_t)env->ws_bytes,
                                    (auvrrt_astar_record_t *)dr.p, (double *)dp.p, (uint8_t *)dk.p, (int32_t *)de.p, (double *)dn.p, env->stream);
    if (rc != AUVRRT_OK) { cudaStreamSynchronize(env->stream); return rc; }
    AUV_CUDA(cudaMemcpyAsync(records, dr.p, sizeof(auvrrt_astar_record_t) * q, cudaMemcpyDeviceToHost, env->stream));
    if (paths) {
        AUV_CUDA(cudaMemcpyAsync(paths, dp.p, 48 * q * (size_t)path_cap, cudaMemcpyDeviceToHost, env->stream));
        AUV_CUDA(cudaMemcpyAsync(keep, dk.p, q * (size_t)path_cap, cudaMemcpyDeviceToHost, env->stream));
    }
    if (expand_order) AUV_CUDA(cudaMemcpyAsync(expand_order, de.p, 4 * q * (size_t)node_cap, cudaMemcpyDeviceToHost, env->stream));
    if (node_xy) AUV_CUDA(cudaMemcpyAsync(node_xy, dn.p, 16 * q * (size_t)node_cap, cudaMemcpyDeviceToHost, env->stream));
    AUV_CUDA(cudaStreamSynchronize(env->stream));
    return AUVRRT_OK;
}
