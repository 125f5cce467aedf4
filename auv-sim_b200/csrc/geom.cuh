// geom.cuh -- point-in-polygon, circle collision, per-point cost contribution (device).
#pragma once
#include "env.cuh"

namespace auv {

// ---------------------------------------------------------------- exact orientation (fp64)
// Sign of (ax-cx)(by-cy) - (ay-cy)(bx-cx).  Float filter with Shewchuk's error bound; when it is
// inconclusive the six exact products are summed as a non-overlapping expansion.  This is what
// "Point.within" needs to be decided exactly (rrt_dubins.py:544-547 via GEOS).
__device__ __forceinline__ void two_sum_d(double a, double b, double &s, double &e) {
    s = __dadd_rn(a, b);
    double bv = __dsub_rn(s, a), av = __dsub_rn(s, bv);
    e = __dadd_rn(__dsub_rn(a, av), __dsub_rn(b, bv));
}
static __device__ __noinline__ int orient2d_exact_slow(double ax, double ay, double bx, double by, double cx, double cy) {
    const double pa[6] = {ax, -ax, -cx, -ay, ay, cy};
    const double pb[6] = {by, cy, by, bx, cx, bx};
    double e[16];
    int n = 0;
    for (int i = 0; i < 6; i++) {
        double hi = __dmul_rn(pa[i], pb[i]);
        double lo = fma(pa[i], pb[i], -hi);
        for (int pass = 0; pass < 2; pass++) {
            double q = pass == 0 ? lo : hi;
            int m = 0;
            for (int k = 0; k < n; k++) {
                double s, err;
                two_sum_d(q, e[k], s, err);
                if (err != 0.0) e[m++] = err;
                q = s;
            }
            if (q != 0.0 || m == 0) e[m++] = q;
            n = m;
        }
    }
    double top = e[n - 1];
    return (top > 0.0) - (top < 0.0);
}
__device__ __forceinline__ int orient2d(double ax, double ay, double bx, double by, double cx, double cy) {
    double detl = __dmul_rn(__dsub_rn(ax, cx), __dsub_rn(by, cy));
    double detr = __dmul_rn(__dsub_rn(ay, cy), __dsub_rn(bx, cx));
    double det = __dsub_rn(detl, detr), detsum;
    if (detl > 0.0) { if (detr <= 0.0) return (det > 0.0) - (det < 0.0); detsum = detl + detr; }
    else if (detl < 0.0) { if (detr >= 0.0) return (det > 0.0) - (det < 0.0); detsum = -detl - detr; }
    else detsum = fabs(detr);
    const double errbound = (3.0 + 16.0 * 0x1.0p-53) * 0x1.0p-53;
    if (fabs(det) > errbound * detsum) return (det > 0.0) - (det < 0.0);
    return orient2d_exact_slow(ax, ay, bx, by, cx, cy);
}
__device__ __forceinline__ int orient2d(float ax, float ay, float bx, float by, float cx, float cy) {
    float det = (ax - cx) * (by - cy) - (ay - cy) * (bx - cx);
    return (det > 0.f) - (det < 0.f);
}

// strictly inside the boundary polygon?  (boundary points are NOT within)
template <typename R> __device__ __forceinline__ bool point_within(const EnvView<R> &env, R px, R py) {
    if (!Policy<R>::VERIFY && env.convex != 0) {
        // convex ring: strictly inside <=> strictly on the interior side of every edge
        bool in = true;
        R ax = env.px[env.E - 1], ay = env.py[env.E - 1];
        for (int i = 0; i < env.E; i++) {
            R bx = env.px[i], by = env.py[i];
            R det = (bx - ax) * (py - ay) - (by - ay) * (px - ax);
            in = in && (env.convex > 0 ? det > (R)0 : det < (R)0);
            ax = bx; ay = by;
        }
        return in && env.E >= 3;
    }
    bool inside = false;
    bool boundary = false;
    for (int i = 0; i < env.E; i++) {
        int j = i + 1 == env.E ? 0 : i + 1;
        R ax = env.px[i], ay = env.py[i], bx = env.px[j], by = env.py[j];
        if (px == ax && py == ay) boundary = true;
        if (ay == py && by == py) {
            if (fmin(ax, bx) <= px && px <= fmax(ax, bx)) boundary = true;
            continue;
        }
        if ((ay > py) != (by > py)) {
            int s = orient2d(ax, ay, bx, by, px, py);
            if (s == 0) boundary = true;
            if ((s > 0) == (by > ay)) inside = !inside;
        }
    }
    return inside && !boundary;
}

// the full test out of line, for the fast build's rare "cell needs the whole ring" case: called with scalars and
// pointers only, so the world-model view stays in registers at the call site
template <typename R>
__device__ __noinline__ bool point_within_outlined(const R *vx, const R *vy, int E, int convex, R px, R py) {
    EnvView<R> e;
    e.px = vx; e.py = vy; e.E = E; e.convex = convex;
    return point_within<R>(e, px, py);
}

// same, short-circuited by the classification grid: definitive code, else (fast build, convex ring)
// only the candidate edges of the cell, else the full test
// OUTLINE: call the rare full tests out of line (planner kernels, where they would otherwise sit in the hot loop);
// the thread-per-edge micro-benchmark kernels on dense synthetic worlds keep them inline.
template <typename R, bool OUTLINE = true> __device__ __forceinline__ bool point_within_c(const EnvView<R> &env, const Cls &cl, R px, R py) {
    const unsigned pc = cl.code & 3u;
    if (pc == 1u) return true;
    if (pc == 2u) return false;
    if (Policy<R>::VERIFY) return point_within<R>(env, px, py);
    if (cl.code & AUV_GRID_POLY_FULL)
        return OUTLINE ? point_within_outlined<R>(env.px, env.py, env.E, env.convex, px, py) : point_within<R>(env, px, py);
    if (cl.code & AUV_GRID_POLY_ONE) {
        // one undecided edge (every other half-plane is constant over the cell, on the inner side)
        const int i = (int)((cl.code >> 26) & 0x1Fu), j = i + 1 == env.E ? 0 : i + 1;
        const R ax = env.px[i], ay = env.py[i], bx = env.px[j], by = env.py[j];
        const R det = (bx - ax) * (py - ay) - (by - ay) * (px - ax);
        return env.convex > 0 ? det > (R)0 : det < (R)0;
    }
    const unsigned w2 = env.word2(cl);
    bool in = true;
#pragma unroll
    for (int s = 0; s < 2; s++) {
        const int i = (int)((w2 >> (18 + 5 * s)) & 0x1Fu);
        if (i != 0x1F) {
            const int j = i + 1 == env.E ? 0 : i + 1;
            const R ax = env.px[i], ay = env.py[i], bx = env.px[j], by = env.py[j];
            const R det = (bx - ax) * (py - ay) - (by - ay) * (px - ax);
            in = in && (env.convex > 0 ? det > (R)0 : det < (R)0);
        }
    }
    return in;
}

// does the point hit any (inflated, see env.cuh) circle?   thread-level, all circles
template <typename R> __device__ __forceinline__ bool point_hits_circles(const EnvView<R> &env, R x, R y) {
    typedef typename Policy<R>::A A;
    bool hit = false;
    for (int k = 0; k < env.K; k++) {
        R q = A::sq2(A::sub(x, env.cx[k]), A::sub(y, env.cy[k]));
        if (Policy<R>::VERIFY) hit = hit || (A::sqrt(q) <= env.creff[k]);
        else hit = hit || (q <= env.creff2[k]);
    }
    return hit;
}

// the all-circles loop out of line for the fast build's rare "more than 3 candidate circles" cells
template <typename R>
__device__ __noinline__ bool point_hits_circles_outlined(const R *cx, const R *cy, const R *creff2, int K, R x, R y) {
    typedef typename Policy<R>::A A;
    bool hit = false;
#pragma unroll 1
    for (int k = 0; k < K; k++) hit = hit || (A::sq2(A::sub(x, cx[k]), A::sub(y, cy[k])) <= creff2[k]);
    return hit;
}

// same through the classification grid: clear cell, else the cell's <= 3 candidate circles, else all
template <typename R, bool OUTLINE = true> __device__ __forceinline__ bool point_hits_circles_c(const EnvView<R> &env, const Cls &cl, R x, R y) {
    typedef typename Policy<R>::A A;
    if (cl.code & 4u) return false;
    if (cl.code & AUV_GRID_CIRC_ONE) {
        const int k = (int)((cl.code >> 16) & 0x3FFu);
        const R q = A::sq2(A::sub(x, env.cx[k]), A::sub(y, env.cy[k]));
        return Policy<R>::VERIFY ? (A::sqrt(q) <= env.creff[k]) : (q <= env.creff2[k]);
    }
    if (cl.code & AUV_GRID_CIRC_MANY) {
        if (Policy<R>::VERIFY || !OUTLINE) return point_hits_circles<R>(env, x, y);
        return point_hits_circles_outlined<R>(env.cx, env.cy, env.creff2, env.K, x, y);
    }
    const unsigned w1 = env.word1(cl);
    bool hit = false;
#pragma unroll
    for (int s = 0; s < 3; s++) {
        const int k = (int)((w1 >> (10 * s)) & 0x3FFu);
        if (k != 0x3FF) {
            R q = A::sq2(A::sub(x, env.cx[k]), A::sub(y, env.cy[k]));
            if (Policy<R>::VERIFY) hit = hit || (A::sqrt(q) <= env.creff[k]);
            else hit = hit || (q <= env.creff2[k]);
        }
    }
    return hit;
}

__device__ __forceinline__ void keep_unconditional(float &a, float &b) { asm volatile("" : "+f"(a), "+f"(b)); }
__device__ __forceinline__ void keep_unconditional(double &, double &) {}

// Fast build, branch-free: the collision test of a cell that is decided by its code or by ONE circle and / or ONE
// boundary edge (code bit 31 clear).  Both candidates are always fetched (a cell without one names row 0) and
// their results masked by the code: on the Catalina map 17 % of the free cells are boundary cells of this kind, so in a
// kernel that runs 32 edges per warp some lane is in one on nearly every step -- a branch would be taken every time,
// for two or three lanes.  Same arithmetic as point_within_c / point_hits_circles_c.
template <typename R>
__device__ __forceinline__ bool point_unsafe_one(const EnvView<R> &env, unsigned code, R x, R y) {
    typedef typename Policy<R>::A A;
    const One<R> ce = env.cone[(code >> 16) & 0x3FFu];
    const One<R> pe = env.pone[(code >> 26) & 0x1Fu];
    R q = A::sq2(A::sub(x, ce.x), A::sub(y, ce.y));
    R det = pe.z * (y - pe.y) - pe.w * (x - pe.x);
    // (the compiler would otherwise sink the two fetches under the code bits that use them: a branch for two or three lanes)
    keep_unconditional(q, det);
    const unsigned hit = ((code >> 14) & 1u) & (q <= ce.z ? 1u : 0u);
    const unsigned in = ((code & 3u) == 1u ? 1u : 0u) | (((code >> 15) & 1u) & (det > (R)0 ? 1u : 0u));
    return ((in ^ 1u) | hit) != 0u;
}
// collision test of a classified point: the branch-free form, the general one only for cells flagged AUV_GRID_SLOW
template <typename R>
__device__ __forceinline__ bool point_unsafe_c(const EnvView<R> &env, const Cls &cl, R x, R y) {
    if (Policy<R>::VERIFY) return !point_within_c<R>(env, cl, x, y) || point_hits_circles_c<R>(env, cl, x, y);
    bool bad = point_unsafe_one<R>(env, cl.code, x, y);
    if (__builtin_expect((cl.code & AUV_GRID_SLOW) != 0u, 0))
        bad = !point_within_c<R>(env, cl, x, y) || point_hits_circles_c<R>(env, cl, x, y);
    return bad;
}

// ---------------------------------------------------------------- cost contribution of a point
// One iteration of the `for mps in path` loop of habitat_shark_cost_func (cost.py:171-191).
struct Contrib {
    int bin;      // first shark-grid bin containing t, -1: none (the point is skipped, cost.py:178)
    int cell;     // first matching cell, -1: none
    int hab;      // first habitat containing the point, -1: none
};

// the rare cases of find_cell: a bucket with several breakpoints, or a point below the first candidate of a piece
// that has more
template <typename R>
__device__ __noinline__ int find_cell_walk(const R *brk, const int *piece, const R *c1, const int *cell, int NB, int lo, R x, R y) {
    if (!(x >= brk[0]) || !(x <= brk[NB - 1])) return -1;
    lo = lo < 0 ? 0 : lo;
    while (lo > 0 && brk[lo] > x) lo--;
    while (lo + 1 < NB && brk[lo + 1] <= x) lo++;
    const int p = 2 * lo + (x == brk[lo] ? 0 : 1);
    for (int k = piece[p]; k < piece[p + 1]; k++)
        if (c1[k] <= y) return cell[k];
    return -1;
}

template <typename R>
__device__ __noinline__ int find_cell_walk_shared(const EnvView<R> *senv, int lo, R x, R y) {
    return find_cell_walk<R>(senv->brk, senv->piece, senv->c1, senv->cell, senv->NB, lo, x, y);
}
template <typename R, bool SHARED = false>
__device__ __forceinline__ int find_cell_rare(const EnvView<R> &env, int lo, R x, R y) {
    if (SHARED || env.shared_self) return find_cell_walk_shared<R>(env.shared_self, lo, x, y);
    return find_cell_walk<R>(env.brk, env.piece, env.c1, env.cell, env.NB, lo, x, y);
}

// first cell (dict order) with x >= c0 and x <= c2 and y >= c1 and x <= c3 (sic), -1 if none     cost.py:181-184
// Straight-line code but for two rare cases (a bucket with several breakpoints; a point below the first candidate
// of a piece that has more): sentinels brk[-1] = -inf, brk[NB] = +inf, pfirst[-2] = pfirst[-1] = none (api.cu).
// HAS_XB: the caller knows the bucket table exists (nxb > 0), checked once on the host
template <typename R, bool HAS_XB = false>
__device__ __forceinline__ int find_cell(const EnvView<R> &env, R x, R y) {
    if (!HAS_XB && env.nxb == 0) return env.NB == 0 ? -1 : find_cell_walk<R>(env.brk, env.piece, env.c1, env.cell, env.NB, 0, x, y);
    // the first and last buckets lie outside every cell.  A NaN x goes to the first bucket, where it matches no piece
    // (fmaxf(NaN, 0) = 0; without it the fp32 form sent NaN to the last bucket and the piece before the last breakpoint)
    int b;
    if (sizeof(R) == 4) b = min(__float_as_int(__fadd_rd(fmaxf(fmaf((float)x, (float)env.xbinv, (float)env.xbo), 0.f), 8388608.f)) - 0x4B000000, env.nxb - 1);
    else { const R fb = (x - env.xb0) * env.xbinv; b = fb >= (R)0 ? (fb < (R)env.nxb ? (int)fb : env.nxb - 1) : 0; }
    const int e = (int)env.xb[b];
    int lo = (e & 0x7FFF) - 1;                   // last breakpoint left of the bucket (-1: none)
    if (__builtin_expect(e & 0x8000, 0)) return find_cell_rare<R, HAS_XB>(env, lo, x, y);
    // at most one breakpoint in the bucket: one compare settles the piece
    const R nxt = env.brk[lo + 1];
    R cur = env.brk[lo];
    if (nxt <= x) { lo++; cur = nxt; }
    const int p = 2 * lo + (x == cur ? 0 : 1);   // the point piece {brk[lo]} or the open interval after it; lo == -1: none
    const PFirst<R> f = env.pfirst[p];
    const bool hit = f.v >= 0 && y >= f.c1;
    if (__builtin_expect(!hit && f.v >= (1 << 30), 0)) return find_cell_rare<R, HAS_XB>(env, lo, x, y);
    return hit ? (f.v & 0x3FFFFFFF) : -1;
}

// first shark-grid time bin (dict order) with b0 <= t <= b1, -1 if none          cost.py:173-177
// UNIFORM: the caller knows the bins are contiguous and equally wide (checked once on the host) and asks for all of them
template <typename R, bool UNIFORM = false>
__device__ __forceinline__ int find_bin(const EnvView<R> &env, R t, unsigned bin_mask) {
    if (UNIFORM || (env.bins_uniform && bin_mask == 0xffffffffu)) {
        // contiguous sorted bins: the containing bins are adjacent; guess (off by at most one), settle
        // on the FIRST containing bin, verify with the reference's own comparisons
        // contiguous bins (b0[i+1] == b1[i]): the first containing bin is the first i with b1[i] >= t, if
        // b0[0] <= t <= b1[T-1].  The arithmetic guess is off by at most one either way.
        // (b1[-1] = the number just below b0[0] is a sentinel: t < b0[0] steps down to -1 like any "an earlier bin
        // holds it"; beyond the last bin the range test below rejects)
        int k;
        if (sizeof(R) == 4) k = __float_as_int(__fadd_rd(fmaf((float)t, (float)env.bin_winv, (float)env.bin_off), 8388608.f)) - 0x4B000000;
        else k = (int)((t - env.bin_s0) * env.bin_winv);
        k = min(max(k, 0), env.T - 1);
        const R up = env.b1[k], dn = env.b1[k - 1];
        k += (t > up ? 1 : 0) - (t <= dn ? 1 : 0);              // t <= b1[k-1]: an earlier bin holds it; t > b1[k]: a later one
        return t <= env.bin_hi ? k : -1;
    }
    for (int b = 0; b < env.T; b++) {
        if (b < 32 && !((bin_mask >> b) & 1u)) continue;
        if (t >= env.b0[b] && t <= env.b1[b]) return b;
    }
    return -1;
}

#ifndef AUV_HAB_ONE
#define AUV_HAB_ONE 0             // warp-per-edge kernels too fetch the single candidate habitat unconditionally: measured slower (edge.cuh, AUV_EDGE_ONE)
#endif
#ifndef AUV_OUTLINE_HAB
#define AUV_OUTLINE_HAB 1         // ambiguous-habitat cells out of line
#endif
// first habitat holding (x, y) in a cell whose habitat code is "ambiguous": out of line, for kernels with a shared view
template <typename R>
__device__ __noinline__ int first_habitat_ambiguous(const EnvView<R> *senv, unsigned code, int idx, int n_hab, R x, R y) {
    typedef typename Policy<R>::A A;
    if (!(code & AUV_GRID_HAB_MANY)) {
        const unsigned w2 = __ldg(senv->grid + 2 * senv->ncell + idx);
        for (int s = 0; s < 3; s++) {
            const int h = (int)((w2 >> (6 * s)) & 0x3Fu);
            if (h != 0x3F && h < n_hab) {
                R q = A::sq2(A::sub(senv->hx[h], x), A::sub(senv->hy[h], y));
                if (Policy<R>::VERIFY ? (A::sqrt(q) <= senv->hr[h]) : (q <= senv->hr2[h])) return h;
            }
        }
        return -1;
    }
    for (int h = 0; h < n_hab; h++) {
        R q = A::sq2(A::sub(senv->hx[h], x), A::sub(senv->hy[h], y));
        if (Policy<R>::VERIFY ? (A::sqrt(q) <= senv->hr[h]) : (q <= senv->hr2[h])) return h;
    }
    return -1;
}

// Time bins along ONE edge: traj_time_stamp never decreases from waypoint to waypoint (rrt_dubins.py:281 adds
// movement / velocity_temp >= 0), so for contiguous increasing bins the first containing bin can only move forward.
// The cursor keeps k = the first bin with b1[k] >= t (T: none left) and up = b1[k]; most waypoints cost one compare.
template <typename R> struct BinCursor {
    int k; R up;
    __device__ __forceinline__ void start(const EnvView<R> &env, R t) {
        k = 0;
        while (k < env.T && env.b1[k] < t) k++;
        up = k < env.T ? env.b1[k] : Policy<R>::A::inf();
    }
    // first bin in dict order with b0 <= t <= b1 (cost.py:173-177), -1 if none; t must not decrease between calls
    __device__ __forceinline__ int at(const EnvView<R> &env, R t) {
        while (__builtin_expect(t > up, 0)) { k++; up = k < env.T ? env.b1[k] : Policy<R>::A::inf(); }
        return (k < env.T && t >= env.bin_lo) ? k : -1;
    }
};

// FASTENV (checked once on the host, edges_tpe.cu / plan_tpt.cu): the bucket table exists, the caller passes the bin
// (known_bin) and published a shared copy of the view -- the run-time flags and the generic fallbacks drop out.
// DEFER: a cell whose habitat code is "ambiguous" is reported as hab = -2 and left to the caller (the thread-per-edge
// kernel queues such points and resolves them warp-wide after the edge, edge_serial.cuh)
template <typename R, bool FASTENV = false, bool DEFER = false>
__device__ __forceinline__ Contrib point_contrib(const EnvView<R> &env, R x, R y, R t,
                                                 unsigned bin_mask, int n_hab, const Cls &cl, int known_bin = -2) {
    typedef typename Policy<R>::A A;
    Contrib c;
    c.cell = -1; c.hab = -1;
    c.bin = (FASTENV || known_bin != -2) ? known_bin : find_bin<R>(env, t, bin_mask);
    if (!FASTENV && c.bin < 0) return c;             // (FASTENV: straight-line code, the result is masked at the end)
    const unsigned code = cl.code;
    c.cell = find_cell<R, FASTENV>(env, x, y);
    const unsigned hc = (code >> 3) & 0xFFu;
    if (!Policy<R>::VERIFY && (FASTENV || AUV_HAB_ONE)) {
        // branch-free: definitive first match (hc < 64), the one habitat a point of this cell can be in (64 + h), or
        // none (128: row 0 is fetched and the result masked)
        const int h = (int)(hc & 63u);
        const One<R> ho = env.hone[h];
        R q = A::sq2(A::sub(ho.x, x), A::sub(ho.y, y)), q_ = q;
        keep_unconditional(q, q_);      // (or the compiler branches around the fetch for the lanes with a definitive code)
        const bool take = (hc < AUV_GRID_HAB_ONE || (hc < 128u && q <= ho.z)) && (FASTENV || h < n_hab);
        c.hab = take ? h : -1;
    } else if (hc < 128u) {
        // definitive first match (hc < 64), or the one habitat a point of this cell can be in (64 + h)
        const int h = (int)(hc & 63u);
        if (h < n_hab) {
            bool in = true;
            if (hc >= AUV_GRID_HAB_ONE) {
                R q = A::sq2(A::sub(env.hx[h], x), A::sub(env.hy[h], y));
                in = Policy<R>::VERIFY ? (A::sqrt(q) <= env.hr[h]) : (q <= env.hr2[h]);
            }
            if (in) c.hab = h;
        }
    }
    if (DEFER) { if (hc == AUV_GRID_HAB_AMBIG) c.hab = -2; }
    else if (__builtin_expect(hc == AUV_GRID_HAB_AMBIG, 0)) {
        if (AUV_OUTLINE_HAB && (FASTENV || env.shared_self)) {
            c.hab = first_habitat_ambiguous<R>(env.shared_self, code, cl.idx, n_hab, x, y);
        } else if (!(code & AUV_GRID_HAB_MANY)) {
            // the cell's candidate habitats, in list order (every habitat that touches the cell, up to
            // and including the first that covers it)
            const unsigned w2 = env.word2(cl);
#pragma unroll
            for (int s = 0; s < 3; s++) {
                const int h = (int)((w2 >> (6 * s)) & 0x3Fu);
                if (h != 0x3F && h < n_hab && c.hab < 0) {
                    R q = A::sq2(A::sub(env.hx[h], x), A::sub(env.hy[h], y));
                    bool in = Policy<R>::VERIFY ? (A::sqrt(q) <= env.hr[h]) : (q <= env.hr2[h]);
                    if (in) c.hab = h;
                }
            }
        } else {
            for (int h = 0; h < n_hab; h++) {
                R q = A::sq2(A::sub(env.hx[h], x), A::sub(env.hy[h], y));
                bool in = Policy<R>::VERIFY ? (A::sqrt(q) <= env.hr[h]) : (q <= env.hr2[h]);
                if (in) { c.hab = h; break; }
            }
        }
    }
    if (FASTENV && c.bin < 0) { c.hab = -1; c.cell = -1; }
    return c;
}

}  // namespace auv
