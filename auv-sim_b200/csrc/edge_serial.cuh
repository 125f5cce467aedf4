// edge_serial.cuh -- one candidate edge evaluated by ONE thread, primitive by primitive, exactly as the
// reference's serial loop runs it:
//   RRT.steer, the random-arc rollout            (/root/reference/path_planning/rrt_dubins.py:252-295)
//   RRT.check_collision on the path so far       (rrt_dubins.py:530-549)
//   the per-waypoint part of cost.habitat_shark_cost_func   (/root/reference/path_planning/cost.py:171-191)
// Used by the thread-per-edge kernel (edges_tpe.cu: independent edges, the north star's "batched
// steer+collide+cost kernel ... one candidate edge per thread") and by the thread-per-tree planner
// (plan_tpt.cu).  edge.cuh is the warp-cooperative evaluation of the same edge.
//
// ALLPAIRS = false: every waypoint is classified by the grid of env.cuh (one load decides most tests).
// ALLPAIRS = true : every waypoint against every circle, polygon edge and habitat -- the all-pairs
//                   work SURVEY.md 8(d) counts (6 W K + 6 W E + ... FLOP per edge), for the roofline.
#pragma once
#include "edge.cuh"

// tuning switches of the one-edge-per-thread hot loop (measured in profiles/r02_tpe_*.txt)
#ifndef AUV_OUTLINE_COLLIDE
#define AUV_OUTLINE_COLLIDE 0     // boundary-cell collision tests out of line: measured SLOWER (4.1e9 vs 4.9e9 edges/s at Catalina
                                  // scale): some lane of a warp is in a boundary cell on most steps, so the call overhead is paid often
#endif
#ifndef AUV_BIN_CURSOR
#define AUV_BIN_CURSOR 0          // forward-only time-bin cursor instead of a lookup per waypoint: measured equal (5.0e9 vs 4.9e9);
                                  // the heavy-tailed time steps make some lane advance the cursor on most steps
#endif

namespace auv {

// circles for the all-pairs test of the fast build, relative to an origin o (the polygon's bounding-box
// centre): |p - c|^2 - r^2 = |p'|^2 + (-2 c').p' + (|c'|^2 - r^2) with p' = p - o, c' = c - o, so a pair
// costs 2 FFMA + 1 FMNMX (half that with the packed FFMA2 / FMNMX3 forms over two circles).  The
// expansion cancels: a minimum within `guard` of the decision is re-evaluated with the direct formula.
struct CircPair {           // two circles a, b
    float2 m2x, m2y;        // -2 c'_x, -2 c'_y
    float2 k;               // |c'|^2 - r_eff^2
};
struct alignas(16) CircQuad { float4 m2x, m2y, k; };     // four circles: three 16-byte loads feed four FFMA2
struct CircTable {
    const CircQuad *pair;   // ceil(K / 4) entries in shared memory; missing circles repeat the quad's first
    int npair;              // number of quads
    float ox, oy;           // origin
    float ccmax;            // max |c'|^2: scale of the rounding error of the expansion
    float rmax1;            // largest inflated radius + 1 m (circ_guard)
    bool buf2;              // enough circles for two waypoints per pass over the table to pay (circles_hit2)
    // the same packed form for the habitats (first match in list order; a missing second habitat has k = +inf) ...
    const CircPair *hpair; int nhpair; float hccmax;
    // ... and for the edges of a convex boundary ring: det_i(p') = A_i x' + B_i y' + C_i as (m2x, m2y, k) = (A, B, C) pairs,
    // signs normalised so that "strictly inside" is det < 0 for every edge; a missing second edge has (0, 0, -1)
    const CircPair *epair; int nepair; float escale, eoff;   // |det| <= escale (|x'| + |y'|) + eoff: too close to call
};
// Deferred slow cases of the thread-per-edge kernel.  Whether a waypoint collides, and which habitat holds it, only
// feed commutative updates of the edge's result (bad |=, cnt +=, mask |=): nothing the rest of the edge depends on.
// A lane that meets a cell needing the general tests (2 % of the waypoints on the Catalina map, i.e. some lane on
// every other step) therefore queues the point and goes on; the warp resolves the queue after its 32 edges, one
// entry per lane, and every lane folds its slot of the result arrays into its edge.
struct SlowEntry { float x, y; int idx; int meta; };      // meta: owner lane | 32: collision test wanted | 64: habitat wanted
#define AUV_SLOWQ_CAP 48
struct SlowQ {               // per warp, shared memory; one pointer (a register) in the hot loop, everything at fixed offsets
    unsigned char *base;     // AUV_SLOWQ_CAP entries | n (entries pushed; beyond the capacity they were resolved in place) | bad[32] cnt[32] mask[32]
    __device__ __forceinline__ SlowEntry *ent() const { return (SlowEntry *)base; }
    __device__ __forceinline__ int *n() const { return (int *)(base + AUV_SLOWQ_CAP * sizeof(SlowEntry)); }
    __device__ __forceinline__ unsigned *bad() const { return (unsigned *)(base + AUV_SLOWQ_CAP * sizeof(SlowEntry) + 16); }
    __device__ __forceinline__ unsigned *cnt() const { return bad() + 32; }
    __device__ __forceinline__ unsigned *mask() const { return bad() + 64; }
};
#define AUV_AP_MAXH 32       // habitat pairs (64 habitats)
#ifndef AUV_AP_BUFFER
#define AUV_AP_BUFFER 1      // all-pairs fp32 build: two waypoints per pass over the circle table (circles_hit2)
#endif
#define AUV_AP_MAXE 16       // polygon edge pairs (32 edges)

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}

// fill a CircTable from the staged world model (all threads of the CTA; caller syncs)
__device__ __forceinline__ void circ_table_fill(CircQuad *dst, const EnvView<float> &env, float ox, float oy) {
    const int nq = (env.K + 3) >> 2;
    for (int j = threadIdx.x; j < nq; j += blockDim.x) {
        float mx[4], my[4], kk[4];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int a = (4 * j + c < env.K) ? 4 * j + c : 4 * j;
            const float ax = env.cx[a] - ox, ay = env.cy[a] - oy;
            mx[c] = -2.f * ax; my[c] = -2.f * ay; kk[c] = fmaf(ay, ay, ax * ax) - env.creff2[a];
        }
        CircQuad q;
        q.m2x = make_float4(mx[0], mx[1], mx[2], mx[3]); q.m2y = make_float4(my[0], my[1], my[2], my[3]);
        q.k = make_float4(kk[0], kk[1], kk[2], kk[3]);
        dst[j] = q;
    }
}
__device__ __forceinline__ float circ_table_ccmax(const EnvView<float> &env, float ox, float oy) {
    float m = 0.f;
    for (int k = 0; k < env.K; k++) {
        const float ax = env.cx[k] - ox, ay = env.cy[k] - oy;
        m = fmaxf(m, fmaf(ay, ay, ax * ax));
    }
    return m;
}

// habitats and boundary edges in the packed form (all threads of the CTA; caller syncs)
__device__ __forceinline__ void allpairs_tables_fill(CircPair *hdst, CircPair *edst, const EnvView<float> &env, float ox, float oy) {
    const int nh = (env.H + 1) >> 1, ne = (env.E + 1) >> 1;
    for (int j = threadIdx.x; j < nh; j += blockDim.x) {
        const int a = 2 * j, b = 2 * j + 1;
        const float ax = env.hx[a] - ox, ay = env.hy[a] - oy;
        CircPair p;
        p.m2x = make_float2(-2.f * ax, 0.f); p.m2y = make_float2(-2.f * ay, 0.f);
        p.k = make_float2(fmaf(ay, ay, ax * ax) - env.hr2[a], Ar<float, false>::inf());
        if (b < env.H) {
            const float bx = env.hx[b] - ox, by = env.hy[b] - oy;
            p.m2x.y = -2.f * bx; p.m2y.y = -2.f * by; p.k.y = fmaf(by, by, bx * bx) - env.hr2[b];
        }
        hdst[j] = p;
    }
    const float sgn = env.convex > 0 ? -1.f : 1.f;       // CCW ring: inside is det > 0 -> flip
    for (int j = threadIdx.x; j < ne; j += blockDim.x) {
        CircPair p;
        p.m2x = make_float2(0.f, 0.f); p.m2y = make_float2(0.f, 0.f); p.k = make_float2(-1.f, -1.f);
        for (int s2 = 0; s2 < 2; s2++) {
            const int i = 2 * j + s2;
            if (i >= env.E) break;
            const int i1 = i + 1 == env.E ? 0 : i + 1;
            const float ax = env.px[i] - ox, ay = env.py[i] - oy, bx = env.px[i1] - ox, by = env.py[i1] - oy;
            const float A = -(by - ay) * sgn, B = (bx - ax) * sgn, Cc = -(B * ay + A * ax);
            if (s2 == 0) { p.m2x.x = A; p.m2y.x = B; p.k.x = Cc; } else { p.m2x.y = A; p.m2y.y = B; p.k.y = Cc; }
        }
        edst[j] = p;
    }
}

// first habitat (list order) holding (x, y): every habitat, packed pairs; -1 none
__device__ __forceinline__ int first_habitat_all_f32(const EnvView<float> &env, const CircTable &ct, float x, float y) {
    const float xr = x - ct.ox, yr = y - ct.oy;
    const float pp = fmaf(yr, yr, xr * xr);
    const float2 x2 = make_float2(xr, xr), y2 = make_float2(yr, yr);
    const float guard = 8e-7f * (pp + ct.hccmax);        // (see point_hits_circles_all)
    int hab = -1;
    bool amb = false;
    for (int j = ct.nhpair - 1; j >= 0; j--) {            // last to first: the earliest match ends up in `hab`
        const CircPair a = ct.hpair[j];
        const float2 q = ffma2(a.m2y, y2, ffma2(a.m2x, x2, a.k));
        const float ta = q.x + pp, tb = q.y + pp;         // d^2 - r^2
        if (tb <= 0.f) hab = 2 * j + 1;
        if (ta <= 0.f) hab = 2 * j;
        amb = amb || fabsf(ta) <= guard || fabsf(tb) <= guard;
    }
    if (__builtin_expect(amb, 0)) {                       // too close to a rim to call: the direct formula, in order
        hab = -1;
        for (int h = 0; h < env.H; h++) {
            const float q = Ar<float, false>::sq2(env.hx[h] - x, env.hy[h] - y);
            if (q <= env.hr2[h]) { hab = h; break; }
        }
    }
    return hab;
}

// strictly inside the convex boundary ring: every edge, packed pairs
__device__ __forceinline__ bool point_within_all_f32(const EnvView<float> &env, const CircTable &ct, float x, float y) {
    const float xr = x - ct.ox, yr = y - ct.oy;
    const float2 x2 = make_float2(xr, xr), y2 = make_float2(yr, yr);
    float dmax = -Ar<float, false>::inf();
    for (int j = 0; j < ct.nepair; j++) {
        const CircPair a = ct.epair[j];
        const float2 d = ffma2(a.m2y, y2, ffma2(a.m2x, x2, a.k));
        dmax = fmaxf(dmax, fmaxf(d.x, d.y));
    }
    // inside <=> every det < 0 <=> dmax < 0; within the rounding error of the expansion: the direct formula
    if (__builtin_expect(fabsf(dmax) <= fmaf(ct.escale, fabsf(xr) + fabsf(yr), ct.eoff), 0)) return point_within<float>(env, x, y);
    return dmax < 0.f;
}

// How close to zero the minimum of the expanded form min_k (|p'|^2 - 2 c_k'.p' + |c_k'|^2 - r_k^2) may be and still be
// trusted.  Circle k's value carries seven roundings of terms bounded by |p'|^2 + |c_k'|^2: an error below
// 4.2e-7 (|p'|^2 + |c_k'|^2).  A circle that can be within 1 m of the point has |c_k'| <= |p'| + r_max + 1; every other
// circle's true value exceeds 2 r + 1 >= 1 m^2, far above its error (< 0.1 m^2 on a 1 km map).  Twice the bound for the
// near circles is therefore a rigorous guard -- about half of 8e-7 (|p'|^2 + max_k |c_k'|^2) for a typical point.
__device__ __forceinline__ float circ_guard(const CircTable &ct, float pp) {
    float root;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(root) : "f"(pp));          // one MUFU; its 2^-22 relative error is nothing next to the factor two
    const float reach = root + ct.rmax1;
    return fminf(8e-7f * fmaf(reach, reach, pp), 8e-7f * (pp + ct.ccmax));
}

// does (x, y) hit any (inflated) circle: every circle, no culling
template <typename R>
__device__ __forceinline__ bool point_hits_circles_all(const EnvView<R> &env, const CircTable &ct, R x, R y) {
    return point_hits_circles<R>(env, x, y);
}
template <>
__device__ __forceinline__ bool point_hits_circles_all<float>(const EnvView<float> &env, const CircTable &ct, float x, float y) {
    if (ct.pair == nullptr) return point_hits_circles<float>(env, x, y);
    const float xr = x - ct.ox, yr = y - ct.oy;
    const float pp = fmaf(yr, yr, xr * xr);
    const float2 x2 = make_float2(xr, xr), y2 = make_float2(yr, yr);
    float q0 = Ar<float, false>::inf(), q1 = q0;
#pragma unroll 4
    for (int j = 0; j < ct.npair; j++) {
        const CircQuad a = ct.pair[j];
        const float2 qa = ffma2(make_float2(a.m2y.x, a.m2y.y), y2, ffma2(make_float2(a.m2x.x, a.m2x.y), x2, make_float2(a.k.x, a.k.y)));
        const float2 qb = ffma2(make_float2(a.m2y.z, a.m2y.w), y2, ffma2(make_float2(a.m2x.z, a.m2x.w), x2, make_float2(a.k.z, a.k.w)));
        q0 = fminf(q0, fminf(qa.x, qa.y));
        q1 = fminf(q1, fminf(qb.x, qb.y));
    }
    const float t = fminf(q0, q1) + pp;                // min_k (d_k^2 - r_k^2)
    // Rounding error of the expansion: seven roundings (k: 3, pp: 2, the two fused multiply-adds) of terms bounded by
    // M = |p'|^2 + max |c'|^2, i.e. <= 7 x 2^-24 M = 4.2e-7 M; the guard is twice that.  (A guard of 4e-6 M, as first
    // written, is 0.7 m^2 on the Catalina map -- a 12 cm band around every rim -- and with 500 circles sent 1 % of the
    // waypoints, hence every fourth warp step, through the scalar loop below: 85 % of the executed instructions.)
    const float guard = circ_guard(ct, pp);
    if (t > guard) return false;
    if (t < -guard) return true;
    return point_hits_circles_outlined<float>(env.cx, env.cy, env.creff2, env.K, x, y);       // too close to call: the direct formula
}

// unsafe point?  (outside the polygon, on its boundary, or inside an inflated circle)
template <typename R> __device__ __forceinline__ bool point_within_all(const EnvView<R> &env, const CircTable &ct, R x, R y) {
    return point_within<R>(env, x, y);
}
template <> __device__ __forceinline__ bool point_within_all<float>(const EnvView<float> &env, const CircTable &ct, float x, float y) {
    if (ct.epair == nullptr) return point_within<float>(env, x, y);
    return point_within_all_f32(env, ct, x, y);
}
template <typename R, bool ALLPAIRS>
__device__ __forceinline__ bool point_unsafe(const EnvView<R> &env, const CircTable &ct, const Cls &cl, R x, R y) {
    if (ALLPAIRS) {
        const bool out = !point_within_all<R>(env, ct, x, y), hit = point_hits_circles_all<R>(env, ct, x, y);     // both, always
        return out || hit;
    }
    return point_unsafe_c<R>(env, cl, x, y);
}

// what one thread carries along an edge
template <typename R> struct ArcEdge;
// Two waypoints per pass over the circle table (all-pairs fp32 build): the three 16-byte loads of a quad feed eight FFMA2
// instead of four.  A warp flushes its lanes' buffers together as soon as one of them holds two waypoints
// (edges_tpe.cu); a lane holding one tests it twice.  Returns "some buffered waypoint hits a circle".
__device__ __forceinline__ bool circles_hit2(const EnvView<float> &env, const CircTable &ct, float xa, float ya, float xb, float yb) {
    const float xra = xa - ct.ox, yra = ya - ct.oy, xrb = xb - ct.ox, yrb = yb - ct.oy;
    const float ppa = fmaf(yra, yra, xra * xra), ppb = fmaf(yrb, yrb, xrb * xrb);
    const float2 xa2 = make_float2(xra, xra), ya2 = make_float2(yra, yra), xb2 = make_float2(xrb, xrb), yb2 = make_float2(yrb, yrb);
    float a0 = Ar<float, false>::inf(), a1 = a0, b0 = a0, b1 = a0;
#pragma unroll 2
    for (int j = 0; j < ct.npair; j++) {
        const CircQuad q = ct.pair[j];
        const float2 mxl = make_float2(q.m2x.x, q.m2x.y), mxh = make_float2(q.m2x.z, q.m2x.w);
        const float2 myl = make_float2(q.m2y.x, q.m2y.y), myh = make_float2(q.m2y.z, q.m2y.w);
        const float2 kl = make_float2(q.k.x, q.k.y), kh = make_float2(q.k.z, q.k.w);
        const float2 al = ffma2(myl, ya2, ffma2(mxl, xa2, kl)), ah = ffma2(myh, ya2, ffma2(mxh, xa2, kh));
        const float2 bl = ffma2(myl, yb2, ffma2(mxl, xb2, kl)), bh = ffma2(myh, yb2, ffma2(mxh, xb2, kh));
        a0 = fminf(a0, fminf(al.x, al.y)); a1 = fminf(a1, fminf(ah.x, ah.y));
        b0 = fminf(b0, fminf(bl.x, bl.y)); b1 = fminf(b1, fminf(bh.x, bh.y));
    }
    const float ta = fminf(a0, a1) + ppa, tb = fminf(b0, b1) + ppb;
    const float ga = circ_guard(ct, ppa), gb = circ_guard(ct, ppb);
    bool hit = ta < -ga || tb < -gb;
    if (__builtin_expect(!hit && fabsf(ta) <= ga, 0)) hit = point_hits_circles_outlined<float>(env.cx, env.cy, env.creff2, env.K, xa, ya);
    if (__builtin_expect(!hit && fabsf(tb) <= gb, 0)) hit = point_hits_circles_outlined<float>(env.cx, env.cy, env.creff2, env.K, xb, yb);
    return hit;
}

// the same out of line through the shared copy of the view (every cell that is not "inside and clear")
template <typename R>
__device__ __noinline__ bool point_unsafe_shared(const EnvView<R> *senv, unsigned code, int idx, R x, R y) {
    Cls cl; cl.code = code; cl.idx = idx;
    return !point_within_c<R>(*senv, cl, x, y) || point_hits_circles_c<R>(*senv, cl, x, y);
}

// one queued point: the general tests, results into the owner's slots
template <typename R>
__device__ __forceinline__ void slowq_resolve(const EnvView<R> &env, const SlowQ &q, const SlowEntry &en) {
    const int owner = en.meta & 31;
    Cls cl; cl.idx = en.idx;
    cl.code = en.idx >= 0 ? __ldg(env.grid + en.idx) : ((AUV_GRID_HAB_AMBIG << 3) | AUV_GRID_HAB_MANY | AUV_GRID_CIRC_MANY | AUV_GRID_POLY_FULL | 2u);
    const R x = (R)en.x, y = (R)en.y;
    if (en.meta & 32) {
        if (!point_within_c<R>(env, cl, x, y) || point_hits_circles_c<R>(env, cl, x, y)) atomicOr(&q.bad()[owner], 1u);
    } else {
        const int hab = first_habitat_ambiguous<R>(env.shared_self, cl.code, cl.idx, env.H, x, y);
        if (hab >= 0) { atomicAdd(&q.cnt()[owner], 1u); atomicOr(&q.mask()[owner], 1u << (hab & 31)); }
    }
}
// queue a point (out of line: the hot loop only sees a call); a full queue resolves the point on the spot
template <typename R>
__device__ __noinline__ void slowq_push(const EnvView<R> *senv, unsigned char *qbase, float x, float y, int idx, int meta) {
    SlowQ q; q.base = qbase;
    __builtin_assume(__isShared(qbase));
    SlowEntry en; en.x = x; en.y = y; en.idx = idx; en.meta = meta;
    const int slot = atomicAdd(q.n(), 1);
    if (slot < AUV_SLOWQ_CAP) q.ent()[slot] = en;
    else slowq_resolve<R>(*senv, q, en);
}
// resolve the queued points: all 32 lanes of the warp, converged; afterwards lane l owns bad[l], cnt[l], mask[l]
template <typename R>
__device__ __forceinline__ void slowq_drain(const EnvView<R> &env, const SlowQ &q) {
    __syncwarp();
    const int lane = threadIdx.x & 31, n = min(*q.n(), AUV_SLOWQ_CAP);
    for (int j = lane; j < n; j += 32) slowq_resolve<R>(env, q, q.ent()[j]);
    __syncwarp();
}

// what one thread carries along an edge
template <typename R> struct ArcEdge {
    R x, y, th, t, len;
    R vt;                      // velocity_temp of the last valid primitive (the v column of a path row)
    R sin0, cos0;              // fp64 build: sin / cos of the heading the next primitive starts from
    int nwp;                   // len(new.path): appended waypoints + 1 (path[0] = parent)
    bool bad, moved, degenerate, last_is_wp;
    R s2; uint32_t cnt; unsigned long long mask;     // cost sums over the APPENDED waypoints
    R self_s2; int self_hab;                         // contribution of the provisional leaf state
    BinCursor<R> bins;                               // shark-grid time bin of the current traj_time_stamp (COST)
    int status;
    // all-pairs fp32 build: waypoints waiting for the circle loop (circles_flush2 takes two per pass over the circle table)
    float pbx0, pby0, pbx1, pby1; int nbuf;
};

// queue a waypoint for the circle loop / run the loop over whatever the lane holds (all-pairs fp32 build)
template <typename R> __device__ __forceinline__ void circles_push(ArcEdge<R> &e, R x, R y) {
    if (e.nbuf == 0) { e.pbx0 = (float)x; e.pby0 = (float)y; } else { e.pbx1 = (float)x; e.pby1 = (float)y; }
    e.nbuf++;
}
template <typename R> __device__ __forceinline__ void circles_flush2(const EnvView<R> &env, const CircTable &ct, ArcEdge<R> &e) {
    if constexpr (sizeof(R) == 4) {
        if (e.nbuf > 0) {
            const bool two = e.nbuf > 1;
            const bool hit = circles_hit2(env, ct, e.pbx0, e.pby0, two ? e.pbx1 : e.pbx0, two ? e.pby1 : e.pby0);
            e.bad = e.bad || hit;
            e.nbuf = 0;
        }
    }
}

// path[0] = the parent node object: tested like any other path point (rrt_dubins.py:537,544)
// FASTENV: contiguous equal time bins, the x-bucket table and a shared copy of the view are all present (the
// launcher checked): the hot loop carries no run-time flags.
template <typename R, bool ALLPAIRS, bool FASTENV = false, bool GRIDS = false, bool DEFER = false>
__device__ __forceinline__ void arc_edge_begin(const EnvView<R> &env, const CircTable &ct, ArcEdge<R> &e, R px, R py, R pth,
                                               R pt, R plen, R parent_self_s2, int parent_self_hab, const SlowQ sq = SlowQ()) {
    typedef typename Policy<R>::A A;
    e.x = px; e.y = py; e.th = pth; e.t = pt; e.len = plen; e.vt = 0;
    e.sin0 = 0; e.cos0 = 0;
    if (Policy<R>::VERIFY) A::sincos(pth, &e.sin0, &e.cos0);
    e.nwp = 1; e.moved = false; e.degenerate = false; e.last_is_wp = false;
    e.s2 = 0; e.cnt = 0; e.mask = 0ull; e.self_s2 = parent_self_s2; e.self_hab = parent_self_hab; e.status = 0;
    e.nbuf = 0; e.pbx0 = e.pby0 = e.pbx1 = e.pby1 = 0.f;
    Cls pcl; pcl.code = 0; pcl.idx = -1;
    if (!ALLPAIRS) pcl = env.template classify<GRIDS>(px, py);
    if (AUV_OUTLINE_COLLIDE && FASTENV && !ALLPAIRS) e.bad = (pcl.code & 7u) != 5u && point_unsafe_shared<R>(env.shared_self, pcl.code, pcl.idx, px, py);
    else if (DEFER && !ALLPAIRS && !Policy<R>::VERIFY) {
        e.bad = point_unsafe_one<R>(env, pcl.code, px, py);
        if (__builtin_expect((pcl.code & AUV_GRID_SLOW) != 0u, 0)) {
            slowq_push<R>(env.shared_self, sq.base, (float)px, (float)py, pcl.idx, (int)(threadIdx.x & 31u) | 32);
            e.bad = false;
        }
    } else if (ALLPAIRS && sizeof(R) == 4 && AUV_AP_BUFFER && ct.buf2) {
        e.bad = !point_within_all<R>(env, ct, px, py);          // the boundary now, the circles together with the next waypoint
        circles_push<R>(e, px, py);
    } else e.bad = point_unsafe<R, ALLPAIRS>(env, ct, pcl, px, py);
    e.bins.k = 0; e.bins.up = 0;
    if (AUV_BIN_CURSOR && (FASTENV || env.bins_uniform)) e.bins.start(env, pt);
}

// one arc primitive (rrt_dubins.py:264-284).  Returns false when the edge must stop (ZeroDivisionError in
// the fp64 build; a degenerate 2^-23 draw in the fp32 build, which rejects the sample).
// DEFER: queue the slow cases in *sq (see SlowQ) instead of resolving them in place
template <typename R, bool COST, bool SELF, bool ALLPAIRS, bool FASTENV = false, bool GRIDS = false, bool DEFER = false>
__device__ __forceinline__ bool arc_edge_step(const EnvView<R> &env, const CircTable &ct, const SteerParams<R> &sp, R w3,
                                              SerialStream<R> &rng, ArcEdge<R> &e, const SlowQ sq = SlowQ()) {
    typedef typename Policy<R>::A A;
    const bool VERIFY = Policy<R>::VERIFY;
    // (fp32: uniform_ab with its two invariants b - a and a - (b - a) taken from the parameter block)
    const R dist = VERIFY ? uniform_ab<R>((R)0, sp.d2e, rng.next()) : A::fma(sp.d2e, rng.next(), sp.o_dist);             // :264
    const R diff = VERIFY ? uniform_ab<R>(sp.neg_dmax, sp.dmax, rng.next()) : A::fma(sp.w_diff, rng.next(), sp.o_diff);  // :265
    if (!(A::fabs(dist) > A::fabs(diff))) { rng.skip(1u); return true; }             // :266; the velocity slot stays unread
    const R vt = VERIFY ? uniform_ab<R>((R)0, sp.two_vel, rng.next()) : A::fma(sp.two_vel, rng.next(), sp.o_vel);        // :279
    R movement;
    if (VERIFY) {
        R s1 = A::add(dist, diff), s2 = A::sub(dist, diff), den = A::add(-s1, s2), num = A::add(s1, s2);
        if (den == (R)0) { e.status = AUVRRT_ST_ZERO_DIV; return false; }
        R radius = A::div(num, den), r2 = A::mul((R)2, radius);                      // :270
        if (r2 == (R)0) { e.status = AUVRRT_ST_ZERO_DIV; return false; }
        e.th = A::add(e.th, A::div(num, r2));                                        // :271, :274
        R s1v, c1v;
        A::sincos(e.th, &s1v, &c1v);
        const R dx = A::mul(radius, A::sub(s1v, e.sin0));                            // :275
        const R dy = A::mul(radius, A::add(-c1v, e.cos0));                           // :276
        e.sin0 = s1v; e.cos0 = c1v;
        movement = A::sqrt(A::sq2(dx, dy));                                          // :280
        if (vt == (R)0) { e.status = AUVRRT_ST_ZERO_DIV; return false; }
        e.x = A::add(e.x, dx); e.y = A::add(e.y, dy);
        e.t = A::add(e.t, A::div(movement, vt));                                     // :281
        e.len = A::add(e.len, movement);
    } else {
        // stable restatement of the arc (edge.cuh): turn angle -diff, chord = dist * sinc(diff / 2), heading
        // at mid-arc; no radius * (sin - sin) cancellation, no sqrt
        if (diff == (R)0 || vt == (R)0) { e.degenerate = true; return false; }
        const R half = (R)0.5 * diff;
        movement = dist * sinc_small((float)half);
        R sm, cm;
        A::sincos(e.th - half, &sm, &cm);
        e.th -= diff;
        e.x = A::fma(movement, cm, e.x); e.y = A::fma(movement, sm, e.y);
        e.t = A::fma(movement, A::div((R)1, vt), e.t);
        e.len += movement;
    }
    e.moved = true;
    e.vt = vt;
    e.last_is_wp = movement >= sp.min_dist;                                          // :283
    if (e.last_is_wp) {
        e.nwp++;
        Cls cl; cl.code = AUV_GRID_ALL_AMBIG; cl.idx = -1;
        if (ALLPAIRS) {
            // every waypoint against everything, also on an edge that is already unsafe: the executed work is the FLOP
            // count the roofline figure uses
            if (sizeof(R) == 4 && AUV_AP_BUFFER && ct.buf2) {
                const bool out = !point_within_all<R>(env, ct, e.x, e.y);
                e.bad = e.bad || out;
                if (e.nbuf >= 2) circles_flush2<R>(env, ct, e);       // (the caller flushes earlier, warp-wide; this keeps the buffer bounded)
                circles_push<R>(e, e.x, e.y);
            } else {
                const bool u = point_unsafe<R, true>(env, ct, cl, e.x, e.y);
                e.bad = e.bad || u;
            }
        }
        else {
            cl = env.template classify<GRIDS>(e.x, e.y);
            if (Policy<R>::VERIFY) {
                // the common cell: strictly inside the polygon (code 1) and clear of every circle (bit 2)
                if (__builtin_expect((cl.code & 7u) != 5u, 0)) e.bad = e.bad || point_unsafe<R, false>(env, ct, cl, e.x, e.y);
            } else {
                // decided cells and single-candidate boundary cells in straight-line code (point_unsafe_one)
                bool bad1 = point_unsafe_one<R>(env, cl.code, e.x, e.y);
                if (__builtin_expect((cl.code & AUV_GRID_SLOW) != 0u && !e.bad, 0)) {       // (an edge that is already unsafe skips the general tests)
                    if (DEFER) { slowq_push<R>(env.shared_self, sq.base, (float)e.x, (float)e.y, cl.idx, (int)(threadIdx.x & 31u) | 32); bad1 = false; }
                    else bad1 = (AUV_OUTLINE_COLLIDE && (FASTENV || env.shared_self)) ? point_unsafe_shared<R>(env.shared_self, cl.code, cl.idx, e.x, e.y)
                                                                                      : (!point_within_c<R>(env, cl, e.x, e.y) || point_hits_circles_c<R>(env, cl, e.x, e.y));
                }
                e.bad = e.bad || bad1;
            }
        }
        if (COST) {
            int kb = -2;
            if (AUV_BIN_CURSOR) { if (FASTENV || env.bins_uniform) kb = e.bins.at(env, e.t); }
            else if (FASTENV) kb = find_bin<R, true>(env, e.t, 0xffffffffu);
            Contrib c;
            if constexpr (ALLPAIRS && sizeof(R) == 4) {
                // every habitat in the packed form (the grid code for "no habitat test needed" keeps point_contrib off them)
                if (ct.hpair != nullptr) cl.code = (cl.code & ~(0xFFu << 3)) | (AUV_GRID_HAB_NONE << 3);
                c = point_contrib<R, false>(env, e.x, e.y, e.t, 0xffffffffu, env.H, cl, kb);
                if (ct.hpair != nullptr && c.bin >= 0) c.hab = first_habitat_all_f32(env, ct, (float)e.x, (float)e.y);
            } else {
                c = point_contrib<R, FASTENV && !ALLPAIRS, DEFER && FASTENV && !ALLPAIRS>(env, e.x, e.y, e.t, 0xffffffffu, env.H, cl, kb);
                if (DEFER && FASTENV && !ALLPAIRS) {
                    if (__builtin_expect(c.hab == -2, 0)) {          // ambiguous habitat cell (the point lies in a time bin)
                        slowq_push<R>(env.shared_self, sq.base, (float)e.x, (float)e.y, cl.idx, (int)(threadIdx.x & 31u) | 64);
                        c.hab = -1;
                    }
                }
            }
            const R ps2 = (c.bin >= 0 && c.cell >= 0) ? A::mul(w3, env.probs[c.bin * env.C + c.cell]) : (R)0;
            // no bin holds the time stamp: the point is skipped (cost.py:178); point_contrib then reports no cell and no
            // habitat, so the sums below do not move (s2 only ever grows from +0)
            e.s2 = A::add(e.s2, ps2);
            const unsigned hb = c.hab >= 0 ? 1u : 0u, sh = (unsigned)c.hab & 31u;
            e.cnt += hb;
            if (FASTENV) e.mask |= (unsigned long long)(hb << sh);             // FASTENV: at most 32 habitats (checked by the launcher)
            else e.mask |= (unsigned long long)((c.hab & 32) ? 0u : (hb << sh)) | ((unsigned long long)((c.hab & 32) ? (hb << sh) : 0u) << 32);
            if (SELF) { e.self_s2 = c.bin >= 0 ? ps2 : (R)0; e.self_hab = c.bin >= 0 ? c.hab : -1; }
        }
    }
    return true;
}

}  // namespace auv
