// edge.cuh -- one candidate edge, evaluated cooperatively by a group of G lanes:
//   RRT.steer, the random-arc rollout   (/root/reference/path_planning/rrt_dubins.py:252-295)
//   RRT.check_collision                  (rrt_dubins.py:530-549)
//   the per-waypoint part of cost.habitat_shark_cost_func (/root/reference/path_planning/cost.py:171-191)
//
// Lane k of the group owns arc primitive k of the current chunk of G primitives.
// The reference consumes its uniforms serially and data-dependently (2 per primitive, a 3rd only if
// abs(dist) > abs(diff), rrt_dubins.py:264-279).  Here every lane hashes its own stream positions,
// the per-position step (2 or 3) goes to shared memory, and log2(G) rounds of pointer doubling give
// each lane the stream offset of its primitive.  theta/x/y/time/length are then prefix sums over
// the lanes: shuffle scans in the fast build, the reference's exact serial order in the fp64
// verification build.
#pragma once
#include "geom.cuh"

#ifndef AUV_EDGE_ONE
// warp-per-edge evaluation: single-candidate boundary cells in straight-line code (point_unsafe_one).  Measured on B200,
// k_plan config 2: 8.89 ms per step with it (and AUV_HAB_ONE), 8.71 with this one off, 8.65 with both off -- the lanes of a
// warp are consecutive waypoints of ONE edge, mostly in cells of one kind, so the branches cost little here and the
// unconditional fetches cost their instructions.  Off; the thread-per-edge kernels (32 unrelated edges per warp) use it.
#define AUV_EDGE_ONE 0
#endif

namespace auv {

template <typename R> struct SteerParams {
    R d2e, dmax, neg_dmax, freq, min_dist, two_vel;
    // uniform_ab<float>(a, b, d) = fmaf(w, d, o) with w = b - a, o = a - w: the two loop invariants of the three steer draws
    R w_diff, o_dist, o_diff, o_vel;
};

template <int G> struct Log2 { static const int v = (G == 32) ? 5 : (G == 16) ? 4 : (G == 8) ? 3 : (G == 4) ? 2 : 1; };

// per-group shared-memory scratch
// FLAT = false (the counter stream with slot addressing: the planners) needs neither the window of uniforms nor the
// pointer-doubling table: 396 instead of 1148 bytes per 32-lane group in fp32 -- shared memory the L1 gets back
template <typename R, int G, bool FLAT = true> struct GroupScratch {
    R us[FLAT ? 3 * G : 32];              // window of uniforms starting at the chunk's offset (FLAT); 32 words of scratch otherwise (k_plan mode 3)
    R wx[G + 1], wy[G + 1];               // waypoint coordinates for the circle lanes (slot G: parent)
    unsigned char jmp[FLAT ? Log2<G>::v : 1][FLAT ? 3 * G + 4 : 4];
};

template <typename R> struct EdgeOut {
    R x, y, th, t, len;       // the new node (leaf of the edge)
    int nwp;                  // len(new.path): appended waypoints + 1 (path[0] = parent)
    int n_exp;                // primitives drawn
    uint32_t ctr;             // stream position after the edge
    int status;
    bool safe;                // check_collision result
    // cost contributions (only if DO_COST): sums over the APPENDED waypoints ...
    R s2; uint32_t cnt; uint64_t mask;
    // ... and of the new node's own state (valid iff leaf_moved; else identical to the parent's)
    R self_s2; int self_hab; bool leaf_moved;
};

// sin(h)/h for the fast build (|h| = |diff|/2 <= diff_max/2)
__device__ __forceinline__ float sinc_small(float h) {
    float z = h * h;
    if (z > 0.25f) {       // only for diff_max > 1: reduced-argument MUFU sine (abs. error ~4e-7), not the libdevice sinf
        float sn, cs;      // whose slow path would sit inside every edge evaluation
        Ar<float, false>::sincos(h, &sn, &cs);
        return __fdividef(sn, h);
    }
    // 1 - z/6 + z^2/120 - z^3/5040 + z^4/362880     (|err| < 2e-9 for |h| <= 0.5)
    float p = fmaf(z, 2.7557319e-6f, -1.9841270e-4f);
    p = fmaf(z, p, 8.3333333e-3f);
    p = fmaf(z, p, -1.6666667e-1f);
    return fmaf(z, p, 1.0f);
}

// wp_out rows: (x, y, theta, v, traj_time_stamp, length)
// FLAT = false: the counter stream with slot addressing (DESIGN.md section 3): the edge owns 1 + 3 n_expand
//   positions, primitive k reads ctr + 1 + 3k (dist), + 1 (diff) and, only if abs(dist) > abs(diff), + 2
//   (velocity_temp): every lane knows its positions, no offsets to resolve.
// FLAT = true : an explicit recorded stream (e.g. a CPython Mersenne-Twister sequence) consumed back to back,
//   2 or 3 uniforms per primitive: the per-position step goes to shared memory and log2(G) rounds of pointer
//   doubling give each lane the offset of its primitive.
// ONE_CHUNK: the caller guarantees n_expand <= G - 1 (freq <= G, checked on the host): the chunk runs exactly once (no
//   loop-carried state), and lane G - 1, which never holds a primitive, tests the parent point (path[0]) with the same
//   code as the waypoint lanes.
// GRIDS: plane 0 of the classification grid is staged in shared memory (env.grid0s)
template <typename R, int G, bool DO_COLLIDE, bool DO_COST, bool WRITE_WP, bool FLAT = false, bool ONE_CHUNK = false, bool GRIDS = false>
__device__ __forceinline__ void eval_edge(const Grp<G> &g, GroupScratch<R, G, FLAT> &sc, const EnvView<R> &env,
                                          const Stream<R> &rng, uint32_t ctr, const SteerParams<R> &sp,
                                          R px, R py, R pth, R pt, R plen, R w3, int n_hab,
                                          R *wp_out, int wp_cap, EdgeOut<R> &out) {
    typedef typename Policy<R>::A A;
    const bool VERIFY = Policy<R>::VERIFY;
    const int LOG = Log2<G>::v;

    // n_expand = floor(uniform(0, freq) / 1)                                   rrt_dubins.py:259-260
    R u0 = rng.u(ctr);
    ctr += 1;
    int n_exp = (int)A::floor(uniform_ab<R>((R)0, sp.freq, u0));
    out.n_exp = n_exp;
    out.status = 0;

    // carries (group-uniform)
    R cth = pth, cx = px, cy = py, ct = pt, clen = plen;
    R csin = 0, ccos = 0;
    if (VERIFY) A::sincos(pth, &csin, &ccos);
    int nwp = 1;
    bool hit = false, outside = false, zero_div = false, moved = false, degenerate = false, parent_clear = false, parent_many = false;
    R acc_s2 = 0; uint32_t acc_cnt = 0; uint64_t acc_mask = 0;
    R self_s2 = 0; int self_hab = -1;

    if (DO_COLLIDE) {
        // path[0] = the parent node object: tested like any other path point (rrt_dubins.py:537,544)
        // (testing it behind the draws and the steer arithmetic of the first chunk, to run those under the planner's
        // load of the parent row, was measured slower: 9.16 vs 8.75 ms per step on config 2; ONE_CHUNK tests it in
        // lane G - 1 of the chunk instead)
        if (g.gl == 0) { sc.wx[G] = px; sc.wy[G] = py; }
    }
    if (DO_COLLIDE && !ONE_CHUNK) {
        const Cls pcl = env.template classify<GRIDS>(px, py);
        parent_clear = (pcl.code & 4u) != 0u;
        parent_many = (pcl.code & AUV_GRID_CIRC_MANY) != 0u;
        if (VERIFY || !AUV_EDGE_ONE || (pcl.code & AUV_GRID_SLOW)) {
            outside = !point_within_c<R>(env, pcl, px, py);
            if (!parent_clear && !parent_many) hit = point_hits_circles_c<R>(env, pcl, px, py);
        } else outside = point_unsafe_one<R>(env, pcl.code, px, py);     // (either flag makes the edge unsafe)
    }

    for (int base = 0; ONE_CHUNK ? base == 0 : base < n_exp; base += G) {
        const int nact = ONE_CHUNK ? max(min(G, n_exp), 0) : min(G, n_exp - base);     // active primitives in this chunk
        const bool act = g.gl < nact;
        R dist = 0, diff = 0, vt = 1;
        bool valid = false;
        if (FLAT) {
            // ---- 1. window of uniforms, one hash per lane per round
    #pragma unroll
            for (int r = 0; r < 3; r++) {
                int s = g.gl + G * r;
                sc.us[s] = (s < 3 * nact) ? rng.u(ctr + (uint32_t)s) : (R)0;
            }
            g.sync();
            // ---- 2. stream offset of every primitive: pointer doubling over step(s) in {2, 3}
    #pragma unroll
            for (int r = 0; r < 3; r++) {
                int s = g.gl + G * r;
                int nx = 3 * G;
                if (s <= 3 * G - 3) {
                    R dist = uniform_ab<R>((R)0, sp.d2e, sc.us[s]);
                    R diff = uniform_ab<R>(sp.neg_dmax, sp.dmax, sc.us[s + 1]);
                    nx = s + 2 + (A::fabs(dist) > A::fabs(diff) ? 1 : 0);
                    if (nx > 3 * G) nx = 3 * G;
                }
                sc.jmp[0][s] = (unsigned char)nx;
            }
            if (g.gl == 0) {
    #pragma unroll
                for (int d = 0; d < LOG; d++) sc.jmp[d][3 * G] = (unsigned char)(3 * G);
            }
            g.sync();
    #pragma unroll
            for (int d = 1; d < LOG; d++) {
    #pragma unroll
                for (int r = 0; r < 3; r++) {
                    int s = g.gl + G * r;
                    sc.jmp[d][s] = sc.jmp[d - 1][sc.jmp[d - 1][s]];
                }
                g.sync();
            }
            int o = 0;
    #pragma unroll
            for (int d = 0; d < LOG; d++)
                if ((g.gl >> d) & 1) o = sc.jmp[d][o];
                // ---- 3. this lane's primitive                                          rrt_dubins.py:264-284
            if (act) {
                dist = uniform_ab<R>((R)0, sp.d2e, sc.us[o]);
                diff = uniform_ab<R>(sp.neg_dmax, sp.dmax, sc.us[o + 1]);
                valid = A::fabs(dist) > A::fabs(diff);
                if (valid) vt = uniform_ab<R>((R)0, sp.two_vel, sc.us[o + 2]);
            }
            // offset just past the chunk's last active primitive
            int o_end = g.bcast(o + 2 + (valid ? 1 : 0), nact - 1);
            ctr += (uint32_t)o_end;

        } else {
            // ---- 1-3. slot addressing: this lane's primitive reads its own three positions     rrt_dubins.py:264-279
            if (act) {
                const uint32_t p0 = ctr + 3u * (uint32_t)g.gl;
                dist = uniform_ab<R>((R)0, sp.d2e, rng.u(p0));
                diff = uniform_ab<R>(sp.neg_dmax, sp.dmax, rng.u(p0 + 1u));
                valid = A::fabs(dist) > A::fabs(diff);
                if (valid) vt = uniform_ab<R>((R)0, sp.two_vel, rng.u(p0 + 2u));
            }
            ctr += 3u * (uint32_t)nact;
        }
        R phi = 0, radius = 0, chord = 0;
        if (valid) {
            if (VERIFY) {
                R s1 = A::add(dist, diff), s2 = A::sub(dist, diff);
                R den = A::add(-s1, s2);
                R num = A::add(s1, s2);
                if (den == (R)0) zero_div = true;
                radius = A::div(num, den);                                     // :270
                R r2 = A::mul((R)2, radius);
                if (r2 == (R)0) zero_div = true;
                phi = A::div(num, r2);                                         // :271
            } else {
                if (diff == (R)0) zero_div = true;
                phi = -diff;                       // (s1+s2)/(2*radius) with radius = -dist/diff
                chord = dist * sinc_small((float)diff * 0.5f);
            }
            if (vt == (R)0) zero_div = true;
        }
        // theta: inclusive running sum                                           :274
        R th;
        if (VERIFY) th = (R)grp_scan_serial<G>(g, (double)phi, (double)cth);
        else th = grp_scan_incl<G>(g, phi) + cth;
        R dx = 0, dy = 0, movement = 0, dt = 0;
        if (VERIFY) {
            R s1v, c1v;
            A::sincos(th, &s1v, &c1v);
            R s0v = g.up(s1v, 1), c0v = g.up(c1v, 1);
            if (g.gl == 0) { s0v = csin; c0v = ccos; }
            if (valid) {
                dx = A::mul(radius, A::sub(s1v, s0v));                         // :275
                dy = A::mul(radius, A::add(-c1v, c0v));                        // :276
                movement = A::sqrt(A::sq2(dx, dy));                            // :280
                dt = A::div(movement, vt);                                     // :281
            }
            csin = g.bcast(s1v, G - 1); ccos = g.bcast(c1v, G - 1);   // theta(G-1) == theta(last valid) bit for bit
        } else {
            if (valid) {
                R sm, cm;
                A::sincos(th - (R)0.5 * phi, &sm, &cm);       // heading at the middle of the arc
                dx = chord * cm; dy = chord * sm;
                movement = chord;
                dt = A::div(movement, vt);
            }
        }
        R x, y, t, len;
        if (VERIFY) {
            x = (R)grp_scan_serial<G>(g, (double)dx, (double)cx);
            y = (R)grp_scan_serial<G>(g, (double)dy, (double)cy);
            t = (R)grp_scan_serial<G>(g, (double)dt, (double)ct);
            len = (R)grp_scan_serial<G>(g, (double)movement, (double)clen);
        } else {
            x = grp_scan_incl<G>(g, dx) + cx;
            y = grp_scan_incl<G>(g, dy) + cy;
            t = grp_scan_incl<G>(g, dt) + ct;
            len = grp_scan_incl<G>(g, movement) + clen;
        }
        const bool is_wp = valid && (movement >= sp.min_dist);                  // :283
        const unsigned wpm = g.ballot(is_wp);
        const unsigned vm = g.ballot(valid);
        if (vm) moved = true;
        const int last_valid = vm ? 31 - __clz(vm) : -1;   // lane whose state is the chunk's end state

        if (WRITE_WP) {
            if (is_wp) {
                int row = nwp - 1 + __popc(wpm & ((1u << g.gl) - 1u));
                if (row < wp_cap) {
                    R *w = wp_out + 6 * (size_t)row;
                    w[0] = x; w[1] = y; w[2] = th; w[3] = vt; w[4] = t; w[5] = len;
                }
            }
        }
        // ONE_CHUNK: lane G - 1 holds no primitive (n_expand <= G - 1) and tests the parent point
        const bool pl = ONE_CHUNK && DO_COLLIDE && g.gl == G - 1;
        const R tx = pl ? px : x, ty = pl ? py : y;          // the point this lane tests
        // one classification-grid load per waypoint replaces most of the exact tests below
        Cls cl; cl.code = AUV_GRID_ALL_AMBIG | 4u; cl.idx = -1;
        if ((DO_COLLIDE || DO_COST) && (is_wp || g.gl == last_valid || pl)) cl = env.template classify<GRIDS>(tx, ty);
        if (DO_COLLIDE) {
            // lane = waypoint: polygon and the cell's candidate circles
            bool in = true, h1 = false;
            if (is_wp || pl) {
                if (VERIFY || !AUV_EDGE_ONE) {
                    in = point_within_c<R>(env, cl, tx, ty);
                    if (!(cl.code & AUV_GRID_CIRC_MANY)) h1 = point_hits_circles_c<R>(env, cl, tx, ty);
                } else {
                    // decided cells and single-candidate boundary cells in straight-line code; `in` carries the verdict
                    in = !point_unsafe_one<R>(env, cl.code, tx, ty);
                    if (__builtin_expect((cl.code & AUV_GRID_SLOW) != 0u, 0)) {
                        in = point_within_c<R>(env, cl, tx, ty);
                        if (!(cl.code & AUV_GRID_CIRC_MANY)) h1 = point_hits_circles_c<R>(env, cl, tx, ty);
                    }
                }
            }
            if (g.ballot(!in)) outside = true;
            if (g.ballot(h1)) hit = true;
            // cells with more than 3 candidate circles (or points outside the grid): lane = circle over
            // all circles, waypoints broadcast through shared memory; the parent joins them in the first chunk (the
            // chunked form tests a parent in such a cell after the loop when n_expand == 0, and not at all when < 0)
            const bool circles_needed = g.ballot((is_wp || (pl && n_exp >= 0)) && !(cl.code & 4u) && (cl.code & AUV_GRID_CIRC_MANY)) != 0u ||
                                        (!ONE_CHUNK && base == 0 && !parent_clear && parent_many);
            // (an edge that already left the polygon is unsafe whatever the circles say)
            if (env.K > 0 && circles_needed && !outside) {
                if (is_wp) { int slot = __popc(wpm & ((1u << g.gl) - 1u)); sc.wx[slot] = x; sc.wy[slot] = y; }
                g.sync();
                const int nw = __popc(wpm);
                bool h = false;
#pragma unroll 1                       // rare path: keep it small, it sits inside the hot loop
                for (int k = g.gl; k < env.K; k += G) {
                    R ccx = env.cx[k], ccy = env.cy[k];
                    R q = A::inf();
                    if (base == 0) q = A::sq2(A::sub(sc.wx[G], ccx), A::sub(sc.wy[G], ccy));
#pragma unroll 1
                    for (int j = 0; j < nw; j++) {
                        R qq = A::sq2(A::sub(sc.wx[j], ccx), A::sub(sc.wy[j], ccy));
                        q = qq < q ? qq : q;
                    }
                    if (VERIFY) h = h || (A::sqrt(q) <= env.creff[k]);
                    else h = h || (q <= env.creff2[k]);
                }
                if (g.ballot(h)) hit = true;
                g.sync();
            }
        }
        if (DO_COST) {
            // lane = waypoint; the lane holding the chunk's end state also evaluates it as the
            // (provisional) leaf state
            const bool need = is_wp || (g.gl == last_valid);
            Contrib c; c.bin = -1; c.cell = -1; c.hab = -1;
            if (need) c = point_contrib<R>(env, x, y, t, 0xffffffffu, n_hab, cl);
            R ps2 = (R)0;
            if (c.bin >= 0 && c.cell >= 0) ps2 = A::mul(w3, env.probs[(size_t)c.bin * env.C + c.cell]);
            const bool counts = is_wp && c.bin >= 0;
            acc_s2 += grp_sum<G>(g, counts ? ps2 : (R)0);
            unsigned hm = g.ballot(counts && c.hab >= 0);
            acc_cnt += __popc(hm);
            // visited-habitat set: OR of (1 << hab) over counting lanes
            unsigned long long mbits = (counts && c.hab >= 0) ? (1ull << c.hab) : 0ull;
            if (G == 32) {
                // full warp: two REDUX.OR instead of ten shuffles
                const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)mbits), hi = __reduce_or_sync(0xffffffffu, (unsigned)(mbits >> 32));
                mbits = ((unsigned long long)hi << 32) | lo;
            } else {
#pragma unroll
                for (int m = G / 2; m > 0; m >>= 1) mbits |= g.xorv(mbits, m);
            }
            acc_mask |= mbits;
            if (last_valid >= 0) {
                self_s2 = g.bcast((c.bin >= 0) ? ps2 : (R)0, last_valid);
                self_hab = g.bcast((c.bin >= 0) ? c.hab : -1, last_valid);
            }
        }
        nwp += __popc(wpm);
        // carries for the next chunk = state after the last valid primitive.  (Invalid / inactive lanes
        // add zero, but a shuffle scan associates differently per lane, so take the value from the
        // lane whose waypoint it is: the node object and its last waypoint must be the same numbers.)
        if (last_valid >= 0) {
            cth = g.bcast(th, last_valid); cx = g.bcast(x, last_valid); cy = g.bcast(y, last_valid);
            ct = g.bcast(t, last_valid); clen = g.bcast(len, last_valid);
        }
        g.sync();      // scratch (us / wx / wy / jmp) is rewritten by the next chunk
        if (g.ballot(zero_div)) {
            // fp64: mirror the reference's ZeroDivisionError (rrt_dubins.py:270, :281).  fp32: with 24-bit
            // uniforms diff == 0 / velocity == 0 have probability 2^-24 per draw (2^-53 in the
            // reference), an artefact of the build, so the sample is rejected instead of aborting.
            if (VERIFY) out.status = 2; else degenerate = true;
            break;
        }
        if (ONE_CHUNK) break;
    }
    if (!ONE_CHUNK && DO_COLLIDE && n_exp == 0 && env.K > 0 && !parent_clear && parent_many) {
        // the path is [parent] alone: test it against the circles
        bool h = false;
#pragma unroll 1
        for (int k = g.gl; k < env.K; k += G) {
            R q = A::sq2(A::sub(px, env.cx[k]), A::sub(py, env.cy[k]));
            if (VERIFY) h = h || (A::sqrt(q) <= env.creff[k]);
            else h = h || (q <= env.creff2[k]);
        }
        if (g.ballot(h)) hit = true;
    }
    if (!rng.consumed_ok(ctr)) out.status = 4;
    out.x = cx; out.y = cy; out.th = cth; out.t = ct; out.len = clen;
    out.nwp = nwp; out.ctr = ctr;
    out.safe = !(hit || outside || degenerate);
    out.s2 = acc_s2; out.cnt = acc_cnt; out.mask = acc_mask;
    out.self_s2 = self_s2; out.self_hab = self_hab; out.leaf_moved = moved;
}

}  // namespace auv
