// gym.cu -- gym_rrt Planner_RRT (/root/reference/gym_rrt/envs/rrt_dubins.py:30-503), the goal-directed
// tree the RL environment grows one node per step (gym_rrt/envs/rrt_env.py:182-247).  SURVEY.md 8(f) N1.
//
// Q independent episodes live in HBM, one THREAD per episode: the per-step work of one episode is a
// serial chain (pick cell -> pick node -> steer <= freq arcs -> test -> goal arc), and a trainer
// steps thousands of environments at once, so episodes are the parallel axis.  A node is one 64-byte row,
// the rows of an episode are contiguous (lanes are at different slots of their own trees, so a [slot][Q]
// layout would touch one 32-byte sector per 4-byte field); occupied sub-cells are found through a small
// open-addressing table per episode; the goal-arc test is done by the whole warp, arc by arc.
//
//   k_gym_reset   Planner_RRT.__init__ (:34-74): node 0, its sub-cell, occupied list, counts
//   k_gym_reset_masked  the same for the episodes a mask selects, clearing only the cells their last tree held
//   k_gym_run     n_steps x generate_one_node (:198-238), cell from random.choice (planning,
//                 :157-196) or from the agent's action (RRTEnv.step)
//   k_gym_path    generate_final_course (:318-328): waypoints are not stored; each node keeps the
//                 sample-sequence position of its steer, which is replayed here
//
// The reference's check_collision_free (:430-449) never resets dList between obstacles, so obstacle k
// is tested against the minimum distance to obstacles 0..k; that is the same as testing every point
// against the inflated radius r_eff[j] = max_{k >= j} size[k], which is what the kernels do (exact).
#include <math.h>
#include <new>
#include <vector>
#include "launch.h"

struct auvrrt_gym {
    int device, precision;
    int64_t Q;
    auvrrt_gym_params_t p;
    int K, rows, cols, ncells;
    void *d_all;
    size_t bytes;
    void *d_circ;                  // [K][3] R: x, y, r_eff
    unsigned char *S;              // GymS<R> carved from d_all (host copy of the pointer struct)
    int32_t *d_actions;
    auvrrt_gym_record_t *d_recs;
    cudaStream_t stream;
    bool reset_once;               // a full reset has been enqueued: every episode's state is defined
};

namespace auv {

template <typename R> struct GymP {
    R x0, y0, x1, y1, exp_rate, d2e, dmax, neg_dmax, freq, cell_side, delta_theta;
    int ns, rows, cols, K, cap, ncells, hsize, hshift;
    long long Q;
};

// One node = one 64-byte row (two 32-byte sectors), rows of an episode contiguous: appending a node writes
// whole sectors and steering from a node reads one, whichever slot each lane of the warp is at.
template <typename R> struct alignas(16) GymNode {
    R x, y, th, t;                       // mps_list[i]: x, y, theta, traj_time_stamp
    int parent, cell, prev, nwp;         // parent index; sub-cell (-1 none); previous node of the same sub-cell; kept primitives
    unsigned npos;                       // sample-sequence position of its steer (replayed by k_gym_path)
    int pad[(64 - 4 * (int)sizeof(R) - 20) / 4];
};
struct GymOcc { int cell, count, tail, pad; };      // occupied_grid_cells_array[i] + len / last node of its node_array
struct GymHash { int key, val; };                   // open addressing: key = sub-cell id + 1 (0 = empty) -> occupied index

template <typename R> struct GymS {
    // per episode
    R *gx, *gy, *arc;                       // goal; arc [6][Q] = x_C, y_C, radius, ang_vel, theta_0, length
    uint64_t *key;
    int *n_nodes, *n_occ, *steps, *done, *status, *goal_checked, *arc_ne, *npath;
    unsigned *spos;
    GymNode<R> *nodes;                      // [Q][cap]
    GymOcc *occ;                            // [Q][cap]
    GymHash *hash;                          // [Q][hsize]
    uint16_t *counts;                       // [Q][ncells] or nullptr
};

template <typename R> struct GymC;
template <> struct GymC<double> {
    static __device__ __forceinline__ double pi() { return 3.141592653589793; }
    static __device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
    static __device__ __forceinline__ double sin(double a) { return ::sin(a); }
};
template <> struct GymC<float> {
    static __device__ __forceinline__ float pi() { return 3.14159274f; }
    static __device__ __forceinline__ float atan2(float y, float x) { return ::atan2f(y, x); }
    static __device__ __forceinline__ float sin(float a) { float s, c; Ar<float, false>::sincos(a, &s, &c); return s; }
};

// Planner_RRT.angle_wrap (:420-428): the recursion adds -2pi / +2pi until the angle is in [-pi, pi]
template <typename R> __device__ __forceinline__ R gym_wrap(R a) {
    typedef typename Policy<R>::A A;
    const R PI = GymC<R>::pi();
    for (int guard = 0; guard < 64 && !(-PI <= a && a <= PI); guard++) {
        if (a > PI) a = A::add(a, -(R)2 * PI);
        else if (a < -PI) a = A::add(a, (R)2 * PI);
        else break;
    }
    return a;
}

// math.hypot as CPython 3.12 evaluates it (Modules/mathmodule.c vector_norm, n = 2): power-of-two
// scaling, double-length sum of squares, one differential correction.  fp64 build only.
__device__ __forceinline__ double py_hypot(double a, double b) {
    double v0 = fabs(a), v1 = fabs(b);
    const double mx = fmax(v0, v1);
    if (mx == 0.0 || !(mx < __longlong_as_double(0x7ff0000000000000LL))) return mx;
    int e;
    frexp(mx, &e);
    const double scale = ldexp(1.0, -e);
    double csum = 1.0, frac1 = 0.0, frac2 = 0.0;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const double x = __dmul_rn(i ? v1 : v0, scale);
        const double hi = __dmul_rn(x, x), lo = fma(x, x, -hi);
        const double s = __dadd_rn(csum, hi), er = __dadd_rn(__dsub_rn(csum, s), hi);
        csum = s; frac1 = __dadd_rn(frac1, lo); frac2 = __dadd_rn(frac2, er);
    }
    double h = __dsqrt_rn(__dadd_rn(__dsub_rn(csum, 1.0), __dadd_rn(frac1, frac2)));
    const double hi = __dmul_rn(-h, h), lo = fma(-h, h, -hi);
    const double s = __dadd_rn(csum, hi), er = __dadd_rn(__dsub_rn(csum, s), hi);
    csum = s; frac1 = __dadd_rn(frac1, lo); frac2 = __dadd_rn(frac2, er);
    const double x = __dadd_rn(__dsub_rn(csum, 1.0), __dadd_rn(frac1, frac2));
    h = __dadd_rn(h, __ddiv_rn(x, __dmul_rn(2.0, h)));
    return __ddiv_rn(h, scale);
}
template <typename R> __device__ __forceinline__ R gym_hypot(R a, R b);
template <> __device__ __forceinline__ double gym_hypot<double>(double a, double b) { return py_hypot(a, b); }
template <> __device__ __forceinline__ float gym_hypot<float>(float a, float b) { return sqrtf(fmaf(b, b, a * a)); }

// add_node_to_grid (:108-154): flat sub-cell id, -1 past the last row / column (early return),
// -2 IndexError.  Negative rows / columns index from the end like a Python list.
template <typename R> __device__ __forceinline__ int gym_subcell(const GymP<R> &P, R x, R y, R th) {
    typedef typename Policy<R>::A A;
    long long row = (long long)A::div(y, P.cell_side), col = (long long)A::div(x, P.cell_side);   // int(): truncation
    if (row >= P.rows) return -1;
    if (col >= P.cols) return -1;
    if (row < 0) { row += P.rows; if (row < 0) return -2; }
    if (col < 0) { col += P.cols; if (col < 0) return -2; }
    long long sub = (long long)A::floor(A::div(th, P.delta_theta));
    if (sub < 0) sub = P.ns + sub;
    if (sub == P.ns) sub -= 1;
    if (sub < 0) { sub += P.ns; if (sub < 0) return -2; }
    if (sub >= P.ns) return -2;
    return (int)((row * P.cols + col) * P.ns + sub);
}

// one point of check_collision_free: inflated circles, then check_within_boundary (:458-471)
template <typename R> __device__ __forceinline__ bool gym_point_free(const GymP<R> &P, const R *circ, R px, R py) {
    typedef typename Policy<R>::A A;
    bool hit = false;
    for (int k = 0; k < P.K; k++) {
        const R dx = A::sub(px, circ[3 * k]), dy = A::sub(py, circ[3 * k + 1]);
        if (Policy<R>::VERIFY) hit |= A::sqrt(A::sq2(dx, dy)) <= circ[3 * k + 2];
        else hit |= A::sq2(dx, dy) <= circ[3 * k + 2];          // fast build: circ[..+2] holds r_eff^2
    }
    const bool inside = (px >= P.x0) && (px <= P.x1) && (py >= P.y0) && (py <= P.y1);
    return !hit && inside;
}

// steer (:241-283) from (x, y, th, t) on sequence positions pos, pos+1, ...; returns the number of kept
// primitives, updates the state; `free` = every waypoint passed gym_point_free (evaluated until the
// first failure unless `full`).  out != nullptr: write waypoint k (0-based) to out[3 * (base - k)]
// (reverse order, for generate_final_course).
template <typename R>
__device__ __forceinline__ int gym_steer(const GymP<R> &P, const R *circ, const Stream<R> &st, unsigned pos, R &x, R &y,
                                         R &th, R &t, bool &free, bool full, int &status, unsigned &used, double *out,
                                         long long base) {
    typedef typename Policy<R>::A A;
    const int n_expand = (int)A::floor(uniform_ab<R>((R)0, P.freq, st.u(pos)));
    used = 1u + 2u * (unsigned)n_expand;
    R s0, c0;
    A::sincos(th, &s0, &c0);
    int m = 0;
    for (int i = 0; i < n_expand; i++) {
        if (!free && !full) break;
        const R dist = uniform_ab<R>((R)0, P.d2e, st.u(pos + 1 + 2 * i));
        const R diff = uniform_ab<R>(P.neg_dmax, P.dmax, st.u(pos + 2 + 2 * i));
        if (!(A::fabs(dist) > A::fabs(diff))) continue;                                  // :258
        R radius, phi;
        if (Policy<R>::VERIFY) {
            const R s1 = A::add(dist, diff), s2 = A::sub(dist, diff), den = A::add(-s1, s2), sum = A::add(s1, s2);
            if (den == (R)0) { status = AUVRRT_ST_ZERO_DIV; break; }
            radius = A::div(sum, den);
            if (A::mul((R)2, radius) == (R)0) { status = AUVRRT_ST_ZERO_DIV; break; }
            phi = A::div(sum, A::mul((R)2, radius));
        } else {
            if (diff == (R)0) continue;          // fast build: a degenerate draw is dropped
            radius = -A::div(dist, diff);
            phi = -diff;
        }
        th = gym_wrap<R>(A::add(th, phi));                                              // :265
        R s1n, c1n;
        A::sincos(th, &s1n, &c1n);
        const R dx = A::mul(radius, A::sub(s1n, s0)), dy = A::mul(radius, A::add(-c1n, c0));
        s0 = s1n; c0 = c1n;
        x = A::add(x, dx); y = A::add(y, dy);
        t = A::add(t, A::sqrt(A::sq2(dx, dy)));                                         // velocity = 1
        if (out) { double *o = out + 3 * (base - m); o[0] = (double)x; o[1] = (double)y; o[2] = (double)th; }
        m++;
        if (free) free = gym_point_free<R>(P, circ, x, y);
    }
    return m;
}

// connect_to_goal_curve_alt (:375-418): 1 = arc built, 0 = `return None`, else 100 + status
template <typename R>
__device__ __forceinline__ int gym_goal_arc(const GymP<R> &P, R gx, R gy, R x, R y, R th, R arc[6], int &ne) {
    typedef typename Policy<R>::A A;
    const R PI = GymC<R>::pi();
    const R gdx = A::sub(gx, x), gdy = A::sub(gy, y);
    const R theta = GymC<R>::atan2(gdy, gdx);
    const R diff = gym_wrap<R>(A::sub(theta, th));
    if (A::fabs(diff) > A::div(PI, (R)2)) return 0;
    const R r_G = gym_hypot<R>(gdx, gdy);
    const R a = A::sub(theta, th);
    if (a == (R)0) return 0;
    R phi = A::mul((R)2, gym_wrap<R>(a));
    const R sn = GymC<R>::sin(a);
    if (sn == (R)0) return 0;
    const R radius = A::div(r_G, A::mul((R)2, sn));
    R length = A::mul(radius, phi);
    if (phi > PI) { phi = A::sub(phi, A::mul((R)2, PI)); length = A::mul(-radius, phi); }
    else if (phi < -PI) { phi = A::add(phi, A::mul((R)2, PI)); length = A::mul(-radius, phi); }
    const R le = A::div(length, P.exp_rate);
    if (le == (R)0) return 100 + AUVRRT_ST_ZERO_DIV;
    R s, c;
    A::sincos(th, &s, &c);
    arc[0] = A::sub(x, A::mul(radius, s));
    arc[1] = A::add(y, A::mul(radius, c));
    arc[2] = radius; arc[3] = A::div(phi, le); arc[4] = th; arc[5] = length;
    ne = (int)A::floor(le);
    return 1;
}
template <typename R> __device__ __forceinline__ void gym_arc_point(const R arc[6], int i, R &px, R &py, R &pa) {
    typedef typename Policy<R>::A A;
    pa = A::add(A::mul(arc[3], (R)i), arc[4]);
    R s, c;
    A::sincos(pa, &s, &c);
    px = A::add(arc[0], A::mul(arc[2], s));
    py = A::sub(arc[1], A::mul(arc[2], c));
}

#define ND(i) S.nodes[(size_t)q * (size_t)P.cap + (size_t)(i)]
#define OC(i) S.occ[(size_t)q * (size_t)P.cap + (size_t)(i)]
#define HT(h) S.hash[(size_t)q * (size_t)P.hsize + (size_t)(h)]

// Planner_RRT.__init__ for episode q on a clean hash table and counts row (the writes k_gym_reset and
// k_gym_reset_masked share)
template <typename R>
__device__ __forceinline__ void gym_init_episode(const GymP<R> &P, const GymS<R> &S, long long q, const double *starts,
                                                 const double *goals, const uint64_t *seeds) {
    const R x = (R)starts[3 * q], y = (R)starts[3 * q + 1], th = (R)starts[3 * q + 2];
    S.gx[q] = (R)goals[2 * q]; S.gy[q] = (R)goals[2 * q + 1];
    S.key[q] = stream_key(seeds[q]);
    ND(0).x = x; ND(0).y = y; ND(0).th = th; ND(0).t = (R)0;
    ND(0).parent = -1; ND(0).prev = -1; ND(0).nwp = 0; ND(0).npos = 0u;
    const int c = gym_subcell<R>(P, x, y, th);                                          // :57
    ND(0).cell = c;
    int n_occ = 0;
    if (c >= 0) {
        OC(0).cell = c; OC(0).count = 1; OC(0).tail = 0; n_occ = 1;
        const unsigned h = ((unsigned)c * 2654435761u) >> P.hshift;
        HT(h).key = c + 1; HT(h).val = 0;
        if (S.counts) S.counts[(size_t)q * P.ncells + c] = 1;
    }
    S.n_nodes[q] = 1; S.n_occ[q] = n_occ; S.steps[q] = 0; S.done[q] = 0; S.goal_checked[q] = -1; S.arc_ne[q] = -1; S.npath[q] = 0;
    S.spos[q] = 0u;
    S.status[q] = c == -2 ? AUVRRT_ST_KEY_ERROR : AUVRRT_ST_OK;
}

template <typename R>
__global__ void __launch_bounds__(128) k_gym_reset(GymP<R> P, GymS<R> S, const double *starts, const double *goals,
                                                   const uint64_t *seeds) {
    const long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (q >= P.Q) return;
    gym_init_episode<R>(P, S, q, starts, goals, seeds);
}

// occupied-cell lookup: open-addressing table per episode (key = sub-cell id + 1, 0 = empty; value = index into the
// occupied list).  Replaces a linear scan of occupied_grid_cells_array, which streamed ~n_occ/2 rows per step.
template <typename R>
__device__ __forceinline__ int gym_occ_find(const GymP<R> &P, const GymS<R> &S, long long q, int c, unsigned &slot) {
    unsigned h = ((unsigned)c * 2654435761u) >> P.hshift;
    for (;;) {
        const int k = HT(h).key;
        if (k == 0) { slot = h; return -1; }
        if (k == c + 1) { slot = h; return HT(h).val; }
        h = (h + 1) & (unsigned)(P.hsize - 1);
    }
}

// Planner_RRT.__init__ for the episodes with mask[q] != 0, in place: a vectorised environment resets each episode
// when it ends instead of waiting for all Q.  Everything the previous episode wrote outside its own rows is undone
// at the cells it occupied, so the cost is O(n_occ) and not O(ncells + hsize):
//  - counts: only the sub-cells in the occupied list are non-zero (k_gym_run counts a node only in a cell it has
//    put in that list), so those entries are zeroed;
//  - hash: linear probing that never deletes means a key's probe path crosses only slots filled before it, and the
//    occupied list is in insertion order, so clearing keys from the LAST occupied cell to the first, each found by
//    the ordinary probe, always finds it with every earlier key still in place.  This keeps k_gym_run as it is
//    (recording each key's slot at insertion would cost it a store per new cell).
// Node and occupied-list rows are not cleared: n_nodes / n_occ bound every read of them.  An episode's state must
// have been written by an earlier full reset (the host side refuses a masked call before one).
template <typename R>
__global__ void __launch_bounds__(128) k_gym_reset_masked(GymP<R> P, GymS<R> S, const uint8_t *mask, const double *starts,
                                                          const double *goals, const uint64_t *seeds) {
    const long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (q >= P.Q || !mask[q]) return;
    for (int i = S.n_occ[q] - 1; i >= 0; i--) {
        const int c = OC(i).cell;
        unsigned slot;
        gym_occ_find<R>(P, S, q, c, slot);
        HT(slot).key = 0;
        if (S.counts) S.counts[(size_t)q * P.ncells + c] = 0;
    }
    gym_init_episode<R>(P, S, q, starts, goals, seeds);
}

#ifndef AUV_GYM_MINB
#define AUV_GYM_MINB 8
#endif
template <typename R>
__global__ void __launch_bounds__(128, sizeof(R) == 4 ? AUV_GYM_MINB : 4) k_gym_run(GymP<R> P, GymS<R> S, const R *circ_g, const int32_t *actions, int n_steps,
                                                 int full, auvrrt_gym_record_t *recs) {
    typedef typename Policy<R>::A A;
    extern __shared__ __align__(16) unsigned char gym_smem[];
    R *circ = reinterpret_cast<R *>(gym_smem);
    for (int i = threadIdx.x; i < 3 * P.K; i += blockDim.x) circ[i] = circ_g[i];
    __syncthreads();
    const long long q_raw = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool mine = q_raw < P.Q;
    const long long q = mine ? q_raw : P.Q - 1;          // out-of-range lanes stay in the warp for the collectives
    const int lane = threadIdx.x & 31;
    Stream<R> st;
    st.key = S.key[q]; st.ext = nullptr; st.n_ext = 0;
    int n = S.n_nodes[q], n_occ = S.n_occ[q], steps = S.steps[q], done = S.done[q], status = S.status[q];
    int goal_checked = S.goal_checked[q];
    unsigned pos = S.spos[q];
    const R gx = S.gx[q], gy = S.gy[q];
    int last_parent = -1, last_acc = 0, last_nwp = 0, last_used = 0, n_path = done ? S.npath[q] : 0;
    R cx = 0, cy = 0, cth = 0, ct = 0, arc_len = done ? S.arc[(size_t)5 * P.Q + q] : (R)0;
    for (int it = 0; it < n_steps; it++) {
        bool live = mine && !done && status == AUVRRT_ST_OK;
        if (!__any_sync(0xffffffffu, live)) break;
        bool want_arc = false;
        R arc[6] = {0, 0, 0, 0, 0, 0}; int ne = -1;
        if (live) {
            int oi = -1, cellid = 0;
            unsigned hslot;
            last_parent = -1; last_acc = 0; last_nwp = 0; last_used = 0;
            if (!actions) {
                if (n_occ == 0) { status = AUVRRT_ST_KEY_ERROR; live = false; }              // random.choice([])
                else {
                    oi = (int)A::mul(unit(st.u(pos++)), (R)n_occ);                                // :176
                    if (!Policy<R>::VERIFY) oi = min(oi, n_occ - 1);
                    cellid = OC(oi).cell;
                }
            } else {
                cellid = actions[q];
                oi = cellid >= 0 ? gym_occ_find<R>(P, S, q, cellid, hslot) : -1;
                if (oi < 0) live = false;                                                   // node_array == [] (:209-215)
            }
            if (live) {
                const unsigned pos0 = pos;
                const int cnt = OC(oi).count;
                int k = (int)A::mul(unit(st.u(pos++)), (R)cnt);                                   // :217
                if (!Policy<R>::VERIFY) k = min(k, cnt - 1);
                int pn = OC(oi).tail;
                for (int h = cnt - 1 - k; h > 0; h--) pn = ND(pn).prev;
                R x = ND(pn).x, y = ND(pn).y, th = ND(pn).th, t = ND(pn).t;
                bool free = gym_point_free<R>(P, circ, x, y);                               // path[0] = the node steered from
                unsigned used = 0;
                const unsigned steer_pos = pos;
                const int m = gym_steer<R>(P, circ, st, pos, x, y, th, t, free, full != 0, status, used, nullptr, 0);
                pos += used;
                if (status != AUVRRT_ST_OK) live = false;
                else {
                    last_parent = pn; last_nwp = m; last_used = (int)(pos - pos0);
                    cx = x; cy = y; cth = th; ct = t;
                    if (free) {                                                             // :222-227
                        const int c = gym_subcell<R>(P, x, y, th);
                        if (n >= P.cap) { status = AUVRRT_ST_OVERFLOW; live = false; }
                        else if (c == -2) { status = AUVRRT_ST_KEY_ERROR; live = false; }
                        else {
                            ND(n).x = x; ND(n).y = y; ND(n).th = th; ND(n).t = t;
                            ND(n).parent = pn; ND(n).nwp = m; ND(n).npos = steer_pos;
                            ND(n).cell = c;
                            if (c >= 0) {
                                int oj = gym_occ_find<R>(P, S, q, c, hslot);
                                if (oj < 0) {                                               // :153-154
                                    oj = n_occ++;
                                    OC(oj).cell = c; OC(oj).count = 0; OC(oj).tail = -1;
                                    HT(hslot).key = c + 1; HT(hslot).val = oj;
                                }
                                ND(n).prev = OC(oj).tail;
                                OC(oj).tail = n;
                                OC(oj).count = OC(oj).count + 1;
                                if (S.counts) { uint16_t *cp = S.counts + (size_t)q * P.ncells + c; *cp = (uint16_t)(*cp + 1); }
                            } else {
                                ND(n).prev = -1;
                            }
                            n++; last_acc = 1;
                        }
                    }
                    if (live) {
                        steps++;
                        // connect_to_goal_curve_alt(self.mps_list[-1]) (:229) depends on the last node only
                        const int last = n - 1;
                        if (goal_checked != last) {
                            goal_checked = last;
                            const int g = gym_goal_arc<R>(P, gx, gy, ND(last).x, ND(last).y, ND(last).th, arc, ne);
                            if (g >= 100) status = g - 100;
                            else if (g == 1) {
                                if (ne < 0 && P.K > 0) status = AUVRRT_ST_KEY_ERROR;          // min([]) ValueError
                                else want_arc = true;
                            }
                        }
                    }
                }
            }
        }
        // check_collision_free(final_node) (:232), warp-cooperative: the arcs of this warp's episodes are tested one
        // after the other with the 32 lanes taking 32 consecutive arc points each round (a point is a pure function
        // of its index), stopping at the first round that holds a colliding point.
        unsigned pending = __ballot_sync(0xffffffffu, want_arc);
        bool arc_ok = false;
        while (pending) {
            const int src = __ffs(pending) - 1;
            pending &= pending - 1;
            R a6[6];
#pragma unroll
            for (int j = 0; j < 6; j++) a6[j] = __shfl_sync(0xffffffffu, arc[j], src);
            const int ne_s = __shfl_sync(0xffffffffu, ne, src);
            bool ok = true;
            for (int base = 0; base <= ne_s; base += 32) {
                const int i = base + lane;
                bool okp = true;
                if (i <= ne_s) {
                    R px, py, pa;
                    gym_arc_point<R>(a6, i, px, py, pa);
                    okp = gym_point_free<R>(P, circ, px, py);
                }
                if (!__all_sync(0xffffffffu, okp)) { ok = false; break; }
            }
            if (lane == src) arc_ok = ok;
        }
        if (want_arc && arc_ok) {
            const int last = n - 1;
            done = 1; arc_len = arc[5];
#pragma unroll
            for (int j = 0; j < 6; j++) S.arc[(size_t)j * P.Q + q] = arc[j];
            S.arc_ne[q] = ne;
            n_path = 1 + (ne + 1);
            for (int j = last; ND(j).parent >= 0; j = ND(j).parent) n_path += ND(j).nwp + 1;
            S.npath[q] = n_path;
        }
    }
    if (!mine) return;
    S.n_nodes[q] = n; S.n_occ[q] = n_occ; S.steps[q] = steps; S.done[q] = done; S.status[q] = status;
    S.goal_checked[q] = goal_checked; S.spos[q] = pos;
    if (recs) {
        auvrrt_gym_record_t r;
        r.status = status; r.done = done; r.steps = steps; r.n_nodes = n; r.n_occupied = n_occ;
        r.last_parent = last_parent; r.last_accepted = last_acc; r.last_nwp = last_nwp; r.last_uniforms = last_used;
        r.n_path = n_path; r.n_uniforms = (int64_t)pos;
        r.cand[0] = (double)cx; r.cand[1] = (double)cy; r.cand[2] = (double)cth; r.cand[3] = (double)ct;
        r.arc_length = (double)arc_len;
        recs[q] = r;
    }
}

// generate_final_course (:318-328) for one done episode: [final] + reversed(arc points) + for every node
// up the parent chain reversed(its waypoints) + its parent.  One thread; rarely called.
template <typename R>
__global__ void k_gym_path(GymP<R> P, GymS<R> S, const R *circ, long long q, int cap, double *path, int *n_out) {
    if (threadIdx.x || blockIdx.x) return;
    if (!S.done[q]) { *n_out = 0; return; }
    R arc[6];
    for (int j = 0; j < 6; j++) arc[j] = S.arc[(size_t)j * P.Q + q];
    const int ne = S.arc_ne[q];
    const int last = S.n_nodes[q] - 1;
    long long total = 1 + (ne + 1);
    for (int j = last; ND(j).parent >= 0; j = ND(j).parent) total += ND(j).nwp + 1;
    *n_out = (int)total;
    if (total > cap) return;
    long long w = 0;
    R px, py, pa;
    if (ne >= 0) gym_arc_point<R>(arc, ne, px, py, pa); else { px = ND(last).x; py = ND(last).y; pa = ND(last).th; }
    path[0] = (double)px; path[1] = (double)py; path[2] = (double)pa; w = 1;
    for (int i = ne; i >= 0; i--) {
        gym_arc_point<R>(arc, i, px, py, pa);
        path[3 * w] = (double)px; path[3 * w + 1] = (double)py; path[3 * w + 2] = (double)pa; w++;
    }
    Stream<R> st;
    st.key = S.key[q]; st.ext = nullptr; st.n_ext = 0;
    for (int j = last; ND(j).parent >= 0; j = ND(j).parent) {
        const int pj = ND(j).parent, m = ND(j).nwp;
        R x = ND(pj).x, y = ND(pj).y, th = ND(pj).th, t = ND(pj).t;
        bool free = true; int status = 0; unsigned used = 0;
        gym_steer<R>(P, circ, st, ND(j).npos, x, y, th, t, free, true, status, used, path, w + m - 1);   // waypoint k -> row w + m-1-k
        w += m;
        path[3 * w] = (double)ND(pj).x; path[3 * w + 1] = (double)ND(pj).y; path[3 * w + 2] = (double)ND(pj).th; w++;
    }
}

static int gym_hash_size(int cap) {
    int h = 16;
    while (h < 2 * cap) h <<= 1;
    return h;
}

template <typename R> static GymP<R> make_gymp(const auvrrt_gym *g) {
    GymP<R> P;
    const auvrrt_gym_params_t &p = g->p;
    P.x0 = (R)p.x0; P.y0 = (R)p.y0; P.x1 = (R)p.x1; P.y1 = (R)p.y1; P.exp_rate = (R)p.exp_rate;
    P.d2e = (R)p.dist_to_end; P.dmax = (R)p.diff_max; P.neg_dmax = (R)(-p.diff_max); P.freq = (R)p.freq;
    P.cell_side = (R)p.cell_side;
    P.delta_theta = (R)((2.0 * M_PI) / (double)p.subsections);                          // grid_cell_rrt.py:52
    P.ns = p.subsections; P.rows = g->rows; P.cols = g->cols; P.K = g->K; P.cap = p.node_cap; P.ncells = g->ncells;
    P.Q = g->Q;
    P.hsize = gym_hash_size(p.node_cap);
    P.hshift = 32;
    for (int h = P.hsize; h > 1; h >>= 1) P.hshift--;
    return P;
}

template <typename R> static size_t gym_carve(GymS<R> *S, unsigned char *base, int64_t Q, int cap, int ncells, bool counts) {
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char *p = base ? base + off : nullptr; off += (bytes + 255) & ~(size_t)255; return p; };
    const size_t q = (size_t)Q, nq = (size_t)cap * q;
    S->gx = (R *)take(sizeof(R) * q); S->gy = (R *)take(sizeof(R) * q); S->arc = (R *)take(sizeof(R) * 6 * q);
    S->key = (uint64_t *)take(8 * q);
    S->n_nodes = (int *)take(4 * q); S->n_occ = (int *)take(4 * q); S->steps = (int *)take(4 * q); S->done = (int *)take(4 * q);
    S->status = (int *)take(4 * q); S->goal_checked = (int *)take(4 * q); S->arc_ne = (int *)take(4 * q); S->npath = (int *)take(4 * q);
    S->spos = (unsigned *)take(4 * q);
    S->nodes = (GymNode<R> *)take(sizeof(GymNode<R>) * nq);
    S->occ = (GymOcc *)take(sizeof(GymOcc) * nq);
    S->hash = (GymHash *)take(sizeof(GymHash) * (size_t)gym_hash_size(cap) * q);
    S->counts = counts ? (uint16_t *)take(2 * q * (size_t)ncells) : nullptr;
    return off;
}

template <typename R> static int gym_create_t(auvrrt_gym *g, const double *circles) {
    GymS<R> S;
    g->bytes = gym_carve<R>(&S, nullptr, g->Q, g->p.node_cap, g->ncells, g->p.track_counts != 0);
    AUV_CUDA(cudaMalloc(&g->d_all, g->bytes));
    gym_carve<R>(&S, (unsigned char *)g->d_all, g->Q, g->p.node_cap, g->ncells, g->p.track_counts != 0);
    g->S = (unsigned char *)new GymS<R>(S);
    std::vector<R> c((size_t)3 * (g->K > 0 ? g->K : 1));
    double reff = -INFINITY;
    for (int k = g->K - 1; k >= 0; k--) {
        reff = circles[3 * k + 2] > reff ? circles[3 * k + 2] : reff;
        c[3 * k] = (R)circles[3 * k]; c[3 * k + 1] = (R)circles[3 * k + 1];
        const R r = (R)reff;
        c[3 * k + 2] = Policy<R>::VERIFY ? r : (r < (R)0 ? (R)-1 : r * r);              // fast build compares squares
    }
    AUV_CUDA(cudaMalloc(&g->d_circ, sizeof(R) * c.size()));
    AUV_CUDA(cudaMemcpy(g->d_circ, c.data(), sizeof(R) * c.size(), cudaMemcpyHostToDevice));
    return AUVRRT_OK;
}

template <typename R>
static int gym_reset_t(auvrrt_gym *g, const double *d_starts, const double *d_goals, const uint64_t *d_seeds, cudaStream_t s) {
    const GymS<R> &S = *(const GymS<R> *)g->S;
    if (S.counts) AUV_CUDA(cudaMemsetAsync(S.counts, 0, 2 * (size_t)g->Q * g->ncells, s));
    AUV_CUDA(cudaMemsetAsync(S.hash, 0, sizeof(GymHash) * (size_t)gym_hash_size(g->p.node_cap) * (size_t)g->Q, s));
    k_gym_reset<R><<<(unsigned)((g->Q + 127) / 128), 128, 0, s>>>(make_gymp<R>(g), S, d_starts, d_goals, d_seeds);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

template <typename R>
static int gym_reset_masked_t(auvrrt_gym *g, const uint8_t *d_mask, const double *d_starts, const double *d_goals,
                              const uint64_t *d_seeds, cudaStream_t s) {
    const GymS<R> &S = *(const GymS<R> *)g->S;
    k_gym_reset_masked<R><<<(unsigned)((g->Q + 127) / 128), 128, 0, s>>>(make_gymp<R>(g), S, d_mask, d_starts, d_goals, d_seeds);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

template <typename R>
static int gym_run_t(auvrrt_gym *g, const int32_t *d_actions, int n_steps, int full, auvrrt_gym_record_t *d_recs, cudaStream_t s) {
    const GymS<R> &S = *(const GymS<R> *)g->S;
    k_gym_run<R><<<(unsigned)((g->Q + 127) / 128), 128, sizeof(R) * 3 * (size_t)(g->K > 0 ? g->K : 1), s>>>(
        make_gymp<R>(g), S, (const R *)g->d_circ, d_actions, n_steps, full, d_recs);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

template <typename R>
static int gym_path_t(const auvrrt_gym *g, int64_t q, int cap, double *d_path, int *d_n, cudaStream_t s) {
    const GymS<R> &S = *(const GymS<R> *)g->S;
    k_gym_path<R><<<1, 32, 0, s>>>(make_gymp<R>(g), S, (const R *)g->d_circ, (long long)q, cap, d_path, d_n);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

template <typename R>
static int gym_tree_t(const auvrrt_gym *g, int64_t q, int32_t cap, double *nodes, int32_t *parents, int32_t *cells,
                      int32_t *occupied, int32_t *n_nodes, int32_t *n_occupied) {
    const GymS<R> &S = *(const GymS<R> *)g->S;
    int n = 0, no = 0;
    AUV_CUDA(cudaMemcpy(&n, S.n_nodes + q, 4, cudaMemcpyDeviceToHost));
    AUV_CUDA(cudaMemcpy(&no, S.n_occ + q, 4, cudaMemcpyDeviceToHost));
    if (n_nodes) *n_nodes = n;
    if (n_occupied) *n_occupied = no;
    if (n > cap) return set_err(AUVRRT_ERR_ARG, "gym_tree: cap %d < n_nodes %d", cap, n);
    if (nodes || parents || cells) {
        std::vector<GymNode<R>> rows((size_t)(n > 0 ? n : 1));
        AUV_CUDA(cudaMemcpy(rows.data(), S.nodes + (size_t)q * g->p.node_cap, sizeof(GymNode<R>) * (size_t)n, cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; i++) {
            if (nodes) { nodes[4 * i] = (double)rows[i].x; nodes[4 * i + 1] = (double)rows[i].y; nodes[4 * i + 2] = (double)rows[i].th; nodes[4 * i + 3] = (double)rows[i].t; }
            if (parents) parents[i] = rows[i].parent;
            if (cells) cells[i] = rows[i].cell;
        }
    }
    if (occupied) {
        std::vector<GymOcc> rows((size_t)(no > 0 ? no : 1));
        AUV_CUDA(cudaMemcpy(rows.data(), S.occ + (size_t)q * g->p.node_cap, sizeof(GymOcc) * (size_t)no, cudaMemcpyDeviceToHost));
        for (int i = 0; i < no; i++) occupied[i] = rows[i].cell;
    }
    return AUVRRT_OK;
}

}  // namespace auv

using namespace auv;

extern "C" int auvrrt_gym_create(const double *circles, int K, const auvrrt_gym_params_t *params, int64_t Q, int precision,
                                 int device, auvrrt_gym_t **out) {
    if (!params || !out || Q <= 0 || K < 0 || (K > 0 && !circles)) return set_err(AUVRRT_ERR_ARG, "gym_create: bad arguments");
    if (precision != AUVRRT_F32 && precision != AUVRRT_F64) return set_err(AUVRRT_ERR_ARG, "gym_create: bad precision");
    if (params->subsections <= 0 || params->node_cap < 2 || !(params->cell_side > 0) || !(params->exp_rate > 0))
        return set_err(AUVRRT_ERR_ARG, "gym_create: subsections, node_cap >= 2, cell_side and exp_rate must be positive");
    if (K > 2048) return set_err(AUVRRT_ERR_UNSUPPORTED, "gym_create: at most 2048 obstacles");
    AUV_TRY(need_device(device));
    auvrrt_gym *g = new (std::nothrow) auvrrt_gym();
    if (!g) return set_err(AUVRRT_ERR_ARG, "gym_create: out of memory");
    g->device = device; g->precision = precision; g->Q = Q; g->p = *params; g->K = K;
    g->d_all = nullptr; g->d_circ = nullptr; g->S = nullptr; g->d_actions = nullptr; g->d_recs = nullptr; g->stream = nullptr;
    g->reset_once = false;
    // discretize_env (:77-93): int(env_height) // int(cell_side_length)
    const long long cs = (long long)params->cell_side, hh = (long long)(params->y1 - params->y0), ww = (long long)(params->x1 - params->x0);
    if (cs <= 0 || hh < cs || ww < cs) { delete g; return set_err(AUVRRT_ERR_ARG, "gym_create: int(cell_side) must be >= 1 and the boundary at least one cell wide (ZeroDivisionError / IndexError in the reference)"); }
    g->rows = (int)(hh / cs); g->cols = (int)(ww / cs);
    g->ncells = g->rows * g->cols * params->subsections;
    if (params->track_counts && (size_t)2 * Q * g->ncells > ((size_t)64 << 30)) { delete g; return set_err(AUVRRT_ERR_ARG, "gym_create: dense counts would need more than 64 GiB"); }
    int rc = AUV_DISPATCH(g->precision, gym_create_t, g, circles);
    if (rc == AUVRRT_OK) {
        cudaError_t e = cudaMalloc((void **)&g->d_actions, 4 * (size_t)Q);
        if (e == cudaSuccess) e = cudaMalloc((void **)&g->d_recs, sizeof(auvrrt_gym_record_t) * (size_t)Q);
        if (e == cudaSuccess) e = cudaStreamCreate(&g->stream);
        if (e != cudaSuccess) rc = set_err(AUVRRT_ERR_CUDA, "gym_create: %s", cudaGetErrorString(e));
    }
    if (rc != AUVRRT_OK) { auvrrt_gym_destroy(g); return rc; }
    *out = g;
    return AUVRRT_OK;
}

extern "C" void auvrrt_gym_destroy(auvrrt_gym_t *g) {
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->stream) { cudaStreamSynchronize(g->stream); cudaStreamDestroy(g->stream); }
    cudaFree(g->d_all); cudaFree(g->d_circ); cudaFree(g->d_actions); cudaFree(g->d_recs);
    if (g->S) { if (g->precision == AUVRRT_F64) delete (GymS<double> *)g->S; else delete (GymS<float> *)g->S; }
    delete g;
}

extern "C" int auvrrt_gym_grid_shape(const auvrrt_gym_t *g, int *rows, int *cols) {
    if (!g) return set_err(AUVRRT_ERR_ARG, "gym_grid_shape: null handle");
    if (rows) *rows = g->rows;
    if (cols) *cols = g->cols;
    return AUVRRT_OK;
}

extern "C" int auvrrt_gym_reset(auvrrt_gym_t *g, const double *starts, const double *goals, const uint64_t *seeds) {
    if (!g || !starts || !goals || !seeds) return set_err(AUVRRT_ERR_ARG, "gym_reset: null argument");
    AUV_CUDA(cudaSetDevice(g->device));
    const size_t Q = (size_t)g->Q;
    DBuf d;
    AUV_TRY(d.alloc(8 * Q * 6));
    double *d_starts = d.as<double>(), *d_goals = d_starts + 3 * Q;
    uint64_t *d_seeds = (uint64_t *)(d_starts + 5 * Q);
    AUV_CUDA(cudaMemcpyAsync(d_starts, starts, 24 * Q, cudaMemcpyHostToDevice, g->stream));
    AUV_CUDA(cudaMemcpyAsync(d_goals, goals, 16 * Q, cudaMemcpyHostToDevice, g->stream));
    AUV_CUDA(cudaMemcpyAsync(d_seeds, seeds, 8 * Q, cudaMemcpyHostToDevice, g->stream));
    AUV_TRY(AUV_DISPATCH(g->precision, gym_reset_t, g, d_starts, d_goals, d_seeds, g->stream));
    AUV_CUDA(cudaStreamSynchronize(g->stream));
    g->reset_once = true;
    return AUVRRT_OK;
}

extern "C" int auvrrt_gym_reset_dev(auvrrt_gym_t *g, const uint8_t *d_mask, const double *d_starts, const double *d_goals,
                                    const uint64_t *d_seeds, void *stream) {
    if (!g || !d_starts || !d_goals || !d_seeds) return set_err(AUVRRT_ERR_ARG, "gym_reset_dev: null argument");
    if (d_mask && !g->reset_once)
        return set_err(AUVRRT_ERR_ARG, "gym_reset_dev: a masked reset reads each episode's previous tree, which is undefined "
                                       "until the handle has had one full reset (d_mask = NULL or auvrrt_gym_reset)");
    AUV_CUDA(cudaSetDevice(g->device));
    const int rc = d_mask ? AUV_DISPATCH(g->precision, gym_reset_masked_t, g, d_mask, d_starts, d_goals, d_seeds, (cudaStream_t)stream)
                          : AUV_DISPATCH(g->precision, gym_reset_t, g, d_starts, d_goals, d_seeds, (cudaStream_t)stream);
    if (rc == AUVRRT_OK && !d_mask) g->reset_once = true;
    return rc;
}

extern "C" int auvrrt_gym_step_dev(auvrrt_gym_t *g, const int32_t *d_actions, int n_steps, int full_candidates,
                                   auvrrt_gym_record_t *d_records, void *stream) {
    if (!g || n_steps < 0) return set_err(AUVRRT_ERR_ARG, "gym_step: bad arguments");
    if (d_actions && n_steps != 1) return set_err(AUVRRT_ERR_ARG, "gym_step: n_steps must be 1 when actions are given");
    AUV_CUDA(cudaSetDevice(g->device));
    return AUV_DISPATCH(g->precision, gym_run_t, g, d_actions, n_steps, full_candidates, d_records, (cudaStream_t)stream);
}

extern "C" int auvrrt_gym_step(auvrrt_gym_t *g, const int32_t *actions, int n_steps, int full_candidates,
                               auvrrt_gym_record_t *out_records) {
    if (!g) return set_err(AUVRRT_ERR_ARG, "gym_step: null handle");
    AUV_CUDA(cudaSetDevice(g->device));
    if (actions) AUV_CUDA(cudaMemcpyAsync(g->d_actions, actions, 4 * (size_t)g->Q, cudaMemcpyHostToDevice, g->stream));
    int rc = auvrrt_gym_step_dev(g, actions ? g->d_actions : nullptr, n_steps, full_candidates, out_records ? g->d_recs : nullptr, g->stream);
    if (rc != AUVRRT_OK) return rc;
    if (out_records)
        AUV_CUDA(cudaMemcpyAsync(out_records, g->d_recs, sizeof(auvrrt_gym_record_t) * (size_t)g->Q, cudaMemcpyDeviceToHost, g->stream));
    AUV_CUDA(cudaStreamSynchronize(g->stream));
    return AUVRRT_OK;
}

extern "C" int auvrrt_gym_tree(const auvrrt_gym_t *g, int64_t q, int32_t cap, double *nodes, int32_t *parents, int32_t *cells,
                               int32_t *occupied, int32_t *n_nodes, int32_t *n_occupied) {
    if (!g || q < 0 || q >= g->Q) return set_err(AUVRRT_ERR_ARG, "gym_tree: bad episode index");
    AUV_CUDA(cudaSetDevice(g->device));
    AUV_CUDA(cudaStreamSynchronize(g->stream));
    return AUV_DISPATCH(g->precision, gym_tree_t, g, q, cap, nodes, parents, cells, occupied, n_nodes, n_occupied);
}

extern "C" const uint16_t *auvrrt_gym_counts_dev(const auvrrt_gym_t *g) {
    if (!g) return nullptr;
    return g->precision == AUVRRT_F64 ? ((const GymS<double> *)g->S)->counts : ((const GymS<float> *)g->S)->counts;
}

extern "C" int auvrrt_gym_counts(const auvrrt_gym_t *g, int64_t q0, int64_t nq, uint16_t *out) {
    if (!g || !out || q0 < 0 || nq < 0 || q0 + nq > g->Q) return set_err(AUVRRT_ERR_ARG, "gym_counts: bad range");
    const uint16_t *c = auvrrt_gym_counts_dev(g);
    if (!c) return set_err(AUVRRT_ERR_ARG, "gym_counts: handle was created with track_counts = 0");
    AUV_CUDA(cudaSetDevice(g->device));
    AUV_CUDA(cudaStreamSynchronize(g->stream));
    AUV_CUDA(cudaMemcpy(out, c + (size_t)q0 * g->ncells, 2 * (size_t)nq * g->ncells, cudaMemcpyDeviceToHost));
    return AUVRRT_OK;
}

extern "C" int auvrrt_gym_path(const auvrrt_gym_t *g, int64_t q, int32_t cap, double *path, int32_t *n_path) {
    if (!g || q < 0 || q >= g->Q || cap < 0 || !n_path || (cap > 0 && !path)) return set_err(AUVRRT_ERR_ARG, "gym_path: bad arguments");
    AUV_CUDA(cudaSetDevice(g->device));
    DBuf d;
    AUV_TRY(d.alloc(24 * (size_t)(cap > 0 ? cap : 1) + 16));
    double *d_path = d.as<double>();
    int *d_n = (int *)(d_path + 3 * (size_t)(cap > 0 ? cap : 1));
    AUV_TRY(AUV_DISPATCH(g->precision, gym_path_t, g, q, cap, d_path, d_n, g->stream));
    AUV_CUDA(cudaStreamSynchronize(g->stream));
    int n = 0;
    AUV_CUDA(cudaMemcpy(&n, d_n, 4, cudaMemcpyDeviceToHost));
    if (n <= cap && n > 0) AUV_CUDA(cudaMemcpy(path, d_path, 24 * (size_t)n, cudaMemcpyDeviceToHost));
    *n_path = n;
    if (n > cap) return set_err(AUVRRT_ERR_ARG, "gym_path: cap %d < path length %d", cap, n);
    return AUVRRT_OK;
}
