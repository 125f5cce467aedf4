// plan.cu -- RRT.exploring (/root/reference/path_planning/rrt_dubins.py:92-176) for thousands of
// independent planning queries: one group of G lanes grows one tree.
//
// Persistent kernel: the grid is sized to the machine (148 SMs x resident CTAs), every lane group
// owns one tree workspace in HBM and pulls queries off an atomic counter, so memory is
// O(resident groups), not O(queries).  Per query the kernel keeps, in the group's workspace,
//   * the tree as SoA arrays (x, y, theta, t, length | parent, stream position of the edge |
//     cost prefix sums) -- coalesced for the nearest-node scan,
//   * the reference's time bins (rrt_dubins.py:110-114,147-151) as per-bin chains of 32-entry
//     chunks, so "the idx-th node of bin b" is one chunk walk.
// Waypoints are never stored: an edge is a pure function of (parent state, stream position), so
// the optimal path is re-created at the end from the chain of stream positions (also what the
// multi-GPU gather ships instead of paths).
//
// Cost is incremental (SURVEY.md section 8a, C1): habitat_shark_cost_func (cost.py:145-207) is a sum
// over the waypoints of generate_final_course (rrt_dubins.py:321-331) plus a visited-habitat set, so
// every node stores the sums over its root chain; a candidate leaf costs O(1).  For a parentless
// `initial` the planner's bin filter (rrt_dubins.py:161-166) never changes a waypoint's first-match
// bin (every waypoint time lies in [t_initial, t_leaf]).  Totals equal the reference's up to
// summation order (fp64: <= 1e-12 relative).
#include <stdlib.h>
#include "plan_common.cuh"
#include "dubins.cuh"

// Rehearse the next iteration's parent pick and prefetch its row (k_plan, default parent pick).  Measured on B200,
// config 2: 9.77 ms per step with it, 8.89 ms without -- the parent-row load is 17 % of the stall samples, but the
// rehearsal costs ~50 instructions per iteration in a kernel whose issue slots are 68 % busy, and the prefetched line
// competes with the tree's own lines in a 28-warp L1.  Off.
#ifndef AUV_PLAN_PREFETCH
#define AUV_PLAN_PREFETCH 0
#endif

namespace auv {

// CTA shape of k_plan.  Config 2's 4096 trees (one warp each) need 28 resident warps per SM to run in one wave
// (4096 / 148 = 27.7) and get 72 registers per thread.  Every CTA stages its own copy of the world model's hot part
// (11 KB), so fewer, larger CTAs leave more of the SM to the L1 that serves the trees, the classification grid and the
// probability table.  Measured on B200, config 2: 128 threads x 7 CTAs 8.63 ms per step (256 x 4 in round 1: 32 / 24
// warps per SM, the kernel waited for the fuller SMs), 224 x 4 8.45 ms, 448 x 2 8.25 ms, 896 x 1 7.78 ms (1.08e9 edges/s;
// the per-group scratch of the slot-addressed stream is 396 bytes, so 28 groups fit the 48 KB of static shared memory).
// The narrower groups (16 / 8 lanes per tree) keep 128-thread CTAs: their per-group scratch would not fit.
#ifndef AUV_PLAN_THREADS32
#define AUV_PLAN_THREADS32 896
#endif
#ifndef AUV_PLAN_MINB32
#define AUV_PLAN_MINB32 (896 / AUV_PLAN_THREADS32)
#endif
// (the fp64 verification build keeps 128-thread CTAs: it needs more than the 72 registers a 896-thread CTA leaves)
template <typename R, int G> struct PlanCta {
    static const int T = (sizeof(R) == 4 && G == 32) ? AUV_PLAN_THREADS32 : 128, MINB = (sizeof(R) == 4 && G == 32) ? AUV_PLAN_MINB32 : 7;
};

struct WsLayout {
    size_t slot_bytes;
    size_t rows, xy, pool, next, head, tail, count;
};

template <typename R> static WsLayout make_layout(int cap, int nb, int nchunks) {
    WsLayout L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 127) & ~(size_t)127; return r; };
    L.rows = take(sizeof(NodeRow<R>) * (size_t)cap);
    L.xy = take(2 * sizeof(R) * (size_t)cap);                 // SoA copy of (x, y) for the nearest-node scan
    L.pool = take(4 * 32 * (size_t)nchunks); L.next = take(4 * (size_t)nchunks);
    L.head = take(4 * (size_t)(nb + 2)); L.tail = take(4 * (size_t)(nb + 2)); L.count = take(4 * (size_t)(nb + 2));
    L.slot_bytes = o;
    return L;
}

// The group's tree: one slot base; every array is the base plus its WsLayout offset, which are kernel parameters (one
// 64-bit register for the tree instead of eight pointers)
template <typename R> struct Tree {
    unsigned char *b;
    const WsLayout &L;
    int cap;
    __device__ __forceinline__ NodeRow<R> *row() const { return (NodeRow<R> *)(b + L.rows); }
    __device__ __forceinline__ R *nx() const { return (R *)(b + L.xy); }         // coalesced x[] / y[] for RRT.get_closest_mps (mode 1)
    __device__ __forceinline__ R *ny() const { return nx() + cap; }
    __device__ __forceinline__ int *pool() const { return (int *)(b + L.pool); }
    __device__ __forceinline__ int *next() const { return (int *)(b + L.next); }
    __device__ __forceinline__ int *head() const { return (int *)(b + L.head); }
    __device__ __forceinline__ int *tail() const { return (int *)(b + L.tail); }
    __device__ __forceinline__ int *count() const { return (int *)(b + L.count); }
};

// BS: keep the per-bin metadata (count / head chunk / tail chunk) of the group's tree in shared
// memory as u16 (needs <= 126 time bins and <= 65535 nodes / chunks): the rejection loop of the
// parent pick reads count[bin] once per draw, so this takes a global round trip off every draw.
// ---- mode 3: one candidate edge = six-word Dubins path parent -> sample, cut at eta, W waypoints ---------------------
// (the build's own definition, parity unpinned: DESIGN.md section 11; oracle/auvrrt_oracle.c orc_exploring_dubins)
template <typename R> struct DubinsEdge {
    bool ok;                  // a word exists and the parent may be extended
    bool safe;                // check_collision over the W points
    R x, y, th, t, len;       // the new node = waypoint W-1
    R s2; uint32_t cnt; unsigned long long mask;   // cost sums over waypoints 1..W-1
    R self_s2; int self_hab;                       // contribution of the new node's own state
};
// rows != nullptr: also write waypoints 1..W-1 as (x, y, theta, v, t, len) rows (at most `room` of them)
template <typename R>
__device__ __forceinline__ void dubins_edge_eval(const EnvView<R> &env, const PlanP<R> &P, R px, R py, R pth, R pt, R plen,
                                                 R sx, R sy, R sth, bool do_tests, R *rows, int room, DubinsEdge<R> &e) {
    typedef typename Policy<R>::A A;
    e.ok = false; e.safe = false; e.x = px; e.y = py; e.th = pth; e.t = pt; e.len = plen;
    e.s2 = 0; e.cnt = 0; e.mask = 0ull; e.self_s2 = 0; e.self_hab = -1;
    const DubinsPath<R> d = dubins_shortest<R>(px, py, pth, sx, sy, sth, P.rho);
    if (d.word < 0) return;
    e.ok = true;
    const R s_end = d.length < P.eta ? d.length : P.eta;
    const R step = A::div(s_end, (R)(P.W - 1));
    DubinsSampler<R> smp;
    smp.init(d, px, py, pth, P.rho);
    bool bad = false;
    if (do_tests) {                                      // path[0] is the parent node object
        const Cls pcl = env.classify(px, py);
        bad = point_unsafe_c<R>(env, pcl, px, py);
    }
#pragma unroll 1
    for (int k = 1; k < P.W; k++) {
        const R sk = A::mul((R)k, step);
        R x, y, th;
        smp.at(sk, x, y, th);
        const R t = A::add(pt, A::div(sk, P.vel)), len = A::add(plen, sk);
        if (do_tests) {
            const Cls cl = env.classify(x, y);
            bad = bad || point_unsafe_c<R>(env, cl, x, y);
            const Contrib c = point_contrib<R>(env, x, y, t, 0xffffffffu, env.H, cl);
            const R ps2 = (c.bin >= 0 && c.cell >= 0) ? A::mul(P.w3, env.probs[(size_t)c.bin * env.C + c.cell]) : (R)0;
            if (c.bin >= 0) {
                e.s2 = A::add(e.s2, ps2);
                if (c.hab >= 0) { e.cnt++; e.mask |= 1ull << c.hab; }
            }
            e.self_s2 = c.bin >= 0 ? ps2 : (R)0; e.self_hab = c.bin >= 0 ? c.hab : -1;   // the last one is the new node
        }
        if (rows && k - 1 < room) {
            R *w = rows + 6 * (size_t)(k - 1);
            w[0] = x; w[1] = y; w[2] = th; w[3] = P.vel; w[4] = t; w[5] = len;
        }
        e.x = x; e.y = y; e.th = th; e.t = t; e.len = len;
    }
    e.safe = !bad;
}
// the sample of the iteration whose draws start at stream position ctr (get_random_mps, rrt_dubins.py:333-343)
template <typename R>
__device__ __forceinline__ void dubins_sample_at(const EnvView<R> &env, const Stream<R> &rng, uint32_t ctr, R &sx, R &sy, R &sth) {
    sx = uniform_ab<R>(env.minx, env.maxx, rng.u(ctr));
    sy = uniform_ab<R>(env.miny, env.maxy, rng.u(ctr + 1u));
    sth = uniform_ab<R>((R)-3.141592653589793, (R)3.141592653589793, rng.u(ctr + 2u));     // + 3: size, unused
}

#define AUV_BINS_SMEM 128
template <typename R> struct BestPlan { R c0, c1, c2, len, t; int node, iter; };
// a group's shared state, reached from one shared address: edge scratch, the best plan so far and, with BS, the bin
// metadata (count / head chunk / tail chunk)
template <typename R, int G, bool BS> struct GroupSmem {
    GroupScratch<R, G, false> sc;
    BestPlan<R> best;
    unsigned short bins[3][BS ? AUV_BINS_SMEM : 1];
};
// MODE >= 0 compiles the kernel for that parent-pick mode alone (the other modes' code -- about 1000 instructions that
// the compiler otherwise places inside the hot loop -- disappears); MODE < 0 reads P.mode at run time.
// ONE: freq <= G, every edge is a single chunk of primitives (eval_edge ONE_CHUNK)
template <typename R, int G, bool BS, int MODE, bool ONE>
__global__ void __launch_bounds__(PlanCta<R, G>::T, sizeof(R) == 4 ? PlanCta<R, G>::MINB : (PlanCta<R, G>::MINB + 1) / 2)
k_plan(const unsigned char *blob, int hot_bytes, int total_bytes, int stage_mode, const __grid_constant__ EnvView<R> envp,
       const R *starts, const uint64_t *seeds, long long Q, PlanP<R> P, const __grid_constant__ WsLayout L,
       unsigned char *ws, unsigned long long *qcounter, auvrrt_plan_record_t *records, uint32_t *chain_out, R *path_out,
       auvrrt_plan_trace_t tr) {
    typedef typename Policy<R>::A A;
    const bool VERIFY = Policy<R>::VERIFY;
    const int pick_mode = MODE >= 0 ? MODE : P.mode;
    extern __shared__ __align__(16) unsigned char smem[];
    const int PLAN_THREADS = PlanCta<R, G>::T;
    __shared__ GroupSmem<R, G, BS> groups[PlanCta<R, G>::T / G];
    EnvView<R> env;
    {
        // (the single-chunk variant in its one-CTA-per-SM shape always stages this way, plan_geometry: the other modes'
        // views would make the compiler keep every field in registers)
        if ((ONE && PlanCta<R, G>::T >= 896) || stage_mode == 3) {
            // one CTA per SM: the world model, the probability table and plane 0 of the classification grid (two regions,
            // one barrier) -- every lookup of the edge evaluation is then an LDS
            uint64_t *bar = (uint64_t *)smem;
            const EnvHeader *gh = (const EnvHeader *)blob;
            const int plane = (gh->gnx * gh->gny * 4 + 15) & ~15;
            if (threadIdx.x == 0) mbar_init(bar, 1);
            __syncthreads();
            if (threadIdx.x == 0) {
                mbar_expect_tx(bar, (uint32_t)(total_bytes + plane));
                for (int o = 0; o < total_bytes; o += 65536) tma_bulk_g2s(smem + 16 + o, blob + o, (uint32_t)(total_bytes - o < 65536 ? total_bytes - o : 65536), bar);
                const unsigned char *gsrc = blob + gh->off_grid;
                for (int o = 0; o < plane; o += 65536) tma_bulk_g2s(smem + 16 + total_bytes + o, gsrc + o, (uint32_t)(plane - o < 65536 ? plane - o : 65536), bar);
            }
            mbar_wait(bar, 0);
            // (the copy's shared address through volatile asm: the compiler would otherwise rebuild it from SR_CgaCtaId at
            // every lookup inside the loop)
            uint32_t staged = smem_u32(smem + 16);
            asm volatile("" : "+r"(staged));
            const unsigned char *sp = (const unsigned char *)__cvta_shared_to_generic(staged);
            env = envp;
            env.move_staged(blob, sp);
            env.grid0s = (const unsigned *)(sp + total_bytes);
        } else if (stage_mode == 0) {
            env.bind(blob, blob); env.bind_grid(blob, blob);
        } else {
            uint64_t *bar = (uint64_t *)smem;
            stage_env_tma(smem + 16, blob, stage_mode == 2 ? total_bytes : hot_bytes, bar);
            env.bind(smem + 16, stage_mode == 2 ? smem + 16 : blob);
            env.bind_grid(blob, smem + 16);
        }
        // the single-chunk variant is only launched with the hot part staged (launch_plan_g): its loads are LDS
        if (ONE) env.assume_hot_shared(PlanCta<R, G>::T >= 896);     // (896-thread shape: stage mode 3, the probability table is staged too)
    }
    Grp<G> g;
    // The group's shared state and its tree slot, each one address computed once.  (Through volatile asm: the compiler
    // would otherwise rebuild them from SR_TID.X, SR_CTAID.X and SR_CgaCtaId at every use inside the loop.)
    uint32_t gsa = smem_u32(&groups[threadIdx.x / G]);
    asm volatile("" : "+r"(gsa));
    GroupSmem<R, G, BS> &gs = *(GroupSmem<R, G, BS> *)__cvta_shared_to_generic(gsa);
    GroupScratch<R, G, false> &sc = gs.sc;
    unsigned char *slot_base = ws + (size_t)(blockIdx.x * (PLAN_THREADS / G) + threadIdx.x / G) * L.slot_bytes;
    asm volatile("" : "+l"(slot_base));
    const Tree<R> T{slot_base, L, P.cap};
#define BIN_COUNT(b) (BS ? (int)gs.bins[0][b] : T.count()[b])
#define BIN_HEAD(b) (BS ? (int)gs.bins[1][b] : T.head()[b])
#define BIN_TAIL(b) (BS ? (int)gs.bins[2][b] : T.tail()[b])
#define SET_BIN_COUNT(b, v) do { if (BS) gs.bins[0][b] = (unsigned short)(v); else T.count()[b] = (v); } while (0)
#define SET_BIN_HEAD(b, v) do { if (BS) gs.bins[1][b] = (unsigned short)(v); else T.head()[b] = (v); } while (0)
#define SET_BIN_TAIL(b, v) do { if (BS) gs.bins[2][b] = (unsigned short)(v); else T.tail()[b] = (v); } while (0)

    for (;;) {
        long long q = 0;
        if (g.gl == 0) q = (long long)atomicAdd(qcounter, 1ull);
        q = g.bcast(q, 0);
        if (q >= Q) break;

        const R sx = starts[5 * q], sy = starts[5 * q + 1], sth = starts[5 * q + 2], st = starts[5 * q + 3],
                slen = starts[5 * q + 4];
        // ---- init: mps_list = [initial]; time_bin[bin_interval] = [initial]        rrt_dubins.py:105-114
        for (int b = g.gl; b < P.nb + 2; b += G) SET_BIN_COUNT(b, 0);
        if (g.gl == 0) {
            NodeRow<R> r0;
            r0.x = sx; r0.y = sy; r0.th = sth; r0.t = st; r0.len = slen;
            r0.parent = -1; r0.ctr = 0; r0.s2 = (R)0; r0.cnt = 0; r0.mask = 0ull; r0.born = 0;
            Contrib c = point_contrib<R>(env, sx, sy, st, 0xffffffffu, env.H, env.classify(sx, sy));
            r0.self_s2 = (c.bin >= 0 && c.cell >= 0) ? A::mul(P.w3, env.probs[(size_t)c.bin * env.C + c.cell]) : (R)0;
            r0.self_hab = c.bin >= 0 ? c.hab : -1;
            T.row()[0] = r0;
            if (pick_mode == 1 || pick_mode == 3) { T.nx()[0] = sx; T.ny()[0] = sy; }
        }
        g.sync();
        if (g.gl == 0) { SET_BIN_HEAD(1, 0); SET_BIN_TAIL(1, 0); SET_BIN_COUNT(1, 1); T.pool()[0] = 0; T.next()[0] = -1; }
        g.sync();
        Stream<R> rng;                 // (after the root's cost: the key is not live across it)
        rng.key = stream_key(seeds[q]); rng.ext = nullptr; rng.n_ext = 0;
        int n_nodes = 1, n_chunks = 1;
        uint32_t ctr = 0, upos_mark = 0;
        int status = AUVRRT_ST_OK;
        int n_cost_evals = 0;
        unsigned n_waypoints = 0, n_prims = 0;
        // the best plan so far: only its total is compared every iteration; the rest lives in shared memory
        // (written by lane 0 on the rare improvement), which frees registers for the edge evaluation
        R best_total = A::inf();
        if (g.gl == 0) { BestPlan<R> b0; b0.c0 = b0.c1 = b0.c2 = b0.len = b0.t = (R)0; b0.node = -1; b0.iter = -1; gs.best = b0; }
        int it = 0;
        int guard = 0;
        const int guard_max = (int)min(64LL * P.I + 1024, 2147483647LL);

        while (it < P.I && guard++ < guard_max) {
            int parent;
            if (pick_mode == 3) {
                // ================= mode 3: Dubins-RRT with best-parent selection =================
                // lane = candidate parent: each lane evaluates ONE candidate edge (steer + collide + cost), a warp
                // min-reduction on (path cost, node index) picks the parent
                const uint32_t ctr0 = ctr;
                R smx, smy, smth;
                dubins_sample_at<R>(env, rng, ctr, smx, smy, smth);
                ctr += 4;
                // nearest node (get_closest_mps :505-513) and the first G nodes within near_radius, in index order
                int *near = (int *)sc.us;
                R bq = A::inf(), bs = A::inf();
                int bi = 0x7fffffff, nlist = 0;
                for (int i0 = 0; i0 < n_nodes; i0 += G) {
                    const int i = i0 + g.gl;
                    bool in = false;
                    if (i < n_nodes) {
                        const R qq = A::sq2(A::sub(smx, T.nx()[i]), A::sub(smy, T.ny()[i]));
                        if (qq < bq) {
                            if (VERIFY) { R sd = A::sqrt(qq); if (sd < bs) { bs = sd; bi = i; } }
                            else { bs = qq; bi = i; }
                            bq = qq;
                        }
                        in = VERIFY ? (A::sqrt(qq) <= P.near_r) : (qq <= P.near_r2);
                    }
                    const unsigned m = g.ballot(in);
                    if (in) {
                        const int pos = nlist + __popc(m & ((1u << g.gl) - 1u));
                        if (pos < G) near[pos] = i;
                    }
                    nlist += __popc(m);
                }
                nlist = min(nlist, G);
#pragma unroll
                for (int mm = G / 2; mm > 0; mm >>= 1) {
                    R os = g.xorv(bs, mm);
                    int oi = g.xorv(bi, mm);
                    if (os < bs || (os == bs && oi < bi)) { bs = os; bi = oi; }
                }
                const int nearest = bi;
                g.sync();
                if (T.row()[nearest].t > P.max_traj) { upos_mark = ctr; continue; }          // :138-139
                // candidates: [nearest] + the list without it, G at most
                int pn = nlist;                                    // position of the nearest node in the list, if any
                for (int j = g.gl; j < nlist; j += G) if (near[j] == nearest) pn = j;
#pragma unroll
                for (int mm = G / 2; mm > 0; mm >>= 1) pn = min(pn, g.xorv(pn, mm));
                const int ncand = min(G, 1 + nlist - (pn < nlist ? 1 : 0));
                int pidx = -1;
                if (g.gl == 0) pidx = nearest;
                else if (g.gl < ncand) { const int j = g.gl - 1; pidx = near[j < pn ? j : j + 1]; }
                g.sync();
                DubinsEdge<R> de;
                de.ok = false; de.safe = false; de.x = de.y = de.th = de.t = de.len = 0; de.s2 = 0; de.cnt = 0; de.mask = 0ull;
                de.self_s2 = 0; de.self_hab = -1;
                NodeRow<R> pr;
                pr.s2 = 0; pr.self_s2 = 0; pr.cnt = 0; pr.mask = 0ull; pr.self_hab = -1; pr.t = 0;
                if (pidx >= 0) {
                    pr = T.row()[pidx];
                    if (!(pr.t > P.max_traj))
                        dubins_edge_eval<R>(env, P, pr.x, pr.y, pr.th, pr.t, pr.len, smx, smy, smth, true, nullptr, 0, de);
                }
                n_waypoints += (unsigned)(P.W * __popc(g.ballot(de.ok)));
                // path cost root -> new node through this parent                            cost.py:145-207
                R pre_s2 = 0, c0 = 0, c1 = 0, c2 = 0, total = A::inf();
                uint32_t pre_cnt = 0; unsigned long long pre_mask = 0;
                if (de.ok && de.safe) {
                    const int ph = pr.self_hab;
                    pre_s2 = A::add(A::add(pr.s2, pr.self_s2), de.s2);
                    pre_cnt = pr.cnt + (ph >= 0 ? 1u : 0u) + de.cnt;
                    pre_mask = pr.mask | (ph >= 0 ? (1ull << ph) : 0ull) | de.mask;
                    const uint32_t cnt = pre_cnt + (de.self_hab >= 0 ? 1u : 0u);
                    const unsigned long long mk = pre_mask | (de.self_hab >= 0 ? (1ull << de.self_hab) : 0ull);
                    c1 = A::mul(P.w2, (R)cnt);
                    c2 = A::add(pre_s2, de.self_s2);
                    if (de.t > (R)0) { c1 = A::div(c1, de.t); c2 = A::div(c2, de.t); }
                    if (env.H != 0) c0 = A::div(A::mul(P.w1, (R)__popcll(mk)), (R)env.H);
                    total = py_sum3p<R>(c0, c1, c2);
                }
                // best parent: minimum (total, node index) over the lanes
                R bt = total; int bp = (de.ok && de.safe) ? pidx : 0x7fffffff;
#pragma unroll
                for (int mm = G / 2; mm > 0; mm >>= 1) {
                    R ot = g.xorv(bt, mm);
                    int op = g.xorv(bp, mm);
                    if (ot < bt || (ot == bt && op < bp)) { bt = ot; bp = op; }
                }
                const bool any_safe = bp != 0x7fffffff;
                const unsigned wm = g.ballot(any_safe && pidx == bp && de.ok && de.safe);
                const int bl = wm ? __ffs(wm) - 1 : 0;            // the winning lane (lane 0 = the nearest node otherwise)
                const R nx_ = g.bcast(de.x, bl), ny_ = g.bcast(de.y, bl), nth_ = g.bcast(de.th, bl), nt_ = g.bcast(de.t, bl),
                        nlen_ = g.bcast(de.len, bl);
                if (P.trace && g.gl == 0) {
                    size_t r = (size_t)q * P.I + it;
                    tr.parent[r] = any_safe ? bp : -1; tr.safe[r] = any_safe ? 1 : 0; tr.nwp[r] = P.W; tr.upos[r] = upos_mark;
                    R *lf = (R *)tr.leaf + 5 * r;
                    lf[0] = nx_; lf[1] = ny_; lf[2] = nth_; lf[3] = nt_; lf[4] = nlen_;
                }
                if (any_safe) {
                    const int id = n_nodes++;
                    if (g.gl == bl) {
                        NodeRow<R> nr;
                        nr.x = de.x; nr.y = de.y; nr.th = de.th; nr.t = de.t; nr.len = de.len; nr.parent = bp; nr.ctr = ctr0;
                        nr.s2 = pre_s2; nr.cnt = pre_cnt; nr.mask = pre_mask; nr.self_s2 = de.self_s2; nr.self_hab = de.self_hab;
                        nr.born = it;
                        T.row()[id] = nr;
                        T.nx()[id] = de.x; T.ny()[id] = de.y;
                    }
                    if (nt_ >= P.horizon) {                                                  // :158-171
                        n_cost_evals++;
                        if (bt < best_total) {
                            best_total = bt;
                            if (g.gl == bl) {
                                BestPlan<R> b; b.c0 = c0; b.c1 = c1; b.c2 = c2; b.len = de.len; b.t = de.t; b.node = id; b.iter = it;
                                gs.best = b;
                            }
                        }
                    }
                }
                g.sync();
                it++;
                upos_mark = ctr;
                continue;
            }
            if (pick_mode == 0) {
                // ---- pick a random non-empty time bin, then a random node in it           :122-127
                int ran_bin = 0, bincnt = 0;
                bool kerr = false;
                for (;;) {
                    R u = rng.u(ctr + (uint32_t)g.gl);
                    int rb = (int)uniform_ab<R>((R)1, (R)(P.nb + 1), u);
                    bool ke = rb > P.nb || rb < 1;
                    int cn = ke ? 0 : BIN_COUNT(rb);
                    unsigned m = g.ballot(ke || cn > 0);
                    if (m) {
                        int f = __ffs(m) - 1;
                        ran_bin = g.bcast(rb, f); bincnt = g.bcast(cn, f); kerr = g.bcast(ke ? 1 : 0, f) != 0;
                        ctr += (uint32_t)f + 1u;
                        break;
                    }
                    ctr += G;
                }
                if (kerr) { status = AUVRRT_ST_KEY_ERROR; break; }
                g.sync();        // every lane has read the bin counts before lane 0 may update them below
                R u = rng.u(ctr);
                ctr += 1;
                int idx = (int)uniform_ab<R>((R)0, (R)bincnt, u);
                if (idx >= bincnt) { status = AUVRRT_ST_KEY_ERROR; break; }
                int ch = BIN_HEAD(ran_bin);
#pragma unroll 1
                for (int hop = idx >> 5; hop > 0; hop--) ch = T.next()[ch];
                parent = T.pool()[ch * 32 + (idx & 31)];
            } else if (pick_mode == 2) {
                // ---- wall-clock pick on the simulated clock (:129-132): every lane walks the same bisection
                const R ran_time = uniform_ab<R>((R)0, P.ran_time_max, rng.u(ctr));
                ctr += 1;
                parent = closest_mps_time<R>(T.row(), n_nodes, ran_time, P.plan_dt);
                if (T.row()[parent].t > P.max_traj) continue;                               // :131-132
            } else {
                // ---- get_random_mps (:333-343) + get_closest_mps (:505-513)
                R rx = uniform_ab<R>(env.minx, env.maxx, rng.u(ctr));
                R ry = uniform_ab<R>(env.miny, env.maxy, rng.u(ctr + 1));
                ctr += 4;     // theta and size are drawn and never used
                R bq = A::inf(), bs = A::inf();
                int bi = 0x7fffffff;
                for (int i = g.gl; i < n_nodes; i += G) {
                    R qq = A::sq2(A::sub(rx, T.nx()[i]), A::sub(ry, T.ny()[i]));
                    if (qq < bq) {
                        if (VERIFY) { R s = A::sqrt(qq); if (s < bs) { bs = s; bi = i; } }
                        else { bs = qq; bi = i; }
                        bq = qq;
                    }
                }
#pragma unroll
                for (int m = G / 2; m > 0; m >>= 1) {
                    R os = g.xorv(bs, m);
                    int oi = g.xorv(bi, m);
                    if (os < bs || (os == bs && oi < bi)) { bs = os; bi = oi; }
                }
                parent = bi;
                if (T.row()[parent].t > P.max_traj) continue;                               // :138-139
            }
            // ---- steer + check_collision + per-waypoint cost                              :141-143
            // every lane reads the same row (a broadcast): the state now, the cost prefix after the edge and only if it is
            // safe (the line is then in L1), so that the prefix is not live across the edge evaluation
            const NodeRow<R> *prow = T.row() + parent;
            const R ppx = prow->x, ppy = prow->y, ppth = prow->th, ppt = prow->t, pplen = prow->len;
            const uint32_t ctr0 = ctr;
#if AUV_PLAN_PREFETCH
            // Look ahead.  Slot addressing makes the next iteration's stream position known now (this edge owns
            // 1 + 3 n_expand positions), so its parent pick can be rehearsed on the bins as they stand: the pool entry is
            // requested here and the parent's row prefetched behind the edge, while this edge is being evaluated.  The
            // real pick of the next iteration runs unchanged (an append into a rehearsed bin changes it) and finds both
            // lines in cache.
            int spec_parent = -1;
            if (ONE && BS && pick_mode == 0) {
                const int n_exp_now = (int)A::floor(uniform_ab<R>((R)0, P.sp.freq, rng.u(ctr)));
                const uint32_t cn0 = ctr + 1u + 3u * (uint32_t)(n_exp_now > 0 ? n_exp_now : 0);
                const int rb = (int)uniform_ab<R>((R)1, (R)(P.nb + 1), rng.u(cn0 + (uint32_t)g.gl));
                const int cn = (rb >= 1 && rb <= P.nb) ? (int)gs.bins[0][rb] : 0;
                const unsigned m = g.ballot(cn > 0);
                if (m) {
                    const int f = __ffs(m) - 1;
                    const int sb = g.bcast(rb, f), sc_ = g.bcast(cn, f);
                    const int idx = (int)uniform_ab<R>((R)0, (R)sc_, rng.u(cn0 + (uint32_t)f + 1u));
                    if (idx < 32 && idx < sc_) spec_parent = T.pool()[(int)gs.bins[1][sb] * 32 + idx];
                }
            }
#endif
            EdgeOut<R> o;
            eval_edge<R, G, true, true, false, false, ONE, ONE && (PlanCta<R, G>::T >= 896)>(g, sc, env, rng, ctr, P.sp, ppx, ppy, ppth, ppt, pplen, P.w3, env.H,
                                                           nullptr, 0, o);
#if AUV_PLAN_PREFETCH
            if (ONE && BS && pick_mode == 0 && spec_parent >= 0 && g.gl < 2)
                asm volatile("prefetch.global.L1 [%0];" ::"l"((const char *)&T.row()[spec_parent] + 32 * g.gl));
#endif
            ctr = o.ctr;
            n_waypoints += o.nwp; n_prims += o.n_exp;
            if (P.trace && g.gl == 0) {
                size_t r = (size_t)q * P.I + it;
                tr.parent[r] = parent; tr.safe[r] = o.safe ? 1 : 0; tr.nwp[r] = o.nwp; tr.upos[r] = upos_mark;
                R *lf = (R *)tr.leaf + 5 * r;
                lf[0] = o.x; lf[1] = o.y; lf[2] = o.th; lf[3] = o.t; lf[4] = o.len;
            }
            if (o.status != 0) { status = o.status; break; }
            if (o.safe) {
                const int id = n_nodes++;                                                  // :144-145
                // (every lane computes the new node's cost prefix: the leaf cost below needs no broadcast)
                const R pr_s2 = prow->s2, pr_self_s2 = prow->self_s2;
                const uint32_t pr_cnt = prow->cnt;
                const int ph = prow->self_hab;
                const unsigned long long pr_mask = prow->mask;
                const R pre_s2 = A::add(A::add(pr_s2, pr_self_s2), o.s2);
                const uint32_t pre_cnt = pr_cnt + (ph >= 0 ? 1u : 0u) + o.cnt;
                const unsigned long long pre_mask = pr_mask | (ph >= 0 ? (1ull << ph) : 0ull) | o.mask;
                const R self_s2n = o.leaf_moved ? o.self_s2 : pr_self_s2;
                const int self_habn = o.leaf_moved ? o.self_hab : ph;
                if (g.gl == 0) {
                    NodeRow<R> nr;
                    nr.x = o.x; nr.y = o.y; nr.th = o.th; nr.t = o.t; nr.len = o.len; nr.parent = parent; nr.ctr = ctr0;
                    nr.s2 = pre_s2; nr.cnt = pre_cnt; nr.mask = pre_mask; nr.self_s2 = self_s2n; nr.self_hab = self_habn;
                    nr.born = it;
                    T.row()[id] = nr;
                    if (pick_mode == 1 || pick_mode == 3) { T.nx()[id] = o.x; T.ny()[id] = o.y; }
                }
                // ---- time-bin insert (decision is group-uniform, lane 0 writes)            :147-151
                if (pick_mode != 2) {                   // `if traj_time_stamp:` -- mode 2 keeps no bins
                    R fd = floordiv_pos<R>(o.t, P.bin_interval);
                    R fidx = fd + (R)1;
                    R curr_bin = A::mul(fidx, P.bin_interval);
                    int bidx = -1; bool reset = false;
                    if (curr_bin > P.max_traj) {
                        // `self.time_bin[curr_bin] = []` re-creates the key; only reachable if it is a live one
                        if (fidx >= (R)1 && fidx <= (R)P.nb) { bidx = (int)fidx; reset = true; }
                    } else {
                        if (fidx >= (R)1 && fidx <= (R)P.nb) bidx = (int)fidx; else status = AUVRRT_ST_KEY_ERROR;
                    }
                    if (bidx >= 0) {
                        // lane 0 owns the bin metadata: it reads, broadcasts, and writes (no lane may observe
                        // its update early: n_chunks below must stay identical on every lane)
                        const int c_old = g.bcast(g.gl == 0 ? BIN_COUNT(bidx) : 0, 0);
                        const bool reuse_head = reset && c_old > 0;
                        const int c = reset ? 0 : c_old;
                        const bool alloc = ((c & 31) == 0) && !reuse_head;
                        const int nc = n_chunks;
                        if (alloc) n_chunks++;
                        if (g.gl == 0) {
                            int tl = reuse_head ? BIN_HEAD(bidx) : BIN_TAIL(bidx);
                            if (alloc) {
                                T.next()[nc] = -1;
                                if (c == 0) SET_BIN_HEAD(bidx, nc); else T.next()[tl] = nc;
                                tl = nc;
                            }
                            SET_BIN_TAIL(bidx, tl);
                            T.pool()[tl * 32 + (c & 31)] = id;
                            SET_BIN_COUNT(bidx, c + 1);
                        }
                    }
                }
                if (status != AUVRRT_ST_OK) break;              // (status is group-uniform)
                // ---- candidate leaf: cost of the path root -> new node                    :158-171
                if (o.t >= P.horizon) {
                    const uint32_t cnt = pre_cnt + (self_habn >= 0 ? 1u : 0u);
                    const unsigned long long mk = pre_mask | (self_habn >= 0 ? (1ull << self_habn) : 0ull);
                    R c0 = 0, c1 = A::mul(P.w2, (R)cnt), c2 = A::add(pre_s2, self_s2n);
                    if (o.t > (R)0) { c1 = A::div(c1, o.t); c2 = A::div(c2, o.t); }            // cost.py:194-196
                    if (env.H != 0) c0 = A::div(A::mul(P.w1, (R)__popcll(mk)), (R)env.H);      // cost.py:204-205
                    const R total = py_sum3p<R>(c0, c1, c2);
                    n_cost_evals++;
                    if (total < best_total) {                                              // :169 strict <
                        best_total = total;
                        if (g.gl == 0) {
                            BestPlan<R> b; b.c0 = c0; b.c1 = c1; b.c2 = c2; b.len = o.len; b.t = o.t; b.node = id; b.iter = it;
                            gs.best = b;
                        }
                    }
                }
                g.sync();
            }
            it++;
            upos_mark = ctr;
        }
        g.sync();
        rng.key = stream_key(seeds[q]);   // (derived again for the path: the part the loop does not use is not kept across it)
        const BestPlan<R> best = gs.best;
        const int best_node = best.node, best_iter = best.iter;
        const R best_c[4] = {best_total, best.c0, best.c1, best.c2}, best_len = best.len, best_t = best.t;
        if (status == AUVRRT_ST_OK && best_node < 0) status = AUVRRT_ST_NO_PATH;
        // ---- optimal path: chain of stream positions, optional waypoints             :174-176, :321-331
        int depth = 0, n_path = 0;
        if (best_node < 0 && chain_out)
            for (int k = g.gl; k < P.chain_cap; k += G) chain_out[(size_t)q * P.chain_cap + k] = 0u;
        if (best_node >= 0) {
            for (int n = best_node; T.row()[n].parent >= 0; n = T.row()[n].parent) depth++;
            uint32_t *chain = chain_out ? chain_out + (size_t)q * P.chain_cap : nullptr;
            if (depth > P.chain_cap && chain) { if (status == AUVRRT_ST_OK) status = AUVRRT_ST_OVERFLOW; }
            if (chain && g.gl == 0) {
                int n = best_node;
                for (int k = depth - 1; k >= 0; k--) { if (k < P.chain_cap) chain[k] = (uint32_t)n; n = T.row()[n].parent; }
            }
            g.sync();
            if (path_out && P.path_cap > 0 && chain && depth <= P.chain_cap) {
                R *rows = path_out + (size_t)q * P.path_cap * 6;
                for (int e = 0; e < depth; e++) {
                    const int id = (int)chain[e];
                    const NodeRow<R> pn = T.row()[T.row()[id].parent];
                    if (g.gl == 0 && n_path < P.path_cap) {
                        R *w = rows + 6 * (size_t)n_path;
                        w[0] = pn.x; w[1] = pn.y; w[2] = pn.th; w[3] = (pick_mode == 3 && pn.parent >= 0) ? P.vel : (R)0;
                        w[4] = pn.t; w[5] = pn.len;
                    }
                    n_path++;
                    int room = P.path_cap - n_path; if (room < 0) room = 0;
                    if (pick_mode == 3) {
                        if (g.gl == 0) {
                            R smx, smy, smth;
                            dubins_sample_at<R>(env, rng, T.row()[id].ctr, smx, smy, smth);
                            DubinsEdge<R> de;
                            dubins_edge_eval<R>(env, P, pn.x, pn.y, pn.th, pn.t, pn.len, smx, smy, smth, false,
                                                rows + 6 * (size_t)(n_path < P.path_cap ? n_path : 0), room, de);
                        }
                        n_path += P.W - 1;
                        continue;
                    }
                    EdgeOut<R> o;
                    eval_edge<R, G, false, false, true>(g, sc, env, rng, T.row()[id].ctr, P.sp, pn.x, pn.y, pn.th,
                                                        pn.t, pn.len, (R)0, 0,
                                                        rows + 6 * (size_t)(n_path < P.path_cap ? n_path : 0), room, o);
                    n_path += o.nwp - 1;
                }
                if (g.gl == 0 && n_path < P.path_cap) {
                    R *w = rows + 6 * (size_t)n_path;
                    const NodeRow<R> bn = T.row()[best_node];
                    w[0] = bn.x; w[1] = bn.y; w[2] = bn.th; w[3] = (pick_mode == 3 && bn.parent >= 0) ? P.vel : (R)0;
                    w[4] = bn.t; w[5] = bn.len;
                }
                n_path++;
                if (n_path > P.path_cap && status == AUVRRT_ST_OK) status = AUVRRT_ST_OVERFLOW;
            }
            g.sync();
            if (chain && g.gl == 0)
                for (int k = 0; k < depth && k < P.chain_cap; k++) chain[k] = T.row()[chain[k]].ctr;
            if (chain) for (int k = depth + g.gl; k < P.chain_cap; k += G) chain[k] = 0u;
        }
        if (g.gl == 0) {
            auvrrt_plan_record_t rec;
            rec.status = status; rec.n_nodes = n_nodes; rec.best_node = best_node; rec.best_iter = best_iter;
            rec.depth = depth; rec.n_path = n_path; rec.n_cost_evals = n_cost_evals;
            rec.n_waypoints = (int32_t)n_waypoints; rec.n_uniforms = (long long)ctr; rec.n_primitives = (long long)n_prims;
            rec.cost[0] = best_node >= 0 ? (double)best_c[0] : 0.0; rec.cost[1] = (double)best_c[1];
            rec.cost[2] = (double)best_c[2]; rec.cost[3] = (double)best_c[3];
            rec.path_length = (double)best_len; rec.t_leaf = (double)best_t;
            records[q] = rec;
        }
        g.sync();
    }
}

// ---- re-create paths from (start, seed, chain of stream positions): no tree needed ------------
template <typename R, int G>
__global__ void __launch_bounds__(128)
k_materialize(const unsigned char *blob, const R *starts, const uint64_t *seeds, const uint32_t *chain,
              const int32_t *depth, long long Q, PlanP<R> P, R *path_out, int32_t *n_path_out) {
    __shared__ GroupScratch<R, G, false> scratch[128 / G];
    EnvView<R> env;
    env.bind(blob, blob);
    env.bind_grid(blob, blob);
    Grp<G> g;
    GroupScratch<R, G, false> &sc = scratch[threadIdx.x / G];
    const long long groups = (long long)gridDim.x * (128 / G);
    for (long long q = blockIdx.x * (long long)(128 / G) + threadIdx.x / G; q < Q; q += groups) {
        Stream<R> rng;
        rng.key = stream_key(seeds[q]); rng.ext = nullptr; rng.n_ext = 0;
        R x = starts[5 * q], y = starts[5 * q + 1], th = starts[5 * q + 2], t = starts[5 * q + 3], len = starts[5 * q + 4];
        R *rows = path_out + (size_t)q * P.path_cap * 6;
        int n_path = 0;
        const int d = depth[q];
        for (int e = 0; e < d; e++) {
            if (g.gl == 0 && n_path < P.path_cap) {
                R *w = rows + 6 * (size_t)n_path;
                w[0] = x; w[1] = y; w[2] = th; w[3] = (P.mode == 3 && e > 0) ? P.vel : (R)0; w[4] = t; w[5] = len;
            }
            n_path++;
            int room = P.path_cap - n_path; if (room < 0) room = 0;
            if (P.mode == 3) {                      // every lane re-creates the same Dubins edge; lane 0 writes its rows
                R smx, smy, smth;
                dubins_sample_at<R>(env, rng, chain[(size_t)q * P.chain_cap + e], smx, smy, smth);
                DubinsEdge<R> de;
                dubins_edge_eval<R>(env, P, x, y, th, t, len, smx, smy, smth, false,
                                    g.gl == 0 ? rows + 6 * (size_t)(n_path < P.path_cap ? n_path : 0) : nullptr, room, de);
                n_path += P.W - 1;
                x = de.x; y = de.y; th = de.th; t = de.t; len = de.len;
                continue;
            }
            EdgeOut<R> o;
            eval_edge<R, G, false, false, true>(g, sc, env, rng, chain[(size_t)q * P.chain_cap + e], P.sp, x, y, th, t,
                                                len, (R)0, 0, rows + 6 * (size_t)(n_path < P.path_cap ? n_path : 0),
                                                room, o);
            n_path += o.nwp - 1;
            x = o.x; y = o.y; th = o.th; t = o.t; len = o.len;
        }
        if (d >= 0) {
            if (g.gl == 0 && n_path < P.path_cap) {
                R *w = rows + 6 * (size_t)n_path;
                w[0] = x; w[1] = y; w[2] = th; w[3] = (P.mode == 3 && d > 0) ? P.vel : (R)0; w[4] = t; w[5] = len;
            }
            n_path++;
        }
        if (g.gl == 0) n_path_out[q] = n_path;
    }
}

// ---- host side --------------------------------------------------------------------------------
template <typename R, int G, bool BS, int MODE, bool ONE> static int plan_geometry(const auvrrt_env *env, int *grid, int *smem, int *stage_mode) {
    EnvBlob<R> b = env_blob<R>(env);
    // only the small hot part of the world model is staged in shared memory when it is tight: with 4
    // CTAs per SM the probability table (39 KB for Catalina) is better served by the larger L1
    // (one 896-thread CTA per SM: the probability table is staged too -- measured 7.79 -> 7.69 ms per step on config 2)
    int budget = sizeof(R) == 4 ? (PlanCta<R, G>::T >= 896 ? 96 * 1024 : 24 * 1024) : 110 * 1024;
    if (const char *ev = getenv("AUVRRT_PLAN_STAGE_KB")) budget = atoi(ev) * 1024;
    if (const char *ev = getenv("AUVRRT_PLAN_BUDGET_KB")) budget = atoi(ev) * 1024;      // (does not switch the kernel variant)
    int sm = 16, mode = 0;
    if (b.total_bytes + 16 <= budget) { sm = b.total_bytes + 16; mode = 2; }
    else if (b.hot_bytes + 16 <= budget) { sm = b.hot_bytes + 16; mode = 1; }
    if (ONE && PlanCta<R, G>::T >= 896) {
        // the single-chunk kernel in its one-CTA-per-SM shape reads the grid from shared memory (launch_plan_g checked the fit)
        const EnvHeader &hd = sizeof(R) == 4 ? env->h32 : env->h64;
        sm = b.total_bytes + 16 + ((hd.gnx * hd.gny * 4 + 15) & ~15); mode = 3;
    }
    AUV_CUDA(cudaFuncSetAttribute(k_plan<R, G, BS, MODE, ONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
    int per_sm = 0;
    AUV_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_plan<R, G, BS, MODE, ONE>, PlanCta<R, G>::T, sm));
    if (per_sm < 1) return set_err(AUVRRT_ERR_CUDA, "plan: kernel does not fit on an SM (smem %d)", sm);
    int nsm = 0, dev = 0;
    AUV_CUDA(cudaGetDevice(&dev));
    AUV_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    *grid = nsm * per_sm; *smem = sm; *stage_mode = mode;
    return AUVRRT_OK;
}

template <typename R, int G, bool BS, int MODE, bool ONE>
static int launch_plan_gb(const auvrrt_env *env, const R *starts, const uint64_t *seeds, int64_t Q,
                         const auvrrt_plan_params_t *p, void *workspace, int64_t workspace_bytes,
                         auvrrt_plan_record_t *records, uint32_t *chain, R *path, const auvrrt_plan_trace_t *trace,
                         cudaStream_t s, int64_t *need_bytes) {
    PlanP<R> P;
    int rc = make_planp<R>(env, p, &P);
    if (rc) return rc;
    int grid, smem, mode;
    rc = plan_geometry<R, G, BS, MODE, ONE>(env, &grid, &smem, &mode);
    if (rc) return rc;
    WsLayout L = make_layout<R>(P.cap, P.nb, P.nchunks);
    const int gpc = PlanCta<R, G>::T / G;
    int64_t need = 256 + (int64_t)grid * gpc * (int64_t)L.slot_bytes;
    if (need_bytes) { *need_bytes = need; return AUVRRT_OK; }
    if (Q <= 0) return AUVRRT_OK;
    if (workspace_bytes < need) return set_err(AUVRRT_ERR_ARG, "plan: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)need);
    if (P.trace && !trace) return set_err(AUVRRT_ERR_ARG, "plan: trace requested without trace buffers");
    int64_t blocks = (Q + gpc - 1) / gpc;
    if (blocks < grid) grid = (int)blocks;
    AUV_CUDA(cudaMemsetAsync(workspace, 0, 256, s));
    auvrrt_plan_trace_t tr;
    if (trace) tr = *trace; else { tr.parent = nullptr; tr.safe = nullptr; tr.nwp = nullptr; tr.leaf = nullptr; tr.upos = nullptr; }
    EnvBlob<R> b = env_blob<R>(env);
    // the world-model view bound to the blob in HBM (stage mode 3 moves its arrays to the shared-memory copy)
    const EnvHeader &hd = sizeof(R) == 4 ? env->h32 : env->h64;
    EnvView<R> ev;
    ev.bind_header(hd, b.blob, b.blob);
    ev.bind_grid_header(hd, b.blob, b.blob);
    ev.bin_lo = hd.T > 0 ? (R)env->h_bins[0] : (R)1; ev.bin_hi = hd.T > 0 ? (R)env->h_bins[2 * hd.T - 1] : (R)0;
    k_plan<R, G, BS, MODE, ONE><<<grid, PlanCta<R, G>::T, smem, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode, ev, starts, seeds, (long long)Q, P, L,
                                                  (unsigned char *)workspace + 256, (unsigned long long *)workspace,
                                                  records, chain, path, tr);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

template <typename R, int G>
static int launch_plan_g(const auvrrt_env *env, const R *starts, const uint64_t *seeds, int64_t Q,
                         const auvrrt_plan_params_t *p, void *workspace, int64_t workspace_bytes,
                         auvrrt_plan_record_t *records, uint32_t *chain, R *path, const auvrrt_plan_trace_t *trace,
                         cudaStream_t s, int64_t *need_bytes) {
    const double nb = ceil(p->max_traj_time / p->bin_interval);
    const bool bs = nb + 2 <= AUV_BINS_SMEM && p->iterations < 65000 && !getenv("AUVRRT_PLAN_BINS_GLOBAL");
    // the fast build's default mode (time-bin pick) gets its own compilation of the kernel
#define AUV_PLAN_ARGS env, starts, seeds, Q, p, workspace, workspace_bytes, records, chain, path, trace, s, need_bytes
    if constexpr (sizeof(R) == 4) {
        if (p->mode == 0 && !getenv("AUVRRT_PLAN_GENERIC")) {
            // the common shape: every edge one chunk, bins in shared memory, hot part of the world model staged
            // (896-thread shape: world model + probability table + grid plane 0 must fit next to 36 KB of static arrays)
            const bool fits = PlanCta<R, G>::T >= 896
                                  ? (env->h32.gnx > 0 && env->h32.total_bytes + 16 + env->h32.gnx * env->h32.gny * 4 + 16 <= 180 * 1024)
                                  : env->h32.hot_bytes + 16 <= 24 * 1024;
            // n_expand = floor(uniform_ab<float>(0, freq, d)) = floor(fmaf(freq, d, -freq)) with d in [1, 2 - 2^-23]: at
            // most G - 1 for freq <= G, which leaves lane G - 1 of the single chunk to the parent point (eval_edge).
            // The form is monotone in d, so the largest draw bounds it.
            const float fq = (float)p->freq;
            const bool one_chunk = p->freq <= (double)G && floorf(fmaf(fq, 2.0f - 0x1p-23f, -fq)) <= (float)(G - 1);
            if (one_chunk && bs && fits && !getenv("AUVRRT_PLAN_STAGE_KB"))
                return launch_plan_gb<R, G, true, 0, true>(AUV_PLAN_ARGS);
            return bs ? launch_plan_gb<R, G, true, 0, false>(AUV_PLAN_ARGS) : launch_plan_gb<R, G, false, 0, false>(AUV_PLAN_ARGS);
        }
    }
    return bs ? launch_plan_gb<R, G, true, -1, false>(AUV_PLAN_ARGS) : launch_plan_gb<R, G, false, -1, false>(AUV_PLAN_ARGS);
#undef AUV_PLAN_ARGS
}

template <typename R>
int launch_plan(const auvrrt_env *env, const R *starts, const uint64_t *seeds, int64_t Q,
                const auvrrt_plan_params_t *p, void *workspace, int64_t workspace_bytes,
                auvrrt_plan_record_t *records, uint32_t *chain, R *path, const auvrrt_plan_trace_t *trace,
                cudaStream_t s) {
    // group 0 = automatic: a warp per tree shortens the latency of a few thousand queries; from
    // ~3x10^4 queries on, the queries themselves fill the machine and one thread per tree wins
    int G = p->group ? p->group : ((Q >= 32768 && !(path && p->path_cap > 0) && p->mode != 3) ? 1 : 32);
    if (G == 1 && p->mode == 3) return set_err(AUVRRT_ERR_UNSUPPORTED, "plan: mode 3 evaluates one candidate parent per lane; group must be 32, 16 or 8");
    if (G == 1) {
        if (path && p->path_cap > 0) return set_err(AUVRRT_ERR_UNSUPPORTED, "plan: group 1 (thread per tree) writes no paths; use auvrrt_materialize");
        return launch_plan_tpt<R>(env, starts, seeds, Q, p, workspace, workspace_bytes, records, chain, trace, s, nullptr);
    }
    if (G == 32) return launch_plan_g<R, 32>(env, starts, seeds, Q, p, workspace, workspace_bytes, records, chain, path, trace, s, nullptr);
    if (G == 16) return launch_plan_g<R, 16>(env, starts, seeds, Q, p, workspace, workspace_bytes, records, chain, path, trace, s, nullptr);
    if (G == 8) return launch_plan_g<R, 8>(env, starts, seeds, Q, p, workspace, workspace_bytes, records, chain, path, trace, s, nullptr);
    return set_err(AUVRRT_ERR_ARG, "plan: group must be 32, 16, 8 or 1");
}
// Q <= 0: a batch of any size.  Group 0 lets launch_plan pick the kernel per batch (by its size and whether paths are
// written), so the workspace must hold the largest one it can pick for a batch of at most Q queries.
template <typename R>
int64_t plan_workspace_bytes(const auvrrt_env *env, const auvrrt_plan_params_t *p, int64_t Q) {
    int64_t need = -1;
    int rc;
    const int G = p->group ? p->group : 32;
    if (G == 1) rc = launch_plan_tpt<R>(env, nullptr, nullptr, Q, p, nullptr, 0, nullptr, nullptr, nullptr, 0, &need);
    else if (G == 32) rc = launch_plan_g<R, 32>(env, nullptr, nullptr, 0, p, nullptr, 0, nullptr, nullptr, nullptr, nullptr, 0, &need);
    else if (G == 16) rc = launch_plan_g<R, 16>(env, nullptr, nullptr, 0, p, nullptr, 0, nullptr, nullptr, nullptr, nullptr, 0, &need);
    else if (G == 8) rc = launch_plan_g<R, 8>(env, nullptr, nullptr, 0, p, nullptr, 0, nullptr, nullptr, nullptr, nullptr, 0, &need);
    else { set_err(AUVRRT_ERR_ARG, "plan: group must be 32, 16, 8 or 1"); return -1; }
    if (rc) return -1;
    if (p->group == 0 && p->mode != 3 && (Q <= 0 || Q >= 32768)) {
        int64_t tpt = -1;
        if (launch_plan_tpt<R>(env, nullptr, nullptr, Q, p, nullptr, 0, nullptr, nullptr, nullptr, 0, &tpt)) return -1;
        if (tpt > need) need = tpt;
    }
    return need;
}
template int launch_plan<float>(const auvrrt_env *, const float *, const uint64_t *, int64_t, const auvrrt_plan_params_t *,
                                void *, int64_t, auvrrt_plan_record_t *, uint32_t *, float *, const auvrrt_plan_trace_t *, cudaStream_t);
template int launch_plan<double>(const auvrrt_env *, const double *, const uint64_t *, int64_t, const auvrrt_plan_params_t *,
                                 void *, int64_t, auvrrt_plan_record_t *, uint32_t *, double *, const auvrrt_plan_trace_t *, cudaStream_t);
template int64_t plan_workspace_bytes<float>(const auvrrt_env *, const auvrrt_plan_params_t *, int64_t);
template int64_t plan_workspace_bytes<double>(const auvrrt_env *, const auvrrt_plan_params_t *, int64_t);

template <typename R>
int launch_materialize(const auvrrt_env *env, const R *starts, const uint64_t *seeds, const uint32_t *chain,
                       const int32_t *depth, int64_t Q, const auvrrt_plan_params_t *p, R *path, int32_t *n_path,
                       cudaStream_t s) {
    if (Q <= 0) return AUVRRT_OK;
    PlanP<R> P;
    int rc = make_planp<R>(env, p, &P);
    if (rc) return rc;
    // the evaluator of the planner that made the chains: the fp32 group sizes sum an edge's primitives in their own order
    const int G = p->group ? p->group : 32;
    if (G == 1) {
        if (p->mode == 3) return set_err(AUVRRT_ERR_UNSUPPORTED, "materialize: mode 3 has no thread-per-tree plans");
        return launch_materialize_tpt<R>(env, starts, seeds, chain, depth, Q, P, path, n_path, s);
    }
    int64_t blocks = (Q * G + 127) / 128;
    if (blocks > AUV_SMS * 8) blocks = AUV_SMS * 8;
    const unsigned char *blob = env_blob<R>(env).blob;
    if (G == 32) k_materialize<R, 32><<<(unsigned)blocks, 128, 0, s>>>(blob, starts, seeds, chain, depth, (long long)Q, P, path, n_path);
    else if (G == 16) k_materialize<R, 16><<<(unsigned)blocks, 128, 0, s>>>(blob, starts, seeds, chain, depth, (long long)Q, P, path, n_path);
    else if (G == 8) k_materialize<R, 8><<<(unsigned)blocks, 128, 0, s>>>(blob, starts, seeds, chain, depth, (long long)Q, P, path, n_path);
    else return set_err(AUVRRT_ERR_ARG, "materialize: group must be 32, 16, 8 or 1");
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_materialize<float>(const auvrrt_env *, const float *, const uint64_t *, const uint32_t *, const int32_t *,
                                       int64_t, const auvrrt_plan_params_t *, float *, int32_t *, cudaStream_t);
template int launch_materialize<double>(const auvrrt_env *, const double *, const uint64_t *, const uint32_t *, const int32_t *,
                                        int64_t, const auvrrt_plan_params_t *, double *, int32_t *, cudaStream_t);

}  // namespace auv
