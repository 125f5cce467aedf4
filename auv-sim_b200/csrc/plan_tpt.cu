// plan_tpt.cu -- RRT.exploring (/root/reference/path_planning/rrt_dubins.py:92-176), ONE THREAD PER
// TREE: the throughput planner for very large batches of independent queries (config 5: 10^5..10^6
// queries per GPU).
//
// plan.cu spends 32 lanes on one tree to shorten the latency of a single query (what matters at a
// few thousand queries).  With >= 10^5 queries resident the machine is filled by the queries
// themselves, so each thread simply runs the reference's serial loop for its own tree and all the
// cooperative machinery (stream-offset resolution, scans, ballots) disappears.  Same stream, same
// bins, same incremental cost, same statuses: in the fp64 build the traces are identical to
// plan.cu's and to the reference's (tests/test_gpu_parity.py::test_plan_thread_per_tree_*).
//
// Per-tree workspace (private to the thread): AoS node rows (one 64-byte row in fp32: x,y,theta,t |
// len,s2,self_s2,ctr | parent,cnt,self_hab | mask) and the chunked time bins of plan.cu.
#include <stdlib.h>
#include "plan_common.cuh"
#include "edge_serial.cuh"

namespace auv {

#ifndef AUV_TPT_THREADS
#define AUV_TPT_THREADS 128   // finer work units than 256 (measured +1..4 % at 1.3e5 - 2.6e5 queries)
#endif
static const int TPT_THREADS = AUV_TPT_THREADS;
// Tree slots per thread.  With 2, a CTA of T threads owns 2T trees; every trip sorts them by n_expand into 2T/32 groups
// and warp w runs group w and then group 2T/32 - 1 - w (shortest with longest), so that the warps of a CTA reach the
// barrier behind the sort at about the same time: with one group per warp the warp holding the short edges waits
// for the one holding the long ones (29 % of the stall samples in profiles/r02_tpt_fast.txt).
// Measured on B200, 262 144 queries x 2048: one slot per thread 2.04e9 edges/s, two 1.85e9 (2.02e9 at 524 288 queries):
// the barrier stalls do fall (29 % -> 13 % of the samples) and so do the executed instructions (-15 %), but the shared
// memory of 256 slots leaves 4 CTAs = 16 warps per SM, too few for the kernel's dependent global loads.
#ifndef AUV_TPT_SPT
#define AUV_TPT_SPT 1
#endif
#ifndef AUV_TPT_MINB
#define AUV_TPT_MINB (AUV_TPT_SPT == 2 ? 6 : 8)
#endif
static const int TPT_SLOTS = AUV_TPT_THREADS * AUV_TPT_SPT;

struct TptLayout { size_t slot_bytes, nodes, pool, next, bins, hdr; };

// the part of a tree's bookkeeping that is touched rarely (a new best plan, a skipped trip, the trace): in the tree's
// workspace, not in shared memory -- every byte of per-tree shared state costs resident warps
template <typename R> struct TptHdr { int bestnode, bestiter, ncost, guard; uint32_t upos; int pad_; R bc1, bc2, bc3, blen, bt; };

template <typename R> static TptLayout make_tpt_layout(int cap, int nb, int nchunks) {
    TptLayout L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 127) & ~(size_t)127; return r; };
    L.nodes = take(sizeof(NodeRow<R>) * (size_t)cap);
    L.pool = take(4 * 32 * (size_t)nchunks); L.next = take(4 * (size_t)nchunks);
    // time bins: {count, head chunk, tail chunk, -} per bin in ONE 16-byte row: the pick reads count and head, the insert
    // reads and writes all three -- one 32-byte sector each instead of three
    L.bins = take(16 * (size_t)(nb + 2));
    L.hdr = take(sizeof(TptHdr<R>));
    L.slot_bytes = o;
    return L;
}

// Divergence control: an RRT iteration costs O(n_expand) arc primitives and n_expand is uniform in
// [0, freq), so a warp of 32 trees would idle half its lanes in the primitive loop.  Every trip the
// block therefore (A) lets thread i pick the parent and draw n_expand for tree slot i, (sort) orders
// its 256 tree slots by n_expand with a shared-memory counting sort, and (B) lets thread i run the
// steer / collide / cost / append part for the i-th slot in that order, so the lanes of a warp loop
// over nearly the same number of primitives.  The per-tree registers that survive an iteration
// live in shared memory (struct-of-arrays) because a different thread owns the tree every trip.
// FAST: the hot part of the world model is staged and the map has every lookup table (classification grid, x-bucket
// table, equal contiguous time bins, <= 32 habitats): the edge loop runs the straight-line forms of edge_serial.cuh
template <typename R, bool FAST>
__global__ void __launch_bounds__(TPT_THREADS, AUV_TPT_MINB)
k_plan_tpt(const unsigned char *blob, int hot_bytes, int total_bytes, int stage_mode, const R *starts,
           const uint64_t *seeds, long long Q, PlanP<R> P, TptLayout L, unsigned char *ws, unsigned long long *qcounter,
           auvrrt_plan_record_t *records, uint32_t *chain_out, auvrrt_plan_trace_t tr) {
    typedef typename Policy<R>::A A;
    const bool VERIFY = Policy<R>::VERIFY;
    const int T = TPT_THREADS, S = TPT_SLOTS, SPT = AUV_TPT_SPT;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ unsigned long long s_z[S];
    __shared__ long long s_q[S];
    __shared__ uint32_t s_ctr[S];
    __shared__ int s_nnodes[S], s_nchunks[S], s_it[S], s_status[S], s_nwp[S], s_nprims[S],
        s_active[S], s_parent[S], s_nexp[S], s_order[S], s_hist[2][64];
    __shared__ R s_bc0[S];
    // which time bins of each tree are non-empty (<= 128 bins): the rejection loop of the parent pick probes bins until
    // it finds one (rrt_dubins.py:123-125); testing a bit in shared memory instead of reading count[bin] from the tree's
    // workspace takes a dependent global load (and a 32-byte sector) off every probe
    __shared__ unsigned s_nonempty[S][4];
    const bool bin_bits = P.nb + 2 <= 128;
    EnvView<R> env;
    if (stage_mode == 0) { env.bind(blob, blob); env.bind_grid(blob, blob); }
    else {
        uint64_t *bar = (uint64_t *)smem;
        stage_env_tma(smem + 16, blob, stage_mode == 2 ? total_bytes : hot_bytes, bar);
        env.bind(smem + 16, stage_mode == 2 ? smem + 16 : blob);
        env.bind_grid(blob, smem + 16);
        if (FAST) env.assume_hot_shared(stage_mode == 2);
    }
    __shared__ EnvView<R> s_env;                 // for the out-of-line slow paths
    if (threadIdx.x == 0) { s_env = env; s_env.shared_self = &s_env; }
    env.shared_self = &s_env;
    const SteerParams<R> sp = P.sp;
    const int tid = threadIdx.x;
    unsigned char *block_ws = ws + (size_t)blockIdx.x * S * L.slot_bytes;
    for (int i = tid; i < S; i += T) { s_active[i] = 0; s_q[i] = -1; s_nexp[i] = -2; s_order[i] = i; }
    if (tid < 64) { s_hist[0][tid] = 0; s_hist[1][tid] = 0; }
    int trip = 0;
    bool queue_empty = false;
    const int guard_max = 64 * P.I + 1024;
    __syncthreads();

    for (;;) {
        // this trip's slots of the thread: position tid of group w, then of group 2T/32 - 1 - w (read before anyone rewrites s_order)
        const int slot0 = s_order[tid], slot1 = SPT == 2 ? s_order[(2 * (T / 32) - 1 - (tid >> 5)) * 32 + (tid & 31)] : 0;
        int key0 = 63, key1 = 63, any_active = 0;
#pragma unroll 1
        for (int j = 0; j < SPT; j++) {
        // ============ phase B: the thread runs the edge of its j-th slot ===============================
        const int slot = j == 0 ? slot0 : slot1;
        unsigned char *base = block_ws + (size_t)slot * L.slot_bytes;
        NodeRow<R> *nodes = (NodeRow<R> *)(base + L.nodes);
        int *pool = (int *)(base + L.pool), *next = (int *)(base + L.next);
        int4 *bins = (int4 *)(base + L.bins);
        TptHdr<R> *hdr = (TptHdr<R> *)(base + L.hdr);
        const int n_exp = s_nexp[slot];
        if (s_active[slot] && n_exp != -2) {
            const long long q = s_q[slot];
            int status = s_status[slot];
            int it = s_it[slot];
            if (!status && n_exp >= 0) {
                SerialStream<R> rng;
                rng.wa = (uint32_t)s_z[slot]; rng.wb = (uint32_t)(s_z[slot] >> 32); rng.ctr = s_ctr[slot];
                const int parent = s_parent[slot];
                // ---- steer (:237-295) with check_collision (:530-549) and the per-waypoint cost folded in
                const NodeRow<R> pr = nodes[parent];
                const uint32_t ctr0 = rng.ctr - 1;                 // position of the n_expand draw
                ArcEdge<R> ed;
                CircTable ct; ct.pair = nullptr; ct.npair = 0; ct.ox = ct.oy = ct.ccmax = 0.f; ct.rmax1 = 1.f; ct.buf2 = false;
                ct.hpair = nullptr; ct.nhpair = 0; ct.hccmax = 0.f; ct.epair = nullptr; ct.nepair = 0; ct.escale = 0.f; ct.eoff = 0.f;
                arc_edge_begin<R, false, FAST>(env, ct, ed, pr.x, pr.y, pr.th, pr.t, pr.len, pr.self_s2, pr.self_hab);
                for (int k = 0; k < n_exp; k++)
                    if (!arc_edge_step<R, true, true, false, FAST>(env, ct, sp, P.w3, rng, ed)) break;
                status = ed.status;
                const R x = ed.x, y = ed.y, th = ed.th, t = ed.t, len = ed.len;
                const int nwp = ed.nwp;
                const bool bad = ed.bad, moved = ed.moved, degenerate = ed.degenerate, last_is_wp = ed.last_is_wp;
                const R acc_s2 = ed.s2; const uint32_t acc_cnt = ed.cnt; const unsigned long long acc_mask = ed.mask;
                R self_s2 = ed.self_s2; int self_hab = ed.self_hab;
                if (!status) {
                    const bool safe = !(bad || degenerate);
                    s_nwp[slot] += nwp; s_nprims[slot] += n_exp;
                    if (P.trace) {
                        size_t r = (size_t)q * P.I + it;
                        tr.parent[r] = parent; tr.safe[r] = safe ? 1 : 0; tr.nwp[r] = nwp; tr.upos[r] = hdr->upos;
                        R *lf = (R *)tr.leaf + 5 * r;
                        lf[0] = x; lf[1] = y; lf[2] = th; lf[3] = t; lf[4] = len;
                    }
                    if (safe) {
                        if (moved && !last_is_wp) {     // the leaf state is not one of the waypoints: evaluate it
                            Contrib c = point_contrib<R>(env, x, y, t, 0xffffffffu, env.H, env.classify(x, y));
                            self_s2 = (c.bin >= 0 && c.cell >= 0) ? A::mul(P.w3, env.probs[(size_t)c.bin * env.C + c.cell]) : (R)0;
                            self_hab = c.bin >= 0 ? c.hab : -1;
                        }
                        const int id = s_nnodes[slot]++;                                // :144-145
                        NodeRow<R> nr;
                        nr.x = x; nr.y = y; nr.th = th; nr.t = t; nr.len = len; nr.ctr = ctr0; nr.parent = parent; nr.born = it;
                        nr.s2 = A::add(A::add(pr.s2, pr.self_s2), acc_s2);
                        nr.cnt = pr.cnt + (pr.self_hab >= 0 ? 1u : 0u) + acc_cnt;
                        nr.mask = pr.mask | (pr.self_hab >= 0 ? (1ull << pr.self_hab) : 0ull) | acc_mask;
                        nr.self_s2 = self_s2; nr.self_hab = self_hab;
                        nodes[id] = nr;
                        // ---- time-bin insert                                           :147-151
                        R fd = floordiv_pos<R>(t, P.bin_interval), fidx = fd + (R)1, curr_bin = A::mul(fidx, P.bin_interval);
                        int bidx = -1; bool reset = false;
                        if (P.mode == 2) { }                     // `if traj_time_stamp:` -- mode 2 keeps no bins
                        else if (curr_bin > P.max_traj) { if (fidx >= (R)1 && fidx <= (R)P.nb) { bidx = (int)fidx; reset = true; } }
                        else { if (fidx >= (R)1 && fidx <= (R)P.nb) bidx = (int)fidx; else status = AUVRRT_ST_KEY_ERROR; }
                        if (bidx >= 0) {
                            int4 bm = bins[bidx];                      // x: count, y: head chunk, z: tail chunk
                            const int c_old = bm.x;
                            const bool reuse_head = reset && c_old > 0;
                            const int c = reset ? 0 : c_old;
                            if (reuse_head) bm.z = bm.y;
                            if ((c & 31) == 0 && !reuse_head) {
                                const int nc = s_nchunks[slot]++;
                                next[nc] = -1;
                                if (c == 0) bm.y = nc; else next[bm.z] = nc;
                                bm.z = nc;
                            }
                            pool[bm.z * 32 + (c & 31)] = id;
                            bm.x = c + 1;
                            bins[bidx] = bm;
                            if (bin_bits) s_nonempty[slot][bidx >> 5] |= 1u << (bidx & 31);
                        }
                        if (!status && t >= P.horizon) {                                // :158-171
                            const uint32_t cnt = nr.cnt + (self_hab >= 0 ? 1u : 0u);
                            const unsigned long long mk = nr.mask | (self_hab >= 0 ? (1ull << self_hab) : 0ull);
                            R c1 = A::mul(P.w2, (R)cnt), c2 = A::add(nr.s2, self_s2), c0 = 0;
                            if (t > (R)0) { c1 = A::div(c1, t); c2 = A::div(c2, t); }
                            if (env.H != 0) c0 = A::div(A::mul(P.w1, (R)__popcll(mk)), (R)env.H);
                            const R total = py_sum3p<R>(c0, c1, c2);
                            hdr->ncost++;
                            if (total < s_bc0[slot]) {
                                s_bc0[slot] = total; hdr->bc1 = c0; hdr->bc2 = c1; hdr->bc3 = c2;
                                hdr->bestnode = id; hdr->bestiter = it; hdr->blen = len; hdr->bt = t;
                            }
                        }
                    }
                    it++;
                    s_it[slot] = it;
                    s_z[slot] = (unsigned long long)rng.wa | ((unsigned long long)rng.wb << 32); s_ctr[slot] = rng.ctr;
                    if (P.trace) hdr->upos = rng.ctr;
                }
            }
            // ---- query finished (budget spent, or an error): chain + record, free the slot
            if (status || it >= P.I || n_exp == -1) {
                const int best_node = hdr->bestnode;
                if (status == AUVRRT_ST_OK && best_node < 0) status = AUVRRT_ST_NO_PATH;
                int depth = 0;
                if (best_node >= 0) for (int n = best_node; nodes[n].parent >= 0; n = nodes[n].parent) depth++;
                if (chain_out) {
                    uint32_t *chain = chain_out + (size_t)q * P.chain_cap;
                    if (depth > P.chain_cap && status == AUVRRT_ST_OK) status = AUVRRT_ST_OVERFLOW;
                    int n = best_node;
                    for (int k = depth - 1; k >= 0; k--) { if (k < P.chain_cap) chain[k] = nodes[n].ctr; n = nodes[n].parent; }
                    for (int k = depth; k < P.chain_cap; k++) chain[k] = 0u;
                }
                auvrrt_plan_record_t rec;
                rec.status = status; rec.n_nodes = s_nnodes[slot]; rec.best_node = best_node; rec.best_iter = hdr->bestiter;
                rec.depth = depth; rec.n_path = 0; rec.n_cost_evals = hdr->ncost; rec.n_waypoints = s_nwp[slot];
                rec.n_uniforms = (long long)s_ctr[slot]; rec.n_primitives = (long long)s_nprims[slot];
                rec.cost[0] = best_node >= 0 ? (double)s_bc0[slot] : 0.0; rec.cost[1] = (double)hdr->bc1;
                rec.cost[2] = (double)hdr->bc2; rec.cost[3] = (double)hdr->bc3;
                rec.path_length = (double)hdr->blen; rec.t_leaf = (double)hdr->bt;
                records[q] = rec;
                s_active[slot] = 0;
            }
        }

        // ============ phase A, same thread, same tree: refill the slot, pick the next parent and draw
        // n_expand while the tree's rows and bins are still in this SM's L1 ============================
        {
            if (!s_active[slot] && !queue_empty) {
                const long long q = (long long)atomicAdd(qcounter, 1ull);
                if (q >= Q) queue_empty = true;
                else {
                    // ---- init                                                           rrt_dubins.py:105-114
                    for (int b = 0; b < P.nb + 2; b++) bins[b] = make_int4(0, 0, 0, 0);
                    NodeRow<R> r0;
                    r0.x = starts[5 * q]; r0.y = starts[5 * q + 1]; r0.th = starts[5 * q + 2]; r0.t = starts[5 * q + 3];
                    r0.len = starts[5 * q + 4]; r0.s2 = (R)0; r0.ctr = 0; r0.parent = -1; r0.cnt = 0; r0.mask = 0ull; r0.born = 0;
                    Contrib c = point_contrib<R>(env, r0.x, r0.y, r0.t, 0xffffffffu, env.H, env.classify(r0.x, r0.y));
                    r0.self_s2 = (c.bin >= 0 && c.cell >= 0) ? A::mul(P.w3, env.probs[(size_t)c.bin * env.C + c.cell]) : (R)0;
                    r0.self_hab = c.bin >= 0 ? c.hab : -1;
                    nodes[0] = r0;
                    bins[1] = make_int4(1, 0, 0, 0); pool[0] = 0; next[0] = -1;
                    s_nonempty[slot][0] = 2u; s_nonempty[slot][1] = s_nonempty[slot][2] = s_nonempty[slot][3] = 0u;     // bin 1 holds `initial`
                    s_z[slot] = stream_key(seeds[q]); s_ctr[slot] = 0; s_q[slot] = q; s_nprims[slot] = 0;
                    s_nnodes[slot] = 1; s_nchunks[slot] = 1; s_it[slot] = 0; s_status[slot] = AUVRRT_ST_OK;
                    s_nwp[slot] = 0; s_bc0[slot] = A::inf();
                    { TptHdr<R> h0; h0.bestnode = -1; h0.bestiter = -1; h0.ncost = 0; h0.guard = 0; h0.upos = 0; h0.pad_ = 0;
                      h0.bc1 = 0; h0.bc2 = 0; h0.bc3 = 0; h0.blen = 0; h0.bt = 0; *hdr = h0; }
                    s_active[slot] = 1;
                }
            }
            int key = 63;                         // inactive trees and skipped trips sort last
            if (s_active[slot]) {
                SerialStream<R> rng;
                rng.wa = (uint32_t)s_z[slot]; rng.wb = (uint32_t)(s_z[slot] >> 32); rng.ctr = s_ctr[slot];
                int parent = -1, status = AUVRRT_ST_OK;
                bool skip = false;
                if (P.mode == 0) {                                                      // :122-127
                    int rb = 0, cn = 0, ch = 0;
                    for (;;) {
                        rb = (int)uniform_ab<R>((R)1, (R)(P.nb + 1), rng.next());
                        if (rb > P.nb || rb < 1) { status = AUVRRT_ST_KEY_ERROR; break; }
                        if (bin_bits && !((s_nonempty[slot][rb >> 5] >> (rb & 31)) & 1u)) continue;      // empty: draw again
                        const int4 bm = bins[rb];
                        cn = bm.x; ch = bm.y;
                        if (cn > 0) break;
                    }
                    if (!status) {
                        int idx = (int)uniform_ab<R>((R)0, (R)cn, rng.next());
                        if (idx >= cn) status = AUVRRT_ST_KEY_ERROR;
                        else {
                            for (int hop = idx >> 5; hop > 0; hop--) ch = next[ch];
                            parent = pool[ch * 32 + (idx & 31)];
                        }
                    }
                } else if (P.mode == 2) {                                               // :129-132, :515-528
                    const R ran_time = uniform_ab<R>((R)0, P.ran_time_max, rng.next());
                    parent = closest_mps_time<R>(nodes, s_nnodes[slot], ran_time, P.plan_dt);
                    if (nodes[parent].t > P.max_traj) skip = true;
                } else {                                                                // :136-139, :505-513
                    R rx = uniform_ab<R>(env.minx, env.maxx, rng.next());
                    R ry = uniform_ab<R>(env.miny, env.maxy, rng.next());
                    rng.skip(2);                   // theta and size are drawn and never used
                    R bq = A::inf(), bs = A::inf();
                    int bi = 0;
                    const int n_nodes = s_nnodes[slot];
                    for (int i = 0; i < n_nodes; i++) {
                        R qq = A::sq2(A::sub(rx, nodes[i].x), A::sub(ry, nodes[i].y));
                        if (qq < bq) {
                            if (VERIFY) { R s = A::sqrt(qq); if (s < bs) { bs = s; bi = i; } }
                            else bi = i;
                            bq = qq;
                        }
                    }
                    parent = bi;
                    if (nodes[parent].t > P.max_traj) skip = true;                      // `continue`: no steer call
                }
                int n_exp = 0;
                if (!status && !skip) {
                    // the edge's stream position = position of its n_expand draw
                    n_exp = (int)A::floor(uniform_ab<R>((R)0, sp.freq, rng.next()));     // :259-260
                    key = n_exp < 62 ? n_exp : 62;
                }
                // the thread that runs this tree's edge after the sort (any thread of this CTA) finds the parent's row in L1
                if (parent >= 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(&nodes[parent]));
                s_z[slot] = (unsigned long long)rng.wa | ((unsigned long long)rng.wb << 32); s_ctr[slot] = rng.ctr; s_parent[slot] = parent; s_nexp[slot] = n_exp;
                if (status) { s_status[slot] = status; key = 62; s_nexp[slot] = -1; }    // phase B finalises it
                if (skip) {
                    s_nexp[slot] = -2;
                    if (++hdr->guard >= guard_max) { key = 62; s_nexp[slot] = -1; }
                }
            }
            if (j == 0) key0 = key; else key1 = key;
            any_active |= s_active[slot];
        }
        }   // j
        // ============================ counting sort of the slots by n_expand ======================
        // Two barriers per trip: the histogram alternates between two buffers (the idle one is cleared while this one is
        // read), and every warp scans the 64 buckets for itself in registers instead of waiting for one warp to do it.
        int *hist = s_hist[trip & 1];
        const int rank0 = atomicAdd(&hist[key0], 1), rank1 = SPT == 2 ? atomicAdd(&hist[key1], 1) : 0;
        __syncthreads();                          // histogram complete; every thread is past this trip's edges
        {
            const int lane = tid & 31;
            const int a0 = hist[2 * lane], a1 = hist[2 * lane + 1];
            int v = a0 + a1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) v += o; }
            const int e0 = v - a0 - a1, e1 = v - a1;            // exclusive offsets of buckets 2 lane and 2 lane + 1
            const int b0e = __shfl_sync(0xffffffffu, e0, key0 >> 1), b0o = __shfl_sync(0xffffffffu, e1, key0 >> 1);
            s_order[((key0 & 1) ? b0o : b0e) + rank0] = slot0;
            if (SPT == 2) {
                const int b1e = __shfl_sync(0xffffffffu, e0, key1 >> 1), b1o = __shfl_sync(0xffffffffu, e1, key1 >> 1);
                s_order[((key1 & 1) ? b1o : b1e) + rank1] = slot1;
            }
        }
        if (tid < 64) s_hist[(trip + 1) & 1][tid] = 0;
        trip++;
        if (__syncthreads_count(any_active) == 0) break;      // also publishes s_order and the cleared histogram
    }
}

template <typename R>
int launch_plan_tpt(const auvrrt_env *env, const R *starts, const uint64_t *seeds, int64_t Q,
                    const auvrrt_plan_params_t *p, void *workspace, int64_t workspace_bytes,
                    auvrrt_plan_record_t *records, uint32_t *chain, const auvrrt_plan_trace_t *trace,
                    cudaStream_t s, int64_t *need_bytes) {
    PlanP<R> P;
    int rc = make_planp<R>(env, p, &P);
    if (rc) return rc;
    EnvBlob<R> b = env_blob<R>(env);
    // only the hot part of the world model is staged: the per-tree state of 256 trees already takes
    // ~27 KB of shared memory per CTA and 4 CTAs per SM must fit
    int budget = 24 * 1024, sm = 16, mode = 0;
    if (const char *ev = getenv("AUVRRT_TPT_STAGE_KB")) budget = atoi(ev) * 1024;
    if (b.total_bytes + 16 <= budget) { sm = b.total_bytes + 16; mode = 2; }
    else if (b.hot_bytes + 16 <= budget) { sm = b.hot_bytes + 16; mode = 1; }
    const EnvHeader &hd = sizeof(R) == 4 ? env->h32 : env->h64;
    const bool fast = sizeof(R) == 4 && mode >= 1 && hd.gnx > 0 && hd.bins_uniform && hd.nxb > 0 && hd.H <= 32;
    auto kern = fast ? k_plan_tpt<R, true> : k_plan_tpt<R, false>;
    AUV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
    int per_sm = 0, nsm = 0, dev = 0;
    AUV_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TPT_THREADS, sm));
    if (per_sm < 1) return set_err(AUVRRT_ERR_CUDA, "plan_tpt: kernel does not fit on an SM");
    AUV_CUDA(cudaGetDevice(&dev));
    AUV_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    int grid = nsm * per_sm;
    TptLayout L = make_tpt_layout<R>(P.cap, P.nb, P.nchunks);
    // the workspace is sized for the full machine unless the batch (Q > 0) is smaller
    if (Q > 0) {
        int64_t blocks = (Q + TPT_SLOTS - 1) / TPT_SLOTS;
        if (blocks < grid) grid = (int)blocks;
    }
    int64_t need = 256 + (int64_t)grid * TPT_SLOTS * (int64_t)L.slot_bytes;
    if (need_bytes) { *need_bytes = need; return AUVRRT_OK; }
    if (Q <= 0) return AUVRRT_OK;
    if (workspace_bytes < need) return set_err(AUVRRT_ERR_ARG, "plan_tpt: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)need);
    if (P.trace && !trace) return set_err(AUVRRT_ERR_ARG, "plan_tpt: trace requested without trace buffers");
    AUV_CUDA(cudaMemsetAsync(workspace, 0, 256, s));
    auvrrt_plan_trace_t tr;
    if (trace) tr = *trace; else { tr.parent = nullptr; tr.safe = nullptr; tr.nwp = nullptr; tr.leaf = nullptr; tr.upos = nullptr; }
    kern<<<grid, TPT_THREADS, sm, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode, starts, seeds, (long long)Q, P, L,
                                                (unsigned char *)workspace + 256, (unsigned long long *)workspace, records,
                                                chain, tr);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
// ---- re-create paths of thread-per-tree plans from (start, seed, chain of stream positions) ----------------------
// One thread per query, with the edge evaluator k_plan_tpt grew the tree with (arc_edge_step): in fp32 the warp
// evaluator of plan.cu sums the same primitives in another order, so its waypoints, and from the first waypoint count
// that differs on the whole path, would not be the plan that was scored.  Output row m, pick and depth as k_materialize.
// 128 registers, as k_materialize: under the default heuristic both precisions spilled (fp64 148 bytes).
template <typename R>
__global__ void __maxnreg__(128)
k_materialize_tpt(const unsigned char *blob, const R *starts, const uint64_t *seeds, const uint32_t *chain,
                  const int32_t *depth, int depth_stride, long long Q, const int64_t *pick, long long M, PlanP<R> P,
                  R *path_out, int32_t *n_path_out) {
    EnvView<R> env;
    env.bind(blob, blob);
    env.bind_grid(blob, blob);
    CircTable ct; ct.pair = nullptr; ct.npair = 0; ct.ox = ct.oy = ct.ccmax = 0.f; ct.rmax1 = 1.f; ct.buf2 = false;
    ct.hpair = nullptr; ct.nhpair = 0; ct.hccmax = 0.f; ct.epair = nullptr; ct.nepair = 0; ct.escale = 0.f; ct.eoff = 0.f;
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < M; m += gridDim.x * blockDim.x) {   // (M, Q < 2^31)
        const long long pq = pick ? (long long)pick[m] : m;
        if (pq < 0 || pq >= Q) { n_path_out[m] = pq == -1 ? 0 : -1; continue; }
        const int q = (int)pq;
        const int d = depth[(size_t)q * depth_stride];
        if (d < 0 || d > P.chain_cap) { n_path_out[m] = -1; continue; }
        const uint64_t key = stream_key(seeds[q]);
        R x = starts[5 * q], y = starts[5 * q + 1], th = starts[5 * q + 2], t = starts[5 * q + 3], len = starts[5 * q + 4];
        const uint32_t *ch = chain + (size_t)q * P.chain_cap;
        R *rows = path_out + (size_t)m * P.path_cap * 6;
        int n_path = 0;
        auto put = [&](R vx, R vy, R vth, R vv, R vtt, R vlen) {
            if (n_path < P.path_cap) {
                R *w = rows + 6 * (size_t)n_path;
                w[0] = vx; w[1] = vy; w[2] = vth; w[3] = vv; w[4] = vtt; w[5] = vlen;
            }
            n_path++;
        };
        for (int e = 0; e < d; e++) {
            put(x, y, th, (R)0, t, len);
            SerialStream<R> rng;
            rng.seek(key, ch[e]);           // the edge's n_expand draw comes next
            const int n_exp = (int)Policy<R>::A::floor(uniform_ab<R>((R)0, P.sp.freq, rng.next()));
            ArcEdge<R> ed;
            arc_edge_begin<R, false>(env, ct, ed, x, y, th, t, len, (R)0, -1);
            for (int k = 0; k < n_exp; k++) {
                const int nwp = ed.nwp;
                if (!arc_edge_step<R, false, false, false>(env, ct, P.sp, P.w3, rng, ed)) break;
                if (ed.nwp > nwp) put(ed.x, ed.y, ed.th, ed.vt, ed.t, ed.len);
            }
            x = ed.x; y = ed.y; th = ed.th; t = ed.t; len = ed.len;
        }
        put(x, y, th, (R)0, t, len);
        n_path_out[m] = n_path;
    }
}

template <typename R>
int launch_materialize_tpt(const auvrrt_env *env, const R *starts, const uint64_t *seeds, const uint32_t *chain,
                           const int32_t *depth, int depth_stride, int64_t Q, const int64_t *pick, int64_t M,
                           const PlanP<R> &P, R *path, int32_t *n_path, cudaStream_t s) {
    int64_t blocks = (M + 127) / 128;
    if (blocks > AUV_SMS * 8) blocks = AUV_SMS * 8;
    k_materialize_tpt<R><<<(unsigned)blocks, 128, 0, s>>>(env_blob<R>(env).blob, starts, seeds, chain, depth, depth_stride,
                                                          (long long)Q, pick, (long long)M, P, path, n_path);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_materialize_tpt<float>(const auvrrt_env *, const float *, const uint64_t *, const uint32_t *, const int32_t *,
                                           int, int64_t, const int64_t *, int64_t, const PlanP<float> &, float *, int32_t *,
                                           cudaStream_t);
template int launch_materialize_tpt<double>(const auvrrt_env *, const double *, const uint64_t *, const uint32_t *, const int32_t *,
                                            int, int64_t, const int64_t *, int64_t, const PlanP<double> &, double *, int32_t *,
                                            cudaStream_t);

template int launch_plan_tpt<float>(const auvrrt_env *, const float *, const uint64_t *, int64_t, const auvrrt_plan_params_t *,
                                    void *, int64_t, auvrrt_plan_record_t *, uint32_t *, const auvrrt_plan_trace_t *, cudaStream_t, int64_t *);
template int launch_plan_tpt<double>(const auvrrt_env *, const double *, const uint64_t *, int64_t, const auvrrt_plan_params_t *,
                                     void *, int64_t, auvrrt_plan_record_t *, uint32_t *, const auvrrt_plan_trace_t *, cudaStream_t, int64_t *);

}  // namespace auv
