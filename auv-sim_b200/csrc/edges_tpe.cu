// edges_tpe.cu -- the batched steer + collide + cost kernel, ONE CANDIDATE EDGE PER THREAD (sm_100a).
//
//   RRT.steer (random-arc rollout)   /root/reference/path_planning/rrt_dubins.py:252-295
//   RRT.check_collision              rrt_dubins.py:530-549
//   habitat_shark_cost_func, the per-waypoint loop   /root/reference/path_planning/cost.py:171-191
//
// Edge i = (parents[i], seeds[i]): the edge consumes the sample sequence of its seed from position 0
// (n_expand, then 2-3 uniforms per arc primitive, SURVEY.md appendix A).  A thread runs the reference's
// serial loop for its edge (edge_serial.cuh); the world model's hot part (circles, polygon, habitats,
// bins, cell index) and, when it fits, the probability table are staged in shared memory by one TMA
// bulk copy per CTA.
//
// Divergence control.  n_expand is uniform in [0, freq): 32 arbitrary edges in a warp would leave half
// the lanes idle in the primitive loop.  Each CTA therefore takes a batch of NT x AUV_TPE_EPT consecutive
// edges, (1) draws n_expand for all of them with coalesced loads, (2) counting-sorts the batch by
// n_expand in shared memory, (3) lets its warps pull groups of 32 edges of (nearly) equal n_expand off a
// shared counter, longest first.  Inputs and outputs stay in the caller's order.
#include <stdlib.h>
#include "launch.h"
#include "edge_serial.cuh"

namespace auv {

#ifndef AUV_TPE_EPT
#define AUV_TPE_EPT 8             // edges per thread per batch: batch = 8 x threads edges
#endif
#ifndef AUV_TPE_MINB
#define AUV_TPE_MINB 4
#endif
// Queue the waypoints that need the general collision / habitat tests (2 % on the Catalina map) per warp and resolve them
// after the warp's 32 edges (edge_serial.cuh, SlowQ).  Measured on B200, Catalina map, 3.4e7 edges, cost on: off 6.8e9
// edges/s; on, push inline 6.2e9; on, push out of line 5.9e9.  The slow-path share of the executed instructions does
// fall from 14.7 % to 5.5 % and the active lanes rise from 22.3 to 24.7, but at 64 registers the extra live state makes
// the compiler duplicate and spill in the hot loop (+14 % instructions on the main path).  Kept for larger register budgets.
#ifndef AUV_TPE_DEFER
#define AUV_TPE_DEFER 0
#endif
#define AUV_TPE_BUCKETS 64
#define AUV_TPE_QBYTES (AUV_SLOWQ_CAP * 16 + 16 + 3 * 128)      // SlowQ of one warp
#define AUV_TPE_MAXPAIRS 128      // all-pairs circle table in shared memory: 128 quads = up to 512 circles (6 KB)

// STAGE: 1 = the hot part of the world model is in shared memory, 2 = the probability table too (always staged:
// the launcher falls back to the warp-per-edge kernel when even the hot part does not fit)
// NT x MINB: threads per CTA x resident CTAs per SM the register allocation targets (256 x 4, 512 x 2 and 1024 x 1 are all
// 32 warps per SM at 64 registers; fewer, larger CTAs share one staged copy of the world model)
// GRIDS: plane 0 of the classification grid is staged behind the world model (one more bulk copy) and read with LDS
template <typename R, bool COST, bool ALLPAIRS, int STAGE, bool FASTENV, int NT, int MINB, bool GRIDS>
__global__ void __launch_bounds__(NT, MINB)
k_edges_arc_tpe(const unsigned char *blob, int hot_bytes, int total_bytes, const R *__restrict__ parents,
                const uint64_t *__restrict__ seeds, long long n, SteerParams<R> sp, R w3, uint8_t *__restrict__ safe,
                int32_t *__restrict__ counts, R *__restrict__ leaf, R *__restrict__ cost_out) {
    typedef typename Policy<R>::A A;
    const int T = NT, BATCH = NT * AUV_TPE_EPT;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ unsigned short s_order[BATCH];
    __shared__ int s_hist[AUV_TPE_BUCKETS];
    __shared__ int s_next;
    __shared__ CircQuad s_pairs[(ALLPAIRS && sizeof(R) == 4) ? AUV_TPE_MAXPAIRS : 1];
    __shared__ CircPair s_hpairs[(ALLPAIRS && sizeof(R) == 4) ? AUV_AP_MAXH : 1], s_epairs[(ALLPAIRS && sizeof(R) == 4) ? AUV_AP_MAXE : 1];
    EnvView<R> env;
    unsigned char *q_base;
    {
        uint64_t *bar = (uint64_t *)smem;
        const int staged = STAGE == 2 ? total_bytes : hot_bytes;          // multiples of 16 (api.cu)
        if (GRIDS) {
            // world model + plane 0 of the grid: two regions, one barrier
            const EnvHeader *gh = (const EnvHeader *)blob;
            const int plane = (gh->gnx * gh->gny * 4 + 15) & ~15;          // (the blob holds three planes: rounding up stays inside)
            if (threadIdx.x == 0) mbar_init(bar, 1);
            __syncthreads();
            if (threadIdx.x == 0) {
                mbar_expect_tx(bar, (uint32_t)(staged + plane));
                for (int o = 0; o < staged; o += 65536) tma_bulk_g2s(smem + 16 + o, blob + o, (uint32_t)(staged - o < 65536 ? staged - o : 65536), bar);
                const unsigned char *gsrc = blob + gh->off_grid;
                for (int o = 0; o < plane; o += 65536) tma_bulk_g2s(smem + 16 + staged + o, gsrc + o, (uint32_t)(plane - o < 65536 ? plane - o : 65536), bar);
            }
            mbar_wait(bar, 0);
        } else stage_env_tma(smem + 16, blob, staged, bar);
        env.bind(smem + 16, STAGE == 2 ? smem + 16 : blob);
        env.bind_grid(blob, smem + 16);
        env.assume_hot_shared(STAGE == 2);
        if (GRIDS) { env.grid0s = (const unsigned *)(smem + 16 + staged); __builtin_assume(__isShared(env.grid0s)); }
        q_base = smem + 16 + staged + (GRIDS ? ((((const EnvHeader *)blob)->gnx * ((const EnvHeader *)blob)->gny * 4 + 15) & ~15) : 0);
    }
    // deferred slow cases (edge_serial.cuh, SlowQ): one queue per warp behind the staged data
    constexpr bool DEFER = AUV_TPE_DEFER && FASTENV && !ALLPAIRS && sizeof(R) == 4 && NT >= 512;     // (256 x 4: no room next to four staged probability tables)
    SlowQ sq; sq.base = nullptr;
    if (DEFER) {
        sq.base = q_base + (size_t)(threadIdx.x >> 5) * AUV_TPE_QBYTES;
        __builtin_assume(__isShared(sq.base));
        const int l = threadIdx.x & 31;
        sq.bad()[l] = 0u; sq.cnt()[l] = 0u; sq.mask()[l] = 0u;
        if (l == 0) *sq.n() = 0;
        __syncwarp();
    }
    __shared__ EnvView<R> s_env;                 // for the out-of-line slow paths
    if (threadIdx.x == 0) { s_env = env; s_env.shared_self = &s_env; }
    __syncthreads();
    env.shared_self = &s_env;
    CircTable ct; ct.pair = nullptr; ct.npair = 0; ct.ox = ct.oy = ct.ccmax = 0.f; ct.rmax1 = 1.f; ct.buf2 = false;
    ct.hpair = nullptr; ct.nhpair = 0; ct.hccmax = 0.f; ct.epair = nullptr; ct.nepair = 0; ct.escale = 0.f; ct.eoff = 0.f;
    if constexpr (ALLPAIRS && sizeof(R) == 4) {
        ct.ox = 0.5f * (float)(env.minx + env.maxx); ct.oy = 0.5f * (float)(env.miny + env.maxy);
        if (env.K > 0 && env.K <= 4 * AUV_TPE_MAXPAIRS) {
            circ_table_fill(s_pairs, env, ct.ox, ct.oy);
            ct.ccmax = circ_table_ccmax(env, ct.ox, ct.oy);
            ct.pair = s_pairs; ct.npair = (env.K + 3) >> 2;
            float rm = 0.f;
            for (int k = 0; k < env.K; k++) rm = fmaxf(rm, (float)env.creff[k]);
            ct.rmax1 = rm + 1.f;
            // two waypoints per pass over the table from 64 circles up (measured: Catalina's 27 circles 3.54e9 edges/s
            // without, 3.40e9 with; config 4's 500 circles 6.35e8 without, 7.9e8 with)
            ct.buf2 = ct.npair >= 16;
        }
        allpairs_tables_fill(s_hpairs, s_epairs, env, ct.ox, ct.oy);
        if (env.H > 0 && env.H <= 2 * AUV_AP_MAXH) {
            float m = 0.f;
            for (int h = 0; h < env.H; h++) { const float ax = env.hx[h] - ct.ox, ay = env.hy[h] - ct.oy; m = fmaxf(m, fmaf(ay, ay, ax * ax)); }
            ct.hpair = s_hpairs; ct.nhpair = (env.H + 1) >> 1; ct.hccmax = m;
        }
        if (env.convex != 0 && env.E >= 3 && env.E <= 2 * AUV_AP_MAXE) {
            float m = 0.f;                                  // largest edge coefficient: scale of the rounding error
            for (int i = 0; i < env.E; i++) {
                const int i1 = i + 1 == env.E ? 0 : i + 1;
                m = fmaxf(m, fmaxf(fabsf((float)(env.px[i1] - env.px[i])), fabsf((float)(env.py[i1] - env.py[i]))));
            }
            ct.epair = s_epairs; ct.nepair = (env.E + 1) >> 1;
            ct.escale = 1e-6f * m; ct.eoff = ct.escale * ((float)(env.maxx - env.minx) + (float)(env.maxy - env.miny));
        }
        __syncthreads();
    }
    const int tid = threadIdx.x, lane = tid & 31;
    const long long n_batches = (n + BATCH - 1) / BATCH;
    for (long long b = blockIdx.x; b < n_batches; b += gridDim.x) {
        const long long base = b * BATCH;
        const int cnt = (int)((n - base) < (long long)BATCH ? (n - base) : (long long)BATCH);
        // ---- (1) n_expand of every edge of the batch: floor(uniform(0, freq)) on stream position 0   :259-260
        if (tid < AUV_TPE_BUCKETS) s_hist[tid] = 0;
        if (tid == 0) s_next = 0;
        __syncthreads();
        unsigned char key[AUV_TPE_EPT];
        unsigned short rank[AUV_TPE_EPT];
#pragma unroll
        for (int e = 0; e < AUV_TPE_EPT; e++) {
            const int j = e * T + tid;
            key[e] = 255;
            if (j < cnt) {
                const uint64_t k64 = stream_key(seeds[base + j]);
                const int n_exp = (int)A::floor(uniform_ab<R>((R)0, sp.freq, Draw<R>::at(k64, 0u)));
                key[e] = (unsigned char)(n_exp < 0 ? 0 : (n_exp < AUV_TPE_BUCKETS - 1 ? n_exp : AUV_TPE_BUCKETS - 1));
                rank[e] = (unsigned short)atomicAdd(&s_hist[key[e]], 1);
            }
        }
        __syncthreads();
        // ---- (2) counting sort: exclusive scan of the 64 buckets by one warp, then scatter
        if (tid < 32) {
            const int a0 = s_hist[2 * tid], a1 = s_hist[2 * tid + 1];
            int v = a0 + a1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, v, d); if (tid >= d) v += o; }
            s_hist[2 * tid] = v - a0 - a1; s_hist[2 * tid + 1] = v - a1;
        }
        __syncthreads();
#pragma unroll
        for (int e = 0; e < AUV_TPE_EPT; e++)
            if (key[e] != 255) s_order[s_hist[key[e]] + rank[e]] = (unsigned short)(e * T + tid);
        __syncthreads();
        // ---- (3) warps pull groups of 32 edges of (nearly) equal n_expand, longest first
        for (;;) {
            int g = 0;
            if (lane == 0) g = atomicAdd(&s_next, 1);
            g = __shfl_sync(0xffffffffu, g, 0);
            const int pos = cnt - 1 - (g * 32 + lane);
            if (cnt - 1 - g * 32 < 0) break;
            long long i = -1;
            ArcEdge<R> ed;
            if (pos >= 0) {
                i = base + (long long)s_order[pos];
                const R *p = parents + 5 * i;
                const R px = p[0], py = p[1], pth = p[2], pt = p[3], plen = p[4];
                SerialStream<R> rng;
                rng.init(stream_key(seeds[i]));
                const int n_exp = (int)A::floor(uniform_ab<R>((R)0, sp.freq, rng.next()));
                arc_edge_begin<R, ALLPAIRS, FASTENV, GRIDS, DEFER>(env, ct, ed, px, py, pth, pt, plen, (R)0, -1, sq);
                for (int k = 0; k < n_exp; k++) {
                    if (!arc_edge_step<R, COST, false, ALLPAIRS, FASTENV, GRIDS, DEFER>(env, ct, sp, w3, rng, ed, sq)) break;
                    if constexpr (ALLPAIRS && sizeof(R) == 4 && AUV_AP_BUFFER) {
                        // the lanes that are here together run the circle loop together as soon as one of them holds two waypoints
                        if (__any_sync(__activemask(), ed.nbuf >= 2)) circles_flush2<R>(env, ct, ed);
                    }
                }
                if constexpr (ALLPAIRS && sizeof(R) == 4 && AUV_AP_BUFFER) circles_flush2<R>(env, ct, ed);
            }
            if (DEFER) {
                // the queued slow cases of these 32 edges, one per lane; then every lane folds its results in
                __syncwarp();
                if (*(volatile int *)sq.n() > 0) {
                    slowq_drain<R>(env, sq);
                    if (pos >= 0) { ed.bad = ed.bad || sq.bad()[lane] != 0u; ed.cnt += sq.cnt()[lane]; ed.mask |= (unsigned long long)sq.mask()[lane]; }
                    __syncwarp();
                    sq.bad()[lane] = 0u; sq.cnt()[lane] = 0u; sq.mask()[lane] = 0u;
                    if (lane == 0) *sq.n() = 0;
                    __syncwarp();
                }
            }
            if (pos >= 0) {
                safe[i] = (ed.status == 0 && !(ed.bad || ed.degenerate)) ? 1 : 0;
                if (counts) counts[i] = ed.nwp;
                if (leaf) { R *l = leaf + 5 * i; l[0] = ed.x; l[1] = ed.y; l[2] = ed.th; l[3] = ed.t; l[4] = ed.len; }
                if (COST) { R *c = cost_out + 3 * i; c[0] = ed.s2; c[1] = (R)ed.cnt; c[2] = (R)__popcll(ed.mask); }
            }
        }
        __syncthreads();        // s_order / s_hist / s_next are rewritten by the next batch
    }
}

typedef void (*tpe_kernel_f32)(const unsigned char *, int, int, const float *, const uint64_t *, long long, SteerParams<float>, float,
                               uint8_t *, int32_t *, float *, float *);
typedef void (*tpe_kernel_f64)(const unsigned char *, int, int, const double *, const uint64_t *, long long, SteerParams<double>, double,
                               uint8_t *, int32_t *, double *, double *);

// the fp32 instantiations: (threads x resident CTAs) in {256 x 4, 256 x 3, 512 x 2, 1024 x 1}; the grid plane in shared
// memory only for the grid-classified kernel on a map with all the lookup tables (FASTENV)
template <bool COST, bool ALLPAIRS>
static tpe_kernel_f32 pick_f32(bool fast, bool probs_too, int nt, int minb, bool grids) {
#define AUV_TPE_K(ST, F, NT_, MB, G) k_edges_arc_tpe<float, COST, ALLPAIRS, ST, F, NT_, MB, G>
#define AUV_TPE_ST(F, NT_, MB, G) (probs_too ? AUV_TPE_K(2, F, NT_, MB, G) : AUV_TPE_K(1, F, NT_, MB, G))
    if constexpr (!ALLPAIRS) {
        if (fast && grids) {
            if (nt == 1024) return AUV_TPE_ST(true, 1024, 1, true);
            if (nt == 512) return AUV_TPE_ST(true, 512, 2, true);
            return minb >= 4 ? AUV_TPE_ST(true, 256, 4, true) : AUV_TPE_ST(true, 256, 3, true);
        }
        if (fast) {
            if (nt == 1024) return AUV_TPE_ST(true, 1024, 1, false);
            if (nt == 512) return AUV_TPE_ST(true, 512, 2, false);
        }
    }
    if constexpr (ALLPAIRS) {
        // the all-pairs loops are unrolled four quads deep (48 registers of circle data in flight): 2 CTAs per SM = 128 registers
        if (minb <= 2) return fast ? AUV_TPE_ST(true, 256, 2, false) : AUV_TPE_ST(false, 256, 2, false);
    }
    if (minb >= 4) return fast ? AUV_TPE_ST(true, 256, 4, false) : AUV_TPE_ST(false, 256, 4, false);
    return fast ? AUV_TPE_ST(true, 256, 3, false) : AUV_TPE_ST(false, 256, 3, false);
#undef AUV_TPE_ST
#undef AUV_TPE_K
}

template <typename R, bool COST, bool ALLPAIRS>
static int launch_tpe_t(const auvrrt_env *env, const R *parents, const uint64_t *seeds, int64_t n, const double params[5],
                        double w3, uint8_t *safe, int32_t *counts, R *leaf, R *cost_out, cudaStream_t s) {
    EnvBlob<R> b = env_blob<R>(env);
    // FASTENV: equal contiguous time bins, x-bucket table and classification grid all present (any real map)
    const EnvHeader &hd = sizeof(R) == 4 ? env->h32 : env->h64;
    const bool fast = hd.gnx > 0 && (!COST || (hd.bins_uniform && hd.nxb > 0 && hd.H <= 32));
    // CTA shape: threads x resident CTAs per SM (fp32: 32 warps per SM at 64 registers, or 24 at 85 with 256 x 3)
    // fp32, measured on the Catalina map at 3.4e7 edges, cost on (profiles/r02_tpe_shapes.txt): 256 x 4: 5.5e9 edges/s,
    // 512 x 2: 6.3e9, 1024 x 1: 6.6e9, 1024 x 1 with the grid plane in shared memory: 6.8e9 -- one staged copy of the
    // world model per SM instead of four leaves the L1 to the grid and the outputs.  Small batches keep 256-thread CTAs
    // (a CTA works on 8 edges per thread at a time).
    int nt = 256, minb = sizeof(R) == 4 ? AUV_TPE_MINB : 1;
    bool grids = false;
    if (sizeof(R) == 4) {
        int nsm_ = 148, dev_ = 0;
        if (cudaGetDevice(&dev_) == cudaSuccess) cudaDeviceGetAttribute(&nsm_, cudaDevAttrMultiProcessorCount, dev_);
        if (n >= (int64_t)nsm_ * 1024 * AUV_TPE_EPT) { nt = 1024; grids = true; }
        if (const char *ev = getenv("AUVRRT_TPE_THREADS")) { const int v = atoi(ev); if (v == 256 || v == 512 || v == 1024) nt = v; }
        if (const char *ev = getenv("AUVRRT_TPE_MINB")) minb = atoi(ev);
        if (const char *ev = getenv("AUVRRT_TPE_GRIDS")) grids = atoi(ev) != 0;
        // (all pairs, measured at 256 x 2 / 3 / 4: Catalina 3.14 / 3.54 / 3.50e9 edges/s, config 4 6.37 / 6.35 / 6.16e8: 3 unless asked otherwise)
        const int minb256 = ALLPAIRS ? ((getenv("AUVRRT_TPE_MINB") && minb <= 2) ? 2 : ((getenv("AUVRRT_TPE_MINB") && minb >= 4) ? 4 : 3)) : (minb >= 4 ? 4 : 3);
        if (ALLPAIRS || !fast) { grids = false; nt = 256; }
        minb = nt == 512 ? 2 : (nt == 1024 ? 1 : minb256);
        // the grid plane must fit next to the hot part
        if (grids && ((hd.gnx * hd.gny * 4 + 15) & ~15) + b.hot_bytes + 16 > (int)((227 * 1024) / minb) - 2048 - (int)(2 * nt * AUV_TPE_EPT)) grids = false;
    }
    const int plane = grids ? ((hd.gnx * hd.gny * 4 + 15) & ~15) : 0;
    // shared memory per CTA: the hot part, + the probability table when the resident CTAs still fit, + the grid plane
    const int qbytes = (AUV_TPE_DEFER && sizeof(R) == 4 && fast && !ALLPAIRS && nt >= 512) ? (nt / 32) * AUV_TPE_QBYTES : 0;       // the warps' SlowQ
    const int per_cta_max = (int)((227 * 1024) / minb) - 1024 - (int)(2 * nt * AUV_TPE_EPT) - 1024;   // less the static arrays
    int budget = per_cta_max - plane - qbytes;
    if (const char *ev = getenv("AUVRRT_TPE_STAGE_KB")) budget = atoi(ev) * 1024;
    int sm = 16;
    const bool probs_too = COST && b.total_bytes + 16 <= budget;
    if (probs_too) sm = b.total_bytes + 16;
    else if (b.hot_bytes + 16 + plane <= 200 * 1024) sm = b.hot_bytes + 16;
    else return AUVRRT_ERR_UNSUPPORTED;          // the caller falls back to the warp-per-edge kernel
    sm += plane;
    sm += qbytes;
    void (*kern)(const unsigned char *, int, int, const R *, const uint64_t *, long long, SteerParams<R>, R, uint8_t *,
                 int32_t *, R *, R *);
    if constexpr (sizeof(R) == 4) {
        kern = pick_f32<COST, ALLPAIRS>(fast, probs_too, nt, minb, grids);
    } else {
        kern = fast ? (probs_too ? k_edges_arc_tpe<R, COST, ALLPAIRS, 2, true, 256, 1, false> : k_edges_arc_tpe<R, COST, ALLPAIRS, 1, true, 256, 1, false>)
                    : (probs_too ? k_edges_arc_tpe<R, COST, ALLPAIRS, 2, false, 256, 1, false> : k_edges_arc_tpe<R, COST, ALLPAIRS, 1, false, 256, 1, false>);
    }
    AUV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
    int per_sm = 0, nsm = 0, dev = 0;
    AUV_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nt, sm));
    if (per_sm < 1) return set_err(AUVRRT_ERR_CUDA, "edges_arc (thread per edge): kernel does not fit on an SM (smem %d)", sm);
    AUV_CUDA(cudaGetDevice(&dev));
    AUV_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    const int64_t batch = (int64_t)nt * AUV_TPE_EPT;
    int64_t blocks = (n + batch - 1) / batch;
    if (blocks > (int64_t)nsm * per_sm) blocks = (int64_t)nsm * per_sm;
    kern<<<(unsigned)blocks, nt, sm, s>>>(b.blob, b.hot_bytes, b.total_bytes, parents, seeds, (long long)n,
                                          make_steer_params<R>(params), (R)w3, safe, counts, leaf, cost_out);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}

template <typename R>
int launch_edges_arc_tpe(const auvrrt_env *env, const R *parents, const uint64_t *seeds, int64_t n, const double params[5],
                         uint8_t *safe, int32_t *counts, R *leaf, cudaStream_t s, double w3, R *cost_out, bool allpairs) {
    if (n <= 0) return AUVRRT_OK;
    if (cost_out)
        return allpairs ? launch_tpe_t<R, true, true>(env, parents, seeds, n, params, w3, safe, counts, leaf, cost_out, s)
                        : launch_tpe_t<R, true, false>(env, parents, seeds, n, params, w3, safe, counts, leaf, cost_out, s);
    return allpairs ? launch_tpe_t<R, false, true>(env, parents, seeds, n, params, w3, safe, counts, leaf, cost_out, s)
                    : launch_tpe_t<R, false, false>(env, parents, seeds, n, params, w3, safe, counts, leaf, cost_out, s);
}
template int launch_edges_arc_tpe<float>(const auvrrt_env *, const float *, const uint64_t *, int64_t, const double[5], uint8_t *,
                                         int32_t *, float *, cudaStream_t, double, float *, bool);
template int launch_edges_arc_tpe<double>(const auvrrt_env *, const double *, const uint64_t *, int64_t, const double[5],
                                          uint8_t *, int32_t *, double *, cudaStream_t, double, double *, bool);

}  // namespace auv
