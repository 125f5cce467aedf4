// kernels.cu -- batched kernels over independent edges / paths / queries (sm_100a).
//   steer_arc, steer_dubins, collide, cost, fused edges (config-4 micro-benchmark), nearest node,
//   FP32 calibration.  The planner itself is in plan.cu.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include "launch.h"
#include "dubins.cuh"
#include "edge_serial.cuh"

namespace auv {

thread_local char g_err[512] = "";
long long g_launches = 0;
int set_err(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

template <> SteerParams<float> make_steer_params<float>(const double p[5]) {
    SteerParams<float> s;
    s.d2e = (float)p[0]; s.dmax = (float)p[1]; s.neg_dmax = (float)(-p[1]); s.freq = (float)p[2];
    s.min_dist = (float)p[3]; s.two_vel = (float)(2.0 * p[4]);
    { volatile float w = s.d2e - 0.f, o = 0.f - w; s.o_dist = o; }
    { volatile float w = s.dmax - s.neg_dmax, o = s.neg_dmax - w; s.w_diff = w; s.o_diff = o; }
    { volatile float w = s.two_vel - 0.f, o = 0.f - w; s.o_vel = o; }
    return s;
}
template <> SteerParams<double> make_steer_params<double>(const double p[5]) {
    SteerParams<double> s;
    s.d2e = p[0]; s.dmax = p[1]; s.neg_dmax = -p[1]; s.freq = p[2]; s.min_dist = p[3]; s.two_vel = 2.0 * p[4];
    s.w_diff = s.dmax - s.neg_dmax; s.o_dist = -s.d2e; s.o_diff = s.neg_dmax - s.w_diff; s.o_vel = -s.two_vel;    // (fp32 build only)
    return s;
}

// ------------------------------------------------------------------ env staging helper
// dynamic shared memory: [0,16) mbarrier, [16, 16+bytes) env copy
template <typename R>
__device__ __forceinline__ EnvView<R> load_env(unsigned char *smem, const unsigned char *blob, int hot_bytes,
                                               int total_bytes, int stage_mode) {
    EnvView<R> v;
    if (stage_mode == 0) { v.bind(blob, blob); v.bind_grid(blob, blob); return v; }
    uint64_t *bar = (uint64_t *)smem;
    unsigned char *dst = smem + 16;
    stage_env_tma(dst, blob, stage_mode == 2 ? total_bytes : hot_bytes, bar);
    v.bind(dst, stage_mode == 2 ? dst : blob);
    v.bind_grid(blob, dst);
    return v;
}
static inline int env_stage_mode(int hot, int total, int budget, int *smem_bytes) {
    if (total + 16 <= budget) { *smem_bytes = total + 16; return 2; }
    if (hot + 16 <= budget) { *smem_bytes = hot + 16; return 1; }
    *smem_bytes = 16; return 0;
}

// ------------------------------------------------------------------ conversions
template <typename R> __global__ void k_convert(const double *src, R *dst, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (R)src[i];
}
template <typename R> __global__ void k_convert_back(const R *src, double *dst, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (double)src[i];
}
template <typename R> int launch_convert(const double *src, R *dst, int64_t n, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    k_convert<R><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, n);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template <typename R> int launch_convert_back(const R *src, double *dst, int64_t n, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    k_convert_back<R><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, n);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_convert<float>(const double *, float *, int64_t, cudaStream_t);
template int launch_convert<double>(const double *, double *, int64_t, cudaStream_t);
template int launch_convert_back<float>(const float *, double *, int64_t, cudaStream_t);
template int launch_convert_back<double>(const double *, double *, int64_t, cudaStream_t);

// ------------------------------------------------------------------ RRT.steer on explicit streams
template <typename R, int G>
__global__ void __launch_bounds__(128) k_steer_arc(const R *parents, int64_t n, const double *u, const int64_t *uoff,
                                                   SteerParams<R> sp, R *leaf, int32_t *counts, R *wp, int wp_cap,
                                                   int32_t *used, int32_t *status) {
    __shared__ GroupScratch<R, G> scratch[128 / G];
    Grp<G> g;
    GroupScratch<R, G> &sc = scratch[threadIdx.x / G];
    EnvView<R> env;
    env.K = env.E = env.H = env.T = env.C = env.NB = env.NP = env.convex = 0;
    env.gnx = env.gny = env.bins_uniform = env.nxb = 0;
    const int64_t groups = (int64_t)gridDim.x * (128 / G);
    for (int64_t i = blockIdx.x * (int64_t)(128 / G) + threadIdx.x / G; i < n; i += groups) {
        Stream<R> rng;
        rng.key = 0; rng.ext = u + uoff[i]; rng.n_ext = uoff[i + 1] - uoff[i];
        const R *p = parents + 5 * i;
        EdgeOut<R> o;
        eval_edge<R, G, false, false, true, true>(g, sc, env, rng, 0u, sp, p[0], p[1], p[2], p[3], p[4], (R)0, 0,
                                                  wp + (size_t)i * wp_cap * 6, wp_cap, o);   // FLAT: explicit streams
        if (g.gl == 0) {
            R *l = leaf + 5 * i;
            l[0] = o.x; l[1] = o.y; l[2] = o.th; l[3] = o.t; l[4] = o.len;
            counts[i] = o.nwp; used[i] = (int32_t)o.ctr; status[i] = o.status;
        }
    }
}
template <typename R>
int launch_steer_arc(const R *parents, int64_t n, const double *u, const int64_t *uoff, const double params[5],
                     R *leaf, int32_t *counts, R *wp, int wp_cap, int32_t *used, int32_t *status, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    int64_t blocks = (n + 3) / 4;
    if (blocks > AUV_SMS * 16) blocks = AUV_SMS * 16;
    k_steer_arc<R, 32><<<(unsigned)blocks, 128, 0, s>>>(parents, n, u, uoff, make_steer_params<R>(params), leaf,
                                                         counts, wp, wp_cap, used, status);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_steer_arc<float>(const float *, int64_t, const double *, const int64_t *, const double[5], float *,
                                     int32_t *, float *, int, int32_t *, int32_t *, cudaStream_t);
template int launch_steer_arc<double>(const double *, int64_t, const double *, const int64_t *, const double[5],
                                      double *, int32_t *, double *, int, int32_t *, int32_t *, cudaStream_t);

// ------------------------------------------------------------------ Dubins steer (waypoints out)
template <typename R>
__global__ void __launch_bounds__(256) k_steer_dubins(const R *from, const R *to, int64_t n, R rho, int W,
                                                      uint8_t *word, R *seg, R *length, R *wp) {
    typedef typename Policy<R>::A A;
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const R *a = from + 3 * i, *b = to + 3 * i;
    DubinsPath<R> d = dubins_shortest<R>(a[0], a[1], a[2], b[0], b[1], b[2], rho);
    word[i] = d.word < 0 ? 255 : (uint8_t)d.word;
    seg[3 * i] = d.t; seg[3 * i + 1] = d.p; seg[3 * i + 2] = d.q;
    length[i] = d.length;
    if (wp && d.word >= 0 && W >= 2) {
        DubinsSampler<R> smp;
        smp.init(d, a[0], a[1], a[2], rho);
        R step = A::div(d.length, (R)(W - 1));
        R *o = wp + (size_t)i * W * 3;
        for (int k = 0; k < W - 1; k++) smp.at(A::mul((R)k, step), o[3 * k], o[3 * k + 1], o[3 * k + 2]);
        o[3 * (W - 1)] = b[0]; o[3 * (W - 1) + 1] = b[1]; o[3 * (W - 1) + 2] = b[2];
    }
}
template <typename R>
int launch_steer_dubins(const R *from, const R *to, int64_t n, double rho, int W, uint8_t *word, R *seg, R *length,
                        R *wp, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    k_steer_dubins<R><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(from, to, n, (R)rho, W, word, seg, length, wp);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_steer_dubins<float>(const float *, const float *, int64_t, double, int, uint8_t *, float *, float *,
                                        float *, cudaStream_t);
template int launch_steer_dubins<double>(const double *, const double *, int64_t, double, int, uint8_t *, double *,
                                         double *, double *, cudaStream_t);

// ------------------------------------------------------------------ RRT.check_collision on explicit paths
template <typename R>
__global__ void __launch_bounds__(128) k_collide(const unsigned char *blob, int hot_bytes, int total_bytes,
                                                 int stage_mode, const R *pts, const int64_t *off, int64_t n,
                                                 uint8_t *safe) {
    extern __shared__ __align__(16) unsigned char smem[];
    EnvView<R> env = load_env<R>(smem, blob, hot_bytes, total_bytes, stage_mode);
    Grp<32> g;
    const int64_t warps = (int64_t)gridDim.x * 4;
    for (int64_t i = blockIdx.x * 4LL + threadIdx.x / 32; i < n; i += warps) {
        int64_t b = off[i], e = off[i + 1];
        bool bad = false;
        for (int64_t k = b + g.gl; k < e; k += 32) {
            R x = pts[2 * k], y = pts[2 * k + 1];
            const Cls cl = env.classify(x, y);
            bad = bad || point_unsafe_c<R>(env, cl, x, y);
        }
        unsigned any = g.ballot(bad);
        if (g.gl == 0) safe[i] = (e == b && env.K > 0) ? 255 : (any ? 0 : 1);
    }
}
template <typename R>
int launch_collide(const auvrrt_env *env, const R *points, const int64_t *off, int64_t n, uint8_t *safe,
                   cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    EnvBlob<R> b = env_blob<R>(env);
    int smem, mode = env_stage_mode(b.hot_bytes, b.hot_bytes, 100 * 1024, &smem);   // probs not needed
    AUV_CUDA(cudaFuncSetAttribute(k_collide<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int64_t blocks = (n + 3) / 4;
    if (blocks > AUV_SMS * 8) blocks = AUV_SMS * 8;
    k_collide<R><<<(unsigned)blocks, 128, smem, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode ? 1 : 0, points, off, n,
                                                      safe);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_collide<float>(const auvrrt_env *, const float *, const int64_t *, int64_t, uint8_t *, cudaStream_t);
template int launch_collide<double>(const auvrrt_env *, const double *, const int64_t *, int64_t, uint8_t *,
                                    cudaStream_t);

// check_collision_obstacle (rrt_dubins.py:551-556): per-obstacle test with the obstacle's OWN radius
template <typename R>
__global__ void __launch_bounds__(256) k_collide_points(const unsigned char *blob, const R *pts, int64_t n,
                                                        uint8_t *safe) {
    typedef typename Policy<R>::A A;
    EnvView<R> env;
    env.bind(blob, blob);
    env.bind_grid(blob, blob);
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    R x = pts[2 * i], y = pts[2 * i + 1];
    bool hit = false;
    for (int k = 0; k < env.K; k++) {
        R q = A::sq2(A::sub(x, env.cx[k]), A::sub(y, env.cy[k]));
        hit = hit || (A::sqrt(q) <= env.cr[k]);
    }
    safe[i] = hit ? 0 : 1;
}
template <typename R>
int launch_collide_points(const auvrrt_env *env, const R *points, int64_t n, uint8_t *safe, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    k_collide_points<R><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(env_blob<R>(env).blob, points, n, safe);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_collide_points<float>(const auvrrt_env *, const float *, int64_t, uint8_t *, cudaStream_t);
template int launch_collide_points<double>(const auvrrt_env *, const double *, int64_t, uint8_t *, cudaStream_t);

// ------------------------------------------------------------------ habitat_shark_cost_func on explicit paths
// builtin sum([c0, c1, c2]) as CPython >= 3.12 evaluates it (Neumaier-compensated float fast path)
template <typename R> __device__ __forceinline__ R py_sum3(R c0, R c1, R c2) {
    typedef typename Policy<R>::A A;
    R f = A::add((R)0, c0), c = (R)0;
    R xs[2] = {c1, c2};
#pragma unroll
    for (int i = 0; i < 2; i++) {
        R x = xs[i], t = A::add(f, x);
        if (A::fabs(f) >= A::fabs(x)) c = A::add(c, A::add(A::sub(f, t), x));
        else c = A::add(c, A::add(A::sub(x, t), f));
        f = t;
    }
    if (c != (R)0 && isfinite(c)) f = A::add(f, c);
    return f;
}

template <typename R>
__global__ void __launch_bounds__(128) k_cost(const unsigned char *blob, int hot_bytes, int total_bytes, int stage_mode,
                                              const R *pts, const int64_t *off, int64_t n, const R *t_total, R w1, R w2,
                                              R w3, unsigned bin_mask, int n_hab, R *out) {
    typedef typename Policy<R>::A A;
    const bool VERIFY = Policy<R>::VERIFY;
    extern __shared__ __align__(16) unsigned char smem[];
    EnvView<R> env = load_env<R>(smem, blob, hot_bytes, total_bytes, stage_mode);
    Grp<32> g;
    const int64_t warps = (int64_t)gridDim.x * 4;
    for (int64_t i = blockIdx.x * 4LL + threadIdx.x / 32; i < n; i += warps) {
        int64_t b = off[i], e = off[i + 1];
        R c1 = 0, c2 = 0;
        unsigned long long visited = 0;
        for (int64_t k0 = b; k0 < e; k0 += 32) {       // path order is the summation order (cost.py:171)
            int64_t k = k0 + g.gl;
            Contrib c; c.bin = -1; c.cell = -1; c.hab = -1;
            if (k < e) c = point_contrib<R>(env, pts[3 * k], pts[3 * k + 1], pts[3 * k + 2], bin_mask, n_hab,
                                             env.classify(pts[3 * k], pts[3 * k + 1]));
            R v2 = (c.bin >= 0 && c.cell >= 0) ? A::mul(w3, env.probs[(size_t)c.bin * env.C + c.cell]) : (R)0;
            R v1 = (c.bin >= 0 && c.hab >= 0) ? w2 : (R)0;
            if (VERIFY) {
                c2 = (R)grp_scan_serial<32>(g, (double)v2, (double)c2); c2 = g.bcast(c2, 31);
                c1 = (R)grp_scan_serial<32>(g, (double)v1, (double)c1); c1 = g.bcast(c1, 31);
            } else {
                c2 += grp_sum<32>(g, v2); c1 += grp_sum<32>(g, v1);
            }
            unsigned long long m = (c.bin >= 0 && c.hab >= 0) ? (1ull << c.hab) : 0ull;
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) m |= g.xorv(m, s);
            visited |= m;
        }
        if (g.gl == 0) {
            R T = t_total[i], c0 = 0;
            if (T > (R)0) { c1 = A::div(c1, T); c2 = A::div(c2, T); }                 // cost.py:194-196
            int count = __popcll(visited);
            if (n_hab != 0) c0 = A::div(A::mul(w1, (R)count), (R)n_hab);              // cost.py:204-205
            out[4 * i] = py_sum3<R>(c0, c1, c2);
            out[4 * i + 1] = c0; out[4 * i + 2] = c1; out[4 * i + 3] = c2;
        }
    }
}
template <typename R>
int launch_cost(const auvrrt_env *env, const R *points, const int64_t *off, int64_t n, const R *t_total,
                const double weights[3], unsigned bin_mask, int n_hab, R *out, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    EnvBlob<R> b = env_blob<R>(env);
    int smem, mode = env_stage_mode(b.hot_bytes, b.total_bytes, 200 * 1024, &smem);
    AUV_CUDA(cudaFuncSetAttribute(k_cost<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int64_t blocks = (n + 3) / 4;
    if (blocks > AUV_SMS * 4) blocks = AUV_SMS * 4;
    k_cost<R><<<(unsigned)blocks, 128, smem, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode, points, off, n, t_total,
                                                   (R)weights[0], (R)weights[1], (R)weights[2], bin_mask, n_hab, out);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_cost<float>(const auvrrt_env *, const float *, const int64_t *, int64_t, const float *,
                                const double[3], unsigned, int, float *, cudaStream_t);
template int launch_cost<double>(const auvrrt_env *, const double *, const int64_t *, int64_t, const double *,
                                 const double[3], unsigned, int, double *, cudaStream_t);

// habitat_shark_cost_point (cost.py:209-241); `visited[i] == True` there is a no-op comparison
template <typename R>
__global__ void __launch_bounds__(256) k_cost_point(const unsigned char *blob, const R *pts, int64_t n,
                                                    unsigned long long visited, int tb, R w1, R w2, R w3, R *out) {
    typedef typename Policy<R>::A A;
    EnvView<R> env;
    env.bind(blob, blob);
    env.bind_grid(blob, blob);
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    R x = pts[2 * i], y = pts[2 * i + 1], c0 = 0, c1 = 0, c2 = 0;
    for (int h = 0; h < env.H; h++) {
        R q = A::sq2(A::sub(env.hx[h], x), A::sub(env.hy[h], y));
        if (A::sqrt(q) <= env.hr[h]) {
            if (!((visited >> h) & 1ull)) c0 = A::add(c0, A::div(w1, (R)env.H));
            c1 = A::add(c1, A::div(w2, (R)env.H));
        }
    }
    int cell = find_cell<R>(env, x, y);
    if (cell >= 0 && tb >= 0 && tb < env.T) c2 = A::add(c2, A::mul(w3, env.probs[(size_t)tb * env.C + cell]));
    out[i] = py_sum3<R>(c0, c1, c2);
}
template <typename R>
int launch_cost_point(const auvrrt_env *env, const R *points, int64_t n, unsigned long long visited, int tb,
                      const double weights[3], R *out, cudaStream_t s) {
    if (n <= 0) return AUVRRT_OK;
    k_cost_point<R><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(env_blob<R>(env).blob, points, n, visited, tb,
                                                                 (R)weights[0], (R)weights[1], (R)weights[2], out);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_cost_point<float>(const auvrrt_env *, const float *, int64_t, unsigned long long, int,
                                      const double[3], float *, cudaStream_t);
template int launch_cost_point<double>(const auvrrt_env *, const double *, int64_t, unsigned long long, int,
                                       const double[3], double *, cudaStream_t);

// ------------------------------------------------------------------ fused Dubins edges (config 4)
// One thread per edge: six-word solve, W waypoints kept in registers, then every waypoint against
// every (inflated) circle read as a shared-memory broadcast, then the polygon test.
#ifndef AUV_ED_THREADS
#define AUV_ED_THREADS 256
#endif
#ifndef AUV_ED_MINB
#define AUV_ED_MINB 2
#endif
#define AUV_ED_TILE 512      // circles kept as float4 triples in shared memory (8 KB); more circles read the SoA arrays
template <typename R, int WT, int MB>
__global__ void __launch_bounds__(AUV_ED_THREADS, MB) k_edges_dubins(const unsigned char *blob, int hot_bytes, int total_bytes,
                                                      int stage_mode, const R *from, const R *to, int64_t n, R rho,
                                                      int W, uint8_t *safe, uint8_t *word, R *length, int wp_off) {
    typedef typename Policy<R>::A A;
    const bool VERIFY = Policy<R>::VERIFY;
    extern __shared__ __align__(16) unsigned char smem[];
    EnvView<R> env = load_env<R>(smem, blob, hot_bytes, total_bytes, stage_mode);
    // fast build: the W waypoints of this thread's edge pass through shared memory, so that a ROLLED loop can compute
    // them (the unrolled sampler + polygon test was 10 k instructions of straight-line code streamed from L2 for every
    // edge: 15 % of the stall cycles were instruction fetch) and an unrolled one loads them into packed registers
    float2 *s_wp = (float2 *)(smem + wp_off) + threadIdx.x;
    __shared__ float4 circ4[AUV_ED_TILE];
    if (!VERIFY) {
        for (int j = threadIdx.x; j < env.K && j < AUV_ED_TILE; j += blockDim.x)
            circ4[j] = make_float4((float)env.cx[j], (float)env.cy[j], (float)env.creff2[j], 0.f);
        __syncthreads();
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        const R *a = from + 3 * i, *b = to + 3 * i;
        DubinsPath<R> d = dubins_shortest<R>(a[0], a[1], a[2], b[0], b[1], b[2], rho);
        bool ok = d.word >= 0;
        if (ok) {
            DubinsSampler<R> smp;
            smp.init(d, a[0], a[1], a[2], rho);
            R step = A::div(d.length, (R)(W - 1));
            bool in = true;
            bool hit = false;
            if (VERIFY) {
                R wx[WT], wy[WT];
#pragma unroll
                for (int k = 0; k < WT; k++) {
                    R th;
                    if (k < W - 1) smp.at(A::mul((R)k, step), wx[k], wy[k], th);
                    else { wx[k] = b[0]; wy[k] = b[1]; }       // k == W-1 is `to`; k >= W duplicates it
                }
#pragma unroll
                for (int k = 0; k < WT; k++) in = in && point_within<R>(env, wx[k], wy[k]);
                for (int c = 0; c < env.K; c++) {
                    R ccx = env.cx[c], ccy = env.cy[c];
                    R q = A::inf();
#pragma unroll
                    for (int k = 0; k < WT; k++) {
                        R qq = A::sq2(A::sub(wx[k], ccx), A::sub(wy[k], ccy));
                        q = qq < q ? qq : q;
                    }
                    hit = hit || (A::sqrt(q) <= env.creff[c]);
                }
            } else {
                // fast build: |p - c|^2 = |p|^2 - 2 p.c + |c|^2 in coordinates relative to the edge's first
                // waypoint: 2 FFMA + 1 FMNMX per (waypoint, circle) instead of 2 FADD + FMUL + FFMA + FMNMX.
                // The expansion cancels, so a result within `guard` of the decision is re-evaluated with
                // the direct formula (far circles never get there: their |c|^2 dwarfs r^2).
#pragma unroll 1
                for (int k = 0; k < WT; k++) {
                    R x, y, th;
                    if (k < W - 1) smp.at(A::mul((R)k, step), x, y, th);
                    else { x = b[0]; y = b[1]; }               // k == W-1 is `to`; k >= W duplicates it
                    in = in && point_within<R>(env, x, y);
                    s_wp[k * AUV_ED_THREADS] = make_float2((float)x, (float)y);
                }
                const R ox = s_wp[0].x, oy = s_wp[0].y;
                // waypoints packed in pairs for the Blackwell packed-FP32 pipe (fma.rn.f32x2 -> FFMA2): one instruction
                // evaluates two (waypoint, circle) pairs, FMNMX3 folds both into the running minimum: 1.5 issue slots
                // per pair instead of 3.  Two circles per iteration keep four independent chains in flight.
                float2 wx2[WT / 2], wy2[WT / 2], pp2[WT / 2];
                R ppmax = (R)0;
#pragma unroll
                for (int k = 0; k < WT / 2; k++) {
                    const float2 wa = s_wp[(2 * k) * AUV_ED_THREADS], wb = s_wp[(2 * k + 1) * AUV_ED_THREADS];
                    const R ax = wa.x - ox, ay = wa.y - oy, bx = wb.x - ox, by = wb.y - oy;
                    pp2[k] = make_float2(fmaf(ay, ay, ax * ax), fmaf(by, by, bx * bx));
                    ppmax = fmaxf(ppmax, fmaxf(pp2[k].x, pp2[k].y));
                    wx2[k] = make_float2((R)-2 * ax, (R)-2 * bx);            // exact scaling: -2 p.c = c.(-2p)
                    wy2[k] = make_float2((R)-2 * ay, (R)-2 * by);
                }
                const R g0 = (R)4e-6 * ppmax;
                const int KT = env.K < AUV_ED_TILE ? env.K : AUV_ED_TILE;       // circles in the shared-memory tile
                for (int c = 0; c < KT; c += 2) {
                    // circles as (x, y, r_eff^2) in shared memory: one 16-byte load each; an odd last circle is paired with itself
                    const int c1 = c + 1 < KT ? c + 1 : c;
                    const float4 ca = circ4[c], cb = circ4[c1];
                    const R axr = ca.x - ox, ayr = ca.y - oy, bxr = cb.x - ox, byr = cb.y - oy;
                    const float2 ax2 = make_float2(axr, axr), ay2 = make_float2(ayr, ayr), bx2 = make_float2(bxr, bxr), by2 = make_float2(byr, byr);
                    R qa0 = A::inf(), qa1 = A::inf(), qb0 = A::inf(), qb1 = A::inf();
#pragma unroll
                    for (int k = 0; k < WT / 2; k += 2) {
                        const float2 a0 = ffma2(ay2, wy2[k], ffma2(ax2, wx2[k], pp2[k]));
                        const float2 b0 = ffma2(by2, wy2[k], ffma2(bx2, wx2[k], pp2[k]));
                        qa0 = fminf(qa0, fminf(a0.x, a0.y));
                        qb0 = fminf(qb0, fminf(b0.x, b0.y));
                        if (k + 1 < WT / 2) {
                            const float2 a1 = ffma2(ay2, wy2[k + 1], ffma2(ax2, wx2[k + 1], pp2[k + 1]));
                            const float2 b1 = ffma2(by2, wy2[k + 1], ffma2(bx2, wx2[k + 1], pp2[k + 1]));
                            qa1 = fminf(qa1, fminf(a1.x, a1.y));
                            qb1 = fminf(qb1, fminf(b1.x, b1.y));
                        }
                    }
                    // d^2 - r_eff^2 for both circles; the expansion cancels, so a result within `guard` of the decision is
                    // re-evaluated with the direct formula (far circles never get there: their |c|^2 dwarfs r^2)
                    const R cca = fmaf(ayr, ayr, axr * axr), ccb = fmaf(byr, byr, bxr * bxr);
                    const R ta = (fminf(qa0, qa1) + cca) - ca.z, tb = (fminf(qb0, qb1) + ccb) - cb.z;
                    const R ga = fmaf((R)4e-6, cca, g0), gb = fmaf((R)4e-6, ccb, g0);
                    if (ta <= ga || tb <= gb) {
                        if (ta < -ga || tb < -gb) hit = true;
                        else {
#pragma unroll 1
                            for (int s = 0; s < 2; s++) {                 // too close to call: direct formula
                                const R cxr = s ? bxr : axr, cyr = s ? byr : ayr, r2 = s ? cb.z : ca.z;
                                R qd = A::inf();
#pragma unroll
                                for (int k = 0; k < WT / 2; k++) {
                                    qd = fminf(qd, A::sq2((R)-0.5 * wx2[k].x - cxr, (R)-0.5 * wy2[k].x - cyr));
                                    qd = fminf(qd, A::sq2((R)-0.5 * wx2[k].y - cxr, (R)-0.5 * wy2[k].y - cyr));
                                }
                                hit = hit || (qd <= r2);
                            }
                        }
                    }
                }
                // circles beyond the tile (K > 512): the direct formula on the SoA arrays
                for (int c = KT; c < env.K; c++) {
                    const R cxr = (R)env.cx[c] - ox, cyr = (R)env.cy[c] - oy;
                    R qd = A::inf();
#pragma unroll
                    for (int k = 0; k < WT / 2; k++) {
                        qd = fminf(qd, A::sq2((R)-0.5 * wx2[k].x - cxr, (R)-0.5 * wy2[k].x - cyr));
                        qd = fminf(qd, A::sq2((R)-0.5 * wx2[k].y - cxr, (R)-0.5 * wy2[k].y - cyr));
                    }
                    hit = hit || (qd <= (R)env.creff2[c]);
                }
            }
            ok = !hit && in;
        }
        safe[i] = ok ? 1 : 0;
        word[i] = d.word < 0 ? 255 : (uint8_t)d.word;
        length[i] = d.length;
    }
}
// Same edges, same booleans, with the broad-phase cull of the classification grid: every waypoint
// is tested only against the <= 3 circles that can touch its grid cell (all circles if the cell has
// more).  Exact by construction (env.cuh); ~70x fewer instructions than the all-pairs loop at K=500.
// COST: also the edge's share of cost.habitat_shark_cost_func (cost.py:171-191) over the appended waypoints 1..W-1
// (waypoint 0 is the parent), with traj_time_stamp = arclength / vel from 0 -- config 4 "cost on" for Dubins edges.
template <typename R, bool COST>
__global__ void __launch_bounds__(256, 4) k_edges_dubins_culled(const unsigned char *blob, int hot_bytes, int total_bytes,
                                                             int stage_mode, const R *from, const R *to, int64_t n,
                                                             R rho, int W, uint8_t *safe, uint8_t *word, R *length,
                                                             R vel, R w3, R *cost_out) {
    typedef typename Policy<R>::A A;
    extern __shared__ __align__(16) unsigned char smem[];
    EnvView<R> env = load_env<R>(smem, blob, hot_bytes, total_bytes, stage_mode);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        const R *a = from + 3 * i, *b = to + 3 * i;
        DubinsPath<R> d = dubins_shortest<R>(a[0], a[1], a[2], b[0], b[1], b[2], rho);
        bool ok = d.word >= 0;
        R s2 = 0; unsigned cnt = 0; unsigned long long mask = 0ull;
        if (ok) {
            DubinsSampler<R> smp;
            smp.init(d, a[0], a[1], a[2], rho);
            const R step = A::div(d.length, (R)(W - 1));
            bool bad = false;
            for (int k = 0; k < W; k++) {
                R x, y, th;
                const R sk = k < W - 1 ? A::mul((R)k, step) : d.length;
                if (k < W - 1) smp.at(sk, x, y, th); else { x = b[0]; y = b[1]; }
                const Cls cl = env.classify(x, y);
                bad = bad || !point_within_c<R, false>(env, cl, x, y) || point_hits_circles_c<R, false>(env, cl, x, y);   // polygon first: one grid code decides most points
                if (COST && k > 0) {
                    const Contrib c = point_contrib<R>(env, x, y, A::div(sk, vel), 0xffffffffu, env.H, cl);
                    if (c.bin >= 0) {
                        if (c.cell >= 0) s2 = A::add(s2, A::mul(w3, env.probs[(size_t)c.bin * env.C + c.cell]));
                        if (c.hab >= 0) { cnt++; mask |= 1ull << c.hab; }
                    }
                }
            }
            ok = !bad;
        }
        safe[i] = ok ? 1 : 0;
        word[i] = d.word < 0 ? 255 : (uint8_t)d.word;
        length[i] = d.length;
        if (COST) { R *c = cost_out + 3 * i; c[0] = s2; c[1] = (R)cnt; c[2] = (R)__popcll(mask); }
    }
}
template <typename R>
int launch_edges_dubins(const auvrrt_env *env, const R *from, const R *to, int64_t n, double rho, int W,
                        uint8_t *safe, uint8_t *word, R *length, cudaStream_t s, double vel, double w3, R *cost_out) {
    if (n <= 0) return AUVRRT_OK;
    EnvBlob<R> b = env_blob<R>(env);
    // default: broad-phase culled kernel; AUVRRT_EDGES_BRUTE=1 selects the all-pairs kernel (the
    // config-4 roofline measurement: every waypoint against every circle)
    const char *brute = getenv("AUVRRT_EDGES_BRUTE");
    if (cost_out && !(env->h32.gnx > 0)) return set_err(AUVRRT_ERR_UNSUPPORTED, "edges_dubins_cost: the world has no classification grid (no boundary polygon)");
    if (cost_out && !(vel > 0.0)) return set_err(AUVRRT_ERR_ARG, "edges_dubins_cost: velocity must be positive, got %g", vel);
    if ((cost_out || !(brute && brute[0] == '1')) && env->h32.gnx > 0) {
        if (W < 2) return set_err(AUVRRT_ERR_ARG, "edges_dubins: W must be >= 2, got %d", W);
        int smem_c, mode_c = env_stage_mode(b.hot_bytes, b.hot_bytes, 64 * 1024, &smem_c);
        mode_c = mode_c ? 1 : 0;
        int64_t blocks_c = (n + 255) / 256;
        if (blocks_c > AUV_SMS * 16) blocks_c = AUV_SMS * 16;
        if (cost_out) {
            AUV_CUDA(cudaFuncSetAttribute(k_edges_dubins_culled<R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_c));
            k_edges_dubins_culled<R, true><<<(unsigned)blocks_c, 256, smem_c, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode_c, from, to,
                                                                                  n, (R)rho, W, safe, word, length, (R)vel, (R)w3, cost_out);
        } else {
            AUV_CUDA(cudaFuncSetAttribute(k_edges_dubins_culled<R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_c));
            k_edges_dubins_culled<R, false><<<(unsigned)blocks_c, 256, smem_c, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode_c, from, to,
                                                                                   n, (R)rho, W, safe, word, length, (R)1, (R)0, nullptr);
        }
        AUV_LAUNCH_CHECK();
        return AUVRRT_OK;
    }
    if (W < 2 || W > 32) return set_err(AUVRRT_ERR_UNSUPPORTED, "edges_dubins (all-pairs): W must be in [2, 32], got %d", W);
    int smem, mode = env_stage_mode(b.hot_bytes, b.hot_bytes, 64 * 1024, &smem);
    mode = mode ? 1 : 0;
    int64_t blocks = (n + AUV_ED_THREADS - 1) / AUV_ED_THREADS;
    if (blocks > AUV_SMS * 12 * (256 / AUV_ED_THREADS)) blocks = AUV_SMS * 12 * (256 / AUV_ED_THREADS);   // a multiple of 1, 2 and 3 CTAs per SM
    // resident CTAs per SM the register allocation targets (fp32): 2 -> 118 registers, 3 -> 80 registers (48 B spilled)
    int mb = AUV_ED_MINB;
    if (const char *ev = getenv("AUVRRT_ED_MINB")) mb = atoi(ev);
    if (sizeof(R) == 8) mb = 1;
#define AUV_ED_L(WT, MB)                                                                                           \
    {                                                                                                              \
        const int wp_off = (smem + 15) & ~15, smem_all = wp_off + (sizeof(R) == 4 ? WT * AUV_ED_THREADS * 8 : 0);      \
        AUV_CUDA(cudaFuncSetAttribute(k_edges_dubins<R, WT, MB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_all));  \
        k_edges_dubins<R, WT, MB><<<(unsigned)blocks, AUV_ED_THREADS, smem_all, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode, from,  \
                                                                   to, n, (R)rho, W, safe, word, length, wp_off);  \
    }
#define AUV_ED(WT) { if (mb >= 3) AUV_ED_L(WT, 3) else if (mb == 2) AUV_ED_L(WT, 2) else AUV_ED_L(WT, 1) }
    if (W <= 8) AUV_ED(8) else if (W <= 12) AUV_ED(12) else if (W <= 16) AUV_ED(16) else if (W <= 20) AUV_ED(20)
    else if (W <= 24) AUV_ED(24) else AUV_ED(32)
#undef AUV_ED
#undef AUV_ED_L
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_edges_dubins<float>(const auvrrt_env *, const float *, const float *, int64_t, double, int,
                                        uint8_t *, uint8_t *, float *, cudaStream_t, double, double, float *);
template int launch_edges_dubins<double>(const auvrrt_env *, const double *, const double *, int64_t, double, int,
                                         uint8_t *, uint8_t *, double *, cudaStream_t, double, double, double *);

// ------------------------------------------------------------------ fused arc edges on the counter stream
// COST: also the edge's share of cost.habitat_shark_cost_func over its appended waypoints (cost.py:171-191):
// cost_out[i] = { sum of w3 * prob, waypoints inside a habitat, distinct habitats visited }.
#ifndef AUV_EA_MINB
#define AUV_EA_MINB 4      // 64 registers, 32 warps per SM (measured: 1.33e9 edges/s vs 1.0e9 at the default 89 registers)
#endif
template <typename R, int G, bool COST>
__global__ void __launch_bounds__(256, sizeof(R) == 4 ? AUV_EA_MINB : 1) k_edges_arc(const unsigned char *blob, int hot_bytes, int total_bytes,
                                                   int stage_mode, const R *parents, const uint64_t *seeds, int64_t n,
                                                   SteerParams<R> sp, R w3, uint8_t *safe, int32_t *counts, R *leaf,
                                                   R *cost_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    EnvView<R> env = load_env<R>(smem, blob, hot_bytes, total_bytes, stage_mode);
    __shared__ GroupScratch<R, G, false> scratch[256 / G];
    Grp<G> g;
    GroupScratch<R, G, false> &sc = scratch[threadIdx.x / G];
    const int64_t groups = (int64_t)gridDim.x * (256 / G);
    for (int64_t i = blockIdx.x * (int64_t)(256 / G) + threadIdx.x / G; i < n; i += groups) {
        Stream<R> rng;
        rng.key = stream_key(seeds[i]); rng.ext = nullptr; rng.n_ext = 0;
        const R *p = parents + 5 * i;
        EdgeOut<R> o;
        eval_edge<R, G, true, COST, false>(g, sc, env, rng, 0u, sp, p[0], p[1], p[2], p[3], p[4], w3, env.H, nullptr,
                                           0, o);
        if (g.gl == 0) {
            safe[i] = o.safe ? 1 : 0;
            if (counts) counts[i] = o.nwp;
            if (leaf) { R *l = leaf + 5 * i; l[0] = o.x; l[1] = o.y; l[2] = o.th; l[3] = o.t; l[4] = o.len; }
            if (COST) { R *c = cost_out + 3 * i; c[0] = o.s2; c[1] = (R)o.cnt; c[2] = (R)__popcll(o.mask); }
        }
    }
}
template <typename R, bool COST>
static int launch_edges_arc_t(const auvrrt_env *env, const R *parents, const uint64_t *seeds, int64_t n,
                              const double params[5], double w3, uint8_t *safe, int32_t *counts, R *leaf, R *cost_out,
                              cudaStream_t s) {
    EnvBlob<R> b = env_blob<R>(env);
    int smem, mode = env_stage_mode(b.hot_bytes, b.hot_bytes, 64 * 1024, &smem);
    mode = mode ? 1 : 0;
    AUV_CUDA(cudaFuncSetAttribute(k_edges_arc<R, 32, COST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int64_t blocks = (n + 7) / 8;
    if (blocks > AUV_SMS * 8) blocks = AUV_SMS * 8;
    k_edges_arc<R, 32, COST><<<(unsigned)blocks, 256, smem, s>>>(b.blob, b.hot_bytes, b.total_bytes, mode, parents, seeds, n,
                                                                  make_steer_params<R>(params), (R)w3, safe, counts, leaf,
                                                                  cost_out);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template <typename R>
int launch_edges_arc(const auvrrt_env *env, const R *parents, const uint64_t *seeds, int64_t n,
                     const double params[5], uint8_t *safe, int32_t *counts, R *leaf, cudaStream_t s, double w3,
                     R *cost_out) {
    if (n <= 0) return AUVRRT_OK;
    // default: one thread per edge (edges_tpe.cu).  AUVRRT_EDGES_VARIANT=warp selects the warp-per-edge kernel
    // above (lower latency for a handful of edges); AUVRRT_EDGES_BRUTE=1 the all-pairs variant of the
    // thread-per-edge kernel (every waypoint against every circle / polygon edge / habitat: the roofline run).
    const char *variant = getenv("AUVRRT_EDGES_VARIANT"), *brute = getenv("AUVRRT_EDGES_BRUTE");
    if (!(variant && variant[0] == 'w')) {
        int rc = launch_edges_arc_tpe<R>(env, parents, seeds, n, params, safe, counts, leaf, s, w3, cost_out,
                                         brute && brute[0] == '1');
        if (rc != AUVRRT_ERR_UNSUPPORTED) return rc;      // world model too large for shared memory: warp per edge
    }
    return cost_out ? launch_edges_arc_t<R, true>(env, parents, seeds, n, params, w3, safe, counts, leaf, cost_out, s)
                    : launch_edges_arc_t<R, false>(env, parents, seeds, n, params, w3, safe, counts, leaf, cost_out, s);
}
template int launch_edges_arc<float>(const auvrrt_env *, const float *, const uint64_t *, int64_t, const double[5],
                                     uint8_t *, int32_t *, float *, cudaStream_t, double, float *);
template int launch_edges_arc<double>(const auvrrt_env *, const double *, const uint64_t *, int64_t, const double[5],
                                      uint8_t *, int32_t *, double *, cudaStream_t, double, double *);

// ------------------------------------------------------------------ RRT.get_closest_mps
// SoA tree streamed once from HBM with vector loads; all arithmetic in fp64 (exact on fp32 inputs),
// compared as sqrt(dx*dx + dy*dy) with strict < and lowest-index ties, like the reference.
struct NNBest { double s; double q; long long i; };
__device__ __forceinline__ void nn_consider(NNBest &b, double dx, double dy, long long i) {
    double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    if (q < b.q) {
        double s = __dsqrt_rn(q);
        if (s < b.s) { b.s = s; b.i = i; }
        b.q = q;
    }
}
__device__ __forceinline__ void nn_merge(NNBest &a, double s, long long i) {
    if (s < a.s || (s == a.s && i < a.i)) { a.s = s; a.i = i; }
}
template <typename R, int NN_QT>
__global__ void __launch_bounds__(256) k_nn_partial(const R *__restrict__ tx, const R *__restrict__ ty, int64_t n,
                                                    const R *__restrict__ qx, const R *__restrict__ qy, int nq,
                                                    double *part_s, long long *part_i) {
    __shared__ double sh_s[8][4];
    __shared__ long long sh_i[8][4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int q0 = 0; q0 < nq; q0 += NN_QT) {
        double qxs[NN_QT], qys[NN_QT];
        float qxf[NN_QT], qyf[NN_QT], thr[NN_QT];
        NNBest best[NN_QT];
#pragma unroll
        for (int j = 0; j < NN_QT; j++) {
            int qi = min(q0 + j, nq - 1);
            qxs[j] = (double)qx[qi]; qys[j] = (double)qy[qi];
            best[j].s = __longlong_as_double(0x7ff0000000000000LL); best[j].q = best[j].s; best[j].i = 0x7fffffffffffffffLL;
            qxf[j] = (float)qxs[j]; qyf[j] = (float)qys[j]; thr[j] = __int_as_float(0x7f800000);
        }
        // 4 consecutive nodes per thread per 16-byte load (fp32), NN_UNROLL independent loads per
        // array in flight per thread: the scan is HBM-bound, so memory-level parallelism is what counts
        const int64_t n4 = n / 4;
        const int64_t stride = (int64_t)gridDim.x * blockDim.x;
#ifndef AUV_NN_UNROLL
#define AUV_NN_UNROLL 3      // loads in flight per thread and array; measured on 2^27 nodes: 2 -> 5.72, 3 -> 5.85, 4 -> 5.42, 5 -> 5.37 TB/s
#endif
        const int NN_UNROLL = AUV_NN_UNROLL;
        for (int64_t v0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v0 < n4; v0 += stride * NN_UNROLL) {
            R xs[NN_UNROLL][4], ys[NN_UNROLL][4];
#pragma unroll
            for (int u = 0; u < NN_UNROLL; u++) {
                const int64_t v = v0 + u * stride;
                if (v < n4) {
                    if (sizeof(R) == 4) {
                        float4 a = __ldcs((const float4 *)tx + v), b = __ldcs((const float4 *)ty + v);
                        xs[u][0] = a.x; xs[u][1] = a.y; xs[u][2] = a.z; xs[u][3] = a.w;
                        ys[u][0] = b.x; ys[u][1] = b.y; ys[u][2] = b.z; ys[u][3] = b.w;
                    } else {
                        double2 a0 = __ldcs((const double2 *)tx + 2 * v), a1 = __ldcs((const double2 *)tx + 2 * v + 1);
                        double2 b0 = __ldcs((const double2 *)ty + 2 * v), b1 = __ldcs((const double2 *)ty + 2 * v + 1);
                        xs[u][0] = a0.x; xs[u][1] = a0.y; xs[u][2] = a1.x; xs[u][3] = a1.y;
                        ys[u][0] = b0.x; ys[u][1] = b0.y; ys[u][2] = b1.x; ys[u][3] = b1.y;
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < NN_UNROLL; u++) {
                const int64_t v = v0 + u * stride;
                if (v < n4) {
#pragma unroll
                    for (int e = 0; e < 4; e++)
#pragma unroll
                        for (int j = 0; j < NN_QT; j++) {
                            if (sizeof(R) == 4) {
                                // fp32 filter in front of the exact fp64 evaluation: q32 is within 3e-7 relative
                                // of the exact q, thr[j] >= 1.000001 * best exact q, so q32 > thr cannot win or tie
                                const float fx = qxf[j] - (float)xs[u][e], fy = qyf[j] - (float)ys[u][e];
                                const float q32 = fmaf(fy, fy, fx * fx);
                                if (q32 <= thr[j]) {
                                    nn_consider(best[j], __dsub_rn(qxs[j], (double)xs[u][e]), __dsub_rn(qys[j], (double)ys[u][e]), 4 * v + e);
                                    thr[j] = __double2float_ru(best[j].q * 1.000001);
                                }
                            } else {
                                nn_consider(best[j], __dsub_rn(qxs[j], (double)xs[u][e]), __dsub_rn(qys[j], (double)ys[u][e]), 4 * v + e);
                            }
                        }
                }
            }
        }
        if (blockIdx.x == 0 && threadIdx.x < (int)(n - 4 * n4)) {     // tail
            int64_t i = 4 * n4 + threadIdx.x;
#pragma unroll
            for (int j = 0; j < NN_QT; j++)
                nn_consider(best[j], __dsub_rn(qxs[j], (double)tx[i]), __dsub_rn(qys[j], (double)ty[i]), i);
        }
        // NOTE per-thread indices are visited in increasing order, so strict < keeps the lowest index
#pragma unroll
        for (int j = 0; j < NN_QT; j++) {
            double s = best[j].s; long long bi = best[j].i;
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) {
                double os = __shfl_xor_sync(0xffffffffu, s, m);
                long long oi = __shfl_xor_sync(0xffffffffu, bi, m);
                if (os < s || (os == s && oi < bi)) { s = os; bi = oi; }
            }
            if (lane == 0) { sh_s[warp][j] = s; sh_i[warp][j] = bi; }
        }
        __syncthreads();
        if (threadIdx.x < NN_QT && q0 + threadIdx.x < nq) {
            NNBest a; a.s = sh_s[0][threadIdx.x]; a.i = sh_i[0][threadIdx.x];
            for (int w = 1; w < 8; w++) nn_merge(a, sh_s[w][threadIdx.x], sh_i[w][threadIdx.x]);
            part_s[(size_t)(q0 + threadIdx.x) * gridDim.x + blockIdx.x] = a.s;
            part_i[(size_t)(q0 + threadIdx.x) * gridDim.x + blockIdx.x] = a.i;
        }
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) k_nn_final(const double *part_s, const long long *part_i, int nparts, int nq,
                                                  int32_t *out_idx) {
    __shared__ double sh_s[8];
    __shared__ long long sh_i[8];
    const int q = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (q >= nq) return;
    double s = __longlong_as_double(0x7ff0000000000000LL); long long bi = 0x7fffffffffffffffLL;
    for (int p = threadIdx.x; p < nparts; p += blockDim.x) {
        double os = part_s[(size_t)q * nparts + p]; long long oi = part_i[(size_t)q * nparts + p];
        if (os < s || (os == s && oi < bi)) { s = os; bi = oi; }
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
        double os = __shfl_xor_sync(0xffffffffu, s, m);
        long long oi = __shfl_xor_sync(0xffffffffu, bi, m);
        if (os < s || (os == s && oi < bi)) { s = os; bi = oi; }
    }
    if (lane == 0) { sh_s[warp] = s; sh_i[warp] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++)
            if (sh_s[w] < s || (sh_s[w] == s && sh_i[w] < bi)) { s = sh_s[w]; bi = sh_i[w]; }
        out_idx[q] = (int32_t)bi;
    }
}
#ifndef AUV_NN_BPS
#define AUV_NN_BPS 8
#endif
static const int NN_BLOCKS = AUV_SMS * AUV_NN_BPS;
int64_t nn_scratch_bytes(int nq) { return (int64_t)nq * NN_BLOCKS * 16 + 256; }
template <typename R>
int launch_nn(const R *tx, const R *ty, int64_t n, const R *qx, const R *qy, int nq, void *scratch,
              int64_t scratch_bytes, int32_t *out_idx, cudaStream_t s) {
    if (nq <= 0) return AUVRRT_OK;
    if (n <= 0) return set_err(AUVRRT_ERR_ARG, "nn: empty tree");
    if (scratch_bytes < nn_scratch_bytes(nq)) return set_err(AUVRRT_ERR_ARG, "nn: scratch too small");
    if (((uintptr_t)tx | (uintptr_t)ty) & 15) return set_err(AUVRRT_ERR_ARG, "nn: tree arrays must be 16-byte aligned");
    int blocks = (int)((n / 4 + 255) / 256);
    if (blocks < 1) blocks = 1;
    if (blocks > NN_BLOCKS) blocks = NN_BLOCKS;
    double *ps = (double *)scratch;
    long long *pi = (long long *)(ps + (size_t)nq * NN_BLOCKS);
    if (nq == 1) k_nn_partial<R, 1><<<blocks, 256, 0, s>>>(tx, ty, n, qx, qy, nq, ps, pi);
    else if (nq == 2) k_nn_partial<R, 2><<<blocks, 256, 0, s>>>(tx, ty, n, qx, qy, nq, ps, pi);
    else k_nn_partial<R, 4><<<blocks, 256, 0, s>>>(tx, ty, n, qx, qy, nq, ps, pi);
    AUV_LAUNCH_CHECK();
    k_nn_final<<<nq, 256, 0, s>>>(ps, pi, blocks, nq, out_idx);
    AUV_LAUNCH_CHECK();
    return AUVRRT_OK;
}
template int launch_nn<float>(const float *, const float *, int64_t, const float *, const float *, int, void *, int64_t,
                              int32_t *, cudaStream_t);
template int launch_nn<double>(const double *, const double *, int64_t, const double *, const double *, int, void *,
                               int64_t, int32_t *, cudaStream_t);

// ------------------------------------------------------------------ FP32 issue-rate calibration
__global__ void __launch_bounds__(256) k_ffma(float *out, int iters, float a, float b) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f,
          x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    float r = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (r == 123.456f) out[0] = r;
}
int launch_calibrate_fp32(int iters, double *flops, double *ms_out) {
    DBuf d;
    AUV_TRY(d.alloc(4));
    cudaEvent_t e0, e1;
    AUV_CUDA(cudaEventCreate(&e0));
    AUV_CUDA(cudaEventCreate(&e1));
    const int blocks = AUV_SMS * 8;
    k_ffma<<<blocks, 256>>>(d.as<float>(), 64, 0.999f, 0.001f);   // warm-up
    AUV_LAUNCH_CHECK();
    AUV_CUDA(cudaEventRecord(e0));
    k_ffma<<<blocks, 256>>>(d.as<float>(), iters, 0.999f, 0.001f);
    AUV_LAUNCH_CHECK();
    AUV_CUDA(cudaEventRecord(e1));
    AUV_CUDA(cudaEventSynchronize(e1));
    float ms;
    AUV_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *ms_out = ms;
    *flops = (double)blocks * 256.0 * (double)iters * 16.0 * 8.0 * 2.0 / (ms * 1e-3);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return AUVRRT_OK;
}

}  // namespace auv
