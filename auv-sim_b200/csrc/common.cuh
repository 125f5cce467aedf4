// common.cuh -- arithmetic policy, counter-based uniform stream, lane-group helpers.
//
// Two builds of every kernel live in the same library (include/auvrrt.h `precision`):
//   R = float,  VERIFY = false : fast build.  FMA contraction allowed, numerically stable
//                                restatements of the reference's formulas, MUFU where accurate.
//   R = double, VERIFY = true  : verification build.  Every operation the reference (CPython
//                                float arithmetic) performs is a separately rounded IEEE operation
//                                here too (__dadd_rn / __dmul_rn / __ddiv_rn are never contracted),
//                                in the reference's order, so booleans and indices match it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#define AUV_SMS 148

namespace auv {

// ------------------------------------------------------------------ strict / relaxed arithmetic
template <typename R, bool VERIFY> struct Ar;

template <> struct Ar<double, true> {
    typedef double R;
    static __device__ __forceinline__ R add(R a, R b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ R sub(R a, R b) { return __dsub_rn(a, b); }
    static __device__ __forceinline__ R mul(R a, R b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ R div(R a, R b) { return __ddiv_rn(a, b); }
    static __device__ __forceinline__ R sqrt(R a) { return __dsqrt_rn(a); }
    // dx**2 + dy**2 : two rounded squares, one rounded sum (rrt_dubins.py:562)
    static __device__ __forceinline__ R sq2(R dx, R dy) { return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)); }
    static __device__ __forceinline__ void sincos(R a, R *s, R *c) { ::sincos(a, s, c); }
    static __device__ __forceinline__ R floor(R a) { return ::floor(a); }
    static __device__ __forceinline__ R fabs(R a) { return ::fabs(a); }
    static __device__ __forceinline__ R fma(R a, R b, R c) { return ::fma(a, b, c); }
    static __device__ __forceinline__ R inf() { return __longlong_as_double(0x7ff0000000000000LL); }
};

template <> struct Ar<float, false> {
    typedef float R;
    static __device__ __forceinline__ R add(R a, R b) { return a + b; }
    static __device__ __forceinline__ R sub(R a, R b) { return a - b; }
    static __device__ __forceinline__ R mul(R a, R b) { return a * b; }
    // a * rcp.approx.ftz(b): <= 2 ulp; no denormal-divisor fix-up code (divisors here are lengths / velocities
    // bounded away from the denormal range)
    static __device__ __forceinline__ R div(R a, R b) {
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b));
        return a * r;
    }
    static __device__ __forceinline__ R sqrt(R a) { return sqrtf(a); }
    static __device__ __forceinline__ R sq2(R dx, R dy) { return fmaf(dy, dy, dx * dx); }
    // fast build: two-term Cody-Waite reduction to [-pi, pi] (exact product for |a| < 2^10 * 2pi),
    // then the MUFU sine / cosine (abs. error ~4e-7 on the reduced range): headings here are a few
    // radians, so the error per arc primitive is < 1e-6 m, far inside the 1e-5 relative bar
    static __device__ __forceinline__ void sincos(R a, R *s, R *c) {
        // nearest integer of a / 2pi through the 1.5 * 2^23 magic constant (|a / 2pi| < 2^22): two full-rate
        // instructions instead of FRND on the conversion pipe
        const float k = __fadd_rn(__fmaf_rn(a, 0.15915494309189535f, 12582912.f), -12582912.f);
        float r = fmaf(k, -6.28318548202514648f, a);         // 2pi rounded to fp32 ...
        r = fmaf(k, 1.74845553146951715e-7f, r);             // ... plus its rounding error
        *s = __sinf(r); *c = __cosf(r);
    }
    static __device__ __forceinline__ R floor(R a) { return floorf(a); }
    static __device__ __forceinline__ R fabs(R a) { return fabsf(a); }
    static __device__ __forceinline__ R fma(R a, R b, R c) { return fmaf(a, b, c); }
    static __device__ __forceinline__ R inf() { return __int_as_float(0x7f800000); }
};

template <typename R> struct Policy;
template <> struct Policy<float> { static const bool VERIFY = false; typedef Ar<float, false> A; };
template <> struct Policy<double> { static const bool VERIFY = true; typedef Ar<double, true> A; };

// ------------------------------------------------------------------ the uniform stream
// The pre-generated sample sequence.  Position k of the stream of `seed` is the 64-bit word
//   hi(k) = M32a(c * 0x9E3779B9 + key_lo),  lo(k) = M32b(c * 0x85EBCA77 + key_hi),  c = k + 1 (mod 2^32)
// where M32a / M32b are two 2-round xorshift-multiply mixers on 32-bit words (the constants of the
// hash-prospector "lowbias32" functions, without their last xorshift, which only touches low bits) and
// key = stream_key(seed) (SplitMix64 finaliser, once per query).  32-bit multiplies only: a draw costs
// ~10 instructions in the fp32 build (round 1 hashed with SplitMix64: two 64-bit multiplies per draw, 13 %
// of the planner's instructions).  Pure function of (seed, k): any lane can evaluate any position (what
// makes the warp-parallel steer possible) and the host can pre-generate the identical sequence for the
// reference (auvrrt_stream_u, oracle/harness.py stream_block).
//   fp64 build:  u = (hi:lo >> 11) * 2^-53     (53 bits)
//   fp32 build:  u = (hi >> 9) * 2^-23         (the top 23 bits of the same word; exact in fp32, in [0, 1))
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t stream_key(uint64_t seed) {
    return mix64((seed + 1) * 0x9E3779B97F4A7C15ULL);
}
#define AUV_WEYL_HI 0x9E3779B9u
#define AUV_WEYL_LO 0x85EBCA77u
// w = c * AUV_WEYL_HI + key_lo  ->  hi word
__host__ __device__ __forceinline__ uint32_t mix32a(uint32_t w) {
    w ^= w >> 16; w *= 0x21F0AAADu; w ^= w >> 15; w *= 0x735A2D97u;
    return w;
}
// w = c * AUV_WEYL_LO + key_hi  ->  lo word
__host__ __device__ __forceinline__ uint32_t mix32b(uint32_t w) {
    w ^= w >> 15; w *= 0xD168AAADu; w ^= w >> 15; w *= 0xAF723597u;
    return w;
}
__host__ __device__ __forceinline__ uint32_t stream_hi(uint64_t key, uint32_t k) {
    return mix32a((k + 1u) * AUV_WEYL_HI + (uint32_t)key);
}
__host__ __device__ __forceinline__ uint32_t stream_lo(uint64_t key, uint32_t k) {
    return mix32b((k + 1u) * AUV_WEYL_LO + (uint32_t)(key >> 32));
}
__host__ __device__ __forceinline__ uint64_t stream_bits(uint64_t key, uint32_t k) {
    return ((uint64_t)stream_hi(key, k) << 32) | (uint64_t)stream_lo(key, k);
}

// A DRAW is what the kernels carry for one stream position: u in [0, 1) in the fp64 build, 1 + u in
// [1, 2) in the fp32 build (the 23 bits dropped into a float's mantissa: no integer-to-float
// conversion).  uniform_ab() and unit() are the only consumers.
template <typename R> struct Draw;
template <> struct Draw<double> {
    static __device__ __forceinline__ double at(uint64_t key, uint32_t k) {
        return (double)(stream_bits(key, k) >> 11) * 0x1.0p-53;
    }
    static __device__ __forceinline__ double from_words(uint32_t hi, uint32_t lo) {
        return (double)((((uint64_t)hi << 32) | (uint64_t)lo) >> 11) * 0x1.0p-53;
    }
    static __device__ __forceinline__ double from_unit(double u) { return u; }
};
template <> struct Draw<float> {
    static __device__ __forceinline__ float from_hi(uint32_t hi) { return __uint_as_float((hi >> 9) | 0x3f800000u); }
    static __device__ __forceinline__ float at(uint64_t key, uint32_t k) { return from_hi(stream_hi(key, k)); }
    static __device__ __forceinline__ float from_unit(double u) { return (float)u + 1.0f; }
};
// the draw as a plain u in [0, 1)
__device__ __forceinline__ double unit(double d) { return d; }
__device__ __forceinline__ float unit(float d) { return d - 1.0f; }

// Where a stream comes from: the counter hash, or an explicit pre-generated array (replaying a
// recorded CPython Mersenne-Twister sequence through the same kernels).
template <typename R> struct Stream {
    uint64_t key;
    const double *ext;    // explicit doubles (host-provided), or nullptr
    int64_t n_ext;
    // Positions past the end of an explicit stream read as 0.5: lanes prefetch a window of positions
    // speculatively, so only a CONSUMED position past the end is an error (see consumed_ok()).
    __device__ __forceinline__ R u(uint32_t k) const {      // a draw (see Draw<R>)
        if (ext) return Draw<R>::from_unit(((int64_t)k < n_ext) ? ext[k] : 0.5);
        return Draw<R>::at(key, k);
    }
    __device__ __forceinline__ bool consumed_ok(uint32_t ctr_end) const {
        return !ext || (int64_t)ctr_end <= n_ext;
    }
};

// serial view of the counter stream: u_ctr, u_ctr+1, ... with the two Weyl products kept incrementally
template <typename R> struct SerialStream {
    uint32_t wa, wb;   // c * AUV_WEYL_HI + key_lo, c * AUV_WEYL_LO + key_hi for c = ctr (the next draw adds one step first)
    uint32_t ctr;
    __device__ __forceinline__ void init(uint64_t key) { wa = (uint32_t)key; wb = (uint32_t)(key >> 32); ctr = 0; }
    __device__ __forceinline__ void seek(uint64_t key, uint32_t pos) {
        wa = pos * AUV_WEYL_HI + (uint32_t)key; wb = pos * AUV_WEYL_LO + (uint32_t)(key >> 32); ctr = pos;
    }
    __device__ __forceinline__ R next();
    __device__ __forceinline__ void skip(uint32_t n) { wa += n * AUV_WEYL_HI; wb += n * AUV_WEYL_LO; ctr += n; }
};
template <> __device__ __forceinline__ float SerialStream<float>::next() {
    wa += AUV_WEYL_HI; ctr++;
    return Draw<float>::from_hi(mix32a(wa));
}
template <> __device__ __forceinline__ double SerialStream<double>::next() {
    wa += AUV_WEYL_HI; wb += AUV_WEYL_LO; ctr++;
    return Draw<double>::from_words(mix32a(wa), mix32b(wb));
}

// random.uniform(a, b) = a + (b - a) * random()      (CPython Lib/random.py) on a draw d.
// fp64: the reference's two rounded operations.  fp32: ONE fma on the mantissa form,
// (a - (b - a)) + (b - a) * (1 + u); b - a and a - (b - a) are loop invariants.  Whenever a - (b - a) is
// exact in fp32 (the steer's (0, 2), (-0.5, 0.5), (0, 30), (0, 2v)) this is a + (b - a) * u rounded once.
template <typename R> __device__ __forceinline__ R uniform_ab(R a, R b, R d);
template <> __device__ __forceinline__ double uniform_ab<double>(double a, double b, double d) {
    return __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), d));
}
template <> __device__ __forceinline__ float uniform_ab<float>(float a, float b, float d) {
    const float w = b - a;
    return fmaf(w, d, a - w);
}

// Python float floor division  t // w  for w > 0 (Objects/floatobject.c float_floor_div): the
// floor of the EXACT quotient, not of the rounded one.
template <typename R> __device__ __forceinline__ R floordiv_pos(R t, R w) {
    typedef typename Policy<R>::A A;
    // fp32: any quotient within one of the true floor will do (the residual tests below settle it), so the fast
    // reciprocal replaces the IEEE division
    R q = sizeof(R) == 4 ? A::floor(A::div(t, w)) : A::floor(t / w);
    // exact residual via FMA: r = q*w - t
    if (A::fma(q, w, -t) > (R)0) q -= (R)1;            // rounded quotient overshot
    else if (A::fma(q + (R)1, w, -t) <= (R)0) q += (R)1;  // or undershot
    return q;
}

// ------------------------------------------------------------------ lane groups
// G lanes (8, 16 or 32) cooperate on one tree / edge; a warp holds 32/G groups.
template <int G> struct Grp {
    int lane, gl, gbase;
    unsigned gmask;
    __device__ __forceinline__ Grp() {
        // %laneid through a volatile asm: the compiler may not rematerialise it (it re-read SR_TID.X and masked it all
        // over the planner's hot loop: 3 % of its instructions)
        unsigned l;
        asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
        lane = (int)l;
        gl = lane & (G - 1);
        gbase = lane - gl;
        gmask = (G == 32) ? 0xffffffffu : (((1u << (G & 31)) - 1u) << gbase);
    }
    __device__ __forceinline__ void sync() const { __syncwarp(gmask); }
    __device__ __forceinline__ unsigned ballot(bool p) const {
        unsigned b = __ballot_sync(gmask, p);
        return (G == 32) ? b : ((b >> gbase) & ((1u << (G & 31)) - 1u));
    }
    template <typename T> __device__ __forceinline__ T bcast(T v, int src) const {
        return __shfl_sync(gmask, v, gbase + src);
    }
    template <typename T> __device__ __forceinline__ T up(T v, int d) const {   // lane gl-d (gl >= d)
        return __shfl_up_sync(gmask, v, d, G);
    }
    template <typename T> __device__ __forceinline__ T xorv(T v, int m) const {
        return __shfl_xor_sync(gmask, v, m, G);
    }
};

template <int G, typename T> __device__ __forceinline__ T grp_sum(const Grp<G> &g, T v) {
#pragma unroll
    for (int m = G / 2; m > 0; m >>= 1) v += g.xorv(v, m);
    return v;
}
template <int G, typename T> __device__ __forceinline__ T grp_scan_incl(const Grp<G> &g, T v) {
#pragma unroll
    for (int d = 1; d < G; d <<= 1) {
        T o = g.up(v, d);
        if (g.gl >= d) v += o;
    }
    return v;
}
// inclusive running sum in the reference's serial order: ((carry + v0) + v1) + ...   (VERIFY)
template <int G> __device__ __forceinline__ double grp_scan_serial(const Grp<G> &g, double v, double carry) {
    double acc = carry, mine = carry;
#pragma unroll 1
    for (int j = 0; j < G; j++) {
        double vj = g.bcast(v, j);
        acc = __dadd_rn(acc, vj);
        if (j == g.gl) mine = acc;
    }
    return mine;
}

// ------------------------------------------------------------------ host-side helpers
extern thread_local char g_err[512];
extern long long g_launches;
int set_err(int code, const char *fmt, ...);

#define AUV_CUDA(call)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return auv::set_err(AUVRRT_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,    \
                                cudaGetErrorString(e_));                                       \
    } while (0)

// After every kernel launch: count it (auvrrt_launch_count) and report a failed launch as AUVRRT_ERR_CUDA.
#define AUV_LAUNCH_CHECK()                                                                     \
    do {                                                                                       \
        auv::g_launches++;                                                                     \
        cudaError_t e_ = cudaGetLastError();                                                   \
        if (e_ != cudaSuccess)                                                                 \
            return auv::set_err(AUVRRT_ERR_CUDA, "%s:%d launch: %s", __FILE__, __LINE__,       \
                                cudaGetErrorString(e_));                                       \
    } while (0)

}  // namespace auv
