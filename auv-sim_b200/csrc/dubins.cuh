// dubins.cuh -- six-word Dubins steer (LSL, LSR, RSL, RSR, RLR, LRL), one thread per edge.
//
// Named by the north star; ABSENT from the reference, whose only trace is a commented-out call
// into the third-party PyPI `dubins` module (/root/reference/path_planning/rrt_dubins.py:238-251:
// dubins.shortest_path(q0, q1, turning_radius); path.sample_many(exp_rate)).  PARITY UNPINNED:
// this follows the published normalised formulation (Shkel & Lumelsky 2001; SURVEY.md appendix B)
// and is checked by closure / symmetry properties and against oracle/auvrrt_oracle.c.
#pragma once
#include "geom.cuh"

namespace auv {

template <typename R> struct DMath;
template <> struct DMath<double> {
    static __device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
    static __device__ __forceinline__ double acos(double x) { return ::acos(x); }
    static __device__ __forceinline__ double two_pi() { return 6.283185307179586; }
};
template <> struct DMath<float> {
    static __device__ __forceinline__ float atan2(float y, float x) { return atan2f(y, x); }
    static __device__ __forceinline__ float acos(float x) { return acosf(x); }
    static __device__ __forceinline__ float two_pi() { return 6.2831853071795864769f; }
};

template <typename R> __device__ __forceinline__ R mod2pi(R t) {
    typedef typename Policy<R>::A A;
    const R tp = DMath<R>::two_pi();
    return A::sub(t, A::mul(tp, A::floor(A::div(t, tp))));
}

template <typename R> struct DubinsPath {
    int word;        // 0..5 in evaluation order LSL, LSR, RSL, RSR, RLR, LRL; -1: none
    R t, p, q;       // segment parameters in units of rho
    R length;        // rho * (t + p + q)
};

// segment types packed 2 bits each: L=0, S=1, R=2
__device__ __forceinline__ int dubins_seg_type(int word, int i) {
    const unsigned codes[6] = {0u | (1u << 2) | (0u << 4), 0u | (1u << 2) | (2u << 4), 2u | (1u << 2) | (0u << 4),
                               2u | (1u << 2) | (2u << 4), 2u | (0u << 2) | (2u << 4), 0u | (2u << 2) | (0u << 4)};
    return (codes[word] >> (2 * i)) & 3;
}

template <typename R>
__device__ __forceinline__ DubinsPath<R> dubins_shortest(R x0, R y0, R th0, R x1, R y1, R th1, R rho) {
    typedef typename Policy<R>::A A;
    typedef DMath<R> M;
    DubinsPath<R> best;
    best.word = -1; best.t = best.p = best.q = 0; best.length = A::inf();
    R dx = A::sub(x1, x0), dy = A::sub(y1, y0);
    R D = A::sqrt(A::add(A::mul(dx, dx), A::mul(dy, dy)));
    R d = A::div(D, rho);
    R theta = d > (R)0 ? mod2pi<R>(M::atan2(dy, dx)) : (R)0;
    R alpha = mod2pi<R>(A::sub(th0, theta)), beta = mod2pi<R>(A::sub(th1, theta));
    R sa, ca, sb, cb, sab, cab;
    A::sincos(alpha, &sa, &ca);
    A::sincos(beta, &sb, &cb);
    A::sincos(A::sub(alpha, beta), &sab, &cab);
    (void)sab;
    const R d2 = A::mul(d, d), two = (R)2;
    R bestc = A::inf();
#define AUV_DUBINS_WORD(W, T_, P_, Q_)                                            \
    {                                                                              \
        R tt = (T_), pp = (P_), qq = (Q_);                                         \
        R c = A::add(A::add(tt, pp), qq);                                          \
        if (c < bestc) { bestc = c; best.word = (W); best.t = tt; best.p = pp; best.q = qq; } \
    }
    {   // LSL
        R p2 = A::add(A::sub(A::add(two, d2), A::mul(two, cab)), A::mul(A::mul(two, d), A::sub(sa, sb)));
        if (p2 >= (R)0) {
            R t0 = M::atan2(A::sub(cb, ca), A::sub(A::add(d, sa), sb));
            AUV_DUBINS_WORD(0, mod2pi<R>(A::sub(t0, alpha)), A::sqrt(p2), mod2pi<R>(A::sub(beta, t0)))
        }
    }
    {   // LSR
        R p2 = A::add(A::add(A::add(-two, d2), A::mul(two, cab)), A::mul(A::mul(two, d), A::add(sa, sb)));
        if (p2 >= (R)0) {
            R p = A::sqrt(p2);
            R t0 = A::sub(M::atan2(A::sub(-ca, cb), A::add(A::add(d, sa), sb)), M::atan2(-two, p));
            AUV_DUBINS_WORD(1, mod2pi<R>(A::sub(t0, alpha)), p, mod2pi<R>(A::sub(t0, mod2pi<R>(beta))))
        }
    }
    {   // RSL
        R p2 = A::sub(A::add(A::add(-two, d2), A::mul(two, cab)), A::mul(A::mul(two, d), A::add(sa, sb)));
        if (p2 >= (R)0) {
            R p = A::sqrt(p2);
            R t0 = A::sub(M::atan2(A::add(ca, cb), A::sub(A::sub(d, sa), sb)), M::atan2(two, p));
            AUV_DUBINS_WORD(2, mod2pi<R>(A::sub(alpha, t0)), p, mod2pi<R>(A::sub(beta, t0)))
        }
    }
    {   // RSR
        R p2 = A::add(A::sub(A::add(two, d2), A::mul(two, cab)), A::mul(A::mul(two, d), A::sub(sb, sa)));
        if (p2 >= (R)0) {
            R t0 = M::atan2(A::sub(ca, cb), A::add(A::sub(d, sa), sb));
            AUV_DUBINS_WORD(3, mod2pi<R>(A::sub(alpha, t0)), A::sqrt(p2), mod2pi<R>(A::sub(t0, beta)))
        }
    }
    {   // RLR
        R w = A::div(A::add(A::add(A::sub((R)6, d2), A::mul(two, cab)), A::mul(A::mul(two, d), A::sub(sa, sb))), (R)8);
        if (A::fabs(w) <= (R)1) {
            R ph = M::atan2(A::sub(ca, cb), A::add(A::sub(d, sa), sb));
            R p = mod2pi<R>(A::sub(M::two_pi(), M::acos(w)));
            R t = mod2pi<R>(A::add(A::sub(alpha, ph), mod2pi<R>(A::div(p, two))));
            AUV_DUBINS_WORD(4, t, p, mod2pi<R>(A::add(A::sub(A::sub(alpha, beta), t), mod2pi<R>(p))))
        }
    }
    {   // LRL
        R w = A::div(A::add(A::add(A::sub((R)6, d2), A::mul(two, cab)), A::mul(A::mul(two, d), A::sub(sb, sa))), (R)8);
        if (A::fabs(w) <= (R)1) {
            R ph = M::atan2(A::sub(ca, cb), A::sub(A::add(d, sa), sb));
            R p = mod2pi<R>(A::sub(M::two_pi(), M::acos(w)));
            R t = mod2pi<R>(A::add(A::sub(-alpha, ph), A::div(p, two)));
            AUV_DUBINS_WORD(5, t, p, mod2pi<R>(A::add(A::sub(A::sub(mod2pi<R>(beta), alpha), t), mod2pi<R>(p))))
        }
    }
#undef AUV_DUBINS_WORD
    if (best.word >= 0) best.length = A::mul(bestc, rho);
    return best;
}

// unit-radius propagation along one segment from (x, y, th) by arclength s
template <typename R>
__device__ __forceinline__ void dubins_segment(R s, R x, R y, R th, int type, R &ox, R &oy, R &oth) {
    typedef typename Policy<R>::A A;
    R st, ct;
    A::sincos(th, &st, &ct);
    if (type == 0) {          // L
        R s2, c2; A::sincos(A::add(th, s), &s2, &c2);
        ox = A::add(A::sub(s2, st), x); oy = A::add(A::add(-c2, ct), y); oth = A::add(s, th);
    } else if (type == 2) {   // R
        R s2, c2; A::sincos(A::sub(th, s), &s2, &c2);
        ox = A::add(A::add(-s2, st), x); oy = A::add(A::sub(c2, ct), y); oth = A::add(-s, th);
    } else {                  // S
        ox = A::add(A::mul(ct, s), x); oy = A::add(A::mul(st, s), y); oth = A::add((R)0, th);
    }
}

template <typename R> struct DubinsSampler {
    R x0, y0, rho, th0;
    R ax, ay, ath, bx, by, bth;   // configurations after segments 1 and 2 (unit radius, origin start)
    R t, p;
    int ty0, ty1, ty2;
    __device__ __forceinline__ void init(const DubinsPath<R> &d, R x0_, R y0_, R th0_, R rho_) {
        x0 = x0_; y0 = y0_; rho = rho_; th0 = th0_; t = d.t; p = d.p;
        ty0 = dubins_seg_type(d.word, 0); ty1 = dubins_seg_type(d.word, 1); ty2 = dubins_seg_type(d.word, 2);
        dubins_segment<R>(d.t, (R)0, (R)0, th0, ty0, ax, ay, ath);
        dubins_segment<R>(d.p, ax, ay, ath, ty1, bx, by, bth);
    }
    __device__ __forceinline__ void at(R s, R &x, R &y, R &th) const {
        typedef typename Policy<R>::A A;
        R tp = A::div(s, rho), qx, qy, qth;
        if (tp < t) dubins_segment<R>(tp, (R)0, (R)0, th0, ty0, qx, qy, qth);
        else if (tp < A::add(t, p)) dubins_segment<R>(A::sub(tp, t), ax, ay, ath, ty1, qx, qy, qth);
        else dubins_segment<R>(A::sub(A::sub(tp, t), p), bx, by, bth, ty2, qx, qy, qth);
        x = A::add(A::mul(qx, rho), x0); y = A::add(A::mul(qy, rho), y0); th = mod2pi<R>(qth);
    }
};

}  // namespace auv
