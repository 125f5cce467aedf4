// plan_common.cuh -- pieces shared by the two planner kernels (plan.cu: one lane group per tree;
// plan_tpt.cu: one thread per tree).
#pragma once
#include "launch.h"

namespace auv {

template <typename R> struct PlanP {
    int I, mode, nb, chain_cap, path_cap, trace, cap, nchunks;
    R bin_interval, max_traj, horizon, w1, w2, w3;
    R ran_time_max, plan_dt;      // mode 2: max_plan_time * freq (:129) and max_plan_time / iterations
    R rho, eta, near_r, near_r2, vel;   // mode 3: turning radius, longest edge, neighbourhood radius (and its square), speed
    int W;                              // mode 3: waypoints per edge, the parent included
    SteerParams<R> sp;
};

// builtin sum([c0, c1, c2]) as CPython >= 3.12 evaluates it (Neumaier-compensated float fast path)
template <typename R> __device__ __forceinline__ R py_sum3p(R c0, R c1, R c2) {
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

template <typename R> static inline int make_planp(const auvrrt_env *env, const auvrrt_plan_params_t *p, PlanP<R> *out) {
    if (p->iterations < 1) return set_err(AUVRRT_ERR_ARG, "plan: iterations must be >= 1");
    if (p->mode < 0 || p->mode > 3) return set_err(AUVRRT_ERR_ARG, "plan: mode must be 0, 1, 2 or 3");
    if (p->mode == 3 && (p->dubins_w < 2 || p->dubins_w > 32 || !(p->dubins_rho > 0) || !(p->dubins_eta > 0) || !(p->v > 0) ||
                         !(p->near_radius >= 0)))
        return set_err(AUVRRT_ERR_ARG, "plan: mode 3 needs dubins_w in [2, 32], dubins_rho > 0, dubins_eta > 0, v > 0, near_radius >= 0");
    if (p->mode == 2 && !(p->max_plan_time > 0)) return set_err(AUVRRT_ERR_ARG, "plan: mode 2 needs max_plan_time > 0");
    if (!(p->bin_interval > 0) || !(p->max_traj_time > 0)) return set_err(AUVRRT_ERR_ARG, "plan: bin_interval and max_traj_time must be > 0");
    if (env->H > 64) return set_err(AUVRRT_ERR_UNSUPPORTED, "plan: more than 64 habitats");
    double nbd = ceil(p->max_traj_time / p->bin_interval);                      // rrt_dubins.py:111
    if (nbd > 1e6) return set_err(AUVRRT_ERR_UNSUPPORTED, "plan: more than 1e6 time bins");
    PlanP<R> P;
    P.I = p->iterations; P.mode = p->mode; P.nb = (int)nbd;
    P.chain_cap = p->chain_cap > 0 ? p->chain_cap : 1; P.path_cap = p->path_cap; P.trace = p->trace;
    P.cap = P.I + 1; P.nchunks = P.nb + P.cap / 32 + 4;
    P.bin_interval = (R)p->bin_interval; P.max_traj = (R)p->max_traj_time;
    P.horizon = (R)(p->max_traj_time - 30);                                     // :158
    P.ran_time_max = (R)(p->max_plan_time * p->freq);
    P.plan_dt = (R)(p->max_plan_time / (double)p->iterations);
    P.w1 = (R)p->weights[0]; P.w2 = (R)p->weights[1]; P.w3 = (R)p->weights[2];
    P.rho = (R)p->dubins_rho; P.eta = (R)p->dubins_eta; P.near_r = (R)p->near_radius;
    P.near_r2 = (R)(p->near_radius * p->near_radius); P.vel = (R)p->v; P.W = p->dubins_w;
    double sp[5] = {p->dist_to_end, p->diff_max, p->freq, p->min_dist, p->v};
    P.sp = make_steer_params<R>(sp);
    *out = P;
    return AUVRRT_OK;
}


// One tree node: a 64-byte row in fp32 (x,y,theta,t | len,s2,self_s2,ctr | parent,cnt,self_hab | mask), so
// fetching a parent and appending a node are a few 16-byte accesses to one or two sectors.
template <typename R> struct alignas(16) NodeRow {
    R x, y, th, t;
    R len, s2, self_s2;
    uint32_t ctr;
    int parent;
    uint32_t cnt;
    int self_hab;
    int born;          // steer call that created the node: plan_time_stamp = born * plan_dt (mode 2)
    unsigned long long mask;
};



// RRT.get_closest_mps_time (rrt_dubins.py:515-528): the reference's list-slicing pseudo-bisection on
// plan_time_stamp, restated on the index range [lo, lo + len).  plan_time_stamp of a node is
// (steer call that created it) * plan_dt on the simulated clock (0 for the root).
template <typename R>
__device__ __forceinline__ int closest_mps_time(const NodeRow<R> *rows, int n_nodes, R ran_time, R plan_dt) {
    typedef typename Policy<R>::A A;
    int lo = 0, len = n_nodes;
    while (len > 3) {
        const int half = len >> 1;
        const R ls = A::mul((R)rows[lo + half - 1].born, plan_dt), rs = A::mul((R)rows[lo + half + 1].born, plan_dt);
        const R left_diff = A::fabs(A::sub(ls, ran_time)), right_diff = A::fabs(A::sub(rs, ran_time));
        if (left_diff >= right_diff) { lo += half; len -= half; } else len = half;
    }
    return lo;
}

// thread-per-tree planner (plan_tpt.cu)
template <typename R>
int launch_plan_tpt(const auvrrt_env *env, const R *starts, const uint64_t *seeds, int64_t Q,
                    const auvrrt_plan_params_t *p, void *workspace, int64_t workspace_bytes,
                    auvrrt_plan_record_t *records, uint32_t *chain, const auvrrt_plan_trace_t *trace,
                    cudaStream_t s, int64_t *need_bytes);
// paths of its plans, re-created with its own edge evaluator
template <typename R>
int launch_materialize_tpt(const auvrrt_env *env, const R *starts, const uint64_t *seeds, const uint32_t *chain,
                           const int32_t *depth, int64_t Q, const PlanP<R> &P, R *path, int32_t *n_path, cudaStream_t s);

}  // namespace auv
