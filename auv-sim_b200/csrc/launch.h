// launch.h -- internal host-side interface between the C ABI (api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/auvrrt.h"
#include "env.cuh"
#include "edge.cuh"

struct auvrrt_env {
    int device;
    auv::EnvHeader h32, h64;
    unsigned char *blob32, *blob64;   // device
    int K, E, H, T, C;
    double *h_bins;                   // host copy of bins[T][2] (owned, malloc)
    // host-call scratch (grown on demand, reused across calls)
    void *d_scratch[8];
    size_t d_scratch_bytes[8];
    void *h_pinned[4];
    size_t h_pinned_bytes[4];
    cudaStream_t stream;
};

namespace auv {

#define AUV_TRY(x) do { int rc_ = (x); if (rc_) return rc_; } while (0)

// fn<double>(args...) for AUVRRT_F64, fn<float>(args...) for AUVRRT_F32 (the caller has checked the precision)
#define AUV_DISPATCH(precision, fn, ...) ((precision) == AUVRRT_F64 ? fn<double>(__VA_ARGS__) : fn<float>(__VA_ARGS__))

// AUVRRT_OK with `device` current; "no CUDA device" (AUVRRT_ERR_CUDA) without one, AUVRRT_ERR_ARG out of range
int need_device(int device);

// A device allocation owned by one scope.  Zero bytes allocate 16, so every buffer has a valid address.
struct DBuf {
    void *p = nullptr;
    size_t bytes = 0;
    DBuf() = default;
    DBuf(const DBuf &) = delete;
    DBuf &operator=(const DBuf &) = delete;
    int alloc(size_t n) {
        bytes = n ? n : 16;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { p = nullptr; return set_err(AUVRRT_ERR_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); }
        return AUVRRT_OK;
    }
    template <typename T> T *as() { return (T *)p; }
    ~DBuf() { if (p) cudaFree(p); }
};

template <typename R> struct EnvBlob { const unsigned char *blob; int hot_bytes; int total_bytes; int off_probs; };
template <typename R> inline EnvBlob<R> env_blob(const auvrrt_env *e);
template <> inline EnvBlob<float> env_blob<float>(const auvrrt_env *e) {
    return EnvBlob<float>{e->blob32, e->h32.hot_bytes, e->h32.total_bytes, e->h32.off_probs};
}
template <> inline EnvBlob<double> env_blob<double>(const auvrrt_env *e) {
    return EnvBlob<double>{e->blob64, e->h64.hot_bytes, e->h64.total_bytes, e->h64.off_probs};
}

template <typename R> SteerParams<R> make_steer_params(const double p[5]);   // {d2e, dmax, freq, min_dist, vel}

// ---- kernels.cu
template <typename R>
int launch_steer_arc(const R *parents, int64_t n, const double *u, const int64_t *uoff, const double params[5],
                     R *leaf, int32_t *counts, R *wp, int wp_cap, int32_t *used, int32_t *status, cudaStream_t s);
template <typename R>
int launch_steer_dubins(const R *from, const R *to, int64_t n, double rho, int W, uint8_t *word, R *seg, R *length,
                        R *wp, cudaStream_t s);
template <typename R>
int launch_collide(const auvrrt_env *env, const R *points, const int64_t *off, int64_t n, uint8_t *safe, cudaStream_t s);
template <typename R>
int launch_collide_points(const auvrrt_env *env, const R *points, int64_t n, uint8_t *safe, cudaStream_t s);
template <typename R>
int launch_cost(const auvrrt_env *env, const R *points, const int64_t *off, int64_t n, const R *t_total,
                const double weights[3], unsigned bin_mask, int n_hab, R *out, cudaStream_t s);
template <typename R>
int launch_cost_point(const auvrrt_env *env, const R *points, int64_t n, unsigned long long visited, int tb,
                      const double weights[3], R *out, cudaStream_t s);
template <typename R>
int launch_edges_dubins(const auvrrt_env *env, const R *from, const R *to, int64_t n, double rho, int W,
                        uint8_t *safe, uint8_t *word, R *length, cudaStream_t s, double vel = 1.0, double w3 = 0.0,
                        R *cost_out = nullptr);
template <typename R>
int launch_edges_arc(const auvrrt_env *env, const R *parents, const uint64_t *seeds, int64_t n,
                     const double params[5], uint8_t *safe, int32_t *counts, R *leaf, cudaStream_t s, double w3 = 0.0,
                     R *cost_out = nullptr);
// ---- edges_tpe.cu: the same edges, one thread per edge (default); allpairs: no classification grid
template <typename R>
int launch_edges_arc_tpe(const auvrrt_env *env, const R *parents, const uint64_t *seeds, int64_t n, const double params[5],
                         uint8_t *safe, int32_t *counts, R *leaf, cudaStream_t s, double w3, R *cost_out, bool allpairs);
template <typename R>
int launch_nn(const R *tx, const R *ty, int64_t n, const R *qx, const R *qy, int nq, void *scratch,
              int64_t scratch_bytes, int32_t *out_idx, cudaStream_t s);
int64_t nn_scratch_bytes(int nq);
int launch_calibrate_fp32(int iters, double *flops, double *ms);
template <typename R> int launch_convert(const double *src, R *dst, int64_t n, cudaStream_t s);
template <typename R> int launch_convert_back(const R *src, double *dst, int64_t n, cudaStream_t s);

// ---- occupancy.cu: the one writer of both blobs' probs[T][C]: grid[b][cell_sq[c]] of a [T][RC] grid, or src[b][c]
// when cell_sq is NULL
int launch_probs_to_env(auvrrt_env *env, const double *src, const int *cell_sq, int RC, cudaStream_t s);

// ---- plan.cu
template <typename R>
int64_t plan_workspace_bytes(const auvrrt_env *env, const auvrrt_plan_params_t *p, int64_t Q);
template <typename R>
int launch_plan(const auvrrt_env *env, const R *starts, const uint64_t *seeds, int64_t Q,
                const auvrrt_plan_params_t *p, void *workspace, int64_t workspace_bytes,
                auvrrt_plan_record_t *records, uint32_t *chain, R *path, const auvrrt_plan_trace_t *trace,
                cudaStream_t s);
template <typename R>
int launch_materialize(const auvrrt_env *env, const R *starts, const uint64_t *seeds, const uint32_t *chain,
                       const int32_t *depth, int64_t Q, const auvrrt_plan_params_t *p, R *path, int32_t *n_path,
                       cudaStream_t s);

}  // namespace auv
