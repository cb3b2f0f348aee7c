// Shared host-side helpers for the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include <cstring>

#include "../../include/cppflow_b200.h"
#include "robots.cuh"
#include "geom.cuh"

namespace cppflow {

void set_last_error(const char* msg);
int fail(int code, const char* fmt, ...);

#define CPPFLOW_CHECK_ARG(cond, what)                                        \
    do {                                                                     \
        if (!(cond)) return ::cppflow::fail(CPPFLOW_E_INVALID, "%s: invalid argument: %s", __func__, what); \
    } while (0)

#define CPPFLOW_CHECK_LAUNCH()                                               \
    do {                                                                     \
        cudaError_t e_ = cudaGetLastError();                                 \
        if (e_ != cudaSuccess)                                               \
            return ::cppflow::fail(CPPFLOW_E_CUDA, "%s: CUDA error: %s", __func__, cudaGetErrorString(e_)); \
    } while (0)

// run `body` with `M` bound to the robot model type
#define CPPFLOW_DISPATCH_ROBOT(robot, ...)                                   \
    switch (robot) {                                                         \
        case ::cppflow::ROBOT_FETCH: { using M = ::cppflow::Fetch; __VA_ARGS__; } break;        \
        case ::cppflow::ROBOT_FETCH_ARM: { using M = ::cppflow::FetchArm; __VA_ARGS__; } break; \
        case ::cppflow::ROBOT_PANDA: { using M = ::cppflow::Panda; __VA_ARGS__; } break;        \
        default: return ::cppflow::fail(CPPFLOW_E_INVALID, "%s: unknown robot id %d", __func__, robot); \
    }

inline int make_obstacles(const float* h_cuboids, const float* h_Tcuboids, int n, Obstacles& ob) {
    std::memset(&ob, 0, sizeof(ob));
    if (n < 0 || n > CPPFLOW_MAX_OBSTACLES) return fail(CPPFLOW_E_INVALID, "n_obstacles %d out of range [0,8]", n);
    if (n > 0 && (!h_cuboids || !h_Tcuboids)) return fail(CPPFLOW_E_INVALID, "null obstacle tables");
    ob.n = n;
    for (int o = 0; o < n; ++o) {
        const float* c = h_cuboids + 6 * o;
        const float* T = h_Tcuboids + 16 * o;
        bool rot = false;
        for (int r = 0; r < 3; ++r) {
            ob.lo[o][r] = c[r];
            ob.hi[o][r] = c[3 + r];
            ob.t[o][r] = T[4 * r + 3];
            for (int k = 0; k < 3; ++k) {
                ob.R[o][3 * r + k] = T[4 * r + k];
                if (T[4 * r + k] != (r == k ? 1.f : 0.f)) rot = true;
            }
        }
        ob.has_rot[o] = rot ? 1 : 0;
    }
    return CPPFLOW_OK;
}

// path_metrics_tagged flag (internal, above the public CPPFLOW_METRICS_* bits): take the kernel one path of T waypoints
// gets (the clustered split, or one CTA per path when a path fits one CTA), whatever the number of paths
constexpr int METRICS_AS_ONE_PATH = 1 << 16;

// cppflow_path_metrics with a completion tag in column 7 of every row (k_metrics.cu)
int path_metrics_tagged(int robot, const float* d_q, const float* d_target, int64_t P, int64_t T, const float* h_cuboids,
                        const float* h_Tcuboids, int n_obstacles, float* d_out, float tag, void* stream, int flags = 0);

// pose-only LM step of one path (T <= 1024) fused with the metrics of the new path (k_metrics.cu)
int pose_step_metrics_tagged(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_target, int64_t T,
                             const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, float* d_x_out, float* d_out,
                             float tag, void* stream);
// the same for n_rows paths: path p is row rows[p] of d_q / d_x_out, its metrics go to d_out[p] (k_metrics.cu)
int pose_step_metrics_rows(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_target, int64_t T,
                           const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, const int* d_rows,
                           int64_t n_rows, float* d_x_out, float* d_out, float tag, void* stream);

inline unsigned grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }

// cudaFuncSetAttribute applies to the CURRENT device only: the opt-in to more than 48 KB of dynamic shared memory is
// remembered per (kernel instantiation, device ordinal), not per process.  `granted` is a static of the calling
// launch function; relaxed atomics make concurrent host threads at worst repeat the (idempotent) call.
constexpr int CPPFLOW_MAX_DEVICES = 64;
struct SmemGrant {
    std::atomic<size_t> bytes[CPPFLOW_MAX_DEVICES];
};
template <class K>
inline int ensure_dynamic_smem(K kernel, size_t bytes, SmemGrant& granted) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
    const bool tracked = dev >= 0 && dev < CPPFLOW_MAX_DEVICES;
    if (tracked && granted.bytes[dev].load(std::memory_order_relaxed) >= bytes) return CPPFLOW_OK;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (tracked) granted.bytes[dev].store(bytes, std::memory_order_relaxed);
    return CPPFLOW_OK;
}

}  // namespace cppflow
