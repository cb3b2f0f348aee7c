// Host-side driver of the alternating LM loop for ONE path: the control flow of run_lm_alternating_loss
// (optimization.py:147-373) in C++, on top of the kernels' C entry points.
//
// The reference decides the type of the next step from the validity of the current iterate (pose-only until position
// and rotation errors are inside the constraints, joint-differencing otherwise, :219-260), watches the trajectory length
// after differencing steps for convergence (:268-283) and keeps the last valid iterate (:318-352).  Every iteration
// therefore needs a device -> host read of the path metrics (the reference's `.item()` calls, :175).  Here that read
// is 8 floats into page-locked memory and one cudaStreamSynchronize; the kernel launches, the decision logic and the
// bookkeeping of an iteration cost ~10 us of host time instead of ~55 us when driven from Python through ctypes
// (the per-plan latency of fetch__circle is dominated by these 20 round trips, not by the kernels).
#include <atomic>
#include <chrono>
#include <cmath>
#include <vector>

#include "common.cuh"

using namespace cppflow;

namespace {

inline size_t align256(size_t n) { return (n + 255) / 256 * 256; }

// The differencing step of ONE path is the block solve's dependent chain and nothing else: it takes the segmented
// solve (csrc/lm_segsolve.cuh; 0.098 -> 0.046 ms for T = 300) with 16 segments.  ops.LOOP_SEGMENTS must be the same
// number: the Python loop then takes the same solve and returns the same bits.
constexpr int LOOP_STEP_FLAGS = CPPFLOW_LM_CLAMP | CPPFLOW_LM_SEGMENTS(16);

struct LoopLayout {
    size_t x_bytes, off_xa, off_xb, off_valid, off_metrics, off_lm, total;
    LoopLayout(int robot, int ndof, int64_t T) {
        if (ndof <= 0) { x_bytes = off_xa = off_xb = off_valid = off_metrics = off_lm = total = 0; return; }
        x_bytes = align256((size_t)T * ndof * sizeof(float));
        off_xa = 0;
        off_xb = off_xa + x_bytes;
        off_valid = off_xb + x_bytes;
        off_metrics = off_valid + x_bytes;
        off_lm = off_metrics + 256;
        total = off_lm + align256(cppflow_lm_full_workspace_bytes_ex(robot, 1, T, LOOP_STEP_FLAGS));
    }
};

int robot_ndof(int robot) {
    cppflow_robot_info info;
    if (cppflow_robot_info_get(robot, &info) != CPPFLOW_OK) return -1;
    return info.ndof;
}

}  // namespace

extern "C" size_t cppflow_lm_alternating_workspace_bytes(int robot, int64_t T) {
    const int ndof = robot_ndof(robot);
    if (ndof < 0 || T <= 0) return 0;
    return LoopLayout(robot, ndof, T).total;
}

namespace {

// One path's alternating loop as a state machine: launch() enqueues the next step, the metrics kernel and the
// device -> host copy of the 8 metrics on the job's stream; finish() waits for them and takes the reference's decisions.
// The single-path entry point runs launch/finish in turn; the many-path entry point launches the step of EVERY active
// job before it waits for any of them, so independent problems overlap on the device.
struct LoopState {
    const cppflow_lm_loop_job* job = nullptr;
    LoopLayout L{0, 0, 1};
    int ndof = 0;
    float *x_cur = nullptr, *x_new = nullptr, *x_valid = nullptr, *d_metrics = nullptr;
    void* lm_ws = nullptr;
    size_t lm_ws_bytes = 0, row_bytes = 0;
    bool pose_pos_valid = true, pose_rot_valid = false;  // the reference starts (True, False): first step pose-only (:219-220)
    bool converged = false, has_valid = false, was_differencing = false, done = false;
    int last_valid_idx = -1, n_tls = 0, i = 0, n_sched = 0;
    double last_tl = 0.0;
    std::chrono::steady_clock::time_point t0;
    float tag = 0.f;               // completion tag of the iteration in flight: (per-call nonce << 8) + (i mod 255) + 1
    unsigned nonce = 0;            // distinguishes this call's tags from stale ones of an earlier (failed) call that
                                   // shared the pinned buffer; < 2^12, so every tag is an exact float below 2^20
    float* metrics_dst = nullptr;  // where the metrics kernel writes: the pinned host buffer itself when the device can
    bool zero_copy = false;        // address it (no copy engine round trip per iteration), the device scratch otherwise

    int init(const cppflow_lm_loop_job* j) {
        job = j;
        if (!(j->params_diff && j->params_pose && j->constraints && j->result)) return fail(CPPFLOW_E_INVALID, "lm_alternating_loss: null parameter struct");
        if (!(j->d_x_seed && j->d_target && j->d_x_out && j->d_workspace && j->h_pinned_metrics)) return fail(CPPFLOW_E_INVALID, "lm_alternating_loss: null pointer");
        if (!(j->T > 0 && j->max_n_steps >= 0)) return fail(CPPFLOW_E_INVALID, "lm_alternating_loss: T, max_n_steps");
        ndof = robot_ndof(j->robot);
        if (ndof < 0) return CPPFLOW_E_INVALID;
        L = LoopLayout(j->robot, ndof, j->T);
        if (j->workspace_bytes < L.total)
            return fail(CPPFLOW_E_WORKSPACE, "lm_alternating_loss: workspace too small (%zu < %zu)", j->workspace_bytes, L.total);
        if (((uintptr_t)j->d_workspace & 255) != 0) return fail(CPPFLOW_E_INVALID, "lm_alternating_loss: workspace must be 256-byte aligned");
        unsigned char* ws = (unsigned char*)j->d_workspace;
        x_cur = (float*)(ws + L.off_xa);
        x_new = (float*)(ws + L.off_xb);
        x_valid = (float*)(ws + L.off_valid);
        d_metrics = (float*)(ws + L.off_metrics);
        lm_ws = ws + L.off_lm;
        lm_ws_bytes = L.total - L.off_lm;
        row_bytes = (size_t)j->T * ndof * sizeof(float);
        cudaError_t e = cudaMemcpyAsync(x_cur, j->d_x_seed, row_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)j->stream);
        if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_alternating_loss: %s", cudaGetErrorString(e));
        // page-locked host memory is device-addressable under unified addressing: let the 8 metrics of an iterate land
        // there directly (a 32-byte write over PCIe at the end of the kernel) instead of copying them afterwards
        cudaPointerAttributes pa;
        zero_copy = cudaPointerGetAttributes(&pa, j->h_pinned_metrics) == cudaSuccess && pa.type == cudaMemoryTypeHost &&
                    pa.devicePointer != nullptr;
        if (!zero_copy) cudaGetLastError();  // unregistered host memory reports an error: not fatal, copy instead
        metrics_dst = zero_copy ? (float*)pa.devicePointer : d_metrics;
        static std::atomic<unsigned> call_counter{0};
        nonce = (call_counter.fetch_add(1, std::memory_order_relaxed) & 0xfffu) + 1u;
        t0 = std::chrono::steady_clock::now();
        done = j->max_n_steps == 0;
        return CPPFLOW_OK;
    }

    int launch() {
        const cppflow_lm_loop_job* j = job;
        tag = (float)((nonce << 8) + (unsigned)(i % 255) + 1u);
        if (zero_copy) *reinterpret_cast<volatile float*>(j->h_pinned_metrics + 7) = 0.f;  // not this iteration's tag
        bool metrics_done = false;
        if (pose_pos_valid && pose_rot_valid) {
            // virtual configs = the current iterate (:253): their residual is identically zero -> d_xv = NULL
            if (int rc = cppflow_lm_full_step(j->robot, j->params_diff, x_cur, nullptr, j->d_target, 1, j->T, j->h_cuboids,
                                              j->h_Tcuboids, j->n_obstacles, LOOP_STEP_FLAGS, lm_ws, lm_ws_bytes, x_new, j->stream))
                return rc;
            was_differencing = true;
        } else if (j->T <= 1024) {
            // pose-only step and the metrics of its result in ONE launch (both kernels are launch-bound for one path)
            if (int rc = pose_step_metrics_tagged(j->robot, j->params_pose, x_cur, j->d_target, j->T, j->h_cuboids, j->h_Tcuboids,
                                                  j->n_obstacles, x_new, metrics_dst, tag, j->stream))
                return rc;
            was_differencing = false;
            metrics_done = true;
        } else {
            if (int rc = cppflow_lm_pose_step(j->robot, j->params_pose, x_cur, j->d_target, j->T, j->T, 1, x_new, nullptr, nullptr, j->stream))
                return rc;
            was_differencing = false;
        }
        if (n_sched < CPPFLOW_LM_SCHEDULE_MAX - 1) j->result->schedule[n_sched++] = was_differencing ? 'd' : 'p';
        float* tmp = x_cur; x_cur = x_new; x_new = tmp;  // clamp_to_joint_limits is fused into both steps (:259)
        if (!metrics_done)
            if (int rc = path_metrics_tagged(j->robot, x_cur, j->d_target, 1, j->T, j->h_cuboids, j->h_Tcuboids, j->n_obstacles,
                                             metrics_dst, tag, j->stream))
                return rc;
        if (!zero_copy) {
            cudaError_t e = cudaMemcpyAsync(j->h_pinned_metrics, d_metrics, 8 * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)j->stream);
            if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_alternating_loss: %s", cudaGetErrorString(e));
        }
        return CPPFLOW_OK;
    }

    int finish() {
        const cppflow_lm_loop_job* j = job;
        // the one host round trip of the iteration.  With the metrics landing in host memory the CPU polls their tag
        // (~1 us after the kernel's last store) instead of going through cudaStreamSynchronize; if the tag does not
        // show up within a second - a faulting kernel never writes it - the stream is synchronised for the error.
        cudaError_t e = cudaSuccess;
        bool seen = false;
        if (zero_copy) {
            const volatile float* flag = j->h_pinned_metrics + 7;
            const auto t_poll = std::chrono::steady_clock::now();
            for (unsigned spin = 0; !(seen = (*flag == tag)); ++spin) {
                if ((spin & 0xfff) == 0xfff &&
                    std::chrono::duration<double>(std::chrono::steady_clock::now() - t_poll).count() > 1.0)
                    break;
            }
            std::atomic_thread_fence(std::memory_order_acquire);
        }
        if (!seen) e = cudaStreamSynchronize((cudaStream_t)j->stream);
        if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_alternating_loss: %s", cudaGetErrorString(e));
        const float* m = j->h_pinned_metrics;  // max_pos_cm, max_rot_deg, mjac_deg, mjac_cm, tl, min_self, min_env
        const double tl_new = m[4];
        if (was_differencing) {
            if (!converged && n_tls > 0) {
                if (std::fabs(tl_new - last_tl) < j->convergence_threshold) {
                    converged = true;
                    if (last_valid_idx == i - 1) { done = true; return CPPFLOW_OK; }
                }
            }
            last_tl = tl_new;
            ++n_tls;
        }
        // x_is_valid (:836-923): strict '<' thresholds (evaluation_utils.py:29-75), then the collision check
        const cppflow_constraints* c = j->constraints;
        // float32 metrics against double thresholds, as the reference's `tensor < python float` comparisons do
        pose_pos_valid = (double)m[0] < c->max_allowed_position_error_cm;
        pose_rot_valid = (double)m[1] < c->max_allowed_rotation_error_deg;
        const bool mjac_ok = (double)m[2] < c->max_allowed_mjac_deg && (double)m[3] < c->max_allowed_mjac_cm;
        const bool is_valid = pose_pos_valid && pose_rot_valid && mjac_ok && !(m[5] < 0.f) && !(m[6] < 0.f);
        if (is_valid) {
            last_valid_idx = i;
            has_valid = true;
            e = cudaMemcpyAsync(x_valid, x_cur, row_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)j->stream);
            if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_alternating_loss: %s", cudaGetErrorString(e));
            if (converged) { done = true; return CPPFLOW_OK; }
        }
        const double elapsed = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (elapsed > j->tmax_sec) { done = true; return CPPFLOW_OK; }
        if (has_valid && (i > j->return_if_valid_after_n_steps || i > j->max_n_steps)) { done = true; return CPPFLOW_OK; }
        if (i + 1 >= j->max_n_steps) { done = true; return CPPFLOW_OK; }  // Python's range() exhausted: i stays at the last value
        ++i;
        return CPPFLOW_OK;
    }

    int finalize() {
        const cppflow_lm_loop_job* j = job;
        cudaError_t e = cudaMemcpyAsync(j->d_x_out, has_valid ? x_valid : x_cur, row_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)j->stream);
        if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_alternating_loss: %s", cudaGetErrorString(e));
        j->result->schedule[n_sched] = 0;
        j->result->n_steps_taken = i;
        j->result->is_valid = has_valid ? 1 : 0;
        for (int k = 0; k < 8; ++k) j->result->last_metrics[k] = j->max_n_steps > 0 ? j->h_pinned_metrics[k] : 0.f;
        return CPPFLOW_OK;
    }
};

}  // namespace

extern "C" int cppflow_lm_alternating_loss_many(int n_jobs, const cppflow_lm_loop_job* jobs) {
    CPPFLOW_CHECK_ARG(n_jobs >= 0 && (n_jobs == 0 || jobs != nullptr), "jobs");
    std::vector<LoopState> st((size_t)n_jobs);
    // on an error return no kernel of any job may still be in flight: it would write its tag into a pinned buffer
    // (and its iterate into a workspace) that the caller is about to reuse.  The last error text is kept.
    auto bail = [&](int rc) {
        for (int k = 0; k < n_jobs; ++k) cudaStreamSynchronize((cudaStream_t)jobs[k].stream);
        cudaGetLastError();
        return rc;
    };
    for (int k = 0; k < n_jobs; ++k)
        if (int rc = st[k].init(&jobs[k])) return bail(rc);
    for (;;) {
        int n_active = 0;
        for (int k = 0; k < n_jobs; ++k)
            if (!st[k].done) {
                if (int rc = st[k].launch()) return bail(rc);
                ++n_active;
            }
        if (n_active == 0) break;
        for (int k = 0; k < n_jobs; ++k)
            if (!st[k].done)
                if (int rc = st[k].finish()) return bail(rc);
    }
    for (int k = 0; k < n_jobs; ++k)
        if (int rc = st[k].finalize()) return bail(rc);
    return CPPFLOW_OK;
}

extern "C" int cppflow_lm_alternating_loss(int robot, const cppflow_lm_params* params_diff,
                                           const cppflow_lm_params* params_pose, const cppflow_constraints* constraints,
                                           const float* d_x_seed, const float* d_target, int64_t T,
                                           const float* h_cuboids, const float* h_Tcuboids, int n_obstacles,
                                           int max_n_steps, double tmax_sec, int return_if_valid_after_n_steps,
                                           double convergence_threshold, void* d_workspace, size_t workspace_bytes,
                                           float* h_pinned_metrics, float* d_x_out, cppflow_lm_loop_result* result,
                                           void* stream) {
    cppflow_lm_loop_job job;
    job.robot = robot;
    job.params_diff = params_diff;
    job.params_pose = params_pose;
    job.constraints = constraints;
    job.d_x_seed = d_x_seed;
    job.d_target = d_target;
    job.T = T;
    job.h_cuboids = h_cuboids;
    job.h_Tcuboids = h_Tcuboids;
    job.n_obstacles = n_obstacles;
    job.max_n_steps = max_n_steps;
    job.tmax_sec = tmax_sec;
    job.return_if_valid_after_n_steps = return_if_valid_after_n_steps;
    job.convergence_threshold = convergence_threshold;
    job.d_workspace = d_workspace;
    job.workspace_bytes = workspace_bytes;
    job.h_pinned_metrics = h_pinned_metrics;
    job.d_x_out = d_x_out;
    job.result = result;
    job.stream = stream;
    return cppflow_lm_alternating_loss_many(1, &job);
}
