// The alternating LM loop of lm_loop.cu for N seed paths of ONE problem, with the per-seed state in device memory:
// every kernel launch of an iteration covers all unfinished seeds and the host reads 3 integers per iteration, whatever N.
//
// An iteration, for the seeds listed by the previous one (pose-step seeds first, then differencing seeds):
//   1. pose-only step + metrics of the new path, one clustered launch over the pose list (path_metrics_kernel<FUSE>,
//      cluster c steps seed list[c]; G and the cluster size are the single-path values for T);
//   2. differencing step: gather the listed seeds into a contiguous [n_d, T, D] buffer, cppflow_lm_full_step with the
//      single loop's LOOP_STEP_FLAGS (segmented solve, S = 16: a path's result depends on S only, not on P), and the
//      metrics of the results with the kernel ONE path gets (METRICS_AS_ONE_PATH: path_metrics_tagged would switch to
//      one CTA per path for many paths, whose trajectory-length sum is added in another order);
//   3. decision kernel, one warp per listed seed: LoopState::finish of lm_loop.cu, check for check, in double; the warp
//      scatters a gathered result back and copies a valid iterate into the seed's x_valid row;
//   4. one CTA compacts the unfinished seeds (in seed order) into the next pose list and differencing list and writes
//      the two counts and a completion tag into page-locked host memory, which the host polls.
// Every seed therefore takes exactly the steps, decisions and bits of cppflow_lm_alternating_loss on that seed alone
// (last_metrics[7], which holds no metric, is 0 here and the single loop's completion tag there).
// The iterates live in two [N, T, D] buffers that swap roles every iteration: every unfinished seed steps every
// iteration, so a seed that stopped at iteration i holds its last iterate in buffer (i + 1) & 1.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstring>
#include <vector>

#include "common.cuh"

using namespace cppflow;

namespace {

inline size_t align256(size_t n) { return (n + 255) / 256 * 256; }

// the single-path loop's differencing step (lm_loop.cu): clamp + segmented solve with 16 segments
constexpr int LOOP_STEP_FLAGS = CPPFLOW_LM_CLAMP | CPPFLOW_LM_SEGMENTS(16);
constexpr int FUSED_MAX_T = 1024;  // pose_step_metrics_rows handles T <= 8 * MBLOCK

struct SeedState {
    double last_tl;
    int32_t last_valid_idx, n_tls, i_end;
    float m[8];  // metrics of the last iterate examined
    uint8_t pose_pos_valid, pose_rot_valid, converged, has_valid, done;
};

struct BatchedLayout {
    size_t x_bytes, off_xa, off_xb, off_valid, off_gin, off_gout, off_metrics, off_state, off_list, off_sched, off_counts,
        off_lm, total;
    BatchedLayout(int robot, int ndof, int64_t N, int64_t T) {
        x_bytes = align256((size_t)N * T * ndof * sizeof(float));
        off_xa = 0;
        off_xb = off_xa + x_bytes;
        off_valid = off_xb + x_bytes;
        off_gin = off_valid + x_bytes;
        off_gout = off_gin + x_bytes;
        off_metrics = off_gout + x_bytes;
        off_state = off_metrics + align256((size_t)N * 8 * sizeof(float));
        off_list = off_state + align256((size_t)N * sizeof(SeedState));
        off_sched = off_list + align256((size_t)N * sizeof(int));
        off_counts = off_sched + align256((size_t)N * CPPFLOW_LM_SCHEDULE_MAX);
        off_lm = off_counts + 256;
        total = off_lm + align256(cppflow_lm_full_workspace_bytes_ex(robot, N, T, LOOP_STEP_FLAGS));
    }
};

int robot_ndof(int robot) {
    cppflow_robot_info info;
    if (cppflow_robot_info_get(robot, &info) != CPPFLOW_OK) return -1;
    return info.ndof;
}

__global__ void lmb_init_kernel(int64_t N, SeedState* __restrict__ st, int* __restrict__ list) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= N) return;
    SeedState z;
    z.last_tl = 0.0;
    z.last_valid_idx = -1;
    z.n_tls = 0;
    z.i_end = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) z.m[k] = 0.f;
    z.pose_pos_valid = 1;  // the reference starts (True, False): the first step is pose-only (:219-220)
    z.pose_rot_valid = 0;
    z.converged = 0;
    z.has_valid = 0;
    z.done = 0;
    st[s] = z;
    list[s] = (int)s;
}

// dst row k = src row list[k], k in [0, n); rows of `row` floats
__global__ void lmb_gather_kernel(const float* __restrict__ src, const int* __restrict__ list, int64_t n, int64_t row,
                                  float* __restrict__ dst) {
    const int64_t total = n * row;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = e / row, c = e - k * row;
        dst[e] = __ldg(src + (int64_t)__ldg(list + k) * row + c);
    }
}

struct DecideArgs {
    const int* list;
    const float* metrics;  // [n, 8] in list order
    int64_t n, n_pose;     // slots [0, n_pose) took a pose step, [n_pose, n) a differencing step
    int64_t scatter_from;  // slots >= scatter_from have their new iterate in `gathered` row k, not yet in x_new
    const float* gathered;
    float* x_new;
    float* x_valid;
    int64_t row;  // T * ndof
    int it;
    int max_n_steps, return_if_valid_after_n_steps;
    double convergence_threshold;
    cppflow_constraints c;
    SeedState* st;
    char* sched;  // [N, CPPFLOW_LM_SCHEDULE_MAX]
};

// LoopState::finish (lm_loop.cu) for the seed of slot k: same checks in the same order, float32 metrics against the
// double thresholds and the trajectory-length difference in double.  The time limit is the host's (it stops every
// unfinished seed after this decision, where the single loop checks it).  Returns 1 when x_new is a valid iterate.
__device__ __forceinline__ int lmb_decide(const DecideArgs& a, SeedState& s, const float (&m)[8], bool was_differencing) {
    const int i = a.it;
    const double tl_new = m[4];
    if (was_differencing) {
        if (!s.converged && s.n_tls > 0) {
            if (fabs(tl_new - s.last_tl) < a.convergence_threshold) {
                s.converged = 1;
                if (s.last_valid_idx == i - 1) { s.done = 1; s.i_end = i; return 0; }
            }
        }
        s.last_tl = tl_new;
        ++s.n_tls;
    }
    s.pose_pos_valid = (double)m[0] < a.c.max_allowed_position_error_cm;
    s.pose_rot_valid = (double)m[1] < a.c.max_allowed_rotation_error_deg;
    const bool mjac_ok = (double)m[2] < a.c.max_allowed_mjac_deg && (double)m[3] < a.c.max_allowed_mjac_cm;
    const bool is_valid = s.pose_pos_valid && s.pose_rot_valid && mjac_ok && !(m[5] < 0.f) && !(m[6] < 0.f);
    if (is_valid) {
        s.last_valid_idx = i;
        s.has_valid = 1;
        if (s.converged) { s.done = 1; s.i_end = i; return 1; }
    }
    if (s.has_valid && (i > a.return_if_valid_after_n_steps || i > a.max_n_steps)) { s.done = 1; s.i_end = i; }
    else if (i + 1 >= a.max_n_steps) { s.done = 1; s.i_end = i; }  // Python's range() exhausted: i stays
    return is_valid ? 1 : 0;
}

// one warp per listed seed: lane 0 decides, the warp moves the rows
__global__ void __launch_bounds__(256) lmb_decide_kernel(const DecideArgs a) {
    const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= a.n) return;
    const int64_t s = __ldg(a.list + k);
    int valid = 0;
    if (lane == 0) {
        float m[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = a.metrics[k * 8 + j];
        SeedState st = a.st[s];
        const bool was_differencing = k >= a.n_pose;
        if (a.it < CPPFLOW_LM_SCHEDULE_MAX - 1) a.sched[s * CPPFLOW_LM_SCHEDULE_MAX + a.it] = was_differencing ? 'd' : 'p';
#pragma unroll
        for (int j = 0; j < 8; ++j) st.m[j] = m[j];
        valid = lmb_decide(a, st, m, was_differencing);
        a.st[s] = st;
    }
    valid = __shfl_sync(0xffffffffu, valid, 0);
    const bool scatter = k >= a.scatter_from;
    if (!scatter && !valid) return;
    const float* src = scatter ? a.gathered + k * a.row : a.x_new + s * a.row;
    float* xn = a.x_new + s * a.row;
    float* xv = a.x_valid + s * a.row;
    for (int64_t e = lane; e < a.row; e += 32) {
        const float v = src[e];
        if (scatter) xn[e] = v;
        if (valid) xv[e] = v;
    }
}

// one CTA: unfinished seeds in seed order -> list = [pose seeds..., differencing seeds...]; counts + tag to `out`
constexpr int COMPACT_BLOCK = 1024;
__global__ void __launch_bounds__(COMPACT_BLOCK)
lmb_compact_kernel(const SeedState* __restrict__ st, int64_t N, int* __restrict__ list, int* out, int tag) {
    __shared__ int s_warp[2][COMPACT_BLOCK / 32];
    __shared__ int s_base[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // pass 0 counts the pose seeds (the differencing seeds start after them), pass 1 writes the list
    int n_pose = 0;
    for (int pass = 0; pass < 2; ++pass) {
        if (threadIdx.x == 0) { s_base[0] = 0; s_base[1] = n_pose; }
        __syncthreads();
        for (int64_t c0 = 0; c0 < N; c0 += COMPACT_BLOCK) {
            const int64_t s = c0 + threadIdx.x;
            int kind = 0;  // 0 finished, 1 pose step, 2 differencing step
            if (s < N) {
                const SeedState& x = st[s];
                kind = x.done ? 0 : (x.pose_pos_valid && x.pose_rot_valid ? 2 : 1);
            }
            const unsigned bp = __ballot_sync(0xffffffffu, kind == 1), bd = __ballot_sync(0xffffffffu, kind == 2);
            if (lane == 0) { s_warp[0][warp] = __popc(bp); s_warp[1][warp] = __popc(bd); }
            __syncthreads();
            if (pass == 1 && kind != 0) {
                const int w = kind - 1;
                int off = s_base[w];
                for (int j = 0; j < warp; ++j) off += s_warp[w][j];
                off += __popc((w == 0 ? bp : bd) & ((1u << lane) - 1u));
                list[off] = (int)s;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                for (int j = 0; j < COMPACT_BLOCK / 32; ++j) { s_base[0] += s_warp[0][j]; s_base[1] += s_warp[1][j]; }
            }
            __syncthreads();
        }
        n_pose = s_base[0];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = s_base[0];
        out[1] = s_base[1] - s_base[0];
        __threadfence_system();  // `out` may be host memory polled by the CPU: the tag must not overtake the counts
        *reinterpret_cast<volatile int*>(out + 2) = tag;
    }
}

// result rows: the last valid iterate, else the last iterate; seeds still running (time limit) stop at iteration it_stop
__global__ void lmb_finalize_kernel(SeedState* __restrict__ st, int64_t N, int it_stop, int stepped,
                                    const float* __restrict__ xa, const float* __restrict__ xb,
                                    const float* __restrict__ xv, int64_t row, float* __restrict__ out) {
    const int64_t s = blockIdx.x;
    if (s >= N) return;
    __shared__ int s_src;
    if (threadIdx.x == 0) {
        SeedState& x = st[s];
        if (!x.done) { x.done = 1; x.i_end = it_stop; }
        s_src = x.has_valid ? 2 : (stepped && ((x.i_end + 1) & 1) ? 1 : 0);
    }
    __syncthreads();
    const float* src = (s_src == 2 ? xv : s_src == 1 ? xb : xa) + s * row;
    for (int64_t e = threadIdx.x; e < row; e += blockDim.x) out[s * row + e] = src[e];
}

}  // namespace

extern "C" size_t cppflow_lm_alternating_batched_workspace_bytes(int robot, int64_t n_seeds, int64_t T) {
    const int ndof = robot_ndof(robot);
    if (ndof < 0 || n_seeds <= 0 || T <= 0) return 0;
    return BatchedLayout(robot, ndof, n_seeds, T).total;
}

extern "C" int cppflow_lm_alternating_loss_batched(
    int robot, const cppflow_lm_params* params_diff, const cppflow_lm_params* params_pose,
    const cppflow_constraints* constraints, const float* d_x_seeds, const float* d_target, int64_t n_seeds, int64_t T,
    const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, int max_n_steps, double tmax_sec,
    int return_if_valid_after_n_steps, double convergence_threshold, void* d_workspace, size_t workspace_bytes,
    int32_t* h_pinned, float* d_x_out, cppflow_lm_loop_result* results, void* stream) {
    CPPFLOW_CHECK_ARG(n_seeds >= 0, "n_seeds");
    if (n_seeds == 0) return CPPFLOW_OK;
    CPPFLOW_CHECK_ARG(params_diff && params_pose && constraints && results, "null parameter struct");
    CPPFLOW_CHECK_ARG(d_x_seeds && d_target && d_workspace && h_pinned && d_x_out, "null pointer");
    CPPFLOW_CHECK_ARG(T > 0 && max_n_steps >= 0, "T, max_n_steps");
    CPPFLOW_CHECK_ARG(n_seeds <= INT32_MAX, "n_seeds");
    const int ndof = robot_ndof(robot);
    if (ndof < 0) return CPPFLOW_E_INVALID;
    Obstacles ob_check;
    if (int rc = make_obstacles(h_cuboids, h_Tcuboids, n_obstacles, ob_check)) return rc;
    const BatchedLayout L(robot, ndof, n_seeds, T);
    if (workspace_bytes < L.total)
        return fail(CPPFLOW_E_WORKSPACE, "lm_alternating_loss_batched: workspace too small (%zu < %zu)", workspace_bytes,
                    L.total);
    CPPFLOW_CHECK_ARG(((uintptr_t)d_workspace & 255) == 0, "workspace must be 256-byte aligned");

    cudaStream_t st = (cudaStream_t)stream;
    const int64_t N = n_seeds, row = T * ndof;
    const size_t row_bytes = (size_t)row * sizeof(float);
    unsigned char* ws = (unsigned char*)d_workspace;
    float* xa = (float*)(ws + L.off_xa);
    float* xb = (float*)(ws + L.off_xb);
    float* x_valid = (float*)(ws + L.off_valid);
    float* gin = (float*)(ws + L.off_gin);
    float* gout = (float*)(ws + L.off_gout);
    float* metrics = (float*)(ws + L.off_metrics);
    SeedState* state = (SeedState*)(ws + L.off_state);
    int* list = (int*)(ws + L.off_list);
    char* sched = (char*)(ws + L.off_sched);
    int* d_counts = (int*)(ws + L.off_counts);
    void* lm_ws = ws + L.off_lm;
    const size_t lm_ws_bytes = L.total - L.off_lm;

    // on an error return no kernel may still be in flight: it would write its tag into the pinned buffer (and rows into
    // the workspace) that the caller is about to reuse.  The last error text is kept.
    auto bail = [&](int rc) {
        cudaStreamSynchronize(st);
        cudaGetLastError();
        return rc;
    };
    auto cuda_fail = [&](cudaError_t e) {
        return bail(fail(CPPFLOW_E_CUDA, "lm_alternating_loss_batched: %s", cudaGetErrorString(e)));
    };

    // page-locked host memory is device-addressable under unified addressing: the compaction kernel writes the counts
    // and the tag there directly; otherwise into device scratch, copied after it
    cudaPointerAttributes pa;
    const bool zero_copy = cudaPointerGetAttributes(&pa, h_pinned) == cudaSuccess && pa.type == cudaMemoryTypeHost &&
                           pa.devicePointer != nullptr;
    if (!zero_copy) cudaGetLastError();
    int* counts_dst = zero_copy ? (int*)pa.devicePointer : d_counts;
    static std::atomic<unsigned> call_counter{0};
    const unsigned nonce = (call_counter.fetch_add(1, std::memory_order_relaxed) & 0xfffu) + 1u;

    cudaError_t e = cudaMemcpyAsync(xa, d_x_seeds, (size_t)N * row_bytes, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return cuda_fail(e);
    e = cudaMemsetAsync(sched, 0, (size_t)N * CPPFLOW_LM_SCHEDULE_MAX, st);
    if (e != cudaSuccess) return cuda_fail(e);
    lmb_init_kernel<<<grid_for(N, 256), 256, 0, st>>>(N, state, list);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e);
    const auto t0 = std::chrono::steady_clock::now();

    int64_t n_pose = N, n_diff = 0;
    int it = 0;
    if (max_n_steps > 0) {
        for (;; ++it) {
            float* x_cur = (it & 1) ? xb : xa;
            float* x_new = (it & 1) ? xa : xb;
            const int tag = (int)((nonce << 8) + (unsigned)(it % 255) + 1u);
            if (zero_copy) reinterpret_cast<volatile int*>(h_pinned)[2] = 0;  // not this iteration's tag
            const int64_t n_act = n_pose + n_diff;
            const bool fused = T <= FUSED_MAX_T;
            // slots [g0, n_act) are stepped on the gathered copy: the differencing seeds, and the pose seeds too for long
            // paths (pose step, then the metrics, as in the single loop)
            const int64_t g0 = fused ? n_pose : 0;
            if (fused && n_pose > 0)
                if (int rc = pose_step_metrics_rows(robot, params_pose, x_cur, d_target, T, h_cuboids, h_Tcuboids, n_obstacles,
                                                    list, n_pose, x_new, metrics, 0.f, st))
                    return bail(rc);
            if (n_act > g0) {
                const int64_t n_g = n_act - g0;
                const int64_t total = n_g * row;
                const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, 148 * 16);
                lmb_gather_kernel<<<blocks, 256, 0, st>>>(x_cur, list + g0, n_g, row, gin + g0 * row);
                if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e);
                if (!fused && n_pose > 0)
                    if (int rc = cppflow_lm_pose_step(robot, params_pose, gin, d_target, n_pose * T, T, 1, gout, nullptr,
                                                      nullptr, st))
                        return bail(rc);
                if (n_diff > 0)
                    if (int rc = cppflow_lm_full_step(robot, params_diff, gin + n_pose * row, nullptr, d_target, n_diff, T,
                                                      h_cuboids, h_Tcuboids, n_obstacles, LOOP_STEP_FLAGS, lm_ws, lm_ws_bytes,
                                                      gout + n_pose * row, st))
                        return bail(rc);
                if (int rc = path_metrics_tagged(robot, gout + g0 * row, d_target, n_g, T, h_cuboids, h_Tcuboids, n_obstacles,
                                                 metrics + g0 * 8, 0.f, st, METRICS_AS_ONE_PATH))
                    return bail(rc);
            }
            DecideArgs a;
            a.list = list;
            a.metrics = metrics;
            a.n = n_act;
            a.n_pose = n_pose;
            a.scatter_from = g0;
            a.gathered = gout;
            a.x_new = x_new;
            a.x_valid = x_valid;
            a.row = row;
            a.it = it;
            a.max_n_steps = max_n_steps;
            a.return_if_valid_after_n_steps = return_if_valid_after_n_steps;
            a.convergence_threshold = convergence_threshold;
            a.c = *constraints;
            a.st = state;
            a.sched = sched;
            lmb_decide_kernel<<<grid_for(n_act * 32, 256), 256, 0, st>>>(a);
            if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e);
            lmb_compact_kernel<<<1, COMPACT_BLOCK, 0, st>>>(state, N, list, counts_dst, tag);
            if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e);
            if (!zero_copy) {
                e = cudaMemcpyAsync(h_pinned, d_counts, 3 * sizeof(int), cudaMemcpyDeviceToHost, st);
                if (e != cudaSuccess) return cuda_fail(e);
            }
            // the one host round trip of the iteration: poll the tag (~1 us after the kernel's last store); if it does
            // not show up within a second - a faulting kernel never writes it - synchronise the stream for the error
            bool seen = false;
            if (zero_copy) {
                const volatile int* flag = reinterpret_cast<const volatile int*>(h_pinned) + 2;
                const auto t_poll = std::chrono::steady_clock::now();
                for (unsigned spin = 0; !(seen = (*flag == tag)); ++spin) {
                    if ((spin & 0xfff) == 0xfff &&
                        std::chrono::duration<double>(std::chrono::steady_clock::now() - t_poll).count() > 1.0)
                        break;
                }
                std::atomic_thread_fence(std::memory_order_acquire);
            }
            if (!seen && (e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail(e);
            n_pose = reinterpret_cast<const volatile int*>(h_pinned)[0];
            n_diff = reinterpret_cast<const volatile int*>(h_pinned)[1];
            if (n_pose + n_diff == 0) break;
            // the single loop checks the time after the decisions of the iteration: every seed still running stops here
            const double elapsed = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (elapsed > tmax_sec) break;
        }
    }
    lmb_finalize_kernel<<<(unsigned)N, 256, 0, st>>>(state, N, it, max_n_steps > 0 ? 1 : 0, xa, xb, x_valid, row, d_x_out);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e);
    std::vector<SeedState> h_state((size_t)N);
    std::vector<char> h_sched((size_t)N * CPPFLOW_LM_SCHEDULE_MAX);
    e = cudaMemcpyAsync(h_state.data(), state, (size_t)N * sizeof(SeedState), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(h_sched.data(), sched, h_sched.size(), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e);
    for (int64_t s = 0; s < N; ++s) {
        const SeedState& x = h_state[(size_t)s];
        cppflow_lm_loop_result& r = results[s];
        const int n_sched = max_n_steps > 0 ? std::min(x.i_end + 1, CPPFLOW_LM_SCHEDULE_MAX - 1) : 0;
        std::memcpy(r.schedule, &h_sched[(size_t)s * CPPFLOW_LM_SCHEDULE_MAX], (size_t)n_sched);
        r.schedule[n_sched] = 0;
        r.n_steps_taken = x.i_end;
        r.is_valid = x.has_valid ? 1 : 0;
        for (int k = 0; k < 7; ++k) r.last_metrics[k] = x.m[k];
        r.last_metrics[7] = 0.f;  // no metric: the single loop leaves its completion tag there
    }
    return CPPFLOW_OK;
}
