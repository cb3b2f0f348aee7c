// Exact IK from IKFlow's samples (include/cppflow_b200.h: cppflow_ik_refine, cppflow_ik_round_inputs,
// cppflow_ik_select): per-row pose-only LM refinement with early exit, the latents of a resampling round, and the
// per-target choice of a converged sample with the order-preserving compaction of the targets left unsolved.
//
// Reference being replaced (restated from memory of ikflow's public code, not checked against it):
//   ikflow IKFlowSolver.generate_exact_ik_solutions: sample, batched LM IK, resample the unconverged targets
//   levenberg_marquardt_only_pose + clamp_to_joint_limits     (optimization.py:61-92, optimization_utils.py:823-833)
//   get_6d_pose_errors                                         (optimization_utils.py:802-820)
//   Robot.self_collision_distances                             (collision_detection.py:65)
#include <climits>

#include <cub/device/device_select.cuh>

#include "common.cuh"
#include "collision.cuh"
#include "pose_step.cuh"
#include "rng.cuh"

namespace cppflow {

constexpr int IK_BLOCK = 128;

// |(a, b, c)| rounded step by step, so that a host check in FP32 ((a*a + b*b) + c*c, then sqrt) gives the same bits
__device__ __forceinline__ float norm3_rn(float a, float b, float c) {
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c)));
}

// The stopping rule of a row: pose error inside the tolerances (strict <) and, with SELF, every capsule self pair at
// d > 0.  Pairs whose bounding spheres prove them apart are not evaluated (self_pair_distance with cull_thr = 0).
template <class M, bool SELF>
__device__ __forceinline__ bool ik_converged(const float (&x)[M::NDOF], const float (&tg)[7], float pos_tol, float rot_tol,
                                             float* sm, float& e_pos, float& e_rot) {
    Frame F;
    if constexpr (SELF) {
        CollisionSink<M, IK_BLOCK, false> sink{sm};
        fk_chain<M>(x, sink, F);
    } else {
        NullSink sink;
        fk_chain<M>(x, sink, F);
    }
    float e[6];
    pose_error(tg, F, e);
    e_rot = norm3_rn(e[0], e[1], e[2]);
    e_pos = norm3_rn(e[3], e[4], e[5]);
    bool ok = e_pos < pos_tol && e_rot < rot_tol;
    if constexpr (SELF) {
        for (int p = 0; p < M::NPAIR && ok; ++p) {
            float C2[3], nrm[3];
            ok = self_pair_distance<M, IK_BLOCK>(sm, p, C2, nrm, 0.f) > 0.f;
        }
    }
    return ok;
}

// One thread per row; q and the target stay in registers for all steps.  q_in and q_out may alias: a row is read
// before it is written, by the same thread.
template <class M, bool SELF>
__global__ void __launch_bounds__(IK_BLOCK)
ik_refine_kernel(const float* q_in, const float* __restrict__ target, int64_t n, int64_t n_targets,
                 const cppflow_ik_refine_desc d, float* q_out, uint8_t* __restrict__ status, int32_t* __restrict__ steps,
                 float* __restrict__ err) {
    extern __shared__ float smem[];
    const int64_t i = (int64_t)blockIdx.x * IK_BLOCK + threadIdx.x;
    if (i >= n) return;
    float x[M::NDOF];
    load_q<M>(q_in, i, x);
    float tg[7];
    const float* tp = target + (i % n_targets) * 7;
#pragma unroll
    for (int k = 0; k < 7; ++k) tg[k] = __ldg(tp + k);
    const bool early = !(d.flags & CPPFLOW_IK_NO_EARLY_EXIT);
    const int clamp = d.flags & CPPFLOW_IK_CLAMP;
    float e_pos = 0.f, e_rot = 0.f;
    bool ok = false;
    int s = 0;
    for (;; ++s) {
        if (early || s == d.n_steps) {
            ok = ik_converged<M, SELF>(x, tg, d.pos_tol, d.rot_tol, smem + threadIdx.x, e_pos, e_rot);
            if (ok || s == d.n_steps) break;
        }
        pose_lm_update<M>(x, tg, d.alpha_position, d.alpha_rotation, d.lambdas[s], clamp, nullptr, nullptr, 0);
    }
    store_q<M>(q_out, i, x);
    status[i] = ok ? 1 : 0;
    if (steps) steps[i] = s;
    if (err) {
        err[2 * i] = e_pos;
        err[2 * i + 1] = e_rot;
    }
}

// Row r = t * rep + j: sample j of target unsolved[t].  The key hashes (seed, round, target, j) only.
__global__ void __launch_bounds__(256)
ik_round_inputs_kernel(const int32_t* __restrict__ unsolved, int64_t rows, int rep, const float* __restrict__ poses,
                       uint64_t seed, int rnd, int width, float scale, float* __restrict__ latents,
                       float* __restrict__ cond) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const int64_t t = unsolved[r / rep];
    const uint64_t j = (uint64_t)(r % rep);
    const uint64_t key = mix64(mix64(mix64(seed ^ mix64((uint64_t)rnd)) ^ (uint64_t)t) ^ j);
    auto draw = [&](int k) { return mix64(key + (uint64_t)k * 0x9E3779B97F4A7C15ull); };
    for (int c = 0; c < width; c += 2) {  // Box-Muller pairs
        const float rad = sqrtf(-2.f * logf(u01(draw(c)))), th = 6.2831853f * u01(draw(c + 1));
        latents[r * width + c] = scale * (rad * cosf(th));
        if (c + 1 < width) latents[r * width + c + 1] = scale * (rad * sinf(th));
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) cond[r * 7 + k] = poses[t * 7 + k];
}

// One thread per listed target: the first converged sample (else sample 0) and the flag "still unsolved".
__global__ void __launch_bounds__(256)
ik_select_kernel(const float* __restrict__ q, const uint8_t* __restrict__ status, const int32_t* __restrict__ unsolved,
                 int64_t n_unsolved, int rep, int ndof, float* __restrict__ solutions, uint8_t* __restrict__ valid,
                 uint8_t* __restrict__ still) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_unsolved) return;
    int pick = 0;
    bool found = false;
    for (int j = 0; j < rep; ++j) {
        if (status[t * rep + j]) {
            pick = j;
            found = true;
            break;
        }
    }
    const int64_t tgt = unsolved[t];
    const float* src = q + (t * rep + pick) * ndof;
    for (int k = 0; k < ndof; ++k) solutions[tgt * ndof + k] = src[k];
    valid[tgt] = found ? 1 : 0;
    still[t] = found ? 0 : 1;
}

static size_t align256(size_t b) { return (b + 255) / 256 * 256; }

// 0 when CUB cannot size its temporary storage (no device)
static size_t select_temp_bytes(int64_t n) {
    size_t bytes = 0;
    const cudaError_t e = cub::DeviceSelect::Flagged(nullptr, bytes, (const int32_t*)nullptr, (const uint8_t*)nullptr,
                                                     (int32_t*)nullptr, (int32_t*)nullptr, (int)n);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return bytes;
}

static int robot_ndof(int robot) {
    switch (robot) {
        case ROBOT_FETCH: return Fetch::NDOF;
        case ROBOT_FETCH_ARM: return FetchArm::NDOF;
        case ROBOT_PANDA: return Panda::NDOF;
        default: return 0;
    }
}

}  // namespace cppflow

using namespace cppflow;

extern "C" int cppflow_ik_refine(int robot, const cppflow_ik_refine_desc* desc, const float* d_q, const float* d_target,
                                 int64_t n, int64_t n_targets, float* d_q_out, uint8_t* d_status, int32_t* d_steps,
                                 float* d_err, void* stream) {
    CPPFLOW_CHECK_ARG(desc != nullptr, "desc");
    CPPFLOW_CHECK_ARG(desc->n_steps >= 0 && desc->n_steps <= CPPFLOW_IK_MAX_STEPS, "n_steps outside [0, 32]");
    CPPFLOW_CHECK_ARG(desc->pos_tol >= 0.f && desc->rot_tol >= 0.f, "tolerances must be >= 0");
    CPPFLOW_CHECK_ARG((desc->flags & ~(CPPFLOW_IK_CLAMP | CPPFLOW_IK_CHECK_SELF_COLLISION | CPPFLOW_IK_NO_EARLY_EXIT)) == 0,
                      "unknown flags");
    CPPFLOW_CHECK_ARG(robot_ndof(robot) > 0, "unknown robot id");
    CPPFLOW_CHECK_ARG(n >= 0, "n");
    if (n == 0) return CPPFLOW_OK;
    CPPFLOW_CHECK_ARG(d_q && d_target && d_q_out && d_status, "null pointer");
    CPPFLOW_CHECK_ARG(n_targets > 0, "n_targets");
    const cudaStream_t st = (cudaStream_t)stream;
    const bool self = desc->flags & CPPFLOW_IK_CHECK_SELF_COLLISION;
    CPPFLOW_DISPATCH_ROBOT(robot, {
        if (self) {
            const size_t sh = sizeof(float) * IK_BLOCK * SmemLayout<M>::N_DIST;
            ik_refine_kernel<M, true><<<grid_for(n, IK_BLOCK), IK_BLOCK, sh, st>>>(
                d_q, d_target, n, n_targets, *desc, d_q_out, d_status, d_steps, d_err);
        } else {
            ik_refine_kernel<M, false><<<grid_for(n, IK_BLOCK), IK_BLOCK, 0, st>>>(
                d_q, d_target, n, n_targets, *desc, d_q_out, d_status, d_steps, d_err);
        }
    });
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" int cppflow_ik_round_inputs(const int32_t* d_unsolved, int64_t n_unsolved, int rep, const float* d_poses,
                                       uint64_t seed, int round, int width, float latent_scale, float* d_latents,
                                       float* d_cond, void* stream) {
    CPPFLOW_CHECK_ARG(rep > 0, "rep must be > 0");
    CPPFLOW_CHECK_ARG(round >= 0, "round");
    CPPFLOW_CHECK_ARG(width >= 1 && width <= 16, "width outside [1, 16]");
    CPPFLOW_CHECK_ARG(latent_scale >= 0.f && latent_scale < INFINITY, "latent_scale");
    CPPFLOW_CHECK_ARG(n_unsolved >= 0, "n_unsolved");
    if (n_unsolved == 0) return CPPFLOW_OK;
    CPPFLOW_CHECK_ARG(d_unsolved && d_poses && d_latents && d_cond, "null pointer");
    const int64_t rows = n_unsolved * rep;
    ik_round_inputs_kernel<<<grid_for(rows, 256), 256, 0, (cudaStream_t)stream>>>(
        d_unsolved, rows, rep, d_poses, seed, round, width, latent_scale, d_latents, d_cond);
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" size_t cppflow_ik_select_workspace_bytes(int64_t n_unsolved) {
    if (n_unsolved < 0 || n_unsolved > INT_MAX) return 0;
    const size_t temp = select_temp_bytes(n_unsolved);
    return temp == 0 ? 0 : align256((size_t)n_unsolved) + align256(temp);
}

extern "C" int cppflow_ik_select(int robot, const float* d_q, const uint8_t* d_status, const int32_t* d_unsolved,
                                 int64_t n_unsolved, int rep, float* d_solutions, uint8_t* d_valid,
                                 int32_t* d_unsolved_out, int32_t* d_n_unsolved_out, void* d_workspace,
                                 size_t workspace_bytes, void* stream) {
    const int ndof = robot_ndof(robot);
    CPPFLOW_CHECK_ARG(ndof > 0, "unknown robot id");
    CPPFLOW_CHECK_ARG(rep > 0, "rep must be > 0");
    CPPFLOW_CHECK_ARG(n_unsolved >= 0 && n_unsolved <= INT_MAX, "n_unsolved outside [0, 2^31)");
    CPPFLOW_CHECK_ARG(d_n_unsolved_out != nullptr, "null pointer");
    const cudaStream_t st = (cudaStream_t)stream;
    if (n_unsolved == 0) {
        cudaError_t e = cudaMemsetAsync(d_n_unsolved_out, 0, sizeof(int32_t), st);
        if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "ik_select: %s", cudaGetErrorString(e));
        return CPPFLOW_OK;
    }
    CPPFLOW_CHECK_ARG(d_q && d_status && d_unsolved && d_solutions && d_valid && d_unsolved_out && d_workspace,
                      "null pointer");
    const size_t need = cppflow_ik_select_workspace_bytes(n_unsolved);
    if (need == 0) return fail(CPPFLOW_E_CUDA, "ik_select: cannot size the compaction's temporary storage");
    if (workspace_bytes < need)
        return fail(CPPFLOW_E_WORKSPACE, "ik_select: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    uint8_t* still = static_cast<uint8_t*>(d_workspace);
    void* temp = still + align256((size_t)n_unsolved);
    size_t temp_bytes = workspace_bytes - align256((size_t)n_unsolved);
    ik_select_kernel<<<grid_for(n_unsolved, 256), 256, 0, st>>>(d_q, d_status, d_unsolved, n_unsolved, rep, ndof,
                                                                 d_solutions, d_valid, still);
    CPPFLOW_CHECK_LAUNCH();
    cudaError_t e = cub::DeviceSelect::Flagged(temp, temp_bytes, d_unsolved, still, d_unsolved_out, d_n_unsolved_out,
                                               (int)n_unsolved, st);
    if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "ik_select: DeviceSelect::Flagged: %s", cudaGetErrorString(e));
    return CPPFLOW_OK;
}
