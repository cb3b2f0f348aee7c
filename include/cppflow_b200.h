/* cppflow_b200 - C ABI of the B200-native path-refinement hot path of jstmn/cppflow.
 *
 * The reference is pure Python: it has no FFI.  Its boundary for this path is the Python call surface
 * of cppflow/{search,collision_detection,optimization,optimization_utils}.py plus the jrl.Robot methods
 * those modules call (SURVEY.md section 8b).  Each entry point below names the reference interface it
 * replaces.  The Python host in cppflow_b200/ binds these with ctypes (see INTEGRATION.md for the stub a
 * reference maintainer would add).
 *
 * Conventions
 *  - every pointer named d_* is DEVICE memory (fp32 unless stated), contiguous, row-major;
 *    h_* pointers are HOST memory read during the call (small tables, copied into the kernel parameters);
 *  - `stream` is a cudaStream_t passed as void* (0 = default stream); calls are asynchronous on it;
 *  - no entry point allocates device memory or synchronises: the caller supplies outputs and workspaces;
 *  - return value: 0 on success, a negative CPPFLOW_E_* code otherwise (cppflow_last_error() has the text).
 *  - robot ids: 0 = Fetch (8 dof, prismatic torso + 7 revolute), 1 = FetchArm (7 dof), 2 = Panda (7 dof)
 *    (planners.py:34-41).
 *  - poses are [x, y, z, qw, qx, qy, qz] (README.md:8); Jacobian rows are [wx wy wz vx vy vz]
 *    (optimization.py:77-80).
 */
#ifndef CPPFLOW_B200_H
#define CPPFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPPFLOW_ROBOT_FETCH 0
#define CPPFLOW_ROBOT_FETCH_ARM 1
#define CPPFLOW_ROBOT_PANDA 2

#define CPPFLOW_OK 0
#define CPPFLOW_E_INVALID (-1)   /* bad argument (robot id, sizes, null pointer) */
#define CPPFLOW_E_CUDA (-2)      /* a CUDA runtime call / launch failed */
#define CPPFLOW_E_WORKSPACE (-3) /* workspace too small */

#define CPPFLOW_MAX_DOF 8
#define CPPFLOW_MAX_CAPSULES 10
#define CPPFLOW_MAX_PAIRS 28
#define CPPFLOW_MAX_OBSTACLES 8

/* Mirrors the fields of OptimizationParameters the live parameter sets use
 * (lm_hyper_parameters.py:14-80; ALT_LOSS_V2_1_DIFF :86-118, ALT_LOSS_V2_1_POSE :119-151). */
typedef struct cppflow_lm_params {
    float lm_lambda;
    float alpha_position;
    float alpha_rotation;
    float alpha_differencing;
    float alpha_differencing_prismatic_scaling;
    float alpha_virtual_configs;
    float alpha_self_collision;
    float alpha_env_collision;
    int32_t use_pose;
    int32_t use_differencing;
    int32_t use_virtual_configs;
    int32_t n_virtual_configs;
    int32_t use_self_collisions;
    int32_t use_env_collisions;
} cppflow_lm_params;

/* Static description of a robot model (what the hot path reads from jrl.Robot: ndof, limits,
 * prismatic idxs, capsule table, pair list - SURVEY.md 8b). */
typedef struct cppflow_robot_info {
    int32_t ndof;
    int32_t n_capsules;
    int32_t n_pairs;
    int32_t n_chain;
    float lower[CPPFLOW_MAX_DOF];
    float upper[CPPFLOW_MAX_DOF];
    int32_t is_prismatic[CPPFLOW_MAX_DOF];
    float capsules[CPPFLOW_MAX_CAPSULES][7]; /* x1 y1 z1 x2 y2 z2 r, link frame */
    int32_t capsule_frame[CPPFLOW_MAX_CAPSULES];
    int32_t pairs[CPPFLOW_MAX_PAIRS][2];
    char name[16];
} cppflow_robot_info;

const char* cppflow_version(void);
const char* cppflow_last_error(void);

/* ABI check for foreign-function bindings: out[0] = CPPFLOW_ABI_VERSION, then sizeof of cppflow_lm_params,
 * cppflow_robot_info, cppflow_constraints, cppflow_lm_loop_result, cppflow_lm_loop_job (as many as fit in n).
 * Returns the number of values the library knows (6).  A binding compares them with its own struct sizes after
 * dlopen and refuses a library built from another header. */
#define CPPFLOW_ABI_VERSION 4
int cppflow_abi_info(int64_t* out, int n);

/* jrl.Robot properties (ndof, actuated_joints_limits, prismatic_joint_idxs, _collision_capsules_by_link). */
int cppflow_robot_info_get(int robot, cppflow_robot_info* out);

/* Robot.forward_kinematics(x) -> [n,7]   (optimization_utils.py:811, evaluation_utils.py:115) */
int cppflow_forward_kinematics(int robot, const float* d_q, int64_t n, float* d_poses, void* stream);

/* Robot.jacobian(x) -> [n,6,ndof]   (optimization.py:74, optimization_utils.py:281) */
int cppflow_jacobian(int robot, const float* d_q, int64_t n, float* d_J, void* stream);

/* get_6d_pose_errors(robot, x, target_poses) -> ([n,6], [n,7])   (optimization_utils.py:802-820).
 * target row of config i is i % n_targets (lets one [T,7] path serve P stacked paths). */
int cppflow_pose_errors(int robot, const float* d_q, const float* d_target, int64_t n, int64_t n_targets,
                        float* d_err, float* d_cur_poses, void* stream);

/* levenberg_marquardt_only_pose + clamp_to_joint_limits   (optimization.py:61-92, optimization_utils.py:823-833).
 * d_x_out = clamp(x + dx) when do_clamp, x + dx otherwise.  d_J_out [n,6,ndof] / d_e_out [n,6] (alpha-scaled,
 * as returned with return_residual=True) may be NULL. */
int cppflow_lm_pose_step(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_target,
                         int64_t n, int64_t n_targets, int do_clamp, float* d_x_out, float* d_J_out, float* d_e_out,
                         void* stream);

/* n_steps pose-only LM steps in a row, step i with damping h_lambdas[i] (host array) instead of params->lm_lambda, in
 * place on d_q [n, ndof] with d_tmp [n, ndof] as the second buffer.  No reference counterpart as a single call: it is
 * levenberg_marquardt_only_pose applied repeatedly, which the stand-in candidate generator (planners.py) uses to pull
 * random joint configurations onto the target poses. */
int cppflow_lm_pose_steps(int robot, const cppflow_lm_params* params, const float* h_lambdas, int n_steps, float* d_q,
                          float* d_tmp, const float* d_target, int64_t n, int64_t n_targets, int do_clamp, void* stream);

/* clamp_to_joint_limits(robot, x), in place   (optimization_utils.py:823-833) */
int cppflow_clamp_to_joint_limits(int robot, float* d_q, int64_t n, void* stream);

/* Robot.self_collision_distances(x) -> [n,S] and its Jacobian [n,S,ndof] (d_J may be NULL)
 * (collision_detection.py:65, optimization_utils.py:652,670) */
int cppflow_self_collision_distances(int robot, const float* d_q, int64_t n, float* d_dist, float* d_J, void* stream);

/* Robot.env_collision_distances(x, cuboid, Tcuboid) -> [n,C] and its Jacobian [n,C,ndof] (d_J may be NULL)
 * (collision_detection.py:40, optimization_utils.py:690,710).  h_cuboid[6] = lo,hi; h_Tcuboid[16] row-major 4x4
 * (data_type_utils.py:109-127). */
int cppflow_env_collision_distances(int robot, const float* d_q, int64_t n, const float* h_cuboid,
                                    const float* h_Tcuboid, float* d_dist, float* d_J, void* stream);

/* qpaths_batched_self_collisions / qpaths_batched_env_collisions (collision_detection.py:27-69):
 * flags[i] = min over pairs/capsules (and obstacles) of the distance < 0.  Either output may be NULL.
 * h_cuboids [n_obstacles,6], h_Tcuboids [n_obstacles,16]. */
int cppflow_collision_flags(int robot, const float* d_q, int64_t n, const float* h_cuboids, const float* h_Tcuboids,
                            int n_obstacles, uint8_t* d_self_flags, uint8_t* d_env_flags, void* stream);

/* levenberg_marquardt_full (get_r_and_J + _lm_full_step) + clamp_to_joint_limits, for P independent paths of T
 * waypoints (optimization.py:95-144, optimization_utils.py:486-731).  The normal equations are assembled
 * implicitly as a symmetric block-tridiagonal system (ndof x ndof blocks) and solved by block Cholesky.
 * d_xv = virtual configs [P,T,ndof] (NULL: equal to x, the run_lm_alternating_loss case, optimization.py:253).
 * Workspace: cppflow_lm_full_workspace_bytes(robot, P, T) bytes of device memory. */
size_t cppflow_lm_full_workspace_bytes(int robot, int64_t P, int64_t T);
int cppflow_lm_full_step(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_xv,
                         const float* d_target, int64_t P, int64_t T, const float* h_cuboids, const float* h_Tcuboids,
                         int n_obstacles, int do_clamp, void* d_workspace, size_t workspace_bytes, float* d_x_out,
                         void* stream);

/* The two halves of cppflow_lm_full_step, exposed so a host pipeline can overlap the assembly of one chunk of paths
 * with the solve of another on different streams: assemble writes the packed (A_tt, b_t) blocks to the workspace,
 * solve consumes them and writes clamp(x + dx). */
int cppflow_lm_full_assemble(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_xv,
                             const float* d_target, int64_t P, int64_t T, const float* h_cuboids,
                             const float* h_Tcuboids, int n_obstacles, void* d_workspace, size_t workspace_bytes,
                             void* stream);
int cppflow_lm_full_solve(int robot, const cppflow_lm_params* params, const float* d_q, int64_t P, int64_t T,
                          int do_clamp, void* d_workspace, size_t workspace_bytes, float* d_x_out, void* stream);

/* `do_clamp` of cppflow_lm_full_step / cppflow_lm_full_solve is a bit set: CPPFLOW_LM_CLAMP (= 1, the reference's
 * clamp_to_joint_limits after the step) | CPPFLOW_LM_OVERLAP: the solve is launched with a shared-memory
 * footprint (fits on an SM next to one assembly CTA) and the highest launch priority, so that it runs UNDER the
 * assembly of another chunk of paths enqueued on another stream (same results bit for bit). */
#define CPPFLOW_LM_CLAMP 1
#define CPPFLOW_LM_OVERLAP 2
/* cppflow_lm_full_step only: the assembly CTA of a waypoint also takes the elimination step of that waypoint (the chain
 * runs from CTA to CTA through L2), so the (A, b) blocks never reach HBM; the solve then only back-substitutes.  Same
 * results bit for bit. */
#define CPPFLOW_LM_FUSED 4
/* cppflow_lm_full_step / cppflow_lm_full_solve: bits 8..15 of `do_clamp` ask for the SEGMENTED solve with that many
 * time segments per path (csrc/lm_segsolve.cuh): the segments between S - 1 separator waypoints are eliminated in
 * parallel, the separators' reduced block-tridiagonal system is solved, the segments are back-substituted in parallel.
 * For few paths (<= ~2000) the twisted solve's dependent chain of T steps is the whole solve time; this one's chain is
 * ~ T / S heavy + S + T / S light steps.  The result differs from the twisted solve's by rounding only and depends on
 * S, not on P or the chunking.  S is reduced to T / 4 for short paths (fewer than 2 segments: the twisted solve).
 * Needs the larger workspace of cppflow_lm_full_workspace_bytes_ex(robot, P, T, flags).  Ignored with
 * CPPFLOW_LM_FUSED. */
#define CPPFLOW_LM_SEGMENTS_SHIFT 8
#define CPPFLOW_LM_SEGMENTS(n) (((n) & 0xff) << CPPFLOW_LM_SEGMENTS_SHIFT)
size_t cppflow_lm_full_workspace_bytes_ex(int robot, int64_t P, int64_t T, int flags);

/* run_lm_alternating_loss for ONE path (optimization.py:147-373; called by run_lm_optimization :376-426 with
 * ALT_LOSS_V2_1_DIFF / ALT_LOSS_V2_1_POSE): pose-only steps until the position and rotation errors are inside the
 * constraints, joint-differencing steps otherwise, clamp after every step, convergence on the trajectory length after
 * differencing steps, the last valid iterate is returned (the current one if none was valid).  Validity = the
 * thresholds of evaluation_utils.py:29-75 (strict <) and non-negative capsule distances (the reference's klampt mesh
 * checks, optimization_utils.py:889-900, are out of scope; the Python host keeps a loop with a mesh callback).
 * UNLIKE the other entry points this one BLOCKS: like the reference (`.item()`, :175) it reads the metrics of every
 * iterate on the host - the metrics kernel stores its 8 floats straight into `h_pinned_metrics` (page-locked,
 * device-mapped host memory) followed by a per-call completion tag, which the host polls (no cudaStreamSynchronize per
 * iteration; a stream synchronisation is the fallback when the buffer is not device-addressable or the tag does not
 * show up).  Workspace: cppflow_lm_alternating_workspace_bytes(robot, T) bytes, 256-byte aligned.
 * The thresholds are doubles, like the Python floats the reference compares its float32 metrics with. */
typedef struct cppflow_constraints { /* data_types.py:53-62 */
    double max_allowed_position_error_cm;
    double max_allowed_rotation_error_deg;
    double max_allowed_mjac_deg;
    double max_allowed_mjac_cm;
} cppflow_constraints;
#define CPPFLOW_LM_SCHEDULE_MAX 256
typedef struct cppflow_lm_loop_result { /* OptimizationResult, optimization.py:52-57 */
    int32_t n_steps_taken;
    int32_t is_valid;
    float last_metrics[8];                  /* cppflow_path_metrics row of the last iterate examined */
    char schedule[CPPFLOW_LM_SCHEDULE_MAX]; /* step types taken: 'p' pose-only, 'd' differencing; 0-terminated */
} cppflow_lm_loop_result;
size_t cppflow_lm_alternating_workspace_bytes(int robot, int64_t T);
int cppflow_lm_alternating_loss(int robot, const cppflow_lm_params* params_diff, const cppflow_lm_params* params_pose,
                                const cppflow_constraints* constraints, const float* d_x_seed, const float* d_target,
                                int64_t T, const float* h_cuboids, const float* h_Tcuboids, int n_obstacles,
                                int max_n_steps, double tmax_sec, int return_if_valid_after_n_steps,
                                double convergence_threshold, void* d_workspace, size_t workspace_bytes,
                                float* h_pinned_metrics, float* d_x_out, cppflow_lm_loop_result* result, void* stream);

/* The same loop for several independent paths / problems at once (BASELINE config 4: the 13 benchmark problems in one
 * run).  One job per path, each with its own stream, workspace and pinned metrics buffer; the next step of EVERY
 * unfinished job is enqueued before the host waits for any of them, so the jobs overlap on the device while the host
 * takes each job's decisions exactly as cppflow_lm_alternating_loss does (which is this call with one job). */
typedef struct cppflow_lm_loop_job {
    int32_t robot;
    const cppflow_lm_params* params_diff;
    const cppflow_lm_params* params_pose;
    const cppflow_constraints* constraints;
    const float* d_x_seed; /* [T, ndof] */
    const float* d_target; /* [T, 7] */
    int64_t T;
    const float* h_cuboids;
    const float* h_Tcuboids;
    int32_t n_obstacles;
    int32_t max_n_steps;
    double tmax_sec;
    int32_t return_if_valid_after_n_steps;
    double convergence_threshold;
    void* d_workspace;
    size_t workspace_bytes;
    float* h_pinned_metrics; /* 8 floats, page-locked */
    float* d_x_out;          /* [T, ndof] */
    cppflow_lm_loop_result* result;
    void* stream;
} cppflow_lm_loop_job;
int cppflow_lm_alternating_loss_many(int n_jobs, const cppflow_lm_loop_job* jobs);

/* joint_limit_almost_violations_3d(robot, qs, eps_revolute, eps_prismatic) -> float32 0/1 [n]  (search.py:25-52) */
int cppflow_joint_limit_flags(int robot, const float* d_q, int64_t n, float eps_revolute, float eps_prismatic,
                              float* d_flags, void* stream);

/* dp_search (search.py:128-173): bottleneck DP over k candidate paths.
 * in : d_q [k,T,ndof]; d_self_flags, d_env_flags uint8 [k,T]
 * out: d_best_path [T,ndof]; d_memo int32 [k,T]; d_costs [k,T]; d_chosen int32 [T] (candidate index per waypoint)
 * Workspace: cppflow_dp_search_workspace_bytes(k, T) bytes. */
size_t cppflow_dp_search_workspace_bytes(int64_t k, int64_t T);
int cppflow_dp_search(int robot, const float* d_q, const uint8_t* d_self_flags, const uint8_t* d_env_flags, int64_t k,
                      int64_t T, void* d_workspace, size_t workspace_bytes, float* d_best_path, int32_t* d_memo,
                      float* d_costs, int32_t* d_chosen, void* stream);

/* Per-path validity metrics (x_is_valid without the klampt calls: optimization_utils.py:836-886,
 * evaluation_utils.py:29-75,113-141; TL of optimization.py:173-175).  d_out [P,8] =
 * {max position error cm, max rotation error deg, max |dq| revolute deg, max |dq| prismatic cm,
 *  trajectory length rad, min capsule self distance m, min capsule env distance m (+inf if no obstacles), 0}. */
int cppflow_path_metrics(int robot, const float* d_q, const float* d_target, int64_t P, int64_t T,
                         const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, float* d_out, void* stream);
/* The same with options.  CPPFLOW_METRICS_SIGN_ONLY: x_is_valid (optimization_utils.py:889-900) and the cost ranking only
 * ask whether a path collides, so only capsule pairs that bounding spheres cannot prove apart are evaluated: columns
 * 5 / 6 are the exact minimum distance when it is negative, and otherwise some non-negative number (+inf when every pair
 * was proven apart).  Every other column is unchanged. */
#define CPPFLOW_METRICS_SIGN_ONLY 1
int cppflow_path_metrics_ex(int robot, const float* d_q, const float* d_target, int64_t P, int64_t T,
                            const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, int flags, float* d_out,
                            void* stream);

/* Ranking of refined paths (north star: "gather per-path costs and the argmin"; no reference counterpart - the reference
 * refines one path).  A path is ranked by (invalid, trajectory length, global index): key = invalid << 62 |
 * bits(float32 TL) << 31 | (first_index + p), valid = the four thresholds of x_is_valid (evaluation_utils.py:41-58) and
 * no negative capsule distance.  d_metrics [P,8] = rows of cppflow_path_metrics; d_out int64[3] = {smallest key, number of
 * valid paths, first_index} - what each rank contributes to the all-gather. */
int cppflow_path_key_argmin(const float* d_metrics, int64_t P, const cppflow_constraints* constraints,
                            int64_t first_index, int64_t* d_out, void* stream);

/* Splits the SMs of `device` into two green contexts - the first with at least `min_sms_first` SMs (rounded up to the
 * architecture's granularity, 8 on sm_90+), the second with the rest - and creates streams in each.  Kernels launched
 * on a stream only run on its partition's SMs.  Used by the chunk-pipelined LM iteration to give the block solves a few
 * SMs of their own while the assembly owns the rest (no reference counterpart). */
int cppflow_sm_partition_create(int device, int min_sms_first, int n_streams_first, int n_streams_second,
                                void** streams_first, void** streams_second, int* sms_first, int* sms_second);

/* IKFlow's conditional GLOW network (ikflow/model.py: glow_cNF_model; restated in oracle/ikflow.py), the candidate
 * generator of the reference (planners.py:116-189).  Forward (x -> z) or reverse (z -> x) pass over n rows; row i is
 * conditioned on d_cond[i % n_cond] = [x, y, z, qw, qx, qy, qz] (the softflow scale, when dim_cond = 8, is 0).
 * The first Linear of each subnet and its hidden Linears run on the tensor cores (tcgen05, BF16 operands, FP32
 * accumulation); the subnet input [half | cond] and the hidden activations are stored in BF16.  The last Linear and
 * the coupling arithmetic are FP32.  A row's result does not depend on n or on the other rows.
 * Supported: ndof <= 8 (the robot's), ndof <= width <= 16, dim_cond 7 or 8, coeff_fn_config 1..4,
 * coeff_fn_internal_size a multiple of 128 up to 1024, nb_nodes >= 1, n >= 1; anything else is CPPFLOW_E_INVALID.
 * Packed weights, with s = 0 for subnet1 and 1 for subnet2 of each coupling block b, H = coeff_fn_internal_size and
 * L = coeff_fn_config (rows beyond a layer's size are zero):
 *   d_w_in     bf16 [nb_nodes, 2, H, 64]          first Linear, [out, in] with `in` zero-padded to 64
 *   d_w_hidden bf16 [nb_nodes, 2, L - 1, H, H]    hidden Linears (NULL when L = 1)
 *   d_b_hidden fp32 [nb_nodes, 2, L, H]           biases of the first and hidden Linears
 *   d_w_out    fp32 [nb_nodes, 2, 16, H]          last Linear, [s | t] rows zero-padded to 16
 *   d_b_out    fp32 [nb_nodes, 2, 16]
 *   d_scale    fp32 [width]                       diagonal of FixedLinearTransform's M
 *   d_perm, d_perm_inv int32 [nb_nodes, width]    PermuteRandom of block b and its inverse
 * Workspace (cppflow_flow_workspace_bytes): four regions, each rounded up to 256 bytes: n x 16 fp32 (state),
 * n x 64 bf16 (subnet input), and min(L, 2) buffers of n x H bf16 (hidden activations); 0 for an invalid desc.
 * d_in, d_out [n, width]; with CPPFLOW_FLOW_CLAMP (reverse only) the first ndof columns of the output are clamped
 * to the robot's joint limits. */
#define CPPFLOW_FLOW_REVERSE 1
#define CPPFLOW_FLOW_CLAMP 2
typedef struct cppflow_flow_desc {
    int32_t robot;
    int32_t width; /* dim_latent_space */
    int32_t ndof;
    int32_t dim_cond;
    int32_t nb_nodes;
    int32_t coeff_fn_config;
    int32_t coeff_fn_internal_size;
    float rnvp_clamp;
    const void* d_w_in;
    const void* d_w_hidden;
    const float* d_b_hidden;
    const float* d_w_out;
    const float* d_b_out;
    const float* d_scale;
    const int32_t* d_perm;
    const int32_t* d_perm_inv;
} cppflow_flow_desc;
size_t cppflow_flow_workspace_bytes(const cppflow_flow_desc* desc, int64_t n);
int cppflow_flow_run(const cppflow_flow_desc* desc, const float* d_in, const float* d_cond, int64_t n, int64_t n_cond,
                     int flags, void* d_workspace, size_t workspace_bytes, float* d_out, void* stream);

/* Training of the network above: ikflow's train.py (the flow's negative log-likelihood of joint configurations given
 * their poses, minimised with Adam; restated in oracle/ikflow_train.py: forward_with_logdet, nll, training_batch).
 * One cppflow_flow_train_step runs, for a batch of n rows (n a multiple of 128, any network cppflow_flow_run accepts):
 * the forward pass of d_x [n, width] conditioned on d_cond [n, dim_cond] (row i on row i, softflow scale included),
 * whose z is bit-identical to cppflow_flow_run's; *d_loss = mean(0.5 |z|^2 - log|det dz/dx|); the gradient of the
 * loss with respect to every packed FP32 parameter (tensor-core GEMMs on tcgen05 for the subnets' Linears, fixed-order
 * reductions, no atomics: two runs are bit-identical); then, unless CPPFLOW_FLOW_TRAIN_NO_UPDATE, one step of
 * torch.optim.Adam (weight decay added to the gradient) on the FP32 master weights, which also rewrites the BF16
 * tables of flow and the transposed copies below.  If any gradient element is not finite the update is skipped:
 * weights and moments stay, d_counters[1] counts it.  The learning rate is
 * lr * lr_decay^floor(d_counters[2] / lr_decay_steps) (torch's ExponentialLR stepped every lr_decay_steps steps).
 * No allocation, no host synchronisation; capturable in a CUDA graph.
 * d_params, d_adam_m, d_adam_v: fp32 [P], the tables of cppflow_flow_desc concatenated in the order
 *   w_in [nb, 2, H, 64] | w_hidden [nb, 2, L - 1, H, H] | b_hidden [nb, 2, L, H] | w_out [nb, 2, 16, H] | b_out [nb, 2, 16]
 *   (padding zero); flow.d_b_hidden, d_w_out and d_b_out must point at their segments of d_params.
 * d_grad: NULL, or fp32 [P] that receives the gradient (before weight decay) in the same layout.
 * Rejected (CPPFLOW_E_INVALID): what cppflow_flow_run rejects, n % 128 != 0, width > ndof with dim_cond 7 (the padding
 * columns have no density without softflow's noise), hyperparameters out of range. */
#define CPPFLOW_FLOW_TRAIN_NO_UPDATE 1
typedef struct cppflow_flow_train_desc {
    cppflow_flow_desc flow;
    float* d_params;
    float* d_adam_m;
    float* d_adam_v;
    void* d_w_in_t;      /* bf16 [nb, 2, 64, H]: w_in transposed */
    void* d_w_hidden_t;  /* bf16 [nb, 2, L - 1, H, H]: each hidden weight transposed (NULL when L = 1) */
    void* d_w_out_t;     /* bf16 [nb, 2, H, 64]: w_out transposed, columns >= 16 zero */
    int64_t* d_counters; /* [3]: Adam updates applied, steps skipped (non-finite gradient), steps taken */
    double lr, beta1, beta2, eps, weight_decay, lr_decay;
    int64_t lr_decay_steps;
} cppflow_flow_train_desc;
/* Workspace of cppflow_flow_train_step: all activations of the forward pass plus the backward's buffers; 0 for an
 * invalid desc or batch. */
size_t cppflow_flow_train_workspace_bytes(const cppflow_flow_train_desc* desc, int64_t batch);
int cppflow_flow_train_step(const cppflow_flow_train_desc* desc, const float* d_x, const float* d_cond, int64_t batch,
                            int flags, void* d_workspace, size_t workspace_bytes, float* d_loss, float* d_grad, void* stream);
/* A training batch (jrl's sample_joint_angles_and_poses data, ikflow's softflow; oracle/ikflow_train.py: training_batch):
 * row r takes sample idx of d_q [n_data, ndof] / d_poses [n_data, 7] and draws c ~ U(0, 1), eps ~ N(0, I_width) and a
 * fair coin from a counter-based generator keyed on (seed, d_counters[2], r); then d_x[r] = [q | 0 ...] +
 * softflow_noise_scale * c * eps and d_cond[r] = [pose with its quaternion negated on heads | c] (dim_cond 8).  With
 * dim_cond 7, c = 0 and eps = 0.  Optional outputs: d_idx int64 [batch], d_noise fp32 [batch, width + 2] = [eps | c | coin]. */
int cppflow_flow_train_batch(const cppflow_flow_train_desc* desc, const float* d_q, const float* d_poses, int64_t n_data,
                             int64_t batch, uint64_t seed, float softflow_noise_scale, float* d_x, float* d_cond,
                             int64_t* d_idx, float* d_noise, void* stream);

/* Measurement aid (no reference counterpart): dependent-free FP32 FMA loop on `blocks` x 1024 threads, used by
 * bench.py to measure the FP32 roofline denominator on the box.  *flops_out = FLOPs of the launch. */
int cppflow_fp32_probe(int blocks, int iters, float* d_scratch, double* flops_out, void* stream);
/* Measurement aid (no reference counterpart): a stand-in neighbour kernel for co-residency experiments - 256-thread CTAs
 * of FMA chains holding `smem_bytes` of shared memory, untouched (touch = 0) or accessed `touch` times per iteration. */
int cppflow_neighbour_probe(int blocks, int iters, int smem_bytes, int touch, float* d_scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CPPFLOW_B200_H */
