// K4: dp_search - the bottleneck dynamic program over k candidate joint-space paths.
//
// Reference being replaced:
//   joint_limit_almost_violations_3d   search.py:25-52
//   _get_mjacs                         search.py:100-125   (materialises [k,k,T-1,D]; here [T-1,k,k] only)
//   dp_search                          search.py:128-173   (T-1 dependent k x k steps + backtrack)
// Bit-exactness contract (DESIGN.md): memo / costs / best_path equal the reference's fp32 results exactly.  Every
// arithmetic op is an explicit round-to-nearest fp32 op in the reference's order (no FMA contraction):
//   dq = q[i,t+1,d] - q[j,t,d];  dq *= 5 for prismatic d (before the wrap);  w = |remainder(dq + pi, 2 pi) - pi|
//   mjac = max_d w;  c = max(mjac, cost[j,t-1]) + ext[i,t];  cost[i,t], memo[i,t] = min_j / first argmin_j.
#include "common.cuh"
#include "kinematics.cuh"
#include <cooperative_groups.h>

namespace cppflow {

template <class M>
__device__ __forceinline__ bool near_joint_limit(const float* __restrict__ q, float eps_rev, float eps_pris) {
    bool bad = false;
    static_for<M::NDOF>([&](auto Dd) {
        constexpr int d = decltype(Dd)::value;
        const float eps = dof_is_prismatic<M>(d) ? eps_pris : eps_rev;
        const float lo = __fadd_rn(dof_lower<M>(d), eps);  // l_lim[idx] += eps in fp32 (search.py:48-49)
        const float hi = __fsub_rn(dof_upper<M>(d), eps);
        const float v = q[d];
        bad = bad || (v < lo) || (v > hi);
    });
    return bad;
}

template <class M>
__global__ void joint_limit_flags_kernel(const float* __restrict__ q, int64_t n, float eps_rev, float eps_pris,
                                         float* __restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flags[i] = near_joint_limit<M>(q + i * M::NDOF, eps_rev, eps_pris) ? 1.f : 0.f;
}

// ext[t][i] = 100 * jlim + 1000 * env + 1000 * self   (search.py:146-150), stored t-major for the DP sweep
template <class M>
__global__ void dp_ext_kernel(const float* __restrict__ q, const uint8_t* __restrict__ self_f,
                              const uint8_t* __restrict__ env_f, int k, int T, float eps_rev, float eps_pris,
                              float* __restrict__ ext) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)k * T) return;
    const int i = (int)(idx / T), t = (int)(idx % T);
    const float jl = near_joint_limit<M>(q + idx * M::NDOF, eps_rev, eps_pris) ? 1.f : 0.f;
    float c = __fmul_rn(100.f, jl);
    c = __fadd_rn(c, env_f[idx] ? 1000.f : 0.f);
    c = __fadd_rn(c, self_f[idx] ? 1000.f : 0.f);
    ext[(int64_t)t * k + i] = c;
}

// mj[t][i][j] = max_d |wrap(s_d (q[i,t+1,d] - q[j,t,d]))|, t in [0, T-1)
constexpr int MJ_ROWS = 16;
template <class M>
__global__ void __launch_bounds__(256)
dp_mjac_kernel(const float* __restrict__ q, int k, int T, float* __restrict__ mj) {
    constexpr int D = M::NDOF;
    __shared__ float qto[MJ_ROWS][D];
    const int t = blockIdx.x;
    const int i0 = blockIdx.y * MJ_ROWS;
    const int rows = min(MJ_ROWS, k - i0);
    for (int e = threadIdx.x; e < rows * D; e += blockDim.x) {
        const int r = e / D, d = e % D;
        qto[r][d] = q[((int64_t)(i0 + r) * T + (t + 1)) * D + d];
    }
    __syncthreads();
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        float qf[D];
#pragma unroll
        for (int d = 0; d < D; ++d) qf[d] = q[((int64_t)j * T + t) * D + d];
        for (int r = 0; r < rows; ++r) {
            float m = 0.f;
            static_for<D>([&](auto Dd) {
                constexpr int d = decltype(Dd)::value;
                float dq = __fsub_rn(qto[r][d], qf[d]);
                if constexpr (dof_is_prismatic<M>(d)) dq = __fmul_rn(dq, 5.0f);
                m = fmaxf(m, fabsf(wrap_pi(dq)));
            });
            mj[((int64_t)t * k + (i0 + r)) * k + j] = m;
        }
    }
}

// Sequential sweep over t.  One CTA; warp w owns rows i = w, w + nwarps, ...; lanes stride over j and keep the
// first minimum; the cross-lane reduction orders (value, index) lexicographically so ties pick the lowest j, as
// torch.min does.  memo is also kept in shared memory (uint16) when it fits so the backtrack never leaves the SM.
template <bool MEMO_SMEM>
__global__ void __launch_bounds__(1024)
dp_sweep_kernel(const float* __restrict__ q, const float* __restrict__ ext, const float* __restrict__ mj, int k, int T,
                int D, float* __restrict__ costs, int32_t* __restrict__ memo, int32_t* __restrict__ chosen,
                float* __restrict__ best_path) {
    extern __shared__ unsigned char dsm[];
    float* cost_a = reinterpret_cast<float*>(dsm);
    float* cost_b = cost_a + k;
    uint16_t* memo_s = reinterpret_cast<uint16_t*>(cost_b + k);
    __shared__ int s_best;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;

    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const float c = ext[i];
        cost_a[i] = c;
        costs[(int64_t)i * T] = c;
        memo[(int64_t)i * T] = 0;
        if (MEMO_SMEM) memo_s[i] = 0;
    }
    __syncthreads();
    float* prev = cost_a;
    float* next = cost_b;
    for (int t = 1; t < T; ++t) {
        const float* mjt = mj + (int64_t)(t - 1) * k * k;
        const float* ext_t = ext + (int64_t)t * k;
        for (int i = warp; i < k; i += nwarps) {
            const float* row = mjt + (int64_t)i * k;
            const float e = ext_t[i];
            float best = INFINITY;
            int bj = 0x7fffffff;
            for (int j = lane; j < k; j += 32) {
                const float v = __fadd_rn(fmaxf(row[j], prev[j]), e);
                if (v < best) { best = v; bj = j; }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float ov = __shfl_down_sync(0xffffffffu, best, off);
                const int oj = __shfl_down_sync(0xffffffffu, bj, off);
                if (ov < best || (ov == best && oj < bj)) { best = ov; bj = oj; }
            }
            if (lane == 0) {
                next[i] = best;
                costs[(int64_t)i * T + t] = best;
                memo[(int64_t)i * T + t] = bj;
                if (MEMO_SMEM) memo_s[(int64_t)t * k + i] = (uint16_t)bj;
            }
        }
        __syncthreads();
        float* tmp = prev; prev = next; next = tmp;
    }
    // final argmin over the last column (first index on ties), then backtrack (search.py:162-173)
    if (warp == 0) {
        float best = INFINITY;
        int bi = 0x7fffffff;
        for (int i = lane; i < k; i += 32) {
            const float v = prev[i];
            if (v < best) { best = v; bi = i; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float ov = __shfl_down_sync(0xffffffffu, best, off);
            const int oi = __shfl_down_sync(0xffffffffu, bi, off);
            if (ov < best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) {
            int i = bi;
            for (int t = T - 1; t >= 0; --t) {
                chosen[t] = i;
                i = MEMO_SMEM ? (int)memo_s[(int64_t)t * k + i] : memo[(int64_t)i * T + t];
            }
        }
    }
    __threadfence_block();
    __syncthreads();
    for (int e = threadIdx.x; e < T * D; e += blockDim.x) {
        const int t = e / D, d = e % D;
        best_path[e] = q[((int64_t)chosen[t] * T + t) * D + d];
    }
    (void)s_best;
}


// ----------------------------------------------------------------------------------------------------------------
// Cluster sweep (k <= 512).  The sweep is a chain of T-1 dependent k x k min-max steps: it is bound by the latency of
// one step, not by throughput.  Eight CTAs of one thread-block cluster split the rows i; a warp owns RPW rows and keeps
// the mjac values of its rows for the NEXT PF steps in registers (they do not depend on the DP state, so their L2
// latency is off the critical path).  The (cost, argmin) pair of a finished row is sent to every CTA of the cluster
// with st.async into distributed shared memory; the store itself signals the destination CTA's mbarrier
// (complete_tx), so a step needs no cluster barrier and no memory fence: every CTA waits until k pairs have arrived.
// Two pair buffers, each with its own mbarrier, alternate; a CTA can only start writing buffer b (and signalling its
// barrier) again after it has received every row of the step in between, i.e. after every warp of the cluster has
// finished reading b and has seen the previous phase of that barrier complete.  Arithmetic and tie-breaking are those
// of dp_sweep_kernel (bit-exact with search.py:156-159).
constexpr int DP_CLUSTER = 8;

__device__ __forceinline__ unsigned dp_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned dp_map_remote(unsigned local_addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}

template <int RPW, int VPL, int PF, bool MEMO_SMEM>
__global__ void __cluster_dims__(DP_CLUSTER, 1, 1) __launch_bounds__(1024)
dp_sweep_cluster_kernel(const float* __restrict__ q, const float* __restrict__ ext, const float* __restrict__ mj, int k,
                        int T, int D, float* __restrict__ costs, int32_t* __restrict__ memo,
                        int32_t* __restrict__ chosen, float* __restrict__ best_path) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int rpc = (k + DP_CLUSTER - 1) / DP_CLUSTER;  // rows per CTA
    extern __shared__ __align__(16) unsigned char dsm[];
    float2* pairs = reinterpret_cast<float2*>(dsm);                  // [2][k] (cost, argmin bits) of the last two steps
    float* ext_s = reinterpret_cast<float*>(pairs + 2 * (size_t)k);  // [rpc][T] penalties of this CTA's rows
    uint16_t* memo_s = reinterpret_cast<uint16_t*>(ext_s + (size_t)rpc * T);  // [T][k] all back-pointers (CTA 0 only)
    __shared__ __align__(8) uint64_t bar[2];  // bar[t & 1] counts the bytes of step t
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dp_smem_u32(&bar[0])) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dp_smem_u32(&bar[1])) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int e = threadIdx.x; e < rpc * T; e += blockDim.x) {
        const int li = e / T, t = e % T, i = rank * rpc + li;
        ext_s[e] = i < k ? ext[(int64_t)t * k + i] : 0.f;
    }
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const float c = ext[i];
        pairs[i] = make_float2(c, 0.f);
        if (MEMO_SMEM && rank == 0) memo_s[i] = 0;
        if (i / rpc == rank) {
            costs[(int64_t)i * T] = c;
            memo[(int64_t)i * T] = 0;
        }
    }
    // register ring of mjac values: slot s holds the values of step t + s for this warp's rows
    float ring[PF + 1][RPW][VPL];
    auto load_step = [&](int t, float (&dst)[RPW][VPL]) {  // t = index of the step being computed (uses mj[t-1])
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            const int li = warp * RPW + r, i = rank * rpc + li;
            const bool row_ok = li < rpc && i < k && t < T;
            const float* row = mj + ((int64_t)(t - 1) * k + i) * k;
#pragma unroll
            for (int v = 0; v < VPL; ++v) {
                const int j = lane + 32 * v;
                dst[r][v] = (row_ok && j < k) ? __ldg(row + j) : INFINITY;
            }
        }
    };
#pragma unroll
    for (int s = 0; s <= PF; ++s) load_step(1 + s, ring[s]);
    // remote addresses of the pair buffers / barrier of CTA `lane` (lanes 0..7 publish)
    const unsigned peer = lane < DP_CLUSTER ? lane : 0;
    const unsigned r_pairs = dp_map_remote(dp_smem_u32(pairs), peer);
    const unsigned r_bar0 = dp_map_remote(dp_smem_u32(&bar[0]), peer);
    cluster.sync();  // barriers initialised and first buffers filled before the first remote store

    // one step of the sweep; `cur` is the register slot holding the mjac values of step t, refilled with those of step
    // t + PF + 1 once they have been used.  The step loop below is unrolled by the ring depth so that the slots are
    // static registers: rotating the ring with moves made the loads issued one step earlier a dependency of the
    // rotation (14 % of the kernel's stall samples).
    auto dp_step = [&](int t, float (&cur)[RPW][VPL]) {
        const int ph = t - 1;
        const float2* prev = pairs + (size_t)(ph & 1) * k;
        const int wr = (ph + 1) & 1;
        const unsigned my_bar = dp_smem_u32(&bar[t & 1]);
        const unsigned r_bar = r_bar0 + (unsigned)((t & 1) * sizeof(uint64_t));
        if (threadIdx.x == 0)  // arm this step's phase: k pairs of 8 bytes will arrive
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(my_bar), "r"(k * 8) : "memory");
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            const int li = warp * RPW + r, i = rank * rpc + li;
            if (li < rpc && i < k) {
                const float e = ext_s[li * T + t];
                float best = INFINITY;
                int bj = 0x7fffffff;
#pragma unroll
                for (int v = 0; v < VPL; ++v) {
                    const int j = lane + 32 * v;
                    if (j < k) {
                        const float val = __fadd_rn(fmaxf(cur[r][v], prev[j].x), e);
                        if (val < best) { best = val; bj = j; }
                    }
                }
                // lexicographic (value, index) minimum over the warp with two REDUX instead of twelve shuffles: costs are
                // non-negative floats (|.| maxima plus non-negative penalties; +inf for padding), whose bit patterns
                // order like unsigned integers; the lowest index among the lanes holding the minimum breaks ties
                const unsigned kb = __reduce_min_sync(0xffffffffu, __float_as_uint(best));
                bj = (int)__reduce_min_sync(0xffffffffu, __float_as_uint(best) == kb ? (unsigned)bj : 0x7fffffffu);
                best = __uint_as_float(kb);
                if (lane < DP_CLUSTER) {  // lane c sends the pair into CTA c and signals its barrier
                    const unsigned dst = r_pairs + (unsigned)(((size_t)wr * k + i) * sizeof(float2));
                    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];"
                                 ::"r"(dst), "r"(__float_as_uint(best)), "r"((unsigned)bj), "r"(r_bar) : "memory");
                } else if (lane == DP_CLUSTER) {
                    costs[(int64_t)i * T + t] = best;
                    memo[(int64_t)i * T + t] = bj;
                }
            }
        }
        load_step(t + PF + 1, cur);  // the slot is free again: fetch step t + PF + 1
        {  // wait until all k pairs of step t have landed in this CTA
            const unsigned parity = (unsigned)(((t - 1) >> 1) & 1);  // n-th use of bar[t & 1], n = (t - 1) / 2 or t / 2 - 1
            asm volatile(
                "{\n"
                ".reg .pred p;\n"
                "DPWAIT_%=:\n"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                "@p bra DPDONE_%=;\n"
                "bra DPWAIT_%=;\n"
                "DPDONE_%=:\n"
                "}\n" ::"r"(my_bar), "r"(parity) : "memory");
        }
        if (MEMO_SMEM && rank == 0) {
            const float2* curp = pairs + (size_t)wr * k;
            for (int i = threadIdx.x; i < k; i += blockDim.x) memo_s[(int64_t)t * k + i] = (uint16_t)__float_as_uint(curp[i].y);
        }
    };
    for (int t = 1; t < T; t += PF + 1) {
        static_for<PF + 1>([&](auto Ss) {
            constexpr int s = decltype(Ss)::value;
            if (t + s < T) dp_step(t + s, ring[s]);
        });
    }
    // final argmin over the last column (first index on ties), then backtrack (search.py:162-173) in CTA 0
    if (rank == 0) {
        const float2* last = pairs + (size_t)((T - 1) & 1) * k;
        __syncthreads();  // memo_s complete
        if (warp == 0) {
            float best = INFINITY;
            int bi = 0x7fffffff;
            for (int i = lane; i < k; i += 32) {
                const float v = last[i].x;
                if (v < best) { best = v; bi = i; }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float ov = __shfl_down_sync(0xffffffffu, best, off);
                const int oi = __shfl_down_sync(0xffffffffu, bi, off);
                if (ov < best || (ov == best && oi < bi)) { best = ov; bi = oi; }
            }
            if (lane == 0) {
                int i = bi;
                for (int t = T - 1; t >= 0; --t) {
                    chosen[t] = i;
                    i = MEMO_SMEM ? (int)memo_s[(int64_t)t * k + i] : __ldcg(memo + (int64_t)i * T + t);
                }
            }
        }
        __threadfence_block();
        __syncthreads();
        for (int e = threadIdx.x; e < T * D; e += blockDim.x) {
            const int t = e / D, d = e % D;
            best_path[e] = q[((int64_t)chosen[t] * T + t) * D + d];
        }
    }
    if (!MEMO_SMEM) __threadfence();  // the other CTAs' memo stores are read by CTA 0's backtrack
    cluster.sync();  // nobody exits while a peer may still address its shared memory
}

inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

}  // namespace cppflow

using namespace cppflow;

extern "C" int cppflow_joint_limit_flags(int robot, const float* d_q, int64_t n, float eps_revolute,
                                         float eps_prismatic, float* d_flags, void* stream) {
    CPPFLOW_CHECK_ARG(n >= 0, "n");
    if (n == 0) return CPPFLOW_OK;
    CPPFLOW_CHECK_ARG(d_q && d_flags, "null pointer");
    CPPFLOW_DISPATCH_ROBOT(robot, joint_limit_flags_kernel<M><<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
                                      d_q, n, eps_revolute, eps_prismatic, d_flags));
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" size_t cppflow_dp_search_workspace_bytes(int64_t k, int64_t T) {
    if (k <= 0 || T <= 0) return 0;
    return align256((size_t)T * k * sizeof(float)) + align256((size_t)(T > 1 ? T - 1 : 0) * k * k * sizeof(float));
}

extern "C" int cppflow_dp_search(int robot, const float* d_q, const uint8_t* d_self_flags, const uint8_t* d_env_flags,
                                 int64_t k, int64_t T, void* d_workspace, size_t workspace_bytes, float* d_best_path,
                                 int32_t* d_memo, float* d_costs, int32_t* d_chosen, void* stream) {
    CPPFLOW_CHECK_ARG(k > 0 && T > 0, "k, T must be positive");
    CPPFLOW_CHECK_ARG(k <= 65535 && T <= 65535, "k, T must be <= 65535");
    CPPFLOW_CHECK_ARG(d_q && d_self_flags && d_env_flags && d_workspace && d_best_path && d_memo && d_costs && d_chosen,
                      "null pointer");
    CPPFLOW_CHECK_ARG(((uintptr_t)d_workspace & 255) == 0, "workspace must be 256-byte aligned");
    if (workspace_bytes < cppflow_dp_search_workspace_bytes(k, T))
        return fail(CPPFLOW_E_WORKSPACE, "cppflow_dp_search: workspace too small (%zu < %zu)", workspace_bytes,
                    cppflow_dp_search_workspace_bytes(k, T));
    cudaStream_t st = (cudaStream_t)stream;
    float* ext = (float*)d_workspace;
    float* mj = (float*)((char*)d_workspace + align256((size_t)T * k * sizeof(float)));
    // DEFAULT_JLIM_SAFETY_PADDING_REVOLUTE = deg2rad(1.5), _PRISMATIC = 3 cm (search.py:20-21)
    const float eps_rev = (float)(1.5 * 3.14159265358979323846 / 180.0);
    const float eps_pris = 0.03f;
    int D = 0;
    CPPFLOW_DISPATCH_ROBOT(robot, {
        D = M::NDOF;
        dp_ext_kernel<M><<<grid_for(k * T, 256), 256, 0, st>>>(d_q, d_self_flags, d_env_flags, (int)k, (int)T, eps_rev,
                                                              eps_pris, ext);
        if (T > 1) {
            dim3 grid((unsigned)(T - 1), (unsigned)((k + MJ_ROWS - 1) / MJ_ROWS));
            dp_mjac_kernel<M><<<grid, 256, 0, st>>>(d_q, (int)k, (int)T, mj);
        }
    });
    CPPFLOW_CHECK_LAUNCH();
    const size_t sh_cost = 2 * (size_t)k * sizeof(float);
    const size_t sh_memo = (size_t)T * k * sizeof(uint16_t);
    cudaError_t e = cudaSuccess;
    // cluster sweep: 8 CTAs split the rows, mjac prefetched in registers; its per-CTA penalties [rows][T] live in shared
    // memory, so very long paths (no limit in the reference's dp_search) take the single-CTA sweep below instead
    const size_t rpc = (size_t)(k + DP_CLUSTER - 1) / DP_CLUSTER;
    const size_t sh_base = 2 * sh_cost + rpc * T * sizeof(float);  // two (cost, argmin) pair buffers + penalties
    if (k <= 512 && T > 1 && sh_base <= 200 * 1024) {
        const bool memo_smem = sh_base + sh_memo <= 200 * 1024;
        const size_t sh = sh_base + (memo_smem ? sh_memo : 0);
#define CPPFLOW_DP_LAUNCH(RPW, VPL, PF, MS)                                                                              \
    do {                                                                                                                 \
        e = cudaFuncSetAttribute(dp_sweep_cluster_kernel<RPW, VPL, PF, MS>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                 (int)sh);                                                                               \
        if (e == cudaSuccess)                                                                                            \
            dp_sweep_cluster_kernel<RPW, VPL, PF, MS><<<DP_CLUSTER, 1024, sh, st>>>(d_q, ext, mj, (int)k, (int)T, D,     \
                                                                                   d_costs, d_memo, d_chosen, d_best_path); \
    } while (0)
        if (k <= 192) {  // the planner's k = 175 (scripts/evaluate.py:266): 6 values per lane
            if (memo_smem) CPPFLOW_DP_LAUNCH(1, 6, 2, true); else CPPFLOW_DP_LAUNCH(1, 6, 2, false);
        } else if (k <= 256) {
            if (memo_smem) CPPFLOW_DP_LAUNCH(1, 8, 2, true); else CPPFLOW_DP_LAUNCH(1, 8, 2, false);
        } else if (k <= 320) {
            if (memo_smem) CPPFLOW_DP_LAUNCH(2, 10, 1, true); else CPPFLOW_DP_LAUNCH(2, 10, 1, false);
        } else {
            if (memo_smem) CPPFLOW_DP_LAUNCH(2, 16, 1, true); else CPPFLOW_DP_LAUNCH(2, 16, 1, false);
        }
#undef CPPFLOW_DP_LAUNCH
        if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    } else {
        const bool memo_smem = sh_cost + sh_memo <= 200 * 1024;
        const size_t sh = sh_cost + (memo_smem ? sh_memo : 0);
        const int threads = k >= 512 ? 1024 : (k >= 128 ? 512 : 256);
        if (memo_smem) {
            e = cudaFuncSetAttribute(dp_sweep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh);
            if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            dp_sweep_kernel<true><<<1, threads, sh, st>>>(d_q, ext, mj, (int)k, (int)T, D, d_costs, d_memo, d_chosen,
                                                          d_best_path);
        } else {
            dp_sweep_kernel<false><<<1, threads, sh, st>>>(d_q, ext, mj, (int)k, (int)T, D, d_costs, d_memo, d_chosen,
                                                           d_best_path);
        }
    }
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

// ----------------------------------------------------------------------------------------------------------------
// Backtrack from chosen terminals (the planner's lm_seeds: the DP's best paths ending at its n cheapest terminals).
// One warp per terminal walks memo from T - 1 to 0 exactly as dp_sweep_kernel's backtrack does (search.py:162-173) and
// gathers the waypoints as it goes: lane d copies joint d of waypoint t of the chosen candidate.  A terminal is a
// candidate index; memo entries are candidate indices, so every step stays inside [0, k).
namespace cppflow {
__global__ void __launch_bounds__(256)
dp_backtrack_kernel(const float* __restrict__ q, const int32_t* __restrict__ memo, int k, int T, int D,
                    const int32_t* __restrict__ terminals, int64_t n, float* __restrict__ out) {
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (j >= n) return;
    int i = __ldg(terminals + j);
    float* o = out + j * (int64_t)T * D;
    for (int t = T - 1; t >= 0; --t) {
        if (lane < D) o[(int64_t)t * D + lane] = __ldg(q + ((int64_t)i * T + t) * D + lane);
        i = __ldg(memo + (int64_t)i * T + t);
    }
}
}  // namespace cppflow

extern "C" int cppflow_dp_backtrack(const float* d_q, const int32_t* d_memo, int64_t k, int64_t T, int ndof,
                                    const int32_t* d_terminals, int64_t n, float* d_out, void* stream) {
    CPPFLOW_CHECK_ARG(k > 0 && T > 0 && n >= 0, "k, T, n");
    CPPFLOW_CHECK_ARG(k <= 65535 && T <= 65535, "k, T must be <= 65535");
    CPPFLOW_CHECK_ARG(ndof > 0 && ndof <= 32, "ndof");
    if (n == 0) return CPPFLOW_OK;
    CPPFLOW_CHECK_ARG(d_q && d_memo && d_terminals && d_out, "null pointer");
    dp_backtrack_kernel<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(d_q, d_memo, (int)k, (int)T, ndof,
                                                                                 d_terminals, n, d_out);
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}
