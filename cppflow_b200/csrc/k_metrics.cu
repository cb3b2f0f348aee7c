// K5: per-path validity metrics - the tensor part of x_is_valid and the cost the multi-GPU argmin ranks paths by.
//
// Reference being replaced:
//   calculate_pose_error_cm_deg       evaluation_utils.py:113-117 (+ positional_errors / rotational_errors :131-141)
//   angular_changes / prismatic_changes, errors_are_below_threshold   evaluation_utils.py:29-75, :97-98, :144-154
//   calc_TL                           optimization.py:173-175
//   capsule pre-filter for the klampt mesh checks of x_is_valid       optimization_utils.py:889-900
// One CTA per path, threads stride over its waypoints, block reduction at the end.  When there are few paths (the
// alternating LM loop checks ONE path per iteration and waits for the answer) the waypoints of a path are split over
// the CTAs of a thread-block cluster instead, one pass of 128 waypoints each; the per-CTA partial results are written
// into the shared memory of the cluster's CTA 0 (distributed shared memory) and combined there in rank order, so the
// sums stay deterministic; in that variant four lanes share a waypoint's 68 distance tests: 41 -> 20 -> ~12 us for T = 295.
#include <cooperative_groups.h>

#include "common.cuh"
#include "collision.cuh"
#include "pose_step.cuh"

namespace cg = cooperative_groups;

namespace cppflow {

constexpr int MBLOCK = 128;

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// CLUSTERED: gridDim.x = P * S with clusters of S CTAs; CTA `rank` of a cluster takes the waypoints
// rank * MBLOCK + threadIdx.x + j * S * MBLOCK of path blockIdx.x / S
// G lanes per waypoint (clustered variant: 4): every lane of a group runs the FK into its own shared-memory column and
// takes every G-th capsule pair / capsule-cuboid test; the warp reductions at the end combine the lanes (max and min
// are idempotent, the trajectory length is added by lane 0 of a group only).
// FUSE (clustered, one pass over the path, one path): the kernel first takes the pose-only LM step of every waypoint
// (lane 0 of a waypoint's group; pose_step.cuh) from `q` into `pf.x_out`, and then evaluates the metrics of the NEW path -
// one launch per iteration of the single-path LM loop instead of two launch-bound ones.  With `rows` set (the batched
// loop, lm_loop_batched.cu) cluster p steps the path in row rows[p] of `q` / `x_out` (paths of T waypoints); its
// metrics still go to out[p].  G and the cluster size depend on T only, so every path gets the single-path arithmetic.
struct PoseFuse {
    float alpha_pos, alpha_rot, lambda;
    float* x_out;
    const int* rows;
};

template <bool COHERENT>
__device__ __forceinline__ float ld_row(const float* p) {
    if constexpr (COHERENT) return __ldcg(p);  // written earlier in this kernel by another SM of the cluster
    else return __ldg(p);
}

template <class M, bool CLUSTERED, int G, bool FUSE = false>
__global__ void __launch_bounds__(MBLOCK)
path_metrics_kernel(const float* __restrict__ q_in, const float* __restrict__ target, int64_t T, const Obstacles ob,
                    float* __restrict__ out, float tag, const PoseFuse pf) {
    constexpr int D = M::NDOF;
    extern __shared__ float smem[];
    __shared__ float red[7][MBLOCK / 32];
    __shared__ float part[8][8];  // CTA 0 of a cluster: partial results of every rank
    unsigned rank = 0, csize = 1;
    if constexpr (CLUSTERED) {
        cg::cluster_group cluster = cg::this_cluster();
        rank = cluster.block_rank();
        csize = cluster.num_blocks();
    }
    const int64_t p = blockIdx.x / csize;
    int64_t prow = p;  // row of `q` that holds path p
    float* sm = smem + threadIdx.x;
    const float* q = q_in;
    if constexpr (FUSE) {
        prow = pf.rows ? __ldg(pf.rows + p) : p;
        const float* xin = q_in + prow * T * D;
        float* xout = pf.x_out + prow * T * D;
        static_assert(CLUSTERED, "the fused step needs the cluster-wide barrier");
        // every thread takes part in the shuffles and the barrier: threads beyond the path shadow its last waypoint
        const int64_t t0 = rank * (MBLOCK / G) + threadIdx.x / G;
        const bool act = t0 < T;
        const int64_t tc = act ? t0 : T - 1;
        float xs[D], tgs[7];
        load_q<M>(xin, tc, xs);
#pragma unroll
        for (int k = 0; k < 7; ++k) tgs[k] = __ldg(target + tc * 7 + k);
        if (threadIdx.x % G == 0) pose_lm_update<M>(xs, tgs, pf.alpha_pos, pf.alpha_rot, pf.lambda, 1, nullptr, nullptr, 0);
        __syncwarp();
        if (threadIdx.x % G == 0 && act) store_q<M>(xout, tc, xs);
        __threadfence();
        cg::this_cluster().sync();  // the new path is complete (neighbouring waypoints live in other CTAs)
        q = pf.x_out;
    }
    float m_pos = 0.f, m_rot = 0.f, m_rev = 0.f, m_pri = 0.f, tl = 0.f, d_self = INFINITY, d_env = INFINITY;
    const int gl = threadIdx.x % G;  // lane within the waypoint's group
    for (int64_t t = rank * (MBLOCK / G) + threadIdx.x / G; t < T; t += (int64_t)csize * (MBLOCK / G)) {
        const int64_t i = prow * T + t;
        float x[D];
#pragma unroll
        for (int d = 0; d < D; ++d) x[d] = ld_row<FUSE>(q + i * D + d);
        CollisionSink<M, MBLOCK, false> sink{sm};
        Frame F;
        fk_chain<M>(x, sink, F);
        // pose error: 100 * |dt| cm; geodesic quaternion distance in degrees (data_types.py:408-411 formula,
        // taken on |dot| so that q and -q are the same rotation)
        const float* tg = target + t * 7;
        const float dx = __ldg(tg) - F.p[0], dy = __ldg(tg + 1) - F.p[1], dz = __ldg(tg + 2) - F.p[2];
        m_pos = fmaxf(m_pos, 100.f * sqrtf(dx * dx + dy * dy + dz * dz));
        float qc[4];
        rotmat_to_quat(F.R, qc);
        float dot = fabsf(qc[0] * __ldg(tg + 3) + qc[1] * __ldg(tg + 4) + qc[2] * __ldg(tg + 5) + qc[3] * __ldg(tg + 6));
        dot = fminf(dot, 1.f - 1e-7f);
        m_rot = fmaxf(m_rot, 2.f * acosf(dot) * 57.29577951308232f);
        if (t > 0) {
            static_for<D>([&](auto Dd) {
                constexpr int d = decltype(Dd)::value;
                const float prev = ld_row<FUSE>(q + (i - 1) * D + d);
                if constexpr (dof_is_prismatic<M>(d)) {
                    m_pri = fmaxf(m_pri, 100.f * fabsf(x[d] - prev));
                } else {
                    const float w = fabsf(wrap_pi(x[d] - prev));
                    m_rev = fmaxf(m_rev, w * 57.29577951308232f);
                    if (gl == 0) tl += w;
                }
            });
        }
        for (int pr = gl; pr < M::NPAIR; pr += G) {
            float C2[3], nrm[3];
            d_self = fminf(d_self, self_pair_distance<M, MBLOCK>(sm, pr, C2, nrm, d_self));
        }
        for (int it = gl; it < ob.n * M::NCAP; it += G) {
            const int o = it / M::NCAP, c = it - o * M::NCAP;
            float Cw[3], nrm[3];
            d_env = fminf(d_env, env_capsule_distance<M, MBLOCK>(sm, c, ob, o, Cw, nrm, d_env));
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float v[7] = {warp_max(m_pos), warp_max(m_rot), warp_max(m_rev), warp_max(m_pri), warp_sum(tl), warp_min(d_self),
                  warp_min(d_env)};
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 7; ++k) red[k][warp] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float r[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) r[k] = red[k][0];
        for (int w = 1; w < MBLOCK / 32; ++w) {
            r[0] = fmaxf(r[0], red[0][w]); r[1] = fmaxf(r[1], red[1][w]);
            r[2] = fmaxf(r[2], red[2][w]); r[3] = fmaxf(r[3], red[3][w]);
            r[4] += red[4][w];
            r[5] = fminf(r[5], red[5][w]); r[6] = fminf(r[6], red[6][w]);
        }
        if constexpr (CLUSTERED) {
            cg::cluster_group cluster = cg::this_cluster();
            float* dst = cluster.map_shared_rank(&part[0][0], 0) + rank * 8;
#pragma unroll
            for (int k = 0; k < 7; ++k) dst[k] = r[k];
        } else {
            float* o = out + p * 8;
#pragma unroll
            for (int k = 0; k < 7; ++k) o[k] = r[k];
            __threadfence_system();  // `out` may be host memory polled by the CPU: the tag must not overtake the metrics
            *reinterpret_cast<volatile float*>(o + 7) = tag;
        }
    }
    if constexpr (CLUSTERED) {
        cg::cluster_group cluster = cg::this_cluster();
        cluster.sync();  // every rank's partials are in CTA 0 (and nobody exits while its memory may be addressed)
        if (rank == 0 && threadIdx.x == 0) {
            float r[7];
#pragma unroll
            for (int k = 0; k < 7; ++k) r[k] = part[0][k];
            for (unsigned w = 1; w < csize; ++w) {
                r[0] = fmaxf(r[0], part[w][0]); r[1] = fmaxf(r[1], part[w][1]);
                r[2] = fmaxf(r[2], part[w][2]); r[3] = fmaxf(r[3], part[w][3]);
                r[4] += part[w][4];
                r[5] = fminf(r[5], part[w][5]); r[6] = fminf(r[6], part[w][6]);
            }
            float* o = out + p * 8;
#pragma unroll
            for (int k = 0; k < 7; ++k) o[k] = r[k];
            __threadfence_system();
            *reinterpret_cast<volatile float*>(o + 7) = tag;
        }
    }
}


// ----------------------------------------------------------------------------------------------------------------
// Many paths (the batch refinement's cost / validity tail: thousands of paths at once): one CTA per path, BLOCK chosen
// at launch so that the path's waypoints fill the CTA's lanes (T = 300 -> 320 threads, one waypoint per thread).
// The minima over the 28 capsule pairs and the 40 capsule-cuboid tests are EXACT but cost only a few exact evaluations
// per waypoint.  With m = distance of the two capsule midpoints (resp. of a midpoint to the cuboid) and
// reach = half lengths + radii, m - reach is a lower bound of the capsule distance, so a pair whose lower bound is not
// below a threshold `thr` known to be >= the PATH's minimum cannot supply that minimum.  The threshold comes from the
// warp: every lane evaluates exactly the one pair that looks closest for its waypoint (smallest m^2 - reach^2, no
// square root), and the minimum of these 32 exact distances over the warp's lanes (shuffles) is `thr` - the lanes of
// a warp are consecutive waypoints of the same path, so it is usually within millimetres of the path's true minimum.
// Phase 2 tests m^2 < (thr + reach)^2 for every pair from the midpoints in registers (fully unrolled, compile-time
// reach) and runs the closed form only for the survivors - typically 0-2 of 68.  (The first version evaluated every
// pair exactly unless its lower bound exceeded the THREAD's running minimum: 0.64 ms for 8192 x 300 waypoints, more
// than the LM assembly itself.)
template <class M, int BLOCK>
__device__ __forceinline__ float self_min_distance(const float (&mid2)[M::NCAP][3], const float* sm, const CollTables<M>& tb) {
    float dd[M::NPAIR];  // 4 x squared distance of the capsule midpoints
    float key = INFINITY;
    int cand = 0;
    static_for<M::NPAIR>([&](auto Pp) {
        constexpr int p = decltype(Pp)::value;
        constexpr int a = pair_cap<M>(p, 0), b = pair_cap<M>(p, 1);
        constexpr float lim = pair_reach<M>(p);
        const float mx = mid2[a][0] - mid2[b][0], my = mid2[a][1] - mid2[b][1], mz = mid2[a][2] - mid2[b][2];
        dd[p] = fmaf(mz, mz, fmaf(my, my, mx * mx));
        const float kp = dd[p] - 4.f * lim * lim;
        cand = kp < key ? p : cand;
        key = fminf(key, kp);
    });
    float C2[3], nrm[3];
    float d = self_pair_exact<M, BLOCK>(sm, tb, cand, C2, nrm);
    const float thr = warp_min(d);  // >= the path's minimum: exact distances of 32 of its waypoints
    unsigned mask = 0u;
    static_for<M::NPAIR>([&](auto Pp) {
        constexpr int p = decltype(Pp)::value;
        const float lim = thr + pair_reach<M>(p);  // lower bound m - reach < thr  <=>  m < thr + reach
        mask |= (lim > 0.f && dd[p] < 4.f * lim * lim) ? (1u << p) : 0u;
    });
    mask &= ~(1u << cand);
    while (mask) {
        const int p = __ffs(mask) - 1;
        mask &= mask - 1;
        d = fminf(d, self_pair_exact<M, BLOCK>(sm, tb, p, C2, nrm));
    }
    return d;
}

// 4 x squared distances of the NCAP capsule midpoints to cuboid o (the obstacle constants are hoisted out of the capsule loop)
template <class M>
__device__ __forceinline__ void env_midpoint_bounds(const float (&mid2)[M::NCAP][3], const Obstacles& ob, int o,
                                                    float (&dd)[M::NCAP]) {
    const float t2[3] = {2.f * ob.t[o][0], 2.f * ob.t[o][1], 2.f * ob.t[o][2]};
    const float lo2[3] = {2.f * ob.lo[o][0], 2.f * ob.lo[o][1], 2.f * ob.lo[o][2]};
    const float hi2[3] = {2.f * ob.hi[o][0], 2.f * ob.hi[o][1], 2.f * ob.hi[o][2]};
    if (ob.has_rot[o]) {
        static_for<M::NCAP>([&](auto Cc) {
            constexpr int c = decltype(Cc)::value;
            const float v[3] = {mid2[c][0] - t2[0], mid2[c][1] - t2[1], mid2[c][2] - t2[2]};
            float acc = 0.f;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const float m = fmaf(ob.R[o][6 + r], v[2], fmaf(ob.R[o][3 + r], v[1], ob.R[o][r] * v[0]));
                const float e = m - fminf(fmaxf(m, lo2[r]), hi2[r]);
                acc = fmaf(e, e, acc);
            }
            dd[c] = acc;
        });
    } else {
        const float wlo[3] = {lo2[0] + t2[0], lo2[1] + t2[1], lo2[2] + t2[2]};
        const float whi[3] = {hi2[0] + t2[0], hi2[1] + t2[1], hi2[2] + t2[2]};
        static_for<M::NCAP>([&](auto Cc) {
            constexpr int c = decltype(Cc)::value;
            float acc = 0.f;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const float e = mid2[c][r] - fminf(fmaxf(mid2[c][r], wlo[r]), whi[r]);
                acc = fmaf(e, e, acc);
            }
            dd[c] = acc;
        });
    }
}

template <class M, int BLOCK>
__device__ __forceinline__ float env_min_distance(const float (&mid2)[M::NCAP][3], const float* sm, const CollTables<M>& tb,
                                                  const Obstacles& ob) {
    if (ob.n == 0) return INFINITY;
    // phase 1: the closest-looking (obstacle, capsule) test over ALL obstacles; one exact evaluation; warp threshold.
    // The bounds of an obstacle are recomputed in phase 2 (12 instructions per test) rather than kept in 80 registers.
    float key = INFINITY;
    int cand = 0;
    for (int o = 0; o < ob.n; ++o) {
        float dd[M::NCAP];
        env_midpoint_bounds<M>(mid2, ob, o, dd);
        static_for<M::NCAP>([&](auto Cc) {
            constexpr int c = decltype(Cc)::value;
            constexpr float lim = cap_reach<M>(c);
            const float kp = dd[c] - 4.f * lim * lim;
            cand = kp < key ? o * 16 + c : cand;
            key = fminf(key, kp);
        });
    }
    float Cw[3], nrm[3];
    float d = env_capsule_exact<M, BLOCK>(sm, tb, cand & 15, cand >> 4, Cw, nrm);
    const float thr = warp_min(d);
    for (int o = 0; o < ob.n; ++o) {
        float dd[M::NCAP];
        env_midpoint_bounds<M>(mid2, ob, o, dd);
        unsigned mask = 0u;
        static_for<M::NCAP>([&](auto Cc) {
            constexpr int c = decltype(Cc)::value;
            const float lim = thr + cap_reach<M>(c);
            mask |= (lim > 0.f && dd[c] < 4.f * lim * lim) ? (1u << c) : 0u;
        });
        if (o == (cand >> 4)) mask &= ~(1u << (cand & 15));
        while (mask) {
            const int c = __ffs(mask) - 1;
            mask &= mask - 1;
            d = fminf(d, env_capsule_exact<M, BLOCK>(sm, tb, c, o, Cw, nrm));
        }
    }
    return d;
}

// SIGN_ONLY (CPPFLOW_METRICS_SIGN_ONLY): the caller only asks whether a path collides (x_is_valid, the cost key of the
// multi-GPU argmin).  Only the pairs the bounding-sphere culls cannot prove apart are evaluated, exactly as in the
// collision flags and the LM assembly: columns 5 / 6 are then the exact minimum when it is negative and some
// non-negative value (the smallest evaluated distance, +inf if every pair was culled) otherwise - 0.46 -> 0.2x ms for
// 8192 x 300 waypoints.
template <class M, int BLOCK, bool SIGN_ONLY>
__global__ void __launch_bounds__(BLOCK)
path_metrics_many_kernel(const float* __restrict__ q, const float* __restrict__ target, int64_t T, const Obstacles ob,
                         float* __restrict__ out, float tag) {
    constexpr int D = M::NDOF;
    constexpr int NWARP = BLOCK / 32;
    extern __shared__ float smem[];
    __shared__ CollTables<M> tb;
    __shared__ float red[7][NWARP];
    fill_coll_tables<M>(tb, ob, threadIdx.x, BLOCK);
    __syncthreads();
    const int64_t p = blockIdx.x;
    float* sm = smem + threadIdx.x;
    float m_pos = 0.f, m_rot = 0.f, m_rev = 0.f, m_pri = 0.f, tl = 0.f, d_self = INFINITY, d_env = INFINITY;
    for (int64_t t0 = 0; t0 < T; t0 += BLOCK) {
        // every lane runs the body (the distance thresholds are shared through warp shuffles): lanes beyond the path
        // shadow its last waypoint - maxima and minima do not mind the duplicate, the trajectory length skips it
        const bool act = t0 + threadIdx.x < T;
        const int64_t t = act ? t0 + threadIdx.x : T - 1;
        const int64_t i = p * T + t;
        float x[D];
        load_q<M>(q, i, x);
        MidSink<M, BLOCK, false> sink;
        sink.sm = sm;
        Frame F;
        fk_chain<M>(x, sink, F);
        const float* tg = target + t * 7;
        const float dx = __ldg(tg) - F.p[0], dy = __ldg(tg + 1) - F.p[1], dz = __ldg(tg + 2) - F.p[2];
        m_pos = fmaxf(m_pos, 100.f * sqrtf(dx * dx + dy * dy + dz * dz));
        float qc[4];
        rotmat_to_quat(F.R, qc);
        float dot = fabsf(qc[0] * __ldg(tg + 3) + qc[1] * __ldg(tg + 4) + qc[2] * __ldg(tg + 5) + qc[3] * __ldg(tg + 6));
        dot = fminf(dot, 1.f - 1e-7f);
        m_rot = fmaxf(m_rot, 2.f * acosf(dot) * 57.29577951308232f);
        if (t > 0) {
            float xp[D];
            load_q<M>(q, i - 1, xp);
            static_for<D>([&](auto Dd) {
                constexpr int d = decltype(Dd)::value;
                if constexpr (dof_is_prismatic<M>(d)) {
                    m_pri = fmaxf(m_pri, 100.f * fabsf(x[d] - xp[d]));
                } else {
                    const float w = fabsf(wrap_pi(x[d] - xp[d]));
                    m_rev = fmaxf(m_rev, w * 57.29577951308232f);
                    tl += act ? w : 0.f;
                }
            });
        }
        if constexpr (SIGN_ONLY) {
            float Cc[3], nrm[3];
            unsigned mask = self_cull_mask<M>(sink.mid2);
            while (mask) {
                const int pr = __ffs(mask) - 1;
                mask &= mask - 1;
                d_self = fminf(d_self, self_pair_exact<M, BLOCK>(sm, tb, pr, Cc, nrm));
            }
#pragma unroll 1
            for (int o = 0; o < tb.ob.n; ++o) {
                unsigned em = env_cull_mask<M>(sink.mid2, tb.ob, o);
                while (em) {
                    const int c = __ffs(em) - 1;
                    em &= em - 1;
                    d_env = fminf(d_env, env_capsule_exact<M, BLOCK>(sm, tb, c, o, Cc, nrm));
                }
            }
        } else {
            d_self = fminf(d_self, self_min_distance<M, BLOCK>(sink.mid2, sm, tb));
            d_env = fminf(d_env, env_min_distance<M, BLOCK>(sink.mid2, sm, tb, ob));
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float v[7] = {warp_max(m_pos), warp_max(m_rot), warp_max(m_rev), warp_max(m_pri), warp_sum(tl), warp_min(d_self),
                  warp_min(d_env)};
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 7; ++k) red[k][warp] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float r[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) r[k] = red[k][0];
        for (int w = 1; w < NWARP; ++w) {
            r[0] = fmaxf(r[0], red[0][w]); r[1] = fmaxf(r[1], red[1][w]);
            r[2] = fmaxf(r[2], red[2][w]); r[3] = fmaxf(r[3], red[3][w]);
            r[4] += red[4][w];
            r[5] = fminf(r[5], red[5][w]); r[6] = fminf(r[6], red[6][w]);
        }
        float* o = out + p * 8;
#pragma unroll
        for (int k = 0; k < 7; ++k) o[k] = r[k];
        __threadfence_system();  // `out` may be host memory polled by the CPU: the tag must not overtake the metrics
        *reinterpret_cast<volatile float*>(o + 7) = tag;
    }
}

template <class M, int BLOCK, bool SIGN_ONLY>
static int launch_metrics_many_v(const float* d_q, const float* d_target, int64_t P, int64_t T, const Obstacles& ob,
                                 float* d_out, float tag, cudaStream_t st) {
    const size_t sh = sizeof(float) * BLOCK * SmemLayout<M>::N_DIST;
    static SmemGrant granted;  // per template instantiation and device
    if (int rc = ensure_dynamic_smem(path_metrics_many_kernel<M, BLOCK, SIGN_ONLY>, sh, granted)) return rc;
    path_metrics_many_kernel<M, BLOCK, SIGN_ONLY><<<(unsigned)P, BLOCK, sh, st>>>(d_q, d_target, T, ob, d_out, tag);
    return CPPFLOW_OK;
}
template <class M, int BLOCK>
static int launch_metrics_many(const float* d_q, const float* d_target, int64_t P, int64_t T, const Obstacles& ob,
                               float* d_out, float tag, bool sign_only, cudaStream_t st) {
    return sign_only ? launch_metrics_many_v<M, BLOCK, true>(d_q, d_target, P, T, ob, d_out, tag, st)
                     : launch_metrics_many_v<M, BLOCK, false>(d_q, d_target, P, T, ob, d_out, tag, st);
}

}  // namespace cppflow

using namespace cppflow;

// `tag` is written to out[p][7] after the seven metrics (system-scope fence in between): a host thread polling a
// device-mapped output buffer sees a complete row once the tag shows up (lm_loop.cu)
int cppflow::path_metrics_tagged(int robot, const float* d_q, const float* d_target, int64_t P, int64_t T,
                                 const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, float* d_out, float tag,
                                 void* stream, int flags) {
    const bool sign_only = (flags & CPPFLOW_METRICS_SIGN_ONLY) != 0;
    CPPFLOW_CHECK_ARG(P >= 0 && T > 0, "P, T");
    if (P == 0) return CPPFLOW_OK;
    CPPFLOW_CHECK_ARG(d_q && d_target && d_out, "null pointer");
    Obstacles ob;
    if (int rc = make_obstacles(h_cuboids, h_Tcuboids, n_obstacles, ob)) return rc;
    // few paths: split each path over a cluster of up to 8 CTAs with G lanes per waypoint, G the largest of 4 / 2 / 1
    // for which the path still fits ONE pass of the cluster (8 * MBLOCK / G waypoints)
    const int G = T <= 8 * MBLOCK / 4 ? 4 : (T <= 8 * MBLOCK / 2 ? 2 : 1);
    const int64_t per_cta = MBLOCK / G;
    const int csize = (int)((T + per_cta - 1) / per_cta < 8 ? (T + per_cta - 1) / per_cta : 8);
    // many paths: one CTA per path fills the GPU better, but its trajectory-length sum is added in another order.
    // METRICS_AS_ONE_PATH keeps the kernel that ONE path of T waypoints gets, whatever P (the batched LM loop's
    // convergence decisions must see the single-path loop's bits)
    const bool clustered = csize > 1 && ((flags & METRICS_AS_ONE_PATH) != 0 || P * csize <= 2 * 148);
    CPPFLOW_DISPATCH_ROBOT(robot, {
        const size_t sh = sizeof(float) * MBLOCK * SmemLayout<M>::N_DIST;
        if (clustered) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(P * csize));
            cfg.blockDim = dim3(MBLOCK);
            cfg.dynamicSmemBytes = sh;
            cfg.stream = (cudaStream_t)stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = (unsigned)csize;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            cudaError_t e = G == 4   ? cudaLaunchKernelEx(&cfg, path_metrics_kernel<M, true, 4>, d_q, d_target, T, ob, d_out, tag, PoseFuse{})
                            : G == 2 ? cudaLaunchKernelEx(&cfg, path_metrics_kernel<M, true, 2>, d_q, d_target, T, ob, d_out, tag, PoseFuse{})
                                     : cudaLaunchKernelEx(&cfg, path_metrics_kernel<M, true, 1>, d_q, d_target, T, ob, d_out, tag, PoseFuse{});
            if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "path_metrics cluster launch: %s", cudaGetErrorString(e));
        } else {
            // block size with the fewest idle lanes over the passes a path needs (ties: the larger block)
            int best = 128;
            int64_t waste = -1;
            for (int b : {128, 192, 256, 320}) {
                const int64_t w = (T + b - 1) / b * b - T;
                if (waste < 0 || w <= waste) { waste = w; best = b; }
            }
            int rc = CPPFLOW_OK;
            switch (best) {
                case 128: rc = launch_metrics_many<M, 128>(d_q, d_target, P, T, ob, d_out, tag, sign_only, (cudaStream_t)stream); break;
                case 192: rc = launch_metrics_many<M, 192>(d_q, d_target, P, T, ob, d_out, tag, sign_only, (cudaStream_t)stream); break;
                case 256: rc = launch_metrics_many<M, 256>(d_q, d_target, P, T, ob, d_out, tag, sign_only, (cudaStream_t)stream); break;
                default: rc = launch_metrics_many<M, 320>(d_q, d_target, P, T, ob, d_out, tag, sign_only, (cudaStream_t)stream); break;
            }
            if (rc) return rc;
        }
    });
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

// pose-only LM step (+ clamp) of n_rows paths of T <= 8 * MBLOCK waypoints and the metrics of the new paths, one launch:
// cluster p steps the path in row rows[p] of d_q into the same row of d_x_out and writes its metrics to d_out[p]
// (rows = NULL: one path, row 0)
int cppflow::pose_step_metrics_rows(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_target,
                                    int64_t T, const float* h_cuboids, const float* h_Tcuboids, int n_obstacles,
                                    const int* d_rows, int64_t n_rows, float* d_x_out, float* d_out, float tag,
                                    void* stream) {
    CPPFLOW_CHECK_ARG(params && d_q && d_target && d_x_out && d_out, "null pointer");
    CPPFLOW_CHECK_ARG(T > 0 && T <= 8 * MBLOCK, "T");
    CPPFLOW_CHECK_ARG(n_rows >= 0 && (d_rows != nullptr || n_rows <= 1), "rows");
    if (n_rows == 0) return CPPFLOW_OK;
    Obstacles ob;
    if (int rc = make_obstacles(h_cuboids, h_Tcuboids, n_obstacles, ob)) return rc;
    const int G = T <= 8 * MBLOCK / 4 ? 4 : (T <= 8 * MBLOCK / 2 ? 2 : 1);
    const int64_t per_cta = MBLOCK / G;
    const int csize = (int)((T + per_cta - 1) / per_cta);
    const PoseFuse pf{params->alpha_position, params->alpha_rotation, params->lm_lambda, d_x_out, d_rows};
    CPPFLOW_DISPATCH_ROBOT(robot, {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(n_rows * csize));
        cfg.blockDim = dim3(MBLOCK);
        cfg.dynamicSmemBytes = sizeof(float) * MBLOCK * SmemLayout<M>::N_DIST;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)csize;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        cudaError_t e = G == 4   ? cudaLaunchKernelEx(&cfg, path_metrics_kernel<M, true, 4, true>, d_q, d_target, T, ob, d_out, tag, pf)
                        : G == 2 ? cudaLaunchKernelEx(&cfg, path_metrics_kernel<M, true, 2, true>, d_q, d_target, T, ob, d_out, tag, pf)
                                 : cudaLaunchKernelEx(&cfg, path_metrics_kernel<M, true, 1, true>, d_q, d_target, T, ob, d_out, tag, pf);
        if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "pose_step_metrics launch: %s", cudaGetErrorString(e));
    });
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

int cppflow::pose_step_metrics_tagged(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_target,
                                      int64_t T, const float* h_cuboids, const float* h_Tcuboids, int n_obstacles,
                                      float* d_x_out, float* d_out, float tag, void* stream) {
    return pose_step_metrics_rows(robot, params, d_q, d_target, T, h_cuboids, h_Tcuboids, n_obstacles, nullptr, 1, d_x_out,
                                  d_out, tag, stream);
}

extern "C" int cppflow_path_metrics(int robot, const float* d_q, const float* d_target, int64_t P, int64_t T,
                                    const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, float* d_out,
                                    void* stream) {
    return cppflow::path_metrics_tagged(robot, d_q, d_target, P, T, h_cuboids, h_Tcuboids, n_obstacles, d_out, 0.f, stream);
}

// ----------------------------------------------------------------------------------------------------------------
// Ranking key of every path and its minimum (distributed.py: key = invalid << 62 | bits(float32 TL) << 31 | global index):
// one launch instead of the ~25 elementwise torch kernels the same arithmetic takes from Python, whose host-side
// enqueue (0.3 ms) was most of the once-per-job tail.  One CTA strides over the paths; 64-bit minimum and the number of
// valid paths by warp shuffles.  out = {best key, #valid, first_index}.
__global__ void __launch_bounds__(1024)
path_key_argmin_kernel(const float* __restrict__ metrics, int64_t P, float thr_pos, float thr_rot, float thr_deg,
                       float thr_cm, long long first_index, long long* __restrict__ out) {
    __shared__ long long s_key[32];
    __shared__ int s_cnt[32];
    long long best = 0x7fffffffffffffffLL;
    int n_valid = 0;
    for (int64_t p = threadIdx.x; p < P; p += blockDim.x) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(metrics + p * 8));
        const float4 b = __ldg(reinterpret_cast<const float4*>(metrics + p * 8 + 4));
        const float tl = b.x;
        const bool finite = isfinite(tl) && tl >= 0.f;
        const bool valid = a.x < thr_pos && a.y < thr_rot && a.z < thr_deg && a.w < thr_cm && b.y >= 0.f && b.z >= 0.f && finite;
        const long long tl_bits = (long long)__float_as_int(finite ? tl : INFINITY);
        const long long key = ((long long)(valid ? 0 : 1) << 62) | (tl_bits << 31) | (first_index + p);
        best = key < best ? key : best;
        n_valid += valid ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other < best ? other : best;
        n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_key[warp] = best; s_cnt[warp] = n_valid; }
    __syncthreads();
    if (warp == 0) {
        best = lane < (int)(blockDim.x >> 5) ? s_key[lane] : 0x7fffffffffffffffLL;
        n_valid = lane < (int)(blockDim.x >> 5) ? s_cnt[lane] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other < best ? other : best;
            n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
        }
        if (lane == 0) { out[0] = best; out[1] = n_valid; out[2] = first_index; }
    }
}

extern "C" int cppflow_path_key_argmin(const float* d_metrics, int64_t P, const cppflow_constraints* constraints,
                                       int64_t first_index, int64_t* d_out, void* stream) {
    CPPFLOW_CHECK_ARG(d_metrics && constraints && d_out, "null pointer");
    CPPFLOW_CHECK_ARG(P >= 0 && first_index >= 0 && first_index + P < ((int64_t)1 << 31), "global path index must fit 31 bits");
    CPPFLOW_CHECK_ARG(((uintptr_t)d_metrics & 15) == 0, "metrics must be 16-byte aligned");
    path_key_argmin_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(
        d_metrics, P, (float)constraints->max_allowed_position_error_cm, (float)constraints->max_allowed_rotation_error_deg,
        (float)constraints->max_allowed_mjac_deg, (float)constraints->max_allowed_mjac_cm, (long long)first_index,
        reinterpret_cast<long long*>(d_out));
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" int cppflow_path_metrics_ex(int robot, const float* d_q, const float* d_target, int64_t P, int64_t T,
                                       const float* h_cuboids, const float* h_Tcuboids, int n_obstacles, int flags,
                                       float* d_out, void* stream) {
    CPPFLOW_CHECK_ARG((flags & ~CPPFLOW_METRICS_SIGN_ONLY) == 0, "unknown metrics flag");
    return cppflow::path_metrics_tagged(robot, d_q, d_target, P, T, h_cuboids, h_Tcuboids, n_obstacles, d_out, 0.f, stream,
                                        flags);
}
