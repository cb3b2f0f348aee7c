// K3: the full Levenberg-Marquardt step (pose + joint-difference + virtual-config + capsule collision residuals)
// for P independent paths of T waypoints.
//
// Reference being replaced (dense, one path at a time, (T*D)^2 floats per path):
//   LmResidualFns.get_r_and_J           optimization_utils.py:486-731  (terms :264-285, :335-349, :430-483, :643-725)
//   _lm_full_step                       optimization.py:95-113         (J^T J + lambda I, Cholesky, 2 triangular solves)
//   levenberg_marquardt_full            optimization.py:116-144
//   clamp_to_joint_limits               optimization_utils.py:823-833
//
// Structure exploited: every residual row touches the D joints of ONE waypoint, except the differencing rows
// r = alpha * wrap(x[t+1] - x[t]) which couple neighbours with +-alpha * I.  Hence
//     A = J^T J + lambda I  is symmetric block-tridiagonal with dense D x D diagonal blocks
//         A_tt = Jp_t^T Jp_t + sum_active w^2 g g^T + beta * n_t + gamma^2 [t in virtual set] + lambda I
//     and off-diagonal blocks -diag(beta),  beta_d = (alpha_diff * prismatic_scale_d)^2,
//     b_t = Jp_t^T e_t - sum_active w^2 d g + beta * (wrap(x[t+1]-x[t]) - wrap(x[t]-x[t-1])) - gamma^2 wrap(x_t - xv_t).
// Kernel A (assembly) evaluates FK, the Jacobian, all capsule distances and the active gradients of one waypoint per
// thread and writes the packed (A_tt, b_t) block (44 floats for D = 8) to the workspace.
// Kernel B (solve) runs a twisted block-Thomas elimination per path (two lanes per path, one from each end), streaming
// the blocks in with TMA bulk copies, and writes clamp(x + dx).  Nothing of size (T*D)^2 is ever formed.
#include "common.cuh"
#include "collision.cuh"
#include "linalg.cuh"

namespace cppflow {

// 256-thread CTAs, two per SM: the 8 warps of a CTA start together and walk the same 68 KB of straight-line code at
// about the same time, so instruction-cache lines are shared (128-thread CTAs, four per SM: 0.436 ms; 256: 0.409 ms;
// 512: 0.486 ms - one CTA per SM leaves nothing to cover its ramp-up and drain)
constexpr int ABLOCK = 256;

template <int D>
struct BlockLayout {
    static constexpr int NT = D * (D + 1) / 2;             // packed lower triangle
    static constexpr int NW = ((NT + D) + 3) / 4 * 4;      // floats per waypoint block, float4 aligned
};

struct AssembleParams {
    float lambda;
    float a_pos, a_rot;
    float w2_self, w2_env;  // alpha^2
    float gamma2;           // (alpha_virtual * alpha_diff)^2
    float beta[CPPFLOW_MAX_DOF];
    int use_pose, use_diff, use_virtual, n_virtual, use_self, use_env;
    int prefetch;  // waypoints ahead whose q row is pulled into L2 for the CTAs of the next wave (0 = off)
};

// (y0, y1) += s * (x0, x1) as ONE packed FFMA2 (sm_100: two independent round-to-nearest FMAs per instruction, the
// scalar is a broadcast operand).  Same math rate as two FFMAs (measured: 68 vs 72 TFLOP/s) but half the issue slots,
// and the assembly kernel is issue-bound (64 % issue-active, FMA pipe at 35 %).  Bit-identical to two fmaf calls.
__device__ __forceinline__ void axpy2(float s, float x0, float x1, float& y0, float& y1) {
    const float2 r = __ffma2_rn(make_float2(s, s), make_float2(x0, x1), make_float2(y0, y1));
    y0 = r.x;
    y1 = r.y;
}

template <class M>
__device__ __forceinline__ void rank1_update(float (&A)[BlockLayout<M::NDOF>::NT], float (&b)[M::NDOF],
                                             const float (&g)[M::NDOF], float w2, float d) {
    constexpr int D = M::NDOF;
    float wg[D];
#pragma unroll
    for (int i = 0; i < D; ++i) wg[i] = w2 * g[i];
#pragma unroll
    for (int i = 0; i + 1 < D; i += 2) axpy2(-d, wg[i], wg[i + 1], b[i], b[i + 1]);
    if constexpr (D % 2 == 1) b[D - 1] = fmaf(-d, wg[D - 1], b[D - 1]);
#pragma unroll
    for (int i = 0; i < D; ++i) {
#pragma unroll
        for (int j = 0; j + 1 <= i; j += 2) axpy2(wg[i], g[j], g[j + 1], A[tri(i, j)], A[tri(i, j + 1)]);
        if (i % 2 == 0) A[tri(i, i)] = fmaf(wg[i], g[i], A[tri(i, i)]);
    }
}

// one q row -> registers; 16-byte vector loads when the row is 16-byte aligned (D % 4 == 0)
template <int D>
__device__ __forceinline__ void load_row(const float* __restrict__ p, float (&x)[D]) {
    if constexpr (D % 4 == 0) {
#pragma unroll
        for (int d = 0; d < D; d += 4) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(p + d));
            x[d] = v.x; x[d + 1] = v.y; x[d + 2] = v.z; x[d + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int d = 0; d < D; ++d) x[d] = __ldg(p + d);
    }
}

// wrap to [-pi, pi) for the LM residuals (evaluation_utils.py:144-154): one rounding step instead of fmodf.  Within
// 1 ulp of torch.remainder for |d| < 4 pi (joint differences are < 2 pi); the bit-exact wrap_pi stays in dp_search.
__device__ __forceinline__ float wrap_pi_lm(float d) {
    const float k = floorf(fmaf(d, 0.15915494309189535f, 0.5f));
    return fmaf(k, -6.28318548202514648f, d);  // float32(2 pi), the modulus torch uses
}

struct SolveParams {
    float b_rev, b_pri;  // beta of revolute / prismatic dofs
    float pivot_floor;   // lambda: every Schur complement of J^T J + lambda I has pivots >= lambda
    int do_clamp;
    unsigned zero;       // always 0; a run-time value so that dependency tokens built from it survive the optimisers
};

// beta of dof d / product beta_i beta_j with the prismatic pattern folded at compile time (three registers instead of
// D (D + 1) / 2 products): beta_d = b_pri for prismatic dofs, b_rev otherwise (make_params)
template <class M>
struct BetaSel {
    float b_rev, b_pri, rr, rp, pp;
    __device__ __forceinline__ BetaSel(float b_rev_, float b_pri_)
        : b_rev(b_rev_), b_pri(b_pri_), rr(b_rev_ * b_rev_), rp(b_rev_ * b_pri_), pp(b_pri_ * b_pri_) {}
    template <int d>
    __device__ __forceinline__ float b() const { return dof_is_prismatic<M>(d) ? b_pri : b_rev; }
    template <int i, int j>
    __device__ __forceinline__ float bb() const {
        return (dof_is_prismatic<M>(i) && dof_is_prismatic<M>(j)) ? pp
               : (dof_is_prismatic<M>(i) || dof_is_prismatic<M>(j)) ? rp : rr;
    }
};

template <class M>
__global__ void __launch_bounds__(ABLOCK, 2)
lm_assemble_kernel(const float* __restrict__ q, const float* __restrict__ xv, const float* __restrict__ target,
                   int P, int T, const Obstacles ob, const AssembleParams prm, float* __restrict__ ws) {
    constexpr int D = M::NDOF;
    constexpr int NT = BlockLayout<D>::NT;
    constexpr int NW = BlockLayout<D>::NW;
    extern __shared__ float smem[];
    __shared__ CollTables<M> tb;
    fill_coll_tables<M>(tb, ob, threadIdx.x, ABLOCK);
    // grid = (path blocks, waypoints): consecutive threads take consecutive PATHS at the same waypoint t, so the
    // target pose is block-uniform and the block stores below are fully coalesced in the [t][k][path] workspace
    const int t = blockIdx.y, pbx = blockIdx.x;
    const int pth_raw = pbx * ABLOCK + threadIdx.x;
    const bool live = pth_raw < P;
    const int pth = live ? pth_raw : P - 1;  // idle lanes shadow the last path and skip the stores
    const int64_t i = (int64_t)pth * T + t;  // row of q / xv
    float* sm = smem + threadIdx.x;

    // all global loads up front (the neighbour rows are strided across paths, like the row itself); the wrapped
    // differences are formed right away so that only D of the 3 D neighbour values stay live through the FK
    float x[D], dwrap[D], vwrap[D];
    const bool has_prev = t > 0, has_next = t < T - 1;
    const bool in_virtual = prm.use_virtual && (t < prm.n_virtual || t >= T - prm.n_virtual);
    load_row<D>(q + i * D, x);
    // the CTAs of waypoint t + prefetch are dispatched about one wave later: their q rows are pulled into L2 now (a CTA
    // lives ~12k cycles of which the wait for its first loads was 15-25 %)
    if (prm.prefetch > 0 && t + prm.prefetch < T)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(q + (i + prm.prefetch) * D));
    float tg[7];
    if (prm.use_pose) {
#pragma unroll
        for (int k = 0; k < 7; ++k) tg[k] = __ldg(target + (int64_t)t * 7 + k);
    }
    if (prm.use_diff) {
        float xp[D], xn[D];
        load_row<D>(q + (has_prev ? i - 1 : i) * D, xp);
        load_row<D>(q + (has_next ? i + 1 : i) * D, xn);
#pragma unroll
        for (int d = 0; d < D; ++d) dwrap[d] = wrap_pi_lm(xn[d] - x[d]) - wrap_pi_lm(x[d] - xp[d]);  // 0 at the ends
    }
    if (in_virtual && xv) {
        float xvv[D];
        load_row<D>(xv + i * D, xvv);
#pragma unroll
        for (int d = 0; d < D; ++d) vwrap[d] = wrap_pi_lm(x[d] - xvv[d]);
    }
    __syncthreads();  // collision tables visible.  (Moving this barrier below the FK, where the tables are first read,
                      // lets early warps run ahead - and costs 4 %: the warps of a CTA then drift apart in the 68 KB
                      // of straight-line code and stop sharing instruction-cache lines.)

    MidSink<M, ABLOCK, true> sink;
    sink.sm = sm;
    Frame F;
    fk_chain<M>(x, sink, F);

    float A[NT], b[D];
#pragma unroll
    for (int k = 0; k < NT; ++k) A[k] = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) b[d] = 0.f;

    // ---- capsule collisions: register culls -> survivor masks -> exact distance; d < 0 adds w^2 g g^T, -w^2 d g
    if (prm.use_self) {
        unsigned mask = self_cull_mask<M>(sink.mid2);
        while (mask) {
            const int p = __ffs(mask) - 1;
            mask &= mask - 1;
            float C2[3], nrm[3];
            const float d = self_pair_exact<M, ABLOCK>(sm, tb, p, C2, nrm);
            if (d < 0.f) {  // residual -alpha d > 0 (optimization_utils.py:653-660)
                float g[D];
                self_pair_gradient_rt<M, ABLOCK>(sm, tb, p, C2, nrm, g);
                rank1_update<M>(A, b, g, prm.w2_self, d);
            }
        }
    }
    if (prm.use_env) {
        // survivors of up to seven obstacles share one 64-bit mask (bit = oo * NCAP + c): a warp pays the LONGEST survivor
        // list of its lanes per mask, so one list per waypoint (instead of one per three obstacles) keeps the lanes'
        // lists as even as they get.  Capsules on links that no joint moves have a zero distance gradient: an active
        // one adds nothing to (A, b), so they are not tested at all.
        constexpr int OGRP = 64 / M::NCAP;
        for (int o0 = 0; o0 < tb.ob.n; o0 += OGRP) {
            unsigned long long mask = 0ull;
#pragma unroll 1  // one copy of the 9 x 12-instruction cull block (and of its rotated-cuboid variant) in the kernel
            for (int oo = 0; oo < OGRP; ++oo)
                if (o0 + oo < tb.ob.n)
                    mask |= (unsigned long long)env_cull_mask<M, n_static_capsules<M>()>(sink.mid2, tb.ob, o0 + oo) << (oo * M::NCAP);
            while (mask) {
                const int bit = __ffsll((long long)mask) - 1;
                mask &= mask - 1;
                const int oo = bit / M::NCAP, c = bit - oo * M::NCAP;
                float Cw[3], nrm[3];
                const float d = env_capsule_exact<M, ABLOCK>(sm, tb, c, o0 + oo, Cw, nrm);
                if (d < 0.f) {
                    float g[D];
                    env_capsule_gradient_rt<M, ABLOCK>(sm, tb, c, Cw, nrm, g);
                    rank1_update<M>(A, b, g, prm.w2_env, d);
                }
            }
        }
    }

    // ---- pose term: Jp^T Jp, Jp^T e with the alpha-scaled geometric Jacobian (optimization.py:77-87)
    if (prm.use_pose) {
        float e[6];
        pose_error(tg, F, e);
        float J[6][D];
        static_for<D>([&](auto Dd) {
            constexpr int d = decltype(Dd)::value;
            float a[3], o[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                a[r] = sm[(SmemLayout<M>::AXES + d * 3 + r) * ABLOCK];
                o[r] = sm[(SmemLayout<M>::ORIGINS + d * 3 + r) * ABLOCK];
            }
            if constexpr (dof_is_prismatic<M>(d)) {
                J[0][d] = 0.f; J[1][d] = 0.f; J[2][d] = 0.f;
                J[3][d] = a[0] * prm.a_pos; J[4][d] = a[1] * prm.a_pos; J[5][d] = a[2] * prm.a_pos;
            } else {
                const float rr[3] = {F.p[0] - o[0], F.p[1] - o[1], F.p[2] - o[2]};
                float v[3];
                cross3(a, rr, v);
                J[0][d] = a[0] * prm.a_rot; J[1][d] = a[1] * prm.a_rot; J[2][d] = a[2] * prm.a_rot;
                J[3][d] = v[0] * prm.a_pos; J[4][d] = v[1] * prm.a_pos; J[5][d] = v[2] * prm.a_pos;
            }
        });
#pragma unroll
        for (int r = 0; r < 3; ++r) { e[r] *= prm.a_rot; e[r + 3] *= prm.a_pos; }
        // b += Jp^T e, A += Jp^T Jp with packed FFMA2 over column pairs (the zero rows 0-2 of a prismatic column are
        // skipped when both columns of a pair allow it; multiplying by the exact zeros changes nothing otherwise)
#pragma unroll
        for (int r = 0; r < 6; ++r) {
#pragma unroll
            for (int c = 0; c + 1 < D; c += 2) axpy2(e[r], J[r][c], J[r][c + 1], b[c], b[c + 1]);
            if constexpr (D % 2 == 1) b[D - 1] = fmaf(e[r], J[r][D - 1], b[D - 1]);
        }
        static_for<D>([&](auto Cc) {
            constexpr int c = decltype(Cc)::value;
            static_for<(c + 2) / 2>([&](auto Hh) {
                constexpr int c2 = 2 * decltype(Hh)::value;
                if constexpr (c2 + 1 <= c) {
                    constexpr int r0 = (dof_is_prismatic<M>(c) || (dof_is_prismatic<M>(c2) && dof_is_prismatic<M>(c2 + 1))) ? 3 : 0;
#pragma unroll
                    for (int r = r0; r < 6; ++r) axpy2(J[r][c], J[r][c2], J[r][c2 + 1], A[tri(c, c2)], A[tri(c, c2 + 1)]);
                } else {  // c2 == c: the diagonal entry of an even column
                    constexpr int r0 = dof_is_prismatic<M>(c) ? 3 : 0;
                    float v = A[tri(c, c)];
#pragma unroll
                    for (int r = r0; r < 6; ++r) v = fmaf(J[r][c], J[r][c], v);
                    A[tri(c, c)] = v;
                }
            });
        });
    }

    if (prm.use_diff) {
        const float nt = (has_prev ? 1.f : 0.f) + (has_next ? 1.f : 0.f);
#pragma unroll
        for (int d = 0; d < D; ++d) {
            b[d] = fmaf(prm.beta[d], dwrap[d], b[d]);
            A[tri(d, d)] = fmaf(prm.beta[d], nt, A[tri(d, d)]);
        }
    }
    if (in_virtual) {
#pragma unroll
        for (int d = 0; d < D; ++d) {
            A[tri(d, d)] += prm.gamma2;
            if (xv) b[d] = fmaf(-prm.gamma2, vwrap[d], b[d]);
        }
    }
#pragma unroll
    for (int d = 0; d < D; ++d) A[tri(d, d)] += prm.lambda;

    // workspace layout [path / 16][t][k][path % 16] float4: the block of one 16-path group is 16 * NW contiguous floats
    float4* grp = reinterpret_cast<float4*>(ws) + (int64_t)(pth >> 4) * T * (NW / 4 * 16) + (pth & 15);  // + t * (NW / 4 * 16)
    auto block_at = [&](int tt) { return grp + (int64_t)tt * (NW / 4 * 16); };
    auto store_blk = [&](int tt, const float (&S)[NT], const float (&y)[D]) {
        float blk[NW];
#pragma unroll
        for (int k = 0; k < NT; ++k) blk[k] = S[k];
#pragma unroll
        for (int d = 0; d < D; ++d) blk[NT + d] = y[d];
#pragma unroll
        for (int k = NT + D; k < NW; ++k) blk[k] = 0.f;
        float4* out = block_at(tt);
#pragma unroll
        for (int k = 0; k < NW / 4; ++k) out[k * 16] = make_float4(blk[4 * k], blk[4 * k + 1], blk[4 * k + 2], blk[4 * k + 3]);
    };
    if (live) store_blk(t, A, b);
}

template <int NW>
__device__ __forceinline__ void load_block(const float* __restrict__ p, float (&v)[NW]) {
    const float4* s = reinterpret_cast<const float4*>(p);
#pragma unroll
    for (int k = 0; k < NW / 4; ++k) {
        const float4 f = s[k];
        v[4 * k] = f.x; v[4 * k + 1] = f.y; v[4 * k + 2] = f.z; v[4 * k + 3] = f.w;
    }
}
template <int NW>
__device__ __forceinline__ void store_block(float* __restrict__ p, const float (&v)[NW]) {
    float4* s = reinterpret_cast<float4*>(p);
#pragma unroll
    for (int k = 0; k < NW / 4; ++k) s[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}

// ----------------------------------------------------------------------------------------------------------------
// Block-tridiagonal solve.  Two lanes per path run a TWISTED (two-sided) block-Thomas factorisation: lane side 0
// eliminates t = 0, 1, ... upwards, lane side 1 eliminates t = T-1, T-2, ... downwards; they meet at the middle block
// m = T/2, whose Schur complement takes both neighbours' inverses.
//   elimination (per side, "in" = the neighbour already eliminated):
//       S_t = A_t - E S_in^-1 E,  y_t = b_t - E u_in,  u_t = S_t^-1 y_t,  E = -diag(beta);  block t <- (-S_t^-1, u_t)
//   middle:  S_m = A_m - E (S_{m-1}^-1 + S_{m+1}^-1) E,  y_m = b_m - E (u_{m-1} + u_{m+1}),  dx_m = S_m^-1 y_m
//   back-substitution (per side, outwards from m):  dx_t = u_t + S_t^-1 (beta . dx_{inner neighbour})
// The arithmetic is ~5 % of the kernel's time: it is a streaming kernel over the block workspace (read A, write
// (-S^-1, u), read them back).  A warp owns one 16-path group, whose blocks are 2816 contiguous bytes per waypoint
// (BlockLayout), and moves them with TMA bulk copies: one elected lane arms an mbarrier and issues
// cp.async.bulk global -> shared for the two blocks (one per side) of a step, SOLVE_RING steps ahead; results go back
// with coalesced 16-byte stores straight from registers.  Warps are independent (no block-level sync).
constexpr int SOLVE_WARPS_DEFAULT = 4;  // a CTA's warp w runs on SM sub-partition w % 4: single-warp CTAs would pile
                                        // every chain of an SM onto one of its four schedulers
// Two ring depths: 3 slots per warp (80 KB per CTA, two CTAs per SM) is the fastest on its own; 4 slots (109 KB) is
// the deepest that still fits NEXT TO one 256-thread assembly CTA (110 KB, half the register file) and is used with
// CPPFLOW_LM_OVERLAP, where the solve of one path chunk - a latency-bound chain that keeps 4 warps of an SM busy - runs
// under the assembly of another chunk (pipeline.ResidentPipeline) and shares the SM's issue slots with it.
// Measured at P = 8192, T = 300 (single stream / 4 chunks overlapped, ms per iteration): ring 2: 0.665 / 0.639,
// ring 3: 0.646 / 0.568, ring 4: 0.657 / 0.560, ring 6 (one CTA per SM): 0.660 / 0.618.
constexpr int SOLVE_RING_ALONE = 3;
constexpr int SOLVE_RING_OVERLAP = 4;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
template <bool CG = false>
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    if constexpr (CG) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// arrival count 1: the thread that arms the barrier with expect_tx
__device__ __forceinline__ void mbar_init(uint64_t* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* smem, const void* gmem, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem)), "l"(gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// per-warp shared memory: SOLVE_RING load slots, each holding the two blocks of one step
// (side 1's block is shifted by 64 B so that the LDS.128 of the two sides hit different banks), the q rows of
// the back-substitution (the mbarriers of the load slots are static shared memory)
template <int D, int SOLVE_RING>
struct SolveSmem {
    static constexpr int NV = BlockLayout<D>::NW / 4;                      // float4 per block
    static constexpr int BLK_BYTES = NV * 16 * 16;                         // one block of a 16-path group
    static constexpr int SLOT_BYTES = (2 * BLK_BYTES + 64 + 127) / 128 * 128;
    static constexpr int Q_BYTES = ((D + 3) / 4) * 16 * 32;                // q rows of one step, 32 lanes
    static constexpr int OFF_Q = SOLVE_RING * SLOT_BYTES;
    static constexpr int BYTES = (OFF_Q + SOLVE_RING * Q_BYTES + 127) / 128 * 128;
    __device__ static unsigned char* part(unsigned char* slot, int side) { return slot + side * (BLK_BYTES + 64); }
    // float4 k of path l (0..15) of the block held in `part`
    __device__ static float4* blk(unsigned char* part, int k, int l) { return reinterpret_cast<float4*>(part) + k * 16 + l; }
    // q value d of `lane`: groups of 4 dofs are contiguous per lane so a 16-byte cp.async can fill them
    __device__ static float* qv(unsigned char* base, int slot, int d, int lane) {
        return reinterpret_cast<float*>(base + OFF_Q + (size_t)slot * Q_BYTES) + ((d >> 2) * 32 + lane) * 4 + (d & 3);
    }
};

// shared-space (32-bit) address forms of the ring primitives: the ring bookkeeping below runs once per step on the
// critical path of a latency-bound chain, so it is kept to 32-bit adds on precomputed bases (no generic -> shared
// conversions, no 64-bit index arithmetic, no modulo)
__device__ __forceinline__ void mbar_expect_tx_a(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s_a(unsigned dst, const void* gmem, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(gmem), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async16_a(unsigned dst, const void* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async4_a(unsigned dst, const void* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(gmem) : "memory");
}

template <class M, int SOLVE_RING, int SOLVE_WARPS>
__global__ void __launch_bounds__(32 * SOLVE_WARPS, 512 / (32 * SOLVE_WARPS))
lm_block_solve_kernel(const float* __restrict__ q, int64_t P, int64_t T64, const SolveParams prm, float* __restrict__ ws,
                      float* __restrict__ x_out) {
    constexpr int D = M::NDOF;
    constexpr int NT = BlockLayout<D>::NT;
    constexpr int NW = BlockLayout<D>::NW;
    constexpr int NV = NW / 4;
    using SM = SolveSmem<D, SOLVE_RING>;
    extern __shared__ __align__(128) unsigned char smem_all[];
    // the warp index as a value ptxas KNOWS to be warp-uniform (a shuffle from lane 0): everything derived from it - the
    // group's workspace base, the ring and barrier addresses - then lives in uniform registers, and a TMA issue is one
    // UBLKCP.  With threadIdx.x >> 5 each UBLKCP was wrapped in an ELECT + 4 x R2UR.BROADCAST + BRA.U.ANY loop (the
    // compiler's fallback for possibly divergent operands): ~100 cycles per copy, twice per step of a latency-bound chain.
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * SOLVE_WARPS + warp;  // 16-path group of this warp
    __shared__ uint64_t s_bars[SOLVE_WARPS][SOLVE_RING];  // one mbarrier per load slot
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < SOLVE_RING; ++j) mbar_init(s_bars[warp] + j);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();          // the only block-level synchronisation: warps are independent from here on
    if (g * 16 >= P) return;
    const int T = (int)T64;   // <= 65535 (check_common): waypoint indices are 32-bit from here on
    unsigned char* sm = smem_all + (size_t)warp * SM::BYTES;
    const unsigned sm_a = smem_u32(sm);              // shared-space address of this warp's ring ...
    const unsigned bar_a = smem_u32(s_bars[warp]);   // ... and of its mbarriers (8 bytes apart)
    const int side = lane & 1, l = lane >> 1;
    const int64_t p_raw = g * 16 + l;
    const bool active = p_raw < P;
    const int64_t p = active ? p_raw : P - 1;  // idle lanes (P % 16 != 0) work on the group's padding and never store x
    unsigned char* wsg = reinterpret_cast<unsigned char*>(ws) + g * T64 * SM::BLK_BYTES;  // block t at wsg + t * BLK_BYTES
    const float* qp = q + p * T64 * D;
    float* xp = x_out + p * T64 * D;
    const int m = T / 2;
    const int n0 = m, n1 = T - 1 - m;           // blocks eliminated by side 0 / side 1
    const int n_side = side == 0 ? n0 : n1;
    const int n_iter = n0 > n1 ? n0 : n1;
    const BetaSel<M> bs(prm.b_rev, prm.b_pri);

    // Ring state: step s (0 .. 2 n_iter - 1: elimination, then back-substitution) lives in slot s % RING and completes
    // that slot's barrier for the (s / RING)-th time - kept as a running (slot, phase) pair instead of a modulo and a
    // division per step.
    int slot = 0;
    unsigned phase = 0u;
    auto advance = [&]() {
        if (++slot == SOLVE_RING) { slot = 0; phase ^= 1u; }
    };
    // Arm slot `sl` and fetch the blocks t0 (side 0) / t1 (side 1) of a later step into it; a negative t skips that
    // side.  Addresses are computed by every lane (cheap, off the elected lane's serial path); lane 0 issues.
    // `token` is the (always zero, but opaque to the compiler) value of slot_read_token below: folding it into the
    // destination address makes the refill of a slot data-dependent on the completed shared-memory reads of its
    // previous contents.
    auto issue = [&](int sl, int t0, int t1, unsigned token) {
        const unsigned bar = bar_a + (unsigned)sl * 8u;
        const unsigned dst = sm_a + (unsigned)sl * (unsigned)SM::SLOT_BYTES + token;
        const unsigned tx = (unsigned)SM::BLK_BYTES * ((t0 >= 0 ? 1u : 0u) + (t1 >= 0 ? 1u : 0u));
        const unsigned char* s0 = wsg + (t0 >= 0 ? t0 : 0) * SM::BLK_BYTES;
        const unsigned char* s1 = wsg + (t1 >= 0 ? t1 : 0) * SM::BLK_BYTES;
        if (lane == 0) {
            mbar_expect_tx_a(bar, tx);
            if (t0 >= 0) bulk_g2s_a(dst, s0, SM::BLK_BYTES, bar);
            if (t1 >= 0) bulk_g2s_a(dst + (unsigned)(SM::BLK_BYTES + 64), s1, SM::BLK_BYTES, bar);
        }
    };
    auto wait_slot = [&]() { mbar_wait_a(bar_a + (unsigned)slot * 8u, phase); };
    auto read_block = [&](float (&v)[NW]) {
        unsigned char* part = SM::part(sm + slot * SM::SLOT_BYTES, side);
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            const float4 f = *SM::blk(part, k, l);
            v[4 * k] = f.x; v[4 * k + 1] = f.y; v[4 * k + 2] = f.z; v[4 * k + 3] = f.w;
        }
    };
    // WAR hazard between the generic-proxy reads of a ring slot (LDS) and the async-proxy refill of the same slot
    // (TMA): an LDS only has to be ISSUED before the instructions after it run, and __syncwarp() of a converged warp is
    // no instruction at all, so nothing orders the UBLKCP of lane 0 after the reads.  Measured: with two solve CTAs per
    // SM the refill regularly landed first and the back-substitution used rows of the block three steps ahead.
    // The token consumes one register of every LDS.128 of every lane (the warp-wide OR cannot complete before every
    // lane's loads have returned) and is folded into the refill's address.
    auto slot_read_token = [&](const float (&v)[NW], bool valid) -> unsigned {
        unsigned acc = 0u;
        if (valid) {
#pragma unroll
            for (int k = 0; k < NV; ++k) acc |= __float_as_uint(v[4 * k]);
        }
        return __reduce_or_sync(0xffffffffu, acc & prm.zero);  // prm.zero = 0 at run time: neither nvcc nor ptxas can fold it
    };
    auto store_x = [&](int t, float (&xn)[D]) {
        if (prm.do_clamp) {
            static_for<D>([&](auto Dd) {
                constexpr int d = decltype(Dd)::value;
                xn[d] = fminf(fmaxf(xn[d], dof_lower<M>(d)), dof_upper<M>(d));
            });
        }
        float* xo = xp + t * D;
        if constexpr (D % 4 == 0) {
#pragma unroll
            for (int d = 0; d < D; d += 4)
                *reinterpret_cast<float4*>(xo + d) = make_float4(xn[d], xn[d + 1], xn[d + 2], xn[d + 3]);
        } else {
#pragma unroll
            for (int d = 0; d < D; ++d) xo[d] = xn[d];
        }
    };

    // running state of this side: nS = -S^-1 of the block eliminated last (packed lower triangle), u = S^-1 y
    float nS[NT], u[D];
#pragma unroll
    for (int k = 0; k < NT; ++k) nS[k] = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) u[d] = 0.f;

    // ---- elimination sweep (steps s = 0 .. n_iter-1):  S_t = A_t + (beta beta^T) . nS,  y_t = b_t + beta . u_in
#pragma unroll
    for (int j = 0; j < SOLVE_RING; ++j)
        if (j < n_iter) issue(j, j < n0 ? j : -1, j < n1 ? T - 1 - j : -1, 0u);
    for (int k = 0; k < n_iter; ++k) {
        const bool mine = k < n_side;
        float blk[NW];
        wait_slot();
        if (mine) read_block(blk);
        const unsigned token = slot_read_token(blk, mine);  // every lane's reads of the slot have returned
        if (mine) {
            static_for<D>([&](auto Ii) {
                constexpr int i = decltype(Ii)::value;
                u[i] = fmaf(bs.template b<i>(), u[i], blk[NT + i]);
                static_for<i + 1>([&](auto Jj) {
                    constexpr int j = decltype(Jj)::value;
                    nS[tri(i, j)] = fmaf(bs.template bb<i, j>(), nS[tri(i, j)], blk[tri(i, j)]);
                });
            });
            sweep_neg_inverse<D>(nS, u, prm.pivot_floor);
        }
        // refill the slot with step k + RING.  Issued AFTER the sweep: the elected lane's few instructions would
        // otherwise sit between the loads and the first pivot of every step; the slot is not needed for RING more steps.
        {
            const int j = k + SOLVE_RING;
            if (j < n_iter) issue(slot, j < n0 ? j : -1, j < n1 ? T - 1 - j : -1, token);
        }
        // block t <- (-S_t^-1 packed, u_t) with 16-byte generic stores: a warp instruction covers 256 contiguous bytes
        // per side.  (An earlier version staged the block in shared memory and sent it with a TMA bulk store: the
        // staging, fence.proxy.async and bulk-group bookkeeping cost ~500 cycles per step, 0.29 -> 0.24 ms without.)
        // The TMA loads of the back-substitution read these blocks through the async proxy: the fences after the loop
        // make them visible.
        if (mine) {
            float v[NW];
#pragma unroll
            for (int i = 0; i < NT; ++i) v[i] = nS[i];
#pragma unroll
            for (int d = 0; d < D; ++d) v[NT + d] = u[d];
#pragma unroll
            for (int i = NT + D; i < NW; ++i) v[i] = 0.f;
            float4* dstg = reinterpret_cast<float4*>(wsg + (side == 0 ? k : T - 1 - k) * SM::BLK_BYTES) + l;
#pragma unroll
            for (int i = 0; i < NV; ++i) dstg[i * 16] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        }
        advance();
    }
    __threadfence();                                  // the generic stores above are performed ...
    asm volatile("fence.proxy.async;" ::: "memory");  // ... and ordered before the async-proxy (TMA) reads below
    __syncwarp();

    // ---- back-substitution loads (steps s = n_iter .. 2 n_iter - 1, block order k = n_side-1 ... 0) start while the
    // middle block is factorised; they read what the stores above wrote, so those have to be complete
    const unsigned q_a = sm_a + (unsigned)SM::OFF_Q + (unsigned)lane * 16u;  // this lane's 16 bytes of q slot 0, dof group 0
    auto issue_q = [&](int qs, int t) {
        const float* src = qp + t * D;
        const unsigned dst = q_a + (unsigned)qs * (unsigned)SM::Q_BYTES;
        if constexpr (D % 4 == 0) {
#pragma unroll
            for (int d = 0; d < D; d += 4) cp_async16_a(dst + (unsigned)(d >> 2) * 512u, src + d);
        } else {
#pragma unroll
            for (int d = 0; d < D; ++d) cp_async4_a(dst + (unsigned)(d >> 2) * 512u + (unsigned)(d & 3) * 4u, src + d);
        }
    };
    auto t_of = [&](int k) { return side == 0 ? k : T - 1 - k; };
    {
        int sl = slot;  // the slots after the last elimination step, in ring order
#pragma unroll
        for (int r = 0; r < SOLVE_RING; ++r) {
            if (r < n_iter) issue(sl, n0 - 1 - r >= 0 ? n0 - 1 - r : -1, n1 - 1 - r >= 0 ? T - 1 - (n1 - 1 - r) : -1, 0u);
            if (++sl == SOLVE_RING) sl = 0;
        }
    }
#pragma unroll
    for (int r = 0; r < SOLVE_RING; ++r) {
        const int k = n_side - 1 - r;
        if (k >= 0) issue_q(r, t_of(k));
        cp_async_commit();
    }

    // ---- middle block: S_m = A_m + (beta beta^T) . (nS_left + nS_right),  y_m = b_m + beta . (u_left + u_right)
    float dx[D];
    {
        float Sm[NT];
        float blk[NW];
        const float4* src = reinterpret_cast<const float4*>(wsg + m * SM::BLK_BYTES) + l;
#pragma unroll
        for (int k = 0; k < NV; ++k) {  // both lanes of the pair read the middle block (same address)
            const float4 f = src[k * 16];
            blk[4 * k] = f.x; blk[4 * k + 1] = f.y; blk[4 * k + 2] = f.z; blk[4 * k + 3] = f.w;
        }
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            const float uo = __shfl_xor_sync(0xffffffffu, u[i], 1);
            dx[i] = fmaf(bs.template b<i>(), u[i] + uo, blk[NT + i]);
            static_for<i + 1>([&](auto Jj) {
                constexpr int j = decltype(Jj)::value;
                const float so = __shfl_xor_sync(0xffffffffu, nS[tri(i, j)], 1);
                Sm[tri(i, j)] = fmaf(bs.template bb<i, j>(), nS[tri(i, j)] + so, blk[tri(i, j)]);
            });
        });
        sweep_neg_inverse<D>(Sm, dx, prm.pivot_floor);  // both lanes of the pair compute dx_m
        if (side == 0 && active) {
            float xn[D];
#pragma unroll
            for (int i = 0; i < D; ++i) xn[i] = __ldg(qp + m * D + i) + dx[i];
            store_x(m, xn);
        }
    }

    // ---- back-substitution outwards from the middle: dx_t = u_t + S_t^-1 (beta . dx_inner) = u_t - nS_t (beta . dx_inner)
    int qslot = 0;
    for (int r = 0; r < n_iter; ++r) {
        cp_async_wait<SOLVE_RING - 1>();
        const int k = n_side - 1 - r;
        const bool mine = k >= 0;
        float blk[NW], xn[D];
        wait_slot();
        if (mine) {
            read_block(blk);
#pragma unroll
            for (int d = 0; d < D; ++d) xn[d] = *SM::qv(sm, qslot, d, lane);
        }
        const unsigned token = slot_read_token(blk, mine);
        if (mine) {
            const int kn = k - SOLVE_RING;
            if (kn >= 0) issue_q(qslot, t_of(kn));
            float z[D];
            static_for<D>([&](auto Ii) {
                constexpr int i = decltype(Ii)::value;
                z[i] = bs.template b<i>() * dx[i];
            });
            // two partial sums per row halve the dependent FMA chain
#pragma unroll
            for (int i = 0; i < D; ++i) {
                float a0 = blk[NT + i], a1 = 0.f;
#pragma unroll
                for (int j = 0; j < D; j += 2) {
                    a0 = fmaf(-(j <= i ? blk[tri(i, j)] : blk[tri(j, i)]), z[j], a0);
                    if (j + 1 < D) a1 = fmaf(-(j + 1 <= i ? blk[tri(i, j + 1)] : blk[tri(j + 1, i)]), z[j + 1], a1);
                }
                dx[i] = a0 + a1;
            }
#pragma unroll
            for (int i = 0; i < D; ++i) xn[i] += dx[i];
        }
        {
            const int rn = r + SOLVE_RING;  // refill after the arithmetic, as in the elimination
            if (rn < n_iter)
                issue(slot, n0 - 1 - rn >= 0 ? n0 - 1 - rn : -1, n1 - 1 - rn >= 0 ? T - 1 - (n1 - 1 - rn) : -1, token);
        }
        if (mine && active) store_x(t_of(k), xn);
        cp_async_commit();
        advance();
        if (++qslot == SOLVE_RING) qslot = 0;
    }
    cp_async_wait<0>();
}

// ----------------------------------------------------------------------------------------------------------------
// The same solve for a HANDFUL of paths (the alternating LM loop refines one path per call and waits for the answer).
// There the streaming kernel is pure latency: one warp walks a chain of T/2 steps and every step pays the TMA issue,
// the mbarrier wait, the ring bookkeeping and a global store on top of the 8x8 sweep (~1.4 us per step, 0.2 ms for
// T = 295).  A path's blocks are only T x 176 bytes: this kernel gathers them (and the path's q rows) into shared
// memory once with cp.async, then eliminates, factorises the middle block and back-substitutes entirely out of
// shared memory, results overwriting the blocks in place.  One single-warp CTA per path; every lane pair (2k, 2k+1)
// runs the two sides redundantly (same addresses, same values), so the warp never diverges and the shuffles of the
// middle block are the streaming kernel's.  The arithmetic and its order are identical: results are bit-identical.
template <class M>
__global__ void __launch_bounds__(32)
lm_block_solve_resident_kernel(const float* __restrict__ q, int64_t P, int64_t T, const SolveParams prm,
                               const float* __restrict__ ws, float* __restrict__ x_out) {
    constexpr int D = M::NDOF;
    constexpr int NT = BlockLayout<D>::NT;
    constexpr int NW = BlockLayout<D>::NW;
    constexpr int NV = NW / 4;
    constexpr int DQ = (D + 3) / 4 * 4;  // q row padded to float4
    constexpr int BLK_BYTES = NV * 16 * 16;
    extern __shared__ __align__(16) unsigned char smem_all[];
    float4* blk_s = reinterpret_cast<float4*>(smem_all);                 // [T][NV]
    float* q_s = reinterpret_cast<float*>(smem_all + (size_t)T * NV * 16);  // [T][DQ]
    const int lane = threadIdx.x;
    const int64_t p = blockIdx.x;
    const int64_t g = p >> 4;
    const int l = (int)(p & 15);
    const unsigned char* wsg = reinterpret_cast<const unsigned char*>(ws) + g * T * BLK_BYTES;
    const float* qp = q + p * T * D;
    for (int64_t idx = lane; idx < T * NV; idx += 32) {
        const int64_t t = idx / NV;
        const int k = (int)(idx - t * NV);
        cp_async16(blk_s + idx, wsg + t * BLK_BYTES + ((size_t)k * 16 + l) * 16);
    }
    for (int64_t idx = lane; idx < T * D; idx += 32) {
        const int64_t t = idx / D;
        cp_async4(q_s + t * DQ + (idx - t * D), qp + idx);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();

    const int side = lane & 1;
    const int64_t m = T / 2;
    const int64_t n0 = m, n1 = T - 1 - m;
    const int64_t n_side = side == 0 ? n0 : n1;
    const int64_t n_iter = n0 > n1 ? n0 : n1;
    const BetaSel<M> bs(prm.b_rev, prm.b_pri);
    auto t_of = [&](int64_t k) { return side == 0 ? k : T - 1 - k; };
    auto read_block = [&](int64_t t, float (&v)[NW]) {
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            const float4 f = blk_s[t * NV + k];
            v[4 * k] = f.x; v[4 * k + 1] = f.y; v[4 * k + 2] = f.z; v[4 * k + 3] = f.w;
        }
    };
    auto store_x = [&](int64_t t, float (&xn)[D]) {
        if (prm.do_clamp) {
            static_for<D>([&](auto Dd) {
                constexpr int d = decltype(Dd)::value;
                xn[d] = fminf(fmaxf(xn[d], dof_lower<M>(d)), dof_upper<M>(d));
            });
        }
        if (lane < 2) {
            float* xo = x_out + (p * T + t) * D;
#pragma unroll
            for (int d = 0; d < D; ++d) xo[d] = xn[d];
        }
    };

    float nS[NT], u[D];
#pragma unroll
    for (int k = 0; k < NT; ++k) nS[k] = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) u[d] = 0.f;
    for (int64_t k = 0; k < n_side; ++k) {
        const int64_t t = t_of(k);
        float blk[NW];
        read_block(t, blk);
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            u[i] = fmaf(bs.template b<i>(), u[i], blk[NT + i]);
            static_for<i + 1>([&](auto Jj) {
                constexpr int j = decltype(Jj)::value;
                nS[tri(i, j)] = fmaf(bs.template bb<i, j>(), nS[tri(i, j)], blk[tri(i, j)]);
            });
        });
        sweep_neg_inverse<D>(nS, u, prm.pivot_floor);
        float v[NW];
#pragma unroll
        for (int i = 0; i < NT; ++i) v[i] = nS[i];
#pragma unroll
        for (int d = 0; d < D; ++d) v[NT + d] = u[d];
#pragma unroll
        for (int i = NT + D; i < NW; ++i) v[i] = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) blk_s[t * NV + i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }
    __syncwarp();

    float dx[D];
    {
        float Sm[NT];
        float blk[NW];
        read_block(m, blk);
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            const float uo = __shfl_xor_sync(0xffffffffu, u[i], 1);
            dx[i] = fmaf(bs.template b<i>(), u[i] + uo, blk[NT + i]);
            static_for<i + 1>([&](auto Jj) {
                constexpr int j = decltype(Jj)::value;
                const float so = __shfl_xor_sync(0xffffffffu, nS[tri(i, j)], 1);
                Sm[tri(i, j)] = fmaf(bs.template bb<i, j>(), nS[tri(i, j)] + so, blk[tri(i, j)]);
            });
        });
        sweep_neg_inverse<D>(Sm, dx, prm.pivot_floor);
        if (side == 0) {
            float xn[D];
#pragma unroll
            for (int i = 0; i < D; ++i) xn[i] = q_s[m * DQ + i] + dx[i];
            store_x(m, xn);
        }
    }

    for (int64_t k = n_side - 1; k >= 0; --k) {
        const int64_t t = t_of(k);
        float blk[NW], xn[D];
        read_block(t, blk);
#pragma unroll
        for (int d = 0; d < D; ++d) xn[d] = q_s[t * DQ + d];
        float z[D];
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            z[i] = bs.template b<i>() * dx[i];
        });
#pragma unroll
        for (int i = 0; i < D; ++i) {
            float a0 = blk[NT + i], a1 = 0.f;
#pragma unroll
            for (int j = 0; j < D; j += 2) {
                a0 = fmaf(-(j <= i ? blk[tri(i, j)] : blk[tri(j, i)]), z[j], a0);
                if (j + 1 < D) a1 = fmaf(-(j + 1 <= i ? blk[tri(i, j + 1)] : blk[tri(j + 1, i)]), z[j + 1], a1);
            }
            dx[i] = a0 + a1;
        }
#pragma unroll
        for (int i = 0; i < D; ++i) xn[i] += dx[i];
        store_x(t, xn);
    }
}

// ----------------------------------------------------------------------------------------------------------------
// The same twisted sweep with the blocks held in REGISTERS only: every lane loads its own path's block with eleven
// coalesced 16-byte loads (lanes = consecutive paths, so a warp instruction covers 2 x 256 contiguous bytes, one run
// per sweep direction), one step AHEAD of its use, and stores the result straight back.  No shared memory, no
// mbarriers, no TMA: a lane only ever re-reads what it wrote itself (same-thread ordering through global memory), so
// no fence and no read token is needed either.  Per step a warp issues ~11 LDG + S-update + sweep + 11 STG; the
// TMA-ring kernel above spends about as many cycles again on ring bookkeeping (mbarrier wait, LDS, token REDUX,
// re-arming).  Bit-identical to it: same lane <-> (path, side) mapping, same arithmetic in the same order.
// WARPS per CTA: 4 (one per scheduler) or 8 (two per scheduler: the second hides the first one's load and
// fixed-latency stalls).
template <class M, int WARPS, bool PREFETCH>
__global__ void __launch_bounds__(32 * WARPS, 1)
lm_block_solve_v2_kernel(const float* __restrict__ q, int64_t P, int64_t T, const SolveParams prm, float* __restrict__ ws,
                         float* __restrict__ x_out) {
    constexpr int D = M::NDOF;
    constexpr int NT = BlockLayout<D>::NT;
    constexpr int NW = BlockLayout<D>::NW;
    constexpr int NV = NW / 4;
    constexpr int64_t BLK_F4 = NV * 16;  // float4 per 16-path block
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * WARPS + warp;  // 16-path group of this warp
    if (g * 16 >= P) return;
    const int side = lane & 1, l = lane >> 1;
    const int64_t p_raw = g * 16 + l;
    const bool active = p_raw < P;
    const int64_t p = active ? p_raw : P - 1;  // idle lanes (P % 16 != 0) work on the group's padding and never store x
    float4* wsg = reinterpret_cast<float4*>(ws) + g * T * BLK_F4 + l;  // float4 k of block t: wsg[t * BLK_F4 + k * 16]
    const float* qp = q + p * T * D;
    const int64_t m = T / 2;
    const int64_t n0 = m, n1 = T - 1 - m;  // blocks eliminated by side 0 / side 1
    const int64_t n_side = side == 0 ? n0 : n1;
    const BetaSel<M> bs(prm.b_rev, prm.b_pri);
    auto t_of = [&](int64_t k) { return side == 0 ? k : T - 1 - k; };
    auto load_blk = [&](int64_t t, float (&v)[NW]) {
        const float4* src = wsg + t * BLK_F4;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            const float4 f = src[k * 16];
            v[4 * k] = f.x; v[4 * k + 1] = f.y; v[4 * k + 2] = f.z; v[4 * k + 3] = f.w;
        }
    };
    auto store_x = [&](int64_t t, float (&xn)[D]) {
        if (prm.do_clamp) {
            static_for<D>([&](auto Dd) {
                constexpr int d = decltype(Dd)::value;
                xn[d] = fminf(fmaxf(xn[d], dof_lower<M>(d)), dof_upper<M>(d));
            });
        }
        float* xo = x_out + (p * T + t) * D;
        if constexpr (D % 4 == 0) {
#pragma unroll
            for (int d = 0; d < D; d += 4)
                *reinterpret_cast<float4*>(xo + d) = make_float4(xn[d], xn[d + 1], xn[d + 2], xn[d + 3]);
        } else {
#pragma unroll
            for (int d = 0; d < D; ++d) xo[d] = xn[d];
        }
    };

    float nS[NT], u[D];
#pragma unroll
    for (int k = 0; k < NT; ++k) nS[k] = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) u[d] = 0.f;

    // ---- elimination: S_t = A_t + (beta beta^T) . nS,  y_t = b_t + beta . u_in;  block t <- (-S_t^-1, u_t)
    float nxt[NW];
    if (PREFETCH && n_side > 0) load_blk(t_of(0), nxt);
    for (int64_t k = 0; k < n_side; ++k) {
        float blk[NW];
        if constexpr (PREFETCH) {
#pragma unroll
            for (int i = 0; i < NW; ++i) blk[i] = nxt[i];
            if (k + 1 < n_side) load_blk(t_of(k + 1), nxt);
        } else {
            load_blk(t_of(k), blk);
        }
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            u[i] = fmaf(bs.template b<i>(), u[i], blk[NT + i]);
            static_for<i + 1>([&](auto Jj) {
                constexpr int j = decltype(Jj)::value;
                nS[tri(i, j)] = fmaf(bs.template bb<i, j>(), nS[tri(i, j)], blk[tri(i, j)]);
            });
        });
        sweep_neg_inverse<D>(nS, u, prm.pivot_floor);
        float v[NW];
#pragma unroll
        for (int i = 0; i < NT; ++i) v[i] = nS[i];
#pragma unroll
        for (int d = 0; d < D; ++d) v[NT + d] = u[d];
#pragma unroll
        for (int i = NT + D; i < NW; ++i) v[i] = 0.f;
        float4* dst = wsg + t_of(k) * BLK_F4;
#pragma unroll
        for (int i = 0; i < NV; ++i) dst[i * 16] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }

    // first back-substitution block and q row on their way while the middle block is factorised
    float qn[D];
    auto load_qrow = [&](int64_t t, float (&v)[D]) {
        if constexpr (D % 4 == 0) {
#pragma unroll
            for (int d = 0; d < D; d += 4) {
                const float4 f = __ldg(reinterpret_cast<const float4*>(qp + t * D + d));
                v[d] = f.x; v[d + 1] = f.y; v[d + 2] = f.z; v[d + 3] = f.w;
            }
        } else {
#pragma unroll
            for (int d = 0; d < D; ++d) v[d] = __ldg(qp + t * D + d);
        }
    };
    if (PREFETCH && n_side > 0) {
        load_blk(t_of(n_side - 1), nxt);
        load_qrow(t_of(n_side - 1), qn);
    }

    // ---- middle block: S_m = A_m + (beta beta^T) . (nS_left + nS_right),  y_m = b_m + beta . (u_left + u_right)
    __syncwarp();
    float dx[D];
    {
        float Sm[NT];
        float blk[NW];
        load_blk(m, blk);  // both lanes of the pair read the middle block (same address)
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            const float uo = __shfl_xor_sync(0xffffffffu, u[i], 1);
            dx[i] = fmaf(bs.template b<i>(), u[i] + uo, blk[NT + i]);
            static_for<i + 1>([&](auto Jj) {
                constexpr int j = decltype(Jj)::value;
                const float so = __shfl_xor_sync(0xffffffffu, nS[tri(i, j)], 1);
                Sm[tri(i, j)] = fmaf(bs.template bb<i, j>(), nS[tri(i, j)] + so, blk[tri(i, j)]);
            });
        });
        sweep_neg_inverse<D>(Sm, dx, prm.pivot_floor);  // both lanes of the pair compute dx_m
        if (side == 0 && active) {
            float xn[D];
#pragma unroll
            for (int i = 0; i < D; ++i) xn[i] = __ldg(qp + m * D + i) + dx[i];
            store_x(m, xn);
        }
    }

    // ---- back-substitution outwards from the middle: dx_t = u_t - nS_t (beta . dx_inner)
    for (int64_t k = n_side - 1; k >= 0; --k) {
        float blk[NW], xn[D];
        if constexpr (PREFETCH) {
#pragma unroll
            for (int i = 0; i < NW; ++i) blk[i] = nxt[i];
#pragma unroll
            for (int d = 0; d < D; ++d) xn[d] = qn[d];
            if (k > 0) {
                load_blk(t_of(k - 1), nxt);
                load_qrow(t_of(k - 1), qn);
            }
        } else {
            load_blk(t_of(k), blk);
            load_qrow(t_of(k), xn);
        }
        float z[D];
        static_for<D>([&](auto Ii) {
            constexpr int i = decltype(Ii)::value;
            z[i] = bs.template b<i>() * dx[i];
        });
#pragma unroll
        for (int i = 0; i < D; ++i) {
            float a0 = blk[NT + i], a1 = 0.f;
#pragma unroll
            for (int j = 0; j < D; j += 2) {
                a0 = fmaf(-(j <= i ? blk[tri(i, j)] : blk[tri(j, i)]), z[j], a0);
                if (j + 1 < D) a1 = fmaf(-(j + 1 <= i ? blk[tri(i, j + 1)] : blk[tri(j + 1, i)]), z[j + 1], a1);
            }
            dx[i] = a0 + a1;
        }
#pragma unroll
        for (int i = 0; i < D; ++i) xn[i] += dx[i];
        if (active) store_x(t_of(k), xn);
    }
}

}  // namespace cppflow
#include "lm_segsolve.cuh"
namespace cppflow {

constexpr int64_t SOLVE_V2_MAX_PATHS_ALONE = 1024, SOLVE_V2_MAX_PATHS_OVERLAP = 256;  // see launch_solve
constexpr int64_t SOLVE_RESIDENT_MAX_PATHS = 8;  // beyond a handful of paths the streaming kernel's throughput wins

template <class M>
static size_t solve_resident_smem(int64_t T) {
    return (size_t)T * (BlockLayout<M::NDOF>::NW * 4 + (M::NDOF + 3) / 4 * 16);
}

template <class M>
static void make_params(const cppflow_lm_params* p, int n_obstacles, int do_clamp, AssembleParams& ap, SolveParams& sp) {
    ap = AssembleParams{};
    sp = SolveParams{};
    ap.lambda = p->lm_lambda;
    ap.a_pos = p->alpha_position;
    ap.a_rot = p->alpha_rotation;
    ap.w2_self = p->alpha_self_collision * p->alpha_self_collision;
    ap.w2_env = p->alpha_env_collision * p->alpha_env_collision;
    const float gam = p->alpha_virtual_configs * p->alpha_differencing;
    ap.gamma2 = gam * gam;
    for (int d = 0; d < M::NDOF; ++d) {
        float a = p->alpha_differencing;
        if (dof_is_prismatic<M>(d)) a *= p->alpha_differencing_prismatic_scaling;
        ap.beta[d] = p->use_differencing ? a * a : 0.f;
        (dof_is_prismatic<M>(d) ? sp.b_pri : sp.b_rev) = ap.beta[d];
    }
    ap.use_pose = p->use_pose;
    ap.use_diff = p->use_differencing;
    ap.use_virtual = p->use_virtual_configs;
    ap.n_virtual = p->n_virtual_configs;
    ap.use_self = p->use_self_collisions;
    ap.use_env = p->use_env_collisions && n_obstacles > 0;
    ap.prefetch = 4;  // 0.402 -> 0.392 ms (2, 4, 8, 16 alike; 32 is too far ahead)
    sp.do_clamp = do_clamp ? 1 : 0;
    sp.pivot_floor = fmaxf(p->lm_lambda, 1e-30f);
}

template <class M>
static int launch_assemble(const cppflow_lm_params* p, const float* q, const float* xv, const float* target, int64_t P,
                           int64_t T, const Obstacles& ob, float* ws, cudaStream_t st) {
    AssembleParams ap;
    SolveParams sp;
    make_params<M>(p, ob.n, 0, ap, sp);
    const size_t sh = sizeof(float) * ABLOCK * SmemLayout<M>::N_FULL;
    static SmemGrant granted;  // per template instantiation and device
    if (int rc = ensure_dynamic_smem(lm_assemble_kernel<M>, sh, granted)) return rc;
    const dim3 grid(grid_for(P, ABLOCK), (unsigned)T);
    lm_assemble_kernel<M><<<grid, ABLOCK, sh, st>>>(q, xv, target, (int)P, (int)T, ob, ap, ws);
    return CPPFLOW_OK;
}

template <class M, int RING, int WARPS = SOLVE_WARPS_DEFAULT>
static int launch_solve_variant(const SolveParams& sp, const float* q, int64_t P, int64_t T, bool high_priority,
                                float* ws, float* x_out, cudaStream_t st) {
    const size_t sh = SolveSmem<M::NDOF, RING>::BYTES * WARPS;
    auto kern = lm_block_solve_kernel<M, RING, WARPS>;
    static SmemGrant granted;  // per template instantiation and device
    if (int rc = ensure_dynamic_smem(kern, sh, granted)) return rc;
    int prio_high = 0;
    if (high_priority) {
        int least = 0;
        cudaDeviceGetStreamPriorityRange(&least, &prio_high);  // of the current device
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid_for(P, 16 * WARPS));
    cfg.blockDim = dim3(32 * WARPS);
    cfg.dynamicSmemBytes = sh;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributePriority;  // CTAs of this launch are dispatched before pending CTAs of assembly
    at[0].val.priority = prio_high;          // launches on other streams (the block scheduler is otherwise FIFO)
    cfg.attrs = at;
    cfg.numAttrs = high_priority ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, q, P, T, sp, ws, x_out);
    if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_block_solve launch: %s", cudaGetErrorString(e));
    return CPPFLOW_OK;
}

template <class M, int WARPS, bool PREFETCH>
static int launch_solve_v2(const SolveParams& sp, const float* q, int64_t P, int64_t T, bool high_priority, float* ws,
                           float* x_out, cudaStream_t st) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid_for(P, 16 * WARPS));
    cfg.blockDim = dim3(32 * WARPS);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributePriority;
    int least = 0, greatest = 0;
    if (high_priority) cudaDeviceGetStreamPriorityRange(&least, &greatest);
    at[0].val.priority = greatest;
    cfg.attrs = at;
    cfg.numAttrs = high_priority ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, lm_block_solve_v2_kernel<M, WARPS, PREFETCH>, q, P, T, sp, ws, x_out);
    if (e != cudaSuccess) return fail(CPPFLOW_E_CUDA, "lm_block_solve_v2 launch: %s", cudaGetErrorString(e));
    return CPPFLOW_OK;
}

template <class M>
static size_t ws_block_bytes(int64_t P, int64_t T) {
    return ((size_t)((P + 15) / 16 * 16) * (size_t)T * BlockLayout<M::NDOF>::NW * sizeof(float) + 255) / 256 * 256;
}
// segments of the segmented solve asked for by the flags (0 = the twisted solve): at least 4 waypoints per segment
static int seg_count(int64_t T, int flags) {
    int64_t n = (flags >> CPPFLOW_LM_SEGMENTS_SHIFT) & 0xff;
    if (n > SEG_MAX_SEGMENTS) n = SEG_MAX_SEGMENTS;
    const int64_t s = n < T / 4 ? n : T / 4;
    return s >= 2 ? (int)s : 0;
}
template <class M>
static size_t ws_seg_corner_bytes(int64_t P, int S) {
    return (size_t)((P + 15) / 16) * S * 2 * SegLayout<M::NDOF>::corner_f4() * 16;
}
template <class M>
static size_t ws_seg_x_bytes(int64_t P, int S) {
    return ((size_t)((P + 15) / 16) * (S - 1) * SegLayout<M::NDOF>::x_f4() * 16 + 255) / 256 * 256;
}
// [blocks][segmented solve: factors | corners | separator solutions]; the blocks are a multiple of 256 bytes
template <class M>
static size_t ws_bytes(int64_t P, int64_t T, int flags = 0) {
    const size_t n = ws_block_bytes<M>(P, T);
    const int S = seg_count(T, flags);
    if (S == 0) return n;
    return 2 * n + ws_seg_corner_bytes<M>(P, S) + ws_seg_x_bytes<M>(P, S);
}

template <class M>
static int launch_solve_segmented(const SolveParams& sp, const float* q, int64_t P, int64_t T, int S, bool high_priority,
                                  float* ws, float* x_out, cudaStream_t st) {
    unsigned char* base = reinterpret_cast<unsigned char*>(ws);
    size_t off = ws_block_bytes<M>(P, T);
    float* fac = reinterpret_cast<float*>(base + off);
    off += ws_block_bytes<M>(P, T);
    float* corners = reinterpret_cast<float*>(base + off);
    off += ws_seg_corner_bytes<M>(P, S);
    float* sepx = reinterpret_cast<float*>(base + off);
    const SegGeom geo{(int)T, S};
    const int64_t warps = (P + 15) / 16 * S;
    constexpr int W = 1;  // single-warp CTAs spread the chains over the SMs' schedulers (as the register-resident solve)
    // CPPFLOW_LM_OVERLAP: the passes of one chunk run while another chunk's assembly fills the SMs; with the highest
    // launch priority their single-warp CTAs take the registers of every assembly CTA that retires
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributePriority;
    int least = 0, greatest = 0;
    if (high_priority) cudaDeviceGetStreamPriorityRange(&least, &greatest);
    at[0].val.priority = greatest;
    cfg.attrs = at;
    cfg.numAttrs = high_priority ? 1 : 0;
    cfg.stream = st;
    auto launched = [](cudaError_t e, const char* what) {
        return e == cudaSuccess ? CPPFLOW_OK : fail(CPPFLOW_E_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
    };
    cfg.gridDim = dim3(grid_for(warps, W));
    cfg.blockDim = dim3(32 * W);
    cfg.dynamicSmemBytes = 0;
    const float* ws_c = ws;
    if (int rc = launched(cudaLaunchKernelEx(&cfg, lm_seg_eliminate_kernel<M, W>, P, geo, sp, ws_c, fac, corners), "lm_seg_eliminate")) return rc;
    const size_t sh = seg_reduced_smem<M::NDOF>(S);
    static SmemGrant granted;  // per template instantiation and device
    if (int rc = ensure_dynamic_smem(lm_seg_reduced_kernel<M>, seg_reduced_smem<M::NDOF>(SEG_MAX_SEGMENTS), granted)) return rc;
    const float* corners_c = corners;
    cfg.gridDim = dim3(grid_for(P, 16));
    cfg.blockDim = dim3(32 * SEG_REDUCED_WARPS);
    cfg.dynamicSmemBytes = sh;
    if (int rc = launched(cudaLaunchKernelEx(&cfg, lm_seg_reduced_kernel<M>, P, geo, sp, ws_c, corners_c, sepx), "lm_seg_reduced")) return rc;
    const float* sepx_c = sepx;
    // pass 3 out of shared memory when a half-segment's factors fit (T / S <= ~70): every load in flight at once
    int half = 0;
    for (int sgm = 0; sgm < S; ++sgm) {
        const int len = geo.last(sgm) - geo.first(sgm) + 1;
        half = len / 2 > half ? len / 2 : half;
    }
    const size_t stage_bytes = (size_t)(half > 0 ? half : 1) * seg_stage_floats<M::NDOF>() * sizeof(float);
    if (stage_bytes <= 200 * 1024) {
        static SmemGrant granted3;  // per template instantiation and device
        if (int rc = ensure_dynamic_smem(lm_seg_substitute_staged_kernel<M>, 200 * 1024, granted3)) return rc;
        const float* fac_c = fac;
        cfg.gridDim = dim3((unsigned)warps);
        cfg.blockDim = dim3(32);
        cfg.dynamicSmemBytes = stage_bytes;
        return launched(cudaLaunchKernelEx(&cfg, lm_seg_substitute_staged_kernel<M>, q, P, geo, sp, ws_c, fac_c, sepx_c, x_out),
                        "lm_seg_substitute_staged");
    }
    cfg.gridDim = dim3(grid_for(warps, W));
    cfg.blockDim = dim3(32 * W);
    cfg.dynamicSmemBytes = 0;
    return launched(cudaLaunchKernelEx(&cfg, lm_seg_substitute_kernel<M, W>, q, P, geo, sp, ws_c, fac, sepx_c, x_out), "lm_seg_substitute");
}

template <class M>
static int launch_solve(const cppflow_lm_params* p, const float* q, int64_t P, int64_t T, int flags, float* ws,
                        float* x_out, cudaStream_t st) {
    AssembleParams ap;
    SolveParams sp;
    make_params<M>(p, 0, flags & CPPFLOW_LM_CLAMP, ap, sp);
    if (const int S = seg_count(T, flags))
        return launch_solve_segmented<M>(sp, q, P, T, S, (flags & CPPFLOW_LM_OVERLAP) != 0, ws, x_out, st);
    if (P <= SOLVE_RESIDENT_MAX_PATHS && solve_resident_smem<M>(T) <= 200 * 1024) {
        const size_t sh = solve_resident_smem<M>(T);
        static SmemGrant granted;  // per template instantiation and device
        if (int rc = ensure_dynamic_smem(lm_block_solve_resident_kernel<M>, 200 * 1024, granted)) return rc;
        lm_block_solve_resident_kernel<M><<<(unsigned)P, 32, sh, st>>>(q, P, T, sp, ws, x_out);
        return CPPFLOW_OK;
    }
    // few paths: the chain latency is all there is, and the register-resident kernel's step is the shortest (no ring
    // bookkeeping): P = 512 alone 0.128 ms against 0.21; under overlap it only wins for chunks of <= 256 paths
    // (4 chunks of 256: 0.203 ms per iteration against 0.254, of 512: 0.337 against 0.286).  Bit-identical either way.
    // The other variants measured in round 2 (8 or 1 warps per CTA, the register-resident kernel with 2 / 4 / 8 warps
    // or without prefetch) are in profiles/r02_notes.md.
    const bool overlap = (flags & CPPFLOW_LM_OVERLAP) != 0;
    if (P <= (overlap ? SOLVE_V2_MAX_PATHS_OVERLAP : SOLVE_V2_MAX_PATHS_ALONE))
        return launch_solve_v2<M, 1, true>(sp, q, P, T, overlap, ws, x_out, st);
    if (overlap) return launch_solve_variant<M, SOLVE_RING_OVERLAP>(sp, q, P, T, true, ws, x_out, st);
    return launch_solve_variant<M, SOLVE_RING_ALONE>(sp, q, P, T, false, ws, x_out, st);
}

}  // namespace cppflow

using namespace cppflow;

extern "C" size_t cppflow_lm_full_workspace_bytes_ex(int robot, int64_t P, int64_t T, int flags) {
    if (P < 0 || T < 0) return 0;
    switch (robot) {
        case ROBOT_FETCH: return ws_bytes<Fetch>(P, T, flags);
        case ROBOT_FETCH_ARM: return ws_bytes<FetchArm>(P, T, flags);
        case ROBOT_PANDA: return ws_bytes<Panda>(P, T, flags);
        default: return 0;
    }
}

extern "C" size_t cppflow_lm_full_workspace_bytes(int robot, int64_t P, int64_t T) {
    return cppflow_lm_full_workspace_bytes_ex(robot, P, T, 0);
}

// the bits of `do_clamp` that cppflow_lm_full_step / cppflow_lm_full_solve know; any other bit is rejected, so that a
// caller still passing a removed option gets an error instead of a step computed some other way
constexpr int LM_KNOWN_FLAGS = CPPFLOW_LM_CLAMP | CPPFLOW_LM_OVERLAP | CPPFLOW_LM_SEGMENTS(0xff);

static int check_common(int robot, const cppflow_lm_params* params, int64_t P, int64_t T, const void* d_workspace,
                        size_t workspace_bytes, int flags = 0) {
    CPPFLOW_CHECK_ARG(params != nullptr, "params");
    CPPFLOW_CHECK_ARG(P >= 0 && T >= 0, "P, T");
    CPPFLOW_CHECK_ARG(T <= 65535 && P <= (int64_t)1 << 30, "T must be <= 65535 (grid.y) and P <= 2^30");
    CPPFLOW_CHECK_ARG(d_workspace != nullptr, "workspace");
    CPPFLOW_CHECK_ARG(!params->use_virtual_configs || (params->n_virtual_configs > 0 && 2 * params->n_virtual_configs < T),
                      "2 * n_virtual_configs must be < T (optimization_utils.py:457-459)");
    CPPFLOW_CHECK_ARG(((uintptr_t)d_workspace & 15) == 0, "workspace must be 16-byte aligned");
    if (workspace_bytes < cppflow_lm_full_workspace_bytes_ex(robot, P, T, flags))
        return fail(CPPFLOW_E_WORKSPACE, "lm_full: workspace too small (%zu < %zu)", workspace_bytes,
                    cppflow_lm_full_workspace_bytes_ex(robot, P, T, flags));
    return CPPFLOW_OK;
}

extern "C" int cppflow_lm_full_assemble(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_xv,
                                        const float* d_target, int64_t P, int64_t T, const float* h_cuboids,
                                        const float* h_Tcuboids, int n_obstacles, void* d_workspace,
                                        size_t workspace_bytes, void* stream) {
    if (P == 0 || T == 0) return CPPFLOW_OK;
    if (int rc = check_common(robot, params, P, T, d_workspace, workspace_bytes)) return rc;
    CPPFLOW_CHECK_ARG(d_q != nullptr, "null pointer");
    CPPFLOW_CHECK_ARG(!params->use_pose || d_target, "target path required when use_pose");
    Obstacles ob;
    if (int rc = make_obstacles(h_cuboids, h_Tcuboids, n_obstacles, ob)) return rc;
    int rc = CPPFLOW_OK;
    CPPFLOW_DISPATCH_ROBOT(robot, rc = launch_assemble<M>(params, d_q, d_xv, d_target, P, T, ob, (float*)d_workspace,
                                                          (cudaStream_t)stream));
    if (rc) return rc;
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" int cppflow_lm_full_solve(int robot, const cppflow_lm_params* params, const float* d_q, int64_t P, int64_t T,
                                     int do_clamp, void* d_workspace, size_t workspace_bytes, float* d_x_out,
                                     void* stream) {
    CPPFLOW_CHECK_ARG((do_clamp & ~LM_KNOWN_FLAGS) == 0, "unknown do_clamp bits");
    if (P == 0 || T == 0) return CPPFLOW_OK;
    if (int rc = check_common(robot, params, P, T, d_workspace, workspace_bytes, do_clamp)) return rc;
    CPPFLOW_CHECK_ARG(d_q && d_x_out, "null pointer");
    int rc = CPPFLOW_OK;
    CPPFLOW_DISPATCH_ROBOT(robot, rc = launch_solve<M>(params, d_q, P, T, do_clamp, (float*)d_workspace, d_x_out,
                                                       (cudaStream_t)stream));
    if (rc) return rc;
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" int cppflow_lm_full_step(int robot, const cppflow_lm_params* params, const float* d_q, const float* d_xv,
                                    const float* d_target, int64_t P, int64_t T, const float* h_cuboids,
                                    const float* h_Tcuboids, int n_obstacles, int do_clamp, void* d_workspace,
                                    size_t workspace_bytes, float* d_x_out, void* stream) {
    CPPFLOW_CHECK_ARG((do_clamp & ~LM_KNOWN_FLAGS) == 0, "unknown do_clamp bits");
    if (int rc = cppflow_lm_full_assemble(robot, params, d_q, d_xv, d_target, P, T, h_cuboids, h_Tcuboids, n_obstacles,
                                          d_workspace, workspace_bytes, stream))
        return rc;
    return cppflow_lm_full_solve(robot, params, d_q, P, T, do_clamp, d_workspace, workspace_bytes, d_x_out, stream);
}
