// Kernels and host helpers shared by the forward/reverse pass (k_flow.cu) and the training step (k_flow_train.cu).
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cuda_bf16.h>

#include "common.cuh"

namespace cppflow {
namespace flow {

constexpr int MAXW = 16;  // state row stride (floats) and the widest latent
constexpr int KIN = 64;   // first-layer input width (bf16, zero-padded [half | cond])
constexpr int NOUT = 16;  // rows of the packed last Linear
constexpr int BM = 128;   // GEMM tile rows (tensor-memory lanes)
constexpr int BK = 64;    // GEMM k-block: 64 bf16 = one 128-byte swizzle row
constexpr float LEAKY = 0.01f;
constexpr float ATAN_SCALE = 0.636f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, void* dst, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major operand tile in shared memory, 128-byte swizzle: rows of 64 bf16 at 128 B, 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}

// kind::f16 instruction descriptor: D fp32, A and B bf16, both K-major, M x N
template <int N>
constexpr uint32_t instr_desc() {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(a), "l"(b), "r"(idesc), "r"(accumulate));
}

__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

template <int BN>
struct GemmCfg {
    static constexpr int STAGES = BN == 256 ? 4 : 6;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr size_t SMEM = 1024 + (size_t)STAGES * STAGE_BYTES + 256;
};

// What the GEMM epilogue does with acc[m, n] = A[m, :] . W[n, :] for the rows m < n_rows of the tile:
//   EPI_FWD:   out[m, n] = bf16(leaky_relu(acc + bias[n]))                       (a hidden layer of the forward pass)
//   EPI_FWD_T: EPI_FWD, and the same bf16 value to out_t[n, m]                   (training: the input of a weight gradient)
//   EPI_BWD:   out[m, n] = bf16(acc * leaky'(act[m, n])), also to out_t[n, m]    (training: the gradient of a hidden layer)
//   EPI_F32:   out_f[m, n] = acc                                                 (training: weight and input gradients)
// leaky' is 1 where the saved BF16 activation is > 0 and LEAKY elsewhere, as torch's LeakyReLU backward.
enum { EPI_FWD = 0, EPI_FWD_T = 1, EPI_BWD = 2, EPI_F32 = 3 };
struct EpiArgs {
    const float* bias;
    __nv_bfloat16* out;         // row stride ldo
    __nv_bfloat16* out_t;       // row stride ldt
    const __nv_bfloat16* act;   // row stride ldo
    float* out_f;               // row stride ldo
    int ldo;
    int64_t ldt;
};

// A [n_rows, K] and W [N, K] are bf16, K-major, read through the tensor maps; rows >= n_rows read as 0 and are not
// stored.  Warp 0 lane 0 issues the TMA loads, warp 1 lane 0 the MMAs, then all four warps drain tensor memory.
template <int BN, int EPI = EPI_FWD>
__global__ void __launch_bounds__(128, 1) flow_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a,
                                                           const __grid_constant__ CUtensorMap tmap_w, EpiArgs ep,
                                                           int n_rows, int k_blocks) {
    using C = GemmCfg<BN>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* sa = smem;
    uint8_t* sb = smem + C::STAGES * C::A_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
    uint64_t* empty = full + C::STAGES;
    uint64_t* done = empty + C::STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;

    if (threadIdx.x == 0) {
        for (int s = 0; s < C::STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_w)) : "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(BN));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0 && lane == 0) {
        for (int kb = 0; kb < k_blocks; ++kb) {
            const int s = kb % C::STAGES;
            if (kb >= C::STAGES) mbar_wait(&empty[s], ((kb / C::STAGES) - 1) & 1);
            mbar_expect_tx(&full[s], C::STAGE_BYTES);
            tma_load_2d(&tmap_a, sa + s * C::A_BYTES, &full[s], kb * BK, m0);
            tma_load_2d(&tmap_w, sb + s * C::B_BYTES, &full[s], kb * BK, n0);
        }
    } else if (warp == 1 && lane == 0) {
        constexpr uint32_t idesc = instr_desc<BN>();
        for (int kb = 0; kb < k_blocks; ++kb) {
            const int s = kb % C::STAGES;
            mbar_wait(&full[s], (kb / C::STAGES) & 1);
            tc_fence_after();
            const uint64_t da = smem_desc(smem_u32(sa + s * C::A_BYTES));
            const uint64_t db = smem_desc(smem_u32(sb + s * C::B_BYTES));
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)  // 16 bf16 = 32 bytes along the swizzled row: +2 in the address field
                mma_bf16(tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            mma_commit(&empty[s]);
        }
        mma_commit(done);
    }
    __syncwarp();
    mbar_wait(done, 0);
    tc_fence_after();

    const int row = m0 + warp * 32 + lane;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
        uint32_t r[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + c * 32, r);
        if (row < n_rows) {
            const int col = n0 + c * 32;
            if constexpr (EPI == EPI_F32) {
                float4* dst = reinterpret_cast<float4*>(ep.out_f + (size_t)row * ep.ldo + col);
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    dst[q] = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]),
                                         __uint_as_float(r[4 * q + 2]), __uint_as_float(r[4 * q + 3]));
            } else {
                uint4 pk[4];
                uint32_t* pw = reinterpret_cast<uint32_t*>(pk);
                uint4 ak[4];
                if constexpr (EPI == EPI_BWD) {
                    const uint4* src = reinterpret_cast<const uint4*>(ep.act + (size_t)row * ep.ldo + col);
#pragma unroll
                    for (int q = 0; q < 4; ++q) ak[q] = __ldg(src + q);
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    float v0 = __uint_as_float(r[4 * q + 0]), v1 = __uint_as_float(r[4 * q + 1]);
                    float v2 = __uint_as_float(r[4 * q + 2]), v3 = __uint_as_float(r[4 * q + 3]);
                    if constexpr (EPI == EPI_BWD) {
                        const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(ak) + 2 * q;
                        const float2 a01 = __bfloat1622float2(a2[0]), a23 = __bfloat1622float2(a2[1]);
                        v0 = a01.x > 0.f ? v0 : LEAKY * v0;
                        v1 = a01.y > 0.f ? v1 : LEAKY * v1;
                        v2 = a23.x > 0.f ? v2 : LEAKY * v2;
                        v3 = a23.y > 0.f ? v3 : LEAKY * v3;
                    } else {
                        const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + col) + q);
                        v0 += b.x, v1 += b.y, v2 += b.z, v3 += b.w;
                        v0 = v0 > 0.f ? v0 : LEAKY * v0;
                        v1 = v1 > 0.f ? v1 : LEAKY * v1;
                        v2 = v2 > 0.f ? v2 : LEAKY * v2;
                        v3 = v3 > 0.f ? v3 : LEAKY * v3;
                    }
                    __nv_bfloat162 lo = __floats2bfloat162_rn(v0, v1), hi = __floats2bfloat162_rn(v2, v3);
                    pw[2 * q] = *reinterpret_cast<uint32_t*>(&lo);
                    pw[2 * q + 1] = *reinterpret_cast<uint32_t*>(&hi);
                }
                uint4* dst = reinterpret_cast<uint4*>(ep.out + (size_t)row * ep.ldo + col);
#pragma unroll
                for (int q = 0; q < 4; ++q) dst[q] = pk[q];
                if constexpr (EPI != EPI_FWD) {  // lanes hold consecutive rows: each column's store is coalesced
                    const __nv_bfloat16* pb = reinterpret_cast<const __nv_bfloat16*>(pk);
#pragma unroll
                    for (int j = 0; j < 32; ++j) ep.out_t[(size_t)(col + j) * ep.ldt + row] = pb[j];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(BN));
    }
}

// What follows a state update (one warp per row, lane j holds element j of the state v):
//   gather (optional): v'[j] = v[gather[j]];
//   final (out != NULL): out[row, j] = v'[j] (/ scale[j] in reverse, clamped to [lower, upper] for j < ndof with clamp);
//   otherwise: state[row] = v', u[row] = bf16([v'[next_lo .. next_lo + next_len) | cond[row % n_cond] | 0 ...]),
//     and (training) the same bf16 values to the transposed copy u_t[:, row] (row stride ldt).
// cond rows are cond_w floats: 7 (poses; the softflow scale, column 7 when dim_cond = 8, is 0) or dim_cond (training).
struct Emit {
    int width, ndof;
    const int32_t* gather;
    int next_lo, next_len;
    float* state;
    __nv_bfloat16* u;
    const float* cond;
    int64_t n_cond;
    int cond_w;
    __nv_bfloat16* u_t;
    int64_t ldt;
    float* out;
    const float* scale;
    int reverse, clamp;
    float lower[CPPFLOW_MAX_DOF], upper[CPPFLOW_MAX_DOF];
};

__device__ __forceinline__ void emit(float v, int64_t row, bool valid, const Emit& e, int lane) {
    if (e.gather) v = __shfl_sync(0xffffffffu, v, lane < e.width ? __ldg(e.gather + lane) : lane);
    if (e.out) {
        if (valid && lane < e.width) {
            float x = e.reverse ? v / __ldg(e.scale + lane) : v;
            if (e.clamp && lane < e.ndof) {
                float lo = 0.f, hi = 0.f;
#pragma unroll
                for (int j = 0; j < CPPFLOW_MAX_DOF; ++j)
                    if (j == lane) lo = e.lower[j], hi = e.upper[j];
                x = fminf(fmaxf(x, lo), hi);
            }
            e.out[row * e.width + lane] = x;
        }
        return;
    }
    const int q0 = 2 * lane, q1 = 2 * lane + 1;
    const float h0 = __shfl_sync(0xffffffffu, v, min(e.next_lo + q0, 31));
    const float h1 = __shfl_sync(0xffffffffu, v, min(e.next_lo + q1, 31));
    if (!valid) return;
    if (lane < MAXW) e.state[row * MAXW + lane] = v;
    const float* c = e.cond + (row % e.n_cond) * e.cond_w;
    auto elem = [&](int q, float h) {
        if (q < e.next_len) return h;
        const int k = q - e.next_len;
        return k < e.cond_w ? __ldg(c + k) : 0.f;
    };
    const __nv_bfloat162 uq = __floats2bfloat162_rn(elem(q0, h0), elem(q1, h1));
    reinterpret_cast<__nv_bfloat162*>(e.u + row * KIN)[lane] = uq;
    if (e.u_t) {
        e.u_t[q0 * e.ldt + row] = uq.x;
        e.u_t[q1 * e.ldt + row] = uq.y;
    }
}

static __global__ void __launch_bounds__(256) flow_prep_kernel(const float* __restrict__ in, int64_t n, Emit e) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const bool valid = row < n;
    float v = 0.f;
    if (valid && lane < e.width) {
        v = in[row * e.width + lane];
        if (!e.reverse) v *= __ldg(e.scale + lane);
    }
    emit(v, row, valid, e, lane);
}

struct Head {
    const float* state_in;        // [n, MAXW]: the state this step updates (Emit::state receives the next one)
    const __nv_bfloat16* hidden;  // [n, H]
    const float* w_out;           // [16, H]
    const float* b_out;           // [16]
    int H;
    int upd_lo, upd_len;  // the half this step updates: s = outputs [0, upd_len), t = [upd_len, 2 upd_len)
    float clamp;
    int64_t n;
    float* save_s;  // training, else NULL: the raw s of the updated lanes [n, MAXW]
    float* logdet;  // training, else NULL: logdet[row] += sum of the clamped s of the row
};

constexpr int HEAD_ROWS = 4;  // rows per warp and pass: each shared-memory read of the last Linear serves 4 rows

// Last Linear + coupling update + Emit.  The last Linear's weights are staged in shared memory as [16][2][H / 8]
// float4 so that lane l's two float4 of columns 8 q .. 8 q + 7 are consecutive across the warp.
static __global__ void __launch_bounds__(256) flow_head_kernel(Head a, Emit e) {
    extern __shared__ float4 sw[];
    __shared__ float red[8][HEAD_ROWS][NOUT];
    const int H = a.H, H4 = H / 4, H8 = H / 8;
    for (int i = threadIdx.x; i < NOUT * H4; i += blockDim.x) {
        const int o = i / H4, c4 = i % H4;
        sw[o * H4 + (c4 & 1) * H8 + (c4 >> 1)] = __ldg(reinterpret_cast<const float4*>(a.w_out) + i);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int64_t g = (int64_t)blockIdx.x * 8 + warp; g * HEAD_ROWS < a.n; g += (int64_t)gridDim.x * 8) {
        const int64_t row0 = g * HEAD_ROWS;
        float acc[HEAD_ROWS][NOUT];
#pragma unroll
        for (int r = 0; r < HEAD_ROWS; ++r)
#pragma unroll
            for (int o = 0; o < NOUT; ++o) acc[r][o] = 0.f;
        for (int q = lane; q < H8; q += 32) {
            float h[HEAD_ROWS][8];
#pragma unroll
            for (int r = 0; r < HEAD_ROWS; ++r) {
                uint4 raw = make_uint4(0, 0, 0, 0);
                if (row0 + r < a.n) raw = __ldg(reinterpret_cast<const uint4*>(a.hidden + (row0 + r) * H) + q);
                const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 f = __bfloat1622float2(p[k]);
                    h[r][2 * k] = f.x;
                    h[r][2 * k + 1] = f.y;
                }
            }
#pragma unroll
            for (int o = 0; o < NOUT; ++o) {
                const float4 w0 = sw[o * H4 + q], w1 = sw[o * H4 + H8 + q];
#pragma unroll
                for (int r = 0; r < HEAD_ROWS; ++r) {
                    float s = acc[r][o];
                    s = fmaf(h[r][0], w0.x, s);
                    s = fmaf(h[r][1], w0.y, s);
                    s = fmaf(h[r][2], w0.z, s);
                    s = fmaf(h[r][3], w0.w, s);
                    s = fmaf(h[r][4], w1.x, s);
                    s = fmaf(h[r][5], w1.y, s);
                    s = fmaf(h[r][6], w1.z, s);
                    s = fmaf(h[r][7], w1.w, s);
                    acc[r][o] = s;
                }
            }
        }
#pragma unroll
        for (int r = 0; r < HEAD_ROWS; ++r)
#pragma unroll
            for (int o = 0; o < NOUT; ++o) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) acc[r][o] += __shfl_xor_sync(0xffffffffu, acc[r][o], off);
                acc[r][o] += __ldg(a.b_out + o);
            }
        // every lane holds every output now; lane j picks its own s and t through shared memory (a select over the
        // register array would put the array in local memory)
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int r = 0; r < HEAD_ROWS; ++r)
#pragma unroll
                for (int o = 0; o < NOUT; ++o) red[warp][r][o] = acc[r][o];
        }
        __syncwarp();
        const int i = lane - a.upd_lo;
        const bool upd = i >= 0 && i < a.upd_len;
        float sr[HEAD_ROWS], t[HEAD_ROWS];
#pragma unroll
        for (int r = 0; r < HEAD_ROWS; ++r) {
            sr[r] = upd ? red[warp][r][i] : 0.f;
            t[r] = upd ? red[warp][r][i + a.upd_len] : 0.f;
        }
#pragma unroll
        for (int r = 0; r < HEAD_ROWS; ++r) {
            const int64_t row = row0 + r;
            const bool valid = row < a.n;
            float v = valid && lane < e.width ? a.state_in[row * MAXW + lane] : 0.f;
            float sc = 0.f;
            if (upd) {
                const float s = a.clamp * ATAN_SCALE * atanf(sr[r] / a.clamp);
                v = e.reverse ? (v - t[r]) * expf(-s) : fmaf(v, expf(s), t[r]);
                sc = s;
                if (a.save_s && valid) a.save_s[row * MAXW + lane] = sr[r];
            }
            if (a.logdet) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, off);
                if (lane == 0 && valid) a.logdet[row] += sc;
            }
            emit(v, row, valid, e, lane);
        }
    }
}

using EncodeFn = PFN_cuTensorMapEncodeTiled_v12000;

static int encode_fn(EncodeFn* fn) {
    static std::atomic<EncodeFn> cached{nullptr};
    EncodeFn f = cached.load(std::memory_order_relaxed);
    if (!f) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t err = cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q);
        if (err != cudaSuccess || q != cudaDriverEntryPointSuccess || !p)
            return fail(CPPFLOW_E_CUDA, "cppflow_flow_run: cuTensorMapEncodeTiled is not available from the CUDA driver");
        f = reinterpret_cast<EncodeFn>(p);
        cached.store(f, std::memory_order_relaxed);
    }
    *fn = f;
    return CPPFLOW_OK;
}

// bf16 [rows, cols] row-major, read in [box_rows, 64] boxes with the 128-byte swizzle the MMA descriptors expect
static int make_map(EncodeFn enc, CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {cols * 2};
    const cuuint32_t box[2] = {(cuuint32_t)BK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(CPPFLOW_E_CUDA, "cppflow_flow_run: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return CPPFLOW_OK;
}

// A [m_rows, K] . W[n_cols, K]^T through the epilogue EPI; m_rows >= 1, K % 64 == 0, n_cols % BN == 0
template <int BN, int EPI>
static int launch_gemm_epi(EncodeFn enc, const void* a, int64_t m_rows, const void* w, int n_cols, int K,
                           const EpiArgs& ep, cudaStream_t st) {
    static SmemGrant granted;
    int rc = ensure_dynamic_smem(flow_gemm_kernel<BN, EPI>, GemmCfg<BN>::SMEM, granted);
    if (rc) return rc;
    CUtensorMap ma, mw;
    if ((rc = make_map(enc, &ma, a, (uint64_t)m_rows, (uint64_t)K, BM))) return rc;
    if ((rc = make_map(enc, &mw, w, (uint64_t)n_cols, (uint64_t)K, BN))) return rc;
    dim3 grid((unsigned)((m_rows + BM - 1) / BM), (unsigned)(n_cols / BN));
    flow_gemm_kernel<BN, EPI><<<grid, 128, GemmCfg<BN>::SMEM, st>>>(ma, mw, ep, (int)m_rows, K / BK);
    return CPPFLOW_OK;
}

template <int BN>
static int launch_gemm(EncodeFn enc, const void* a, const void* w, const float* bias, __nv_bfloat16* out, int64_t n,
                       int K, int H, cudaStream_t st) {
    EpiArgs ep{};
    ep.bias = bias;
    ep.out = out;
    ep.ldo = H;
    return launch_gemm_epi<BN, EPI_FWD>(enc, a, n, w, H, K, ep, st);
}

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

static int validate(const cppflow_flow_desc* d, int64_t n) {
    if (!d) return fail(CPPFLOW_E_INVALID, "cppflow_flow: desc is NULL");
    int ndof = 0;
    switch (d->robot) {
        case ROBOT_FETCH: ndof = Fetch::NDOF; break;
        case ROBOT_FETCH_ARM: ndof = FetchArm::NDOF; break;
        case ROBOT_PANDA: ndof = Panda::NDOF; break;
        default: return fail(CPPFLOW_E_INVALID, "cppflow_flow: unknown robot id %d", d->robot);
    }
    if (d->ndof != ndof) return fail(CPPFLOW_E_INVALID, "cppflow_flow: ndof %d is not the robot's (%d)", d->ndof, ndof);
    if (d->width < d->ndof || d->width > MAXW)
        return fail(CPPFLOW_E_INVALID, "cppflow_flow: width %d outside [ndof = %d, %d]", d->width, d->ndof, MAXW);
    if (d->dim_cond != 7 && d->dim_cond != 8)
        return fail(CPPFLOW_E_INVALID, "cppflow_flow: dim_cond %d is not 7 or 8", d->dim_cond);
    if (d->coeff_fn_config < 1 || d->coeff_fn_config > 4)
        return fail(CPPFLOW_E_INVALID, "cppflow_flow: coeff_fn_config %d outside [1, 4]", d->coeff_fn_config);
    const int H = d->coeff_fn_internal_size;
    if (H < 128 || H > 1024 || H % 128 != 0)
        return fail(CPPFLOW_E_INVALID, "cppflow_flow: coeff_fn_internal_size %d is not a multiple of 128 in [128, 1024]", H);
    if (d->nb_nodes < 1) return fail(CPPFLOW_E_INVALID, "cppflow_flow: nb_nodes %d < 1", d->nb_nodes);
    if (!(d->rnvp_clamp > 0.f)) return fail(CPPFLOW_E_INVALID, "cppflow_flow: rnvp_clamp must be > 0");
    if (n < 1 || n > INT32_MAX - BM) return fail(CPPFLOW_E_INVALID, "cppflow_flow: n = %lld outside [1, 2^31 - 129]", (long long)n);
    return CPPFLOW_OK;
}

static size_t workspace_bytes(const cppflow_flow_desc* d, int64_t n) {
    const size_t L = d->coeff_fn_config;
    return align256((size_t)n * MAXW * 4) + align256((size_t)n * KIN * 2) +
           (L < 2 ? L : 2) * align256((size_t)n * d->coeff_fn_internal_size * 2);
}

template <class M>
static void fill_limits(Emit& e) {
    for (int j = 0; j < CPPFLOW_MAX_DOF; ++j) {
        e.lower[j] = j < M::NDOF ? dof_lower<M>(j) : 0.f;
        e.upper[j] = j < M::NDOF ? dof_upper<M>(j) : 0.f;
    }
}


}  // namespace flow
}  // namespace cppflow
