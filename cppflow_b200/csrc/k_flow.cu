// IKFlow's conditional GLOW network (oracle/ikflow.py), forward and reverse, for n rows.
//
// One half-coupling (a subnet evaluated on [half | cond], then the affine update of the other half) is
//   L launches of flow_gemm_kernel: the first Linear (K = 64, the input zero-padded) and the L - 1 hidden Linears, on
//     tcgen05 (BF16 operands loaded by TMA, FP32 accumulator in tensor memory, bias + LeakyReLU + BF16 epilogue);
//   one launch of flow_head_kernel: the last Linear (FP32 weights, at most 16 outputs), the clamped scale, the affine
//     update of the state, the permutation between coupling blocks and the BF16 input of the next subnet (or, after
//     the last half-coupling, the output with the joint scale and the optional clamp).
// flow_prep_kernel turns the input into the first state.  Each output row of every kernel depends only on the same
// input row and the weights, through the same sequence of operations for every n: results are bit-identical whatever
// n is and whichever rows share a tile.
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

// out[m, n0 .. n0 + BN) = bf16(leaky_relu(A[m, :] . W[n, :] + bias[n])) for the 128 rows m of the tile.
// A [n_rows, K] and W [H, K] are bf16, K-major, read through the tensor maps; rows >= n_rows read as 0 and are not
// stored.  Warp 0 lane 0 issues the TMA loads, warp 1 lane 0 the MMAs, then all four warps drain tensor memory.
template <int BN>
__global__ void __launch_bounds__(128, 1) flow_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a,
                                                           const __grid_constant__ CUtensorMap tmap_w,
                                                           const float* __restrict__ bias, __nv_bfloat16* __restrict__ out,
                                                           int n_rows, int ldo, int k_blocks) {
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
            const float4* b4 = reinterpret_cast<const float4*>(bias + n0 + c * 32);
            uint4 pk[4];
            uint32_t* pw = reinterpret_cast<uint32_t*>(pk);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 b = __ldg(b4 + q);
                float v0 = __uint_as_float(r[4 * q + 0]) + b.x, v1 = __uint_as_float(r[4 * q + 1]) + b.y;
                float v2 = __uint_as_float(r[4 * q + 2]) + b.z, v3 = __uint_as_float(r[4 * q + 3]) + b.w;
                v0 = v0 > 0.f ? v0 : LEAKY * v0;
                v1 = v1 > 0.f ? v1 : LEAKY * v1;
                v2 = v2 > 0.f ? v2 : LEAKY * v2;
                v3 = v3 > 0.f ? v3 : LEAKY * v3;
                __nv_bfloat162 lo = __floats2bfloat162_rn(v0, v1), hi = __floats2bfloat162_rn(v2, v3);
                pw[2 * q] = *reinterpret_cast<uint32_t*>(&lo);
                pw[2 * q + 1] = *reinterpret_cast<uint32_t*>(&hi);
            }
            uint4* dst = reinterpret_cast<uint4*>(out + (size_t)row * ldo + n0 + c * 32);
#pragma unroll
            for (int q = 0; q < 4; ++q) dst[q] = pk[q];
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
//   otherwise: state[row] = v', u[row] = bf16([v'[next_lo .. next_lo + next_len) | cond[row % n_cond] | 0 ...]).
struct Emit {
    int width, ndof;
    const int32_t* gather;
    int next_lo, next_len;
    float* state;
    __nv_bfloat16* u;
    const float* cond;
    int64_t n_cond;
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
    const float* c = e.cond + (row % e.n_cond) * 7;
    auto elem = [&](int q, float h) {
        if (q < e.next_len) return h;
        const int k = q - e.next_len;
        return k < 7 ? __ldg(c + k) : 0.f;  // the softflow scale (column 7 when dim_cond = 8) is 0
    };
    reinterpret_cast<__nv_bfloat162*>(e.u + row * KIN)[lane] = __floats2bfloat162_rn(elem(q0, h0), elem(q1, h1));
}

__global__ void __launch_bounds__(256) flow_prep_kernel(const float* __restrict__ in, int64_t n, Emit e) {
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
    const __nv_bfloat16* hidden;  // [n, H]
    const float* w_out;           // [16, H]
    const float* b_out;           // [16]
    int H;
    int upd_lo, upd_len;  // the half this step updates: s = outputs [0, upd_len), t = [upd_len, 2 upd_len)
    float clamp;
    int64_t n;
};

constexpr int HEAD_ROWS = 4;  // rows per warp and pass: each shared-memory read of the last Linear serves 4 rows

// Last Linear + coupling update + Emit.  The last Linear's weights are staged in shared memory as [16][2][H / 8]
// float4 so that lane l's two float4 of columns 8 q .. 8 q + 7 are consecutive across the warp.
__global__ void __launch_bounds__(256) flow_head_kernel(Head a, Emit e) {
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
            float v = valid && lane < e.width ? e.state[row * MAXW + lane] : 0.f;
            if (upd) {
                const float s = a.clamp * ATAN_SCALE * atanf(sr[r] / a.clamp);
                v = e.reverse ? (v - t[r]) * expf(-s) : fmaf(v, expf(s), t[r]);
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

template <int BN>
static int launch_gemm(EncodeFn enc, const void* a, const void* w, const float* bias, __nv_bfloat16* out, int64_t n,
                       int K, int H, cudaStream_t st) {
    static SmemGrant granted;
    int rc = ensure_dynamic_smem(flow_gemm_kernel<BN>, GemmCfg<BN>::SMEM, granted);
    if (rc) return rc;
    CUtensorMap ma, mw;
    if ((rc = make_map(enc, &ma, a, (uint64_t)n, (uint64_t)K, BM))) return rc;
    if ((rc = make_map(enc, &mw, w, (uint64_t)H, (uint64_t)K, BN))) return rc;
    dim3 grid((unsigned)((n + BM - 1) / BM), (unsigned)(H / BN));
    flow_gemm_kernel<BN><<<grid, 128, GemmCfg<BN>::SMEM, st>>>(ma, mw, bias, out, (int)n, H, K / BK);
    return CPPFLOW_OK;
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

using namespace cppflow;
using namespace cppflow::flow;

extern "C" size_t cppflow_flow_workspace_bytes(const cppflow_flow_desc* desc, int64_t n) {
    if (validate(desc, n)) return 0;
    return workspace_bytes(desc, n);
}

extern "C" int cppflow_flow_run(const cppflow_flow_desc* d, const float* d_in, const float* d_cond, int64_t n,
                                int64_t n_cond, int flags, void* d_workspace, size_t ws_bytes, float* d_out, void* stream) {
    int rc = validate(d, n);
    if (rc) return rc;
    CPPFLOW_CHECK_ARG(d_in && d_cond && d_out, "d_in / d_cond / d_out");
    CPPFLOW_CHECK_ARG(n_cond >= 1, "n_cond < 1");
    CPPFLOW_CHECK_ARG((flags & ~(CPPFLOW_FLOW_REVERSE | CPPFLOW_FLOW_CLAMP)) == 0, "unknown flag bits");
    CPPFLOW_CHECK_ARG(!(flags & CPPFLOW_FLOW_CLAMP) || (flags & CPPFLOW_FLOW_REVERSE), "CPPFLOW_FLOW_CLAMP needs CPPFLOW_FLOW_REVERSE");
    CPPFLOW_CHECK_ARG(d->d_w_in && d->d_b_hidden && d->d_w_out && d->d_b_out && d->d_scale && d->d_perm && d->d_perm_inv,
                      "null weight table");
    CPPFLOW_CHECK_ARG(d->coeff_fn_config == 1 || d->d_w_hidden, "d_w_hidden is NULL with coeff_fn_config > 1");
    const size_t need = workspace_bytes(d, n);
    if (!d_workspace || ws_bytes < need)
        return fail(CPPFLOW_E_WORKSPACE, "cppflow_flow_run: workspace %zu bytes < %zu", ws_bytes, need);
    EncodeFn enc;
    if ((rc = encode_fn(&enc))) return rc;
    static SmemGrant head_grant;
    const int H = d->coeff_fn_internal_size, L = d->coeff_fn_config, W = d->width, nb = d->nb_nodes;
    const size_t head_smem = (size_t)NOUT * H * 4;
    if ((rc = ensure_dynamic_smem(flow_head_kernel, head_smem, head_grant))) return rc;

    uint8_t* ws = static_cast<uint8_t*>(d_workspace);
    float* state = reinterpret_cast<float*>(ws);
    ws += align256((size_t)n * MAXW * 4);
    __nv_bfloat16* u = reinterpret_cast<__nv_bfloat16*>(ws);
    ws += align256((size_t)n * KIN * 2);
    __nv_bfloat16* hid[2] = {reinterpret_cast<__nv_bfloat16*>(ws),
                             reinterpret_cast<__nv_bfloat16*>(ws + align256((size_t)n * H * 2))};

    const bool rev = flags & CPPFLOW_FLOW_REVERSE;
    Emit e;
    std::memset(&e, 0, sizeof(e));
    e.width = W;
    e.ndof = d->ndof;
    e.state = state;
    e.u = u;
    e.cond = d_cond;
    e.n_cond = n_cond;
    e.scale = d->d_scale;
    e.reverse = rev;
    e.clamp = (flags & CPPFLOW_FLOW_CLAMP) ? 1 : 0;
    CPPFLOW_DISPATCH_ROBOT(d->robot, fill_limits<M>(e));

    // half-couplings in execution order: s = 0 (subnet1) reads half 1 and updates half 2, s = 1 the other way round
    const int len1 = W / 2, len2 = W - W / 2;
    const int in_lo[2] = {0, len1}, in_len[2] = {len1, len2};
    const int upd_lo[2] = {len1, 0}, upd_len[2] = {len2, len1};
    const int n_steps = 2 * nb;
    auto step_block = [&](int i) { return rev ? nb - 1 - i / 2 : i / 2; };
    auto step_subnet = [&](int i) { return rev ? i % 2 : 1 - i % 2; };

    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned row_warps = (unsigned)((n + 7) / 8);

    e.gather = rev ? nullptr : d->d_perm;  // forward: x M, then block 0's permutation
    e.next_lo = in_lo[step_subnet(0)];
    e.next_len = in_len[step_subnet(0)];
    flow_prep_kernel<<<row_warps, 256, 0, st>>>(d_in, n, e);
    CPPFLOW_CHECK_LAUNCH();

    const __nv_bfloat16* w_in = static_cast<const __nv_bfloat16*>(d->d_w_in);
    const __nv_bfloat16* w_hid = static_cast<const __nv_bfloat16*>(d->d_w_hidden);
    for (int i = 0; i < n_steps; ++i) {
        const int b = step_block(i), s = step_subnet(i), bs = 2 * b + s;
        for (int l = 0; l < L; ++l) {
            const void* a = l == 0 ? (const void*)u : (const void*)hid[(l - 1) & 1];
            const void* w = l == 0 ? (const void*)(w_in + (size_t)bs * H * KIN)
                                   : (const void*)(w_hid + ((size_t)bs * (L - 1) + (l - 1)) * H * H);
            const float* bias = d->d_b_hidden + ((size_t)bs * L + l) * H;
            const int K = l == 0 ? KIN : H;
            rc = H % 256 == 0 ? launch_gemm<256>(enc, a, w, bias, hid[l & 1], n, K, H, st)
                              : launch_gemm<128>(enc, a, w, bias, hid[l & 1], n, K, H, st);
            if (rc) return rc;
            CPPFLOW_CHECK_LAUNCH();
        }
        Head h;
        h.hidden = hid[(L - 1) & 1];
        h.w_out = d->d_w_out + (size_t)bs * NOUT * H;
        h.b_out = d->d_b_out + (size_t)bs * NOUT;
        h.H = H;
        h.upd_lo = upd_lo[s];
        h.upd_len = upd_len[s];
        h.clamp = d->rnvp_clamp;
        h.n = n;
        const bool last = i == n_steps - 1, block_end = i % 2 == 1;
        e.gather = nullptr;
        e.out = nullptr;
        if (block_end) e.gather = rev ? d->d_perm_inv + (size_t)b * W : (last ? nullptr : d->d_perm + (size_t)(b + 1) * W);
        if (last) {
            e.out = d_out;
        } else {
            e.next_lo = in_lo[step_subnet(i + 1)];
            e.next_len = in_len[step_subnet(i + 1)];
        }
        const int64_t groups = (n + 8 * HEAD_ROWS - 1) / (8 * HEAD_ROWS);
        const unsigned grid = (unsigned)std::min<int64_t>(groups, (int64_t)sms * 2);
        flow_head_kernel<<<grid, 256, head_smem, st>>>(h, e);
        CPPFLOW_CHECK_LAUNCH();
    }
    return CPPFLOW_OK;
}
