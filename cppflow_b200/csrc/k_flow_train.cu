// One training step of IKFlow's conditional GLOW network (oracle/ikflow_train.py: forward_with_logdet, nll): forward
// with saved activations, the negative log-likelihood, the backward pass and Adam, for a batch of n rows (n % 128 == 0).
//
// Forward: the launches of cppflow_flow_run's forward pass (flow_prep_kernel, flow_gemm_kernel, flow_head_kernel; z is
// bit-identical), except that every state, subnet input and hidden activation gets a buffer of its own, the GEMMs
// also write a transposed [features, n] copy of their output (EPI_FWD_T), the prep and head kernels one of the subnet
// input, and the heads save the raw s and add the clamped s of each row to its log-determinant.
// Backward, per half-coupling from the last: flow_head_bwd_kernel takes the gradient of the state after the step to
// the gradient of the state before it and dA, the gradient of the last Linear's outputs.  Everything a subnet needs
// then runs on the tensor cores through flow_gemm_kernel: dW = dY^T . X (K = n, from the transposed copies),
// dX = dY . W (from transposed BF16 weight tables) with LeakyReLU's derivative in the epilogue (EPI_BWD), and the
// gradient of the subnet input (EPI_F32), which the head backward of the previous step adds to the half it was built
// from.  Bias gradients are column sums of the transposed BF16 gradients.
// Optimizer: one pass checks every gradient for non-finite values, a one-warp kernel decides whether the step is
// skipped and advances the counters, and flow_adam_kernel updates the FP32 master weights and moments and rewrites the
// BF16 tables and their transposed copies.  No kernel uses atomics and every sum has a fixed order: two runs are
// bit-identical.
// Data-parallel training splits a step into its parts: sharded batch draws (cppflow_flow_train_batch_rows), shard
// gradients (NO_UPDATE), their balanced-tree sum (flow_tree_reduce_kernel, on one GPU and on each rank's slice after
// the exchange) and the optimizer tail on the reduced gradient (cppflow_flow_train_apply).
#include "flow.cuh"
#include "rng.cuh"

namespace cppflow {
namespace flow {

constexpr int FLAG_BLOCKS = 256;

// offsets (floats) of the packed tables in the FP32 parameter vector
struct ParamLayout {
    size_t w_in, w_hidden, b_hidden, w_out, b_out, total;
};

static ParamLayout param_layout(const cppflow_flow_desc* d) {
    const size_t nb2 = 2 * (size_t)d->nb_nodes, H = d->coeff_fn_internal_size, L = d->coeff_fn_config;
    ParamLayout p;
    p.w_in = 0;
    p.w_hidden = p.w_in + nb2 * H * KIN;
    p.b_hidden = p.w_hidden + nb2 * (L - 1) * H * H;
    p.w_out = p.b_hidden + nb2 * L * H;
    p.b_out = p.w_out + nb2 * NOUT * H;
    p.total = p.b_out + nb2 * NOUT;
    return p;
}

struct TrainWs {
    float* state;          // [S][n][MAXW]: the state entering half-coupling i (S = 2 nb_nodes)
    float* save_s;         // [S][n][MAXW]
    __nv_bfloat16* u;      // [S][n][KIN]
    __nv_bfloat16* u_t;    // [S][KIN][n]
    __nv_bfloat16* h;      // [S][L][n][H]
    __nv_bfloat16* h_t;    // [S][L][H][n]
    float* logdet;         // [n]
    float* z;              // [n][width]
    float* nll;            // [n]
    float* ds[2];          // [n][MAXW]
    __nv_bfloat16* da;     // [n][KIN]
    __nv_bfloat16* da_t;   // [NOUT][n]
    float* da_t32;         // [NOUT][n]
    __nv_bfloat16* dh[2];  // [n][H]
    __nv_bfloat16* dh_t[2];
    float* du;             // [n][KIN]
    float* grad;           // [P]
    int* flags;            // [FLAG_BLOCKS]
    int* skip;
};

// Lays the workspace out from `base` (nullptr: sizes only); returns the bytes used.
static size_t train_ws(const cppflow_flow_desc* d, int64_t n, uint8_t* base, TrainWs* w) {
    const size_t S = 2 * (size_t)d->nb_nodes, L = d->coeff_fn_config, H = d->coeff_fn_internal_size;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        uint8_t* p = base ? base + off : nullptr;
        off += align256(bytes);
        return p;
    };
    TrainWs t;
    t.state = reinterpret_cast<float*>(take(S * n * MAXW * 4));
    t.save_s = reinterpret_cast<float*>(take(S * n * MAXW * 4));
    t.u = reinterpret_cast<__nv_bfloat16*>(take(S * n * KIN * 2));
    t.u_t = reinterpret_cast<__nv_bfloat16*>(take(S * n * KIN * 2));
    t.h = reinterpret_cast<__nv_bfloat16*>(take(S * L * n * H * 2));
    t.h_t = reinterpret_cast<__nv_bfloat16*>(take(S * L * n * H * 2));
    t.logdet = reinterpret_cast<float*>(take((size_t)n * 4));
    t.z = reinterpret_cast<float*>(take((size_t)n * d->width * 4));
    t.nll = reinterpret_cast<float*>(take((size_t)n * 4));
    for (int k = 0; k < 2; ++k) t.ds[k] = reinterpret_cast<float*>(take((size_t)n * MAXW * 4));
    t.da = reinterpret_cast<__nv_bfloat16*>(take((size_t)n * KIN * 2));
    t.da_t = reinterpret_cast<__nv_bfloat16*>(take((size_t)NOUT * n * 2));
    t.da_t32 = reinterpret_cast<float*>(take((size_t)NOUT * n * 4));
    for (int k = 0; k < 2; ++k) {
        t.dh[k] = reinterpret_cast<__nv_bfloat16*>(take((size_t)n * H * 2));
        t.dh_t[k] = reinterpret_cast<__nv_bfloat16*>(take((size_t)n * H * 2));
    }
    t.du = reinterpret_cast<float*>(take((size_t)n * KIN * 4));
    t.grad = reinterpret_cast<float*>(take(param_layout(d).total * 4));
    t.flags = reinterpret_cast<int*>(take(FLAG_BLOCKS * 4));
    t.skip = reinterpret_cast<int*>(take(4));
    if (w) *w = t;
    return off;
}

static int validate_train(const cppflow_flow_train_desc* t, int64_t n) {
    if (!t) return fail(CPPFLOW_E_INVALID, "cppflow_flow_train: desc is NULL");
    int rc = validate(&t->flow, n);
    if (rc) return rc;
    const cppflow_flow_desc* d = &t->flow;
    if (n % BM != 0) return fail(CPPFLOW_E_INVALID, "cppflow_flow_train: batch %lld is not a multiple of 128", (long long)n);
    if (d->width > d->ndof && d->dim_cond != 8)
        return fail(CPPFLOW_E_INVALID,
                    "cppflow_flow_train: width %d > ndof %d needs softflow (dim_cond 8): the padding's density is degenerate "
                    "without it", d->width, d->ndof);
    if (!(t->lr >= 0.0) || !(t->beta1 >= 0.0 && t->beta1 < 1.0) || !(t->beta2 >= 0.0 && t->beta2 < 1.0) ||
        !(t->eps > 0.0) || !(t->weight_decay >= 0.0) || !(t->lr_decay > 0.0) || t->lr_decay_steps < 1)
        return fail(CPPFLOW_E_INVALID, "cppflow_flow_train: hyperparameter out of range (lr >= 0, 0 <= beta < 1, eps > 0, "
                                       "weight_decay >= 0, lr_decay > 0, lr_decay_steps >= 1)");
    return CPPFLOW_OK;
}

// -------------------------------------------------------------------------------------------------- loss kernels

// nll[row] = 0.5 |z|^2 - (logdet[row] + sum_j log scale[j]); ds[row] = z / n, zero-padded to MAXW
__global__ void __launch_bounds__(256) flow_nll_kernel(const float* __restrict__ z, const float* __restrict__ logdet,
                                                       const float* __restrict__ scale, int width, int64_t n,
                                                       float* __restrict__ nll, float* __restrict__ ds) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const float inv_n = 1.f / (float)n;
    float sq = 0.f, ldm = 0.f;
    for (int j = 0; j < MAXW; ++j) {
        float g = 0.f;
        if (j < width) {
            const float v = z[row * width + j];
            sq = fmaf(v, v, sq);
            ldm += logf(__ldg(scale + j));
            g = v * inv_n;
        }
        ds[row * MAXW + j] = g;
    }
    nll[row] = 0.5f * sq - (logdet[row] + ldm);
}

// *loss = mean(nll): one CTA, thread t sums rows t, t + 1024, ... in order, then a fixed tree
__global__ void __launch_bounds__(1024) flow_loss_kernel(const float* __restrict__ nll, int64_t n, float* __restrict__ loss) {
    __shared__ float part[1024];
    float acc = 0.f;
    for (int64_t r = threadIdx.x; r < n; r += 1024) acc += nll[r];
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) part[threadIdx.x] += part[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) *loss = part[0] / (float)n;
}

// ------------------------------------------------------------------------------------------------ head backward

struct HeadBwd {
    const float* ds_next;  // [n, MAXW]: gradient of the state after this step (of z after the last step)
    const float* du_next;  // [n, KIN]: gradient of the next step's subnet input, NULL after the last step
    int next_lo, next_len;
    const int32_t* ginv;   // inverse of the permutation applied after this step, or NULL
    const float* state;    // [n, MAXW]: the state before this step
    const float* save_s;   // [n, MAXW]: raw s of the updated lanes
    int upd_lo, upd_len, width;
    float clamp, inv_n;
    float* ds;             // [n, MAXW]: gradient of the state before this step (without its subnet's input gradient)
    __nv_bfloat16* da;     // [n, KIN]: [ds | dt | 0 ...]
    __nv_bfloat16* da_t;   // [NOUT, n]
    float* da_t32;         // [NOUT, n]: dA in FP32, for the bias gradient of the last Linear
    int64_t n;
};

// One warp per row, lane j holds element j of the state.  The update of lane j of the updated half is
// y = x exp(sc) + t with sc = clamp 0.636 atan(s / clamp), and the loss holds -sc / n for it.
__global__ void __launch_bounds__(256) flow_head_bwd_kernel(HeadBwd a) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= a.n) return;
    float d = lane < MAXW ? a.ds_next[row * MAXW + lane] : 0.f;
    if (a.du_next) {
        const int q = lane - a.next_lo;
        if (q >= 0 && q < a.next_len) d += a.du_next[row * KIN + q];
    }
    if (a.ginv) d = __shfl_sync(0xffffffffu, d, lane < a.width ? __ldg(a.ginv + lane) : lane);
    const int i = lane - a.upd_lo;
    const bool upd = i >= 0 && i < a.upd_len;
    float dx = d, ds = 0.f, dt = 0.f;
    if (upd) {
        const float s = a.save_s[row * MAXW + lane], x = a.state[row * MAXW + lane];
        const float r = s / a.clamp;
        const float e = expf(a.clamp * ATAN_SCALE * atanf(r));
        dx = d * e;
        dt = d;
        ds = (d * x * e - a.inv_n) * (ATAN_SCALE / fmaf(r, r, 1.f));
    }
    if (lane < MAXW) a.ds[row * MAXW + lane] = lane < a.width ? dx : 0.f;
    auto pick = [&](int q) {
        const float vs = __shfl_sync(0xffffffffu, ds, min(a.upd_lo + q, 31));
        const float vt = __shfl_sync(0xffffffffu, dt, min(max(a.upd_lo + q - a.upd_len, 0), 31));
        return q < a.upd_len ? vs : (q < 2 * a.upd_len ? vt : 0.f);
    };
    const float g0 = pick(2 * lane), g1 = pick(2 * lane + 1);
    const __nv_bfloat162 g = __floats2bfloat162_rn(g0, g1);
    reinterpret_cast<__nv_bfloat162*>(a.da + row * KIN)[lane] = g;
    if (2 * lane < NOUT) {
        a.da_t[(2 * lane) * a.n + row] = g.x;
        a.da_t[(2 * lane + 1) * a.n + row] = g.y;
        a.da_t32[(2 * lane) * a.n + row] = g0;
        a.da_t32[(2 * lane + 1) * a.n + row] = g1;
    }
}

// out[r] = sum over the n columns of row r of t [rows, n] (bf16 or fp32): one warp per row, fixed order
template <class T>
__global__ void __launch_bounds__(256) flow_colsum_kernel(const T* __restrict__ t, int64_t n, int rows,
                                                          float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= rows) return;
    const uint4* p = reinterpret_cast<const uint4*>(t + (size_t)r * n);
    constexpr int PER = 16 / sizeof(T);
    float acc = 0.f;
    for (int64_t k = lane; k < n / PER; k += 32) {
        const uint4 raw = __ldg(p + k);
        if constexpr (sizeof(T) == 2) {
            const __nv_bfloat162* b = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = __bfloat1622float2(b[j]);
                acc += f.x;
                acc += f.y;
            }
        } else {
            acc += __uint_as_float(raw.x);
            acc += __uint_as_float(raw.y);
            acc += __uint_as_float(raw.z);
            acc += __uint_as_float(raw.w);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) out[r] = acc;
}

// ---------------------------------------------------------------------------------------------------- optimizer

__global__ void __launch_bounds__(256) flow_finite_kernel(const float* __restrict__ g, size_t P, int* __restrict__ flags) {
    int bad = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (size_t)gridDim.x * blockDim.x)
        bad |= !isfinite(g[i]);
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) flags[blockIdx.x] = bad;
}

// counters: [0] updates applied (Adam's t), [1] steps skipped for a non-finite gradient, [2] steps taken
__global__ void flow_step_decide_kernel(const int* __restrict__ flags, int* __restrict__ skip, int64_t* __restrict__ counters) {
    int bad = 0;
    for (int k = threadIdx.x; k < FLAG_BLOCKS; k += 32) bad |= flags[k];
    bad = __any_sync(0xffffffffu, bad);
    if (threadIdx.x == 0) {
        *skip = bad;
        counters[bad ? 1 : 0] += 1;
        counters[2] += 1;
    }
}

struct AdamArgs {
    ParamLayout p;
    int H, L;
    const float* grad;
    float* w;
    float* m;
    float* v;
    __nv_bfloat16 *w_in, *w_hidden, *w_in_t, *w_hidden_t, *w_out_t;
    const int* skip;
    const int64_t* counters;
    double lr, beta1, beta2, eps, weight_decay, lr_decay;
    int64_t lr_decay_steps;
};

// torch.optim.Adam (weight decay added to the gradient), then the BF16 tables of the updated weights
__global__ void __launch_bounds__(256) flow_adam_kernel(AdamArgs a) {
    if (*a.skip) return;
    const int64_t t = a.counters[0], taken = a.counters[2] - 1;
    const double lr = a.lr * pow(a.lr_decay, (double)(taken / a.lr_decay_steps));
    const float step_size = (float)(lr / (1.0 - pow(a.beta1, (double)t)));
    const float bc2_sqrt = (float)sqrt(1.0 - pow(a.beta2, (double)t));
    const float wd = (float)a.weight_decay, one_b1 = (float)(1.0 - a.beta1), b2 = (float)a.beta2;
    const float one_b2 = (float)(1.0 - a.beta2), eps = (float)a.eps;
    const size_t H = a.H, HK = H * KIN, HH = H * H;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.p.total; i += (size_t)gridDim.x * blockDim.x) {
        float w = a.w[i], g = a.grad[i];
        if (wd != 0.f) g = __fadd_rn(g, __fmul_rn(wd, w));
        float m = a.m[i], v = a.v[i];
        m = __fadd_rn(m, __fmul_rn(one_b1, __fsub_rn(g, m)));
        v = __fadd_rn(__fmul_rn(v, b2), __fmul_rn(__fmul_rn(one_b2, g), g));
        const float denom = __fadd_rn(__fdiv_rn(sqrtf(v), bc2_sqrt), eps);
        w = __fsub_rn(w, __fmul_rn(step_size, __fdiv_rn(m, denom)));
        a.w[i] = w;
        a.m[i] = m;
        a.v[i] = v;
        const __nv_bfloat16 wb = __float2bfloat16_rn(w);
        if (i < a.p.w_hidden) {
            const size_t bs = i / HK, o = (i / KIN) % H, c = i % KIN;
            a.w_in[i] = wb;
            a.w_in_t[bs * HK + c * H + o] = wb;
        } else if (i < a.p.b_hidden) {
            const size_t k = i - a.p.w_hidden, li = k / HH, o = (k / H) % H, c = k % H;
            a.w_hidden[k] = wb;
            a.w_hidden_t[li * HH + c * H + o] = wb;
        } else if (i >= a.p.w_out && i < a.p.b_out) {
            const size_t k = i - a.p.w_out, bs = k / (NOUT * H), o = (k / H) % NOUT, c = k % H;
            a.w_out_t[bs * HK + c * KIN + o] = wb;
        }
    }
}

// ------------------------------------------------------------------------------------------ gradient reduction

// out[k] = scale * T(in[0 * stride + k], ..., in[(N - 1) * stride + k]) for k < len, T the balanced pairwise tree in
// slice order ((s0 + s1) + (s2 + s3)) + ...; four floats per thread.  out may be slice 0 (each thread reads its
// elements of every slice before it writes them).
template <int N>
__global__ void __launch_bounds__(256) flow_tree_reduce_kernel(const float* in, int64_t len4, int64_t stride4, float scale,
                                                               float* out) {
    const float4* src = reinterpret_cast<const float4*>(in);
    float4* dst = reinterpret_cast<float4*>(out);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < len4; k += (int64_t)gridDim.x * blockDim.x) {
        float4 v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = src[i * stride4 + k];
#pragma unroll
        for (int w = 1; w < N; w *= 2)
#pragma unroll
            for (int i = 0; i < N; i += 2 * w) {
                v[i].x = __fadd_rn(v[i].x, v[i + w].x);
                v[i].y = __fadd_rn(v[i].y, v[i + w].y);
                v[i].z = __fadd_rn(v[i].z, v[i + w].z);
                v[i].w = __fadd_rn(v[i].w, v[i + w].w);
            }
        dst[k] = make_float4(__fmul_rn(v[0].x, scale), __fmul_rn(v[0].y, scale), __fmul_rn(v[0].z, scale),
                             __fmul_rn(v[0].w, scale));
    }
}

// --------------------------------------------------------------------------------------------- batch sampling

// One thread per batch row; the random numbers of (seed, step, first_row + row) do not depend on the batch size, so a
// batch drawn in shards from first_row = 0, B, 2B, ... is the batch drawn at once.
__global__ void __launch_bounds__(256) flow_train_batch_kernel(const float* __restrict__ q, const float* __restrict__ poses,
                                                               int64_t n_data, int64_t batch, int64_t first_row, int ndof,
                                                               int width, int dim_cond, uint64_t seed,
                                                               const int64_t* __restrict__ step, float noise_scale,
                                                               float* __restrict__ x, float* __restrict__ cond,
                                                               int64_t* __restrict__ idx_out, float* __restrict__ noise_out) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= batch) return;
    const uint64_t key = mix64(seed ^ mix64((uint64_t)*step)) ^ mix64((uint64_t)(first_row + row) * 0x2545F4914F6CDD1Dull);
    auto draw = [&](int k) { return mix64(key + (uint64_t)k * 0x9E3779B97F4A7C15ull); };
    const int64_t idx = (int64_t)__umul64hi(draw(0), (uint64_t)n_data);
    const bool soft = dim_cond == 8;
    const float c = soft ? u01(draw(1)) : 0.f;
    const bool flip = draw(2) >> 63;
    const float sc = __fmul_rn(noise_scale, c);
    auto put = [&](int j, float eps) {
        eps = soft ? eps : 0.f;
        const float base = j < ndof ? q[idx * ndof + j] : 0.f;
        x[row * width + j] = __fadd_rn(base, __fmul_rn(sc, eps));
        if (noise_out) noise_out[row * (width + 2) + j] = eps;
    };
    for (int j = 0; j < width; j += 2) {  // Box-Muller pairs
        const float r = sqrtf(-2.f * logf(u01(draw(3 + j)))), th = 6.2831853f * u01(draw(4 + j));
        put(j, r * cosf(th));
        if (j + 1 < width) put(j + 1, r * sinf(th));
    }
    for (int k = 0; k < 7; ++k) {
        const float p = poses[idx * 7 + k];
        cond[row * dim_cond + k] = flip && k >= 3 ? -p : p;
    }
    if (soft) cond[row * dim_cond + 7] = c;
    if (noise_out) {
        noise_out[row * (width + 2) + width] = c;
        noise_out[row * (width + 2) + width + 1] = flip ? 1.f : 0.f;
    }
    if (idx_out) idx_out[row] = idx;
}

static int gemm_f32(EncodeFn enc, const void* a, int64_t m_rows, const void* w, int n_cols, int K, float* out, int ldo,
                    cudaStream_t st) {
    EpiArgs ep{};
    ep.out_f = out;
    ep.ldo = ldo;
    if (n_cols == KIN) return launch_gemm_epi<64, EPI_F32>(enc, a, m_rows, w, n_cols, K, ep, st);
    return n_cols % 256 == 0 ? launch_gemm_epi<256, EPI_F32>(enc, a, m_rows, w, n_cols, K, ep, st)
                             : launch_gemm_epi<128, EPI_F32>(enc, a, m_rows, w, n_cols, K, ep, st);
}

template <int EPI>
static int gemm_bf16(EncodeFn enc, const void* a, int64_t m_rows, const void* w, int n_cols, int K, const EpiArgs& ep,
                     cudaStream_t st) {
    return n_cols % 256 == 0 ? launch_gemm_epi<256, EPI>(enc, a, m_rows, w, n_cols, K, ep, st)
                             : launch_gemm_epi<128, EPI>(enc, a, m_rows, w, n_cols, K, ep, st);
}

// The optimizer tail of a step on the gradient grad [P]: finite check into flags, the skip decision and counters,
// Adam and the BF16 table rewrites.
static int apply_update(const cppflow_flow_train_desc* t, const float* grad, int* flags, int* skip, int sms,
                        cudaStream_t st) {
    const cppflow_flow_desc* d = &t->flow;
    const ParamLayout pl = param_layout(d);
    flow_finite_kernel<<<FLAG_BLOCKS, 256, 0, st>>>(grad, pl.total, flags);
    CPPFLOW_CHECK_LAUNCH();
    flow_step_decide_kernel<<<1, 32, 0, st>>>(flags, skip, t->d_counters);
    CPPFLOW_CHECK_LAUNCH();
    AdamArgs a;
    std::memset(&a, 0, sizeof(a));
    a.p = pl;
    a.H = d->coeff_fn_internal_size;
    a.L = d->coeff_fn_config;
    a.grad = grad;
    a.w = t->d_params;
    a.m = t->d_adam_m;
    a.v = t->d_adam_v;
    a.w_in = static_cast<__nv_bfloat16*>(const_cast<void*>(d->d_w_in));
    a.w_hidden = static_cast<__nv_bfloat16*>(const_cast<void*>(d->d_w_hidden));
    a.w_in_t = static_cast<__nv_bfloat16*>(t->d_w_in_t);
    a.w_hidden_t = static_cast<__nv_bfloat16*>(t->d_w_hidden_t);
    a.w_out_t = static_cast<__nv_bfloat16*>(t->d_w_out_t);
    a.skip = skip;
    a.counters = t->d_counters;
    a.lr = t->lr;
    a.beta1 = t->beta1;
    a.beta2 = t->beta2;
    a.eps = t->eps;
    a.weight_decay = t->weight_decay;
    a.lr_decay = t->lr_decay;
    a.lr_decay_steps = t->lr_decay_steps;
    flow_adam_kernel<<<(unsigned)std::min<size_t>(grid_for((int64_t)pl.total, 256), (size_t)sms * 8), 256, 0, st>>>(a);
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

static int sm_count() {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

}  // namespace flow
}  // namespace cppflow

using namespace cppflow;
using namespace cppflow::flow;

extern "C" size_t cppflow_flow_train_workspace_bytes(const cppflow_flow_train_desc* desc, int64_t batch) {
    if (validate_train(desc, batch)) return 0;
    return train_ws(&desc->flow, batch, nullptr, nullptr);
}

extern "C" int cppflow_flow_train_step(const cppflow_flow_train_desc* t, const float* d_x, const float* d_cond, int64_t n,
                                      int flags, void* d_workspace, size_t ws_bytes, float* d_loss, float* d_grad,
                                      void* stream) {
    int rc = validate_train(t, n);
    if (rc) return rc;
    const cppflow_flow_desc* d = &t->flow;
    CPPFLOW_CHECK_ARG(d_x && d_cond && d_loss, "d_x / d_cond / d_loss");
    CPPFLOW_CHECK_ARG((flags & ~CPPFLOW_FLOW_TRAIN_NO_UPDATE) == 0, "unknown flag bits");
    CPPFLOW_CHECK_ARG(d->d_w_in && d->d_b_hidden && d->d_w_out && d->d_b_out && d->d_scale && d->d_perm && d->d_perm_inv,
                      "null weight table");
    CPPFLOW_CHECK_ARG(d->coeff_fn_config == 1 || (d->d_w_hidden && t->d_w_hidden_t), "null hidden-layer table");
    CPPFLOW_CHECK_ARG(t->d_params && t->d_adam_m && t->d_adam_v && t->d_w_in_t && t->d_w_out_t && t->d_counters,
                      "null training table");
    const ParamLayout pl = param_layout(d);
    CPPFLOW_CHECK_ARG(d->d_b_hidden == t->d_params + pl.b_hidden && d->d_w_out == t->d_params + pl.w_out &&
                          d->d_b_out == t->d_params + pl.b_out,
                      "flow.d_b_hidden / d_w_out / d_b_out must point at their segments of d_params");
    const size_t need = train_ws(d, n, nullptr, nullptr);
    if (!d_workspace || ws_bytes < need)
        return fail(CPPFLOW_E_WORKSPACE, "cppflow_flow_train_step: workspace %zu bytes < %zu", ws_bytes, need);
    EncodeFn enc;
    if ((rc = encode_fn(&enc))) return rc;
    static SmemGrant head_grant;
    const int H = d->coeff_fn_internal_size, L = d->coeff_fn_config, W = d->width, nb = d->nb_nodes, S = 2 * nb;
    const size_t head_smem = (size_t)NOUT * H * 4;
    if ((rc = ensure_dynamic_smem(flow_head_kernel, head_smem, head_grant))) return rc;

    TrainWs ws;
    train_ws(d, n, static_cast<uint8_t*>(d_workspace), &ws);
    float* grad = d_grad ? d_grad : ws.grad;
    const size_t SN = (size_t)n * MAXW, UN = (size_t)n * KIN, HN = (size_t)n * H;
    auto state = [&](int i) { return ws.state + i * SN; };
    auto h_of = [&](int i, int l) { return ws.h + ((size_t)i * L + l) * HN; };
    auto ht_of = [&](int i, int l) { return ws.h_t + ((size_t)i * L + l) * HN; };
    const __nv_bfloat16* w_in = static_cast<const __nv_bfloat16*>(d->d_w_in);
    const __nv_bfloat16* w_hid = static_cast<const __nv_bfloat16*>(d->d_w_hidden);
    const __nv_bfloat16* w_in_t = static_cast<const __nv_bfloat16*>(t->d_w_in_t);
    const __nv_bfloat16* w_hid_t = static_cast<const __nv_bfloat16*>(t->d_w_hidden_t);
    const __nv_bfloat16* w_out_t = static_cast<const __nv_bfloat16*>(t->d_w_out_t);

    const int len1 = W / 2, len2 = W - W / 2;
    const int in_lo[2] = {0, len1}, in_len[2] = {len1, len2};
    const int upd_lo[2] = {len1, 0}, upd_len[2] = {len2, len1};
    auto step_subnet = [&](int i) { return 1 - i % 2; };  // forward order, as cppflow_flow_run

    cudaStream_t st = (cudaStream_t)stream;
    const int sms = sm_count();
    const unsigned row_warps = (unsigned)((n + 7) / 8);

    // ---- forward
    cudaMemsetAsync(ws.logdet, 0, (size_t)n * 4, st);
    CPPFLOW_CHECK_LAUNCH();
    Emit e;
    std::memset(&e, 0, sizeof(e));
    e.width = W;
    e.ndof = d->ndof;
    e.cond = d_cond;
    e.n_cond = n;
    e.cond_w = d->dim_cond;
    e.ldt = n;
    e.scale = d->d_scale;
    e.gather = d->d_perm;
    e.state = state(0);
    e.u = ws.u;
    e.u_t = ws.u_t;
    e.next_lo = in_lo[step_subnet(0)];
    e.next_len = in_len[step_subnet(0)];
    flow_prep_kernel<<<row_warps, 256, 0, st>>>(d_x, n, e);
    CPPFLOW_CHECK_LAUNCH();
    for (int i = 0; i < S; ++i) {
        const int b = i / 2, s = step_subnet(i), bs = 2 * b + s;
        for (int l = 0; l < L; ++l) {
            EpiArgs ep{};
            ep.bias = d->d_b_hidden + ((size_t)bs * L + l) * H;
            ep.out = h_of(i, l);
            ep.out_t = ht_of(i, l);
            ep.ldo = H;
            ep.ldt = n;
            const void* a = l == 0 ? (const void*)(ws.u + i * UN) : (const void*)h_of(i, l - 1);
            const void* w = l == 0 ? (const void*)(w_in + (size_t)bs * H * KIN)
                                   : (const void*)(w_hid + ((size_t)bs * (L - 1) + (l - 1)) * H * H);
            if ((rc = gemm_bf16<EPI_FWD_T>(enc, a, n, w, H, l == 0 ? KIN : H, ep, st))) return rc;
            CPPFLOW_CHECK_LAUNCH();
        }
        Head h;
        std::memset(&h, 0, sizeof(h));
        h.state_in = state(i);
        h.hidden = h_of(i, L - 1);
        h.w_out = d->d_w_out + (size_t)bs * NOUT * H;
        h.b_out = d->d_b_out + (size_t)bs * NOUT;
        h.H = H;
        h.upd_lo = upd_lo[s];
        h.upd_len = upd_len[s];
        h.clamp = d->rnvp_clamp;
        h.n = n;
        h.save_s = ws.save_s + i * SN;
        h.logdet = ws.logdet;
        const bool last = i == S - 1, block_end = i % 2 == 1;
        e.gather = block_end && !last ? d->d_perm + (size_t)(b + 1) * W : nullptr;
        if (last) {
            e.out = ws.z;
        } else {
            e.state = state(i + 1);
            e.u = ws.u + (i + 1) * UN;
            e.u_t = ws.u_t + (i + 1) * UN;
            e.next_lo = in_lo[step_subnet(i + 1)];
            e.next_len = in_len[step_subnet(i + 1)];
        }
        const int64_t groups = (n + 8 * HEAD_ROWS - 1) / (8 * HEAD_ROWS);
        const unsigned grid = (unsigned)std::min<int64_t>(groups, (int64_t)sms * 2);
        flow_head_kernel<<<grid, 256, head_smem, st>>>(h, e);
        CPPFLOW_CHECK_LAUNCH();
    }

    // ---- loss
    flow_nll_kernel<<<grid_for(n, 256), 256, 0, st>>>(ws.z, ws.logdet, d->d_scale, W, n, ws.nll, ws.ds[S & 1]);
    CPPFLOW_CHECK_LAUNCH();
    flow_loss_kernel<<<1, 1024, 0, st>>>(ws.nll, n, d_loss);
    CPPFLOW_CHECK_LAUNCH();

    // ---- backward
    for (int i = S - 1; i >= 0; --i) {
        const int b = i / 2, s = step_subnet(i), bs = 2 * b + s;
        const bool last = i == S - 1, block_end = i % 2 == 1;
        HeadBwd hb;
        std::memset(&hb, 0, sizeof(hb));
        hb.ds_next = ws.ds[(i + 1) & 1];
        hb.du_next = last ? nullptr : ws.du;
        if (!last) {
            hb.next_lo = in_lo[step_subnet(i + 1)];
            hb.next_len = in_len[step_subnet(i + 1)];
        }
        hb.ginv = block_end && !last ? d->d_perm_inv + (size_t)(b + 1) * W : nullptr;
        hb.state = state(i);
        hb.save_s = ws.save_s + i * SN;
        hb.upd_lo = upd_lo[s];
        hb.upd_len = upd_len[s];
        hb.width = W;
        hb.clamp = d->rnvp_clamp;
        hb.inv_n = 1.f / (float)n;
        hb.ds = ws.ds[i & 1];
        hb.da = ws.da;
        hb.da_t = ws.da_t;
        hb.da_t32 = ws.da_t32;
        hb.n = n;
        flow_head_bwd_kernel<<<row_warps, 256, 0, st>>>(hb);
        CPPFLOW_CHECK_LAUNCH();

        // last Linear: dW_out = dA^T . h, db_out = column sums of dA (FP32), dh = (dA . W_out) * leaky'(h)
        if ((rc = gemm_f32(enc, ws.da_t, NOUT, ht_of(i, L - 1), H, (int)n, grad + pl.w_out + (size_t)bs * NOUT * H, H, st)))
            return rc;
        CPPFLOW_CHECK_LAUNCH();
        flow_colsum_kernel<<<grid_for(NOUT, 8), 256, 0, st>>>(ws.da_t32, n, NOUT, grad + pl.b_out + (size_t)bs * NOUT);
        CPPFLOW_CHECK_LAUNCH();
        int cur = 0;
        {
            EpiArgs ep{};
            ep.out = ws.dh[cur];
            ep.out_t = ws.dh_t[cur];
            ep.act = h_of(i, L - 1);
            ep.ldo = H;
            ep.ldt = n;
            if ((rc = gemm_bf16<EPI_BWD>(enc, ws.da, n, w_out_t + (size_t)bs * H * KIN, H, KIN, ep, st))) return rc;
            CPPFLOW_CHECK_LAUNCH();
        }
        for (int l = L - 1; l >= 0; --l) {
            const int Kl = l == 0 ? KIN : H;
            const void* x_t = l == 0 ? (const void*)(ws.u_t + i * UN) : (const void*)ht_of(i, l - 1);
            float* dw = grad + (l == 0 ? pl.w_in + (size_t)bs * H * KIN : pl.w_hidden + ((size_t)bs * (L - 1) + l - 1) * H * H);
            if ((rc = gemm_f32(enc, ws.dh_t[cur], H, x_t, Kl, (int)n, dw, Kl, st))) return rc;
            CPPFLOW_CHECK_LAUNCH();
            flow_colsum_kernel<<<grid_for(H, 8), 256, 0, st>>>(ws.dh_t[cur], n, H, grad + pl.b_hidden + ((size_t)bs * L + l) * H);
            CPPFLOW_CHECK_LAUNCH();
            if (l > 0) {
                EpiArgs ep{};
                ep.out = ws.dh[1 - cur];
                ep.out_t = ws.dh_t[1 - cur];
                ep.act = h_of(i, l - 1);
                ep.ldo = H;
                ep.ldt = n;
                if ((rc = gemm_bf16<EPI_BWD>(enc, ws.dh[cur], n, w_hid_t + ((size_t)bs * (L - 1) + l - 1) * H * H, H, H, ep, st)))
                    return rc;
                CPPFLOW_CHECK_LAUNCH();
                cur = 1 - cur;
            } else if (i > 0) {  // the gradient of x itself is not needed
                if ((rc = gemm_f32(enc, ws.dh[cur], n, w_in_t + (size_t)bs * KIN * H, KIN, H, ws.du, KIN, st))) return rc;
                CPPFLOW_CHECK_LAUNCH();
            }
        }
    }
    if (flags & CPPFLOW_FLOW_TRAIN_NO_UPDATE) return CPPFLOW_OK;
    return apply_update(t, grad, ws.flags, ws.skip, sms, st);
}

extern "C" int cppflow_flow_train_apply(const cppflow_flow_train_desc* t, const float* d_grad, int64_t batch,
                                       void* d_workspace, size_t ws_bytes, void* stream) {
    int rc = validate_train(t, batch);
    if (rc) return rc;
    const cppflow_flow_desc* d = &t->flow;
    CPPFLOW_CHECK_ARG(d_grad, "d_grad");
    CPPFLOW_CHECK_ARG(d->d_w_in && (d->coeff_fn_config == 1 || (d->d_w_hidden && t->d_w_hidden_t)), "null BF16 table");
    CPPFLOW_CHECK_ARG(t->d_params && t->d_adam_m && t->d_adam_v && t->d_w_in_t && t->d_w_out_t && t->d_counters,
                      "null training table");
    const size_t need = train_ws(d, batch, nullptr, nullptr);
    if (!d_workspace || ws_bytes < need)
        return fail(CPPFLOW_E_WORKSPACE, "cppflow_flow_train_apply: workspace %zu bytes < %zu", ws_bytes, need);
    TrainWs ws;
    train_ws(d, batch, static_cast<uint8_t*>(d_workspace), &ws);
    return apply_update(t, d_grad, ws.flags, ws.skip, sm_count(), (cudaStream_t)stream);
}

extern "C" int cppflow_flow_grad_tree_reduce(const float* d_in, int n, int64_t len, int64_t stride, float scale,
                                            float* d_out, void* stream) {
    CPPFLOW_CHECK_ARG(d_in && d_out, "d_in / d_out");
    CPPFLOW_CHECK_ARG(n >= 1 && n <= CPPFLOW_TREE_REDUCE_MAX && (n & (n - 1)) == 0, "n is not a power of two in [1, 32]");
    CPPFLOW_CHECK_ARG(len >= 0 && len % 4 == 0 && stride % 4 == 0 && (n == 1 || stride >= len),
                      "len and stride must be multiples of 4, stride >= len");
    CPPFLOW_CHECK_ARG(reinterpret_cast<uintptr_t>(d_in) % 16 == 0 && reinterpret_cast<uintptr_t>(d_out) % 16 == 0,
                      "d_in / d_out not 16-byte aligned");
    if (len == 0) return CPPFLOW_OK;
    const int64_t len4 = len / 4, stride4 = stride / 4;
    const unsigned grid = (unsigned)std::min<int64_t>(grid_for(len4, 256), (int64_t)sm_count() * 8);
    cudaStream_t st = (cudaStream_t)stream;
    switch (n) {
        case 1: flow_tree_reduce_kernel<1><<<grid, 256, 0, st>>>(d_in, len4, stride4, scale, d_out); break;
        case 2: flow_tree_reduce_kernel<2><<<grid, 256, 0, st>>>(d_in, len4, stride4, scale, d_out); break;
        case 4: flow_tree_reduce_kernel<4><<<grid, 256, 0, st>>>(d_in, len4, stride4, scale, d_out); break;
        case 8: flow_tree_reduce_kernel<8><<<grid, 256, 0, st>>>(d_in, len4, stride4, scale, d_out); break;
        case 16: flow_tree_reduce_kernel<16><<<grid, 256, 0, st>>>(d_in, len4, stride4, scale, d_out); break;
        default: flow_tree_reduce_kernel<32><<<grid, 256, 0, st>>>(d_in, len4, stride4, scale, d_out); break;
    }
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" int cppflow_flow_train_batch_rows(const cppflow_flow_train_desc* t, const float* d_q, const float* d_poses,
                                            int64_t n_data, int64_t batch, int64_t first_row, uint64_t seed,
                                            float softflow_noise_scale, float* d_x, float* d_cond, int64_t* d_idx,
                                            float* d_noise, void* stream) {
    int rc = validate_train(t, batch);
    if (rc) return rc;
    CPPFLOW_CHECK_ARG(d_q && d_poses && d_x && d_cond && t->d_counters, "d_q / d_poses / d_x / d_cond / d_counters");
    CPPFLOW_CHECK_ARG(n_data >= 1, "n_data < 1");
    CPPFLOW_CHECK_ARG(first_row >= 0, "first_row < 0");
    const cppflow_flow_desc* d = &t->flow;
    flow_train_batch_kernel<<<grid_for(batch, 256), 256, 0, (cudaStream_t)stream>>>(
        d_q, d_poses, n_data, batch, first_row, d->ndof, d->width, d->dim_cond, seed, t->d_counters + 2,
        softflow_noise_scale, d_x, d_cond, d_idx, d_noise);
    CPPFLOW_CHECK_LAUNCH();
    return CPPFLOW_OK;
}

extern "C" int cppflow_flow_train_batch(const cppflow_flow_train_desc* t, const float* d_q, const float* d_poses,
                                       int64_t n_data, int64_t batch, uint64_t seed, float softflow_noise_scale,
                                       float* d_x, float* d_cond, int64_t* d_idx, float* d_noise, void* stream) {
    return cppflow_flow_train_batch_rows(t, d_q, d_poses, n_data, batch, 0, seed, softflow_noise_scale, d_x, d_cond,
                                         d_idx, d_noise, stream);
}
