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
#include "flow.cuh"

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
    e.cond_w = 7;
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
        std::memset(&h, 0, sizeof(h));
        h.state_in = state;
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
