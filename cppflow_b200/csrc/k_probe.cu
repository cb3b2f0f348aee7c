// FP32 FMA throughput probe: the roofline denominator for the FP32-bound fused LM kernels
// (MEASURED_PEAKS.json has HBM and bf16 tensor numbers only; SURVEY.md 8d asks for a measured FP32 peak).
// Each thread runs 8 independent FMA chains; FLOPs = 2 * 8 * iters * threads.
#include "common.cuh"

namespace cppflow {

__global__ void __launch_bounds__(1024) fp32_probe_kernel(int iters, float* __restrict__ out) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
    float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.999f, c = 1e-3f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
            a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
        }
    }
    const float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678f) out[0] = s;  // keep the chains alive
}

}  // namespace cppflow

using namespace cppflow;

// Launches `blocks` CTAs of 1024 threads; returns the FLOP count of the launch in *flops_out.
extern "C" int cppflow_fp32_probe(int blocks, int iters, float* d_scratch, double* flops_out, void* stream) {
    CPPFLOW_CHECK_ARG(blocks > 0 && iters > 0 && d_scratch, "blocks, iters, scratch");
    fp32_probe_kernel<<<blocks, 1024, 0, (cudaStream_t)stream>>>(iters, d_scratch);
    CPPFLOW_CHECK_LAUNCH();
    if (flops_out) *flops_out = 2.0 * 8.0 * 8.0 * (double)iters * 1024.0 * (double)blocks;
    return CPPFLOW_OK;
}
