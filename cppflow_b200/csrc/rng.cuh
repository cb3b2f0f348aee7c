// Counter-based random numbers shared by the training batch draw (k_flow_train.cu) and the exact-IK latents (k_ik.cu):
// every draw is a hash of its coordinates, so a value does not depend on the launch shape or on the other rows.
#pragma once
#include <cstdint>

namespace cppflow {

__device__ __forceinline__ uint64_t mix64(uint64_t z) {  // splitmix64's finaliser
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// uniform in (0, 1), never 0 (a Box-Muller radius takes its log)
__device__ __forceinline__ float u01(uint64_t h) { return ((float)(h >> 40) + 0.5f) * (1.f / 16777216.f); }

}  // namespace cppflow
