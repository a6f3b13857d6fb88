// Counter-based random numbers for the draws the shim makes when the caller supplies none (the reference draws fresh
// uniforms with Tensor.uniform_ every decode step, src/generator.py:86-90, and nn.Dropout masks, src/discriminator.py:30).
// Philox4x32-10 (Salmon et al., SC'11): counter = (group index lo, hi, offset, tag), key = seed.  One call yields the four
// uniforms of elements 4c .. 4c+3 of a logical tensor, so a kernel that generates its tile on the fly and
// gic_philox_uniform() filling the whole tensor produce the SAME numbers (tests/test_gpu_tcgen05.py checks that).
#pragma once
#include <stdint.h>

namespace gic {

enum : uint32_t { RNG_TAG_GUMBEL = 0x47u, RNG_TAG_DROPOUT = 0x44u, RNG_TAG_SAMPLE = 0x53u };

struct RngState {
  unsigned long long seed, offset;
  const unsigned long long* dev;     // when non-null: {seed, offset} read from device memory (CUDA-graph replay)
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}

// uniform in [0, 1): the top 24 bits (exactly representable; never 1.0, as Tensor.uniform_(0, 1))
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }

__device__ __forceinline__ void rng_load(const RngState& st, unsigned long long& seed, unsigned long long& offset) {
  if (st.dev) { seed = st.dev[0]; offset = st.dev[1]; } else { seed = st.seed; offset = st.offset; }
}

// the four uniforms of elements 4*group .. 4*group+3 of the logical tensor `tag` at RNG offset `offset`
__device__ __forceinline__ float4 philox_uniform4(unsigned long long seed, unsigned long long offset, uint32_t tag,
                                                  unsigned long long group) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)group, (uint32_t)(group >> 32), (uint32_t)offset,
                                           tag ^ (uint32_t)(offset >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
}

}  // namespace gic
