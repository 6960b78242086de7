// Rotary position embedding arithmetic of K5b, shared with K5e (mxq_kv_cache.cu): transformers' apply_rotary_pos_emb,
//     out = (x * cos) + (rotate_half(x) * sin),   rotate_half(x) = cat(-x2, x1)
// with every bf16 rounding of its elementwise launches reproduced -- each product and the sum is a bf16 tensor.  One copy of
// the rounding sequence keeps both kernels bit-identical to the eager chain by construction.
#pragma once
#include "mxq_common.cuh"

namespace mxq {
namespace glue {

__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }
__device__ __forceinline__ float round_bf16(float f) { return __uint_as_float(pack_bf16x2(f, 0.0f) << 16); }

// two channels of the FIRST half of a head: x1 (these channels), x2 (the channels head_dim / 2 further), cos / sin of x1's channels
__device__ __forceinline__ uint32_t rope_first_half(uint32_t x1, uint32_t x2, uint32_t c, uint32_t s) {
    const float lo = round_bf16(bf16lo(x1) * bf16lo(c)) + round_bf16(-bf16lo(x2) * bf16lo(s));
    const float hi = round_bf16(bf16hi(x1) * bf16hi(c)) + round_bf16(-bf16hi(x2) * bf16hi(s));
    return pack_bf16x2(lo, hi);
}

// two channels of the SECOND half: x2 (these channels), x1 (the channels head_dim / 2 before), cos / sin of x2's channels
__device__ __forceinline__ uint32_t rope_second_half(uint32_t x2, uint32_t x1, uint32_t c, uint32_t s) {
    const float lo = round_bf16(bf16lo(x2) * bf16lo(c)) + round_bf16(bf16lo(x1) * bf16lo(s));
    const float hi = round_bf16(bf16hi(x2) * bf16hi(c)) + round_bf16(bf16hi(x1) * bf16hi(s));
    return pack_bf16x2(lo, hi);
}

}  // namespace glue
}  // namespace mxq
