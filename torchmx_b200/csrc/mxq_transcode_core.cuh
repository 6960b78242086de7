// Exact re-encoding of reference-layout fp6 / fp4 element codes as E4M3 bytes (every e3m2 / e2m3 / e2m1 value is an e4m3
// value), shared by mxq_transcode_to_e4m3 (mxq_transcode.cu) and K5e (mxq_kv_cache.cu), which stores its cache codes in the
// form the attention kernel reads.  fp6: one code per byte in bits [5:0]; fp4: two codes per byte, the even element in the
// high nibble.
#pragma once
#include "mxq_common.cuh"

namespace mxq {

// f16x2 -> two e4m3 bytes (exact: the value set is a subset of e4m3)
__device__ __forceinline__ uint32_t to_e4m3_pair(uint32_t h2) {
    uint16_t r;
    asm("cvt.rn.satfinite.e4m3x2.f16x2 %0, %1;" : "=h"(r) : "r"(h2));
    return r;
}

// one fp4 code byte (elements 2i in the high nibble, 2i + 1 in the low one) -> two e4m3 bytes in element order
__device__ __forceinline__ uint32_t e4m3_pair_from_fp4_byte(uint32_t byte) {
    return to_e4m3_pair(__byte_perm(decode_e2m1_byte_f16x2(byte), 0, 0x1032));  // high nibble (high half) is the earlier element
}

// NW words of codes -> their E4M3 bytes (NW words for fp6, 2 * NW for fp4)
template <int ELEM, int NW>
__device__ __forceinline__ void transcode_words_to_e4m3(const uint32_t (&w)[NW], uint32_t (&o)[(ELEM == MXQ_ELEM_E2M1) ? 2 * NW : NW]) {
#pragma unroll
    for (int j = 0; j < NW; ++j) {
        if constexpr (ELEM == MXQ_ELEM_E2M1) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const uint32_t p0 = e4m3_pair_from_fp4_byte((w[j] >> (16 * k)) & 0xFF), p1 = e4m3_pair_from_fp4_byte((w[j] >> (16 * k + 8)) & 0xFF);
                o[2 * j + k] = p0 | (p1 << 16);
            }
        } else {
            const uint32_t p0 = to_e4m3_pair(decode_pair_f16x2<ELEM>(w[j] & 0xFFFF));
            const uint32_t p1 = to_e4m3_pair(decode_pair_f16x2<ELEM>(w[j] >> 16));
            o[j] = p0 | (p1 << 16);
        }
    }
}

}  // namespace mxq
