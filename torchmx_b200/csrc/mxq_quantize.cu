// K1: fused MX quantize (bf16/fp32 -> element codes + E8M0 scales), one pass over HBM.
//
// Replaces the reference op chain torchmx/mx_tensor.py:72-96 ->
// mx_quantization_utils.py:502-558 (shared exponent) -> :435-499 / :253-412 (element cast) ->
// utils.py:120-145 (fp4 packing), which on a GPU is 33-183 separate aten launches.
//
// Fast path (block_size 32, bf16): the tensor is a flat run of 64-byte blocks.  A thread owns
// EPT = 8, 16 or 32 consecutive elements (one 128/256-bit load, or two 256-bit loads), so
// 32/EPT adjacent lanes own one block: the block amax is a packed-u16 max over the thread's
// registers plus log2(32/EPT) shuffles.  Codes leave as one 64/128/256-bit store per thread and
// the scale byte as one byte store from the block's first lane.  Algorithmic traffic:
// 2 B in + 1 B (0.5 B fp4) + 1/32 B out per element.
#include "mxq_quant_core.cuh"

namespace mxq {

constexpr int kQuantThreads = 256;

// BS = block size: 32 (the MX block; EPT 8 / 16 / 32), or 8 / 16 (EPT = BS: a thread owns a whole block) and 64 / 128 (EPT 32, two /
// four lanes per block) -- same arithmetic, only the number of lanes that share a block maximum changes.
// OPERAND (fp4 / fp6, EPT 16 / 32): the codes leave in the packed tensor-core operand format (include/mxq.h MXQ_OPERAND_*_PACKED:
// fp4 low nibble first, fp6 four codes in three bytes) instead of the reference layout -- what mxq_pack_operand would make of
// them, without the extra launch and round trip; the codes themselves are the same.
// OVER_L2 (block 32, reference layout; the launch's input + code bytes exceed L2): from chunk `hint_from` on -- the chunks
// whose codes are the last l2_handoff_window() bytes the kernel writes -- the input is loaded L2 evict-first while codes and
// scales are stored at normal priority, so the lines the kernel leaves in L2 are those codes, the ones K2, walking back to
// front, reads first.  The chunks before stream as in the plain kernel: their codes cannot stay in L2 anyway.
template <int ELEM, int EPT, int BS = 32, bool OPERAND = false, bool OVER_L2 = false>
__global__ void __launch_bounds__(kQuantThreads) quantize_b32_bf16_kernel(const uint16_t* __restrict__ src, uint8_t* __restrict__ codes,
                                                                           uint8_t* __restrict__ scales, int64_t n_blocks, uint32_t flags,
                                                                           int64_t hint_from = 0) {
    pdl_launch_dependents();       // a dependent MX GEMM may start streaming its weights while the activation is quantized
    constexpr int LPB = BS / EPT;  // lanes per MX block
    constexpr int NW = EPT / 2;    // 32-bit words of bf16 pairs per thread
    constexpr int NO = (ELEM == MXQ_ELEM_E2M1) ? NW / 4 : NW / 2;
    uint64_t pol = 0;
    if constexpr (OVER_L2) pol = l2_evict_first_policy();
    const int64_t n_chunks = n_blocks * LPB;
    const int64_t stride = (int64_t)gridDim.x * kQuantThreads;
    for (int64_t c0 = (int64_t)blockIdx.x * kQuantThreads; c0 < n_chunks; c0 += stride) {
        const int64_t c = c0 + threadIdx.x;
        const bool live = c < n_chunks;  // a block's LPB lanes are live together (n_chunks % LPB == 0)
        const bool ef = OVER_L2 && c0 >= hint_from;  // uniform per CTA
        uint32_t w[NW];
        if (live) {
            const uint8_t* p = reinterpret_cast<const uint8_t*>(src) + c * (EPT * 2);
            if constexpr (EPT == 8) {
                const uint4 v = ef ? ldg128_evict_first(p, pol) : ldg128_stream(p);
                w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < NW / 8; ++j) {
                    const u32x8 v = ef ? ldg256_evict_first(p + 32 * j, pol) : ldg256_stream(p + 32 * j);
#pragma unroll
                    for (int k = 0; k < 8; ++k) w[8 * j + k] = v.v[k];
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < NW; ++i) w[i] = 0;
        }
        uint32_t m = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) m = umax16x2(m, w[i] & 0x7FFF7FFFu);
        m = max(m & 0xFFFFu, m >> 16);
#pragma unroll
        for (int d = 1; d < LPB; d <<= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
        const int s = shared_exp_from_maxE<ELEM>((int)(m >> 7));
        uint32_t out[NO];
        if (s != 255) convert_words<ELEM, NW>(w, s, out);
        else nanblock_words<ELEM, NW>(w, (flags & MXQ_FLAG_HW_EXACT) != 0, out);
        if constexpr (OPERAND && ELEM == MXQ_ELEM_E2M1) {
#pragma unroll
            for (int i = 0; i < NO; ++i) out[i] = ((out[i] & 0x0F0F0F0Fu) << 4) | ((out[i] >> 4) & 0x0F0F0F0Fu);
        }
        if constexpr (OPERAND && (ELEM == MXQ_ELEM_E3M2 || ELEM == MXQ_ELEM_E2M3)) {
            if (live) {
                uint32_t* q = reinterpret_cast<uint32_t*>(codes + c * (EPT * 3 / 4));  // 12 bytes per 16 codes
#pragma unroll
                for (int g = 0; g < EPT / 16; ++g) {
                    uint32_t t[4];  // 24 packed bits per word of four codes
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t v = out[4 * g + j];
                        t[j] = (v & 0x3F) | ((v >> 2) & 0xFC0) | ((v >> 4) & 0x3F000) | ((v >> 6) & 0xFC0000);
                    }
                    q[3 * g + 0] = t[0] | (t[1] << 24);
                    q[3 * g + 1] = (t[1] >> 8) | (t[2] << 16);
                    q[3 * g + 2] = (t[2] >> 16) | (t[3] << 8);
                }
                if ((threadIdx.x & (LPB - 1)) == 0) scales[c / LPB] = (uint8_t)s;
            }
        } else if (live) {
            constexpr int OB = NO * 4;  // output bytes per thread
            uint8_t* q = codes + c * OB;
            if constexpr (OB == 4) *reinterpret_cast<uint32_t*>(q) = out[0];
            else if constexpr (OB == 8) stg64_stream(q, make_uint2(out[0], out[1]));
            else if constexpr (OB == 16) stg128_stream(q, make_uint4(out[0], out[1], out[2], out[3]));
            else {
                u32x8 o;
#pragma unroll
                for (int k = 0; k < 8; ++k) o.v[k] = out[k];
                stg256_stream(q, o);
            }
            if ((threadIdx.x & (LPB - 1)) == 0) scales[c / LPB] = (uint8_t)s;
        }
    }
}

// ---- fp32 input (extension: the reference asserts bf16, torchmx/mx_tensor.py:59-61; the exponent rule is its fp32 branch,
// mx_quantization_utils.py:532-540), block 32: a thread owns 16 consecutive fp32 values (two 256-bit loads), two lanes share a
// block.  code = RNE_satfinite(x * 2^(127-s)) straight from fp32 (one rounding), int8 through the same magic-constant FMA.
// Algorithmic traffic: 4 B in + 1 B (0.5 B fp4) + 1/32 B out per element.
template <int ELEM>
__global__ void __launch_bounds__(kQuantThreads) quantize_b32_f32_kernel(const float* __restrict__ src, uint8_t* __restrict__ codes,
                                                                          uint8_t* __restrict__ scales, int64_t n_blocks) {
    pdl_launch_dependents();
    constexpr int EPT = 16;
    const int64_t n_chunks = n_blocks * 2;
    const int64_t stride = (int64_t)gridDim.x * kQuantThreads;
    for (int64_t c0 = (int64_t)blockIdx.x * kQuantThreads; c0 < n_chunks; c0 += stride) {
        const int64_t c = c0 + threadIdx.x;
        const bool live = c < n_chunks;
        uint32_t w[EPT];
        if (live) {
            const uint8_t* p = reinterpret_cast<const uint8_t*>(src) + c * (EPT * 4);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const u32x8 v = ldg256_stream(p + 32 * j);
#pragma unroll
                for (int k = 0; k < 8; ++k) w[8 * j + k] = v.v[k];
            }
        } else {
#pragma unroll
            for (int i = 0; i < EPT; ++i) w[i] = 0;
        }
        uint32_t m = 0;
#pragma unroll
        for (int i = 0; i < EPT; ++i) m = max(m, w[i] & 0x7FFFFFFFu);
        m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, 1));
        const int s = shared_exp_from_maxE<ELEM>((int)(m >> 23));
        constexpr int NO = (ELEM == MXQ_ELEM_E2M1) ? 2 : 4;
        uint32_t out[NO];
#pragma unroll
        for (int i = 0; i < NO; ++i) out[i] = 0;
        if (s != 255) {  // NaN-scale block: all codes +0 (mx_quantization_utils.py:473)
            const float inv = inv_scale_f32(s);
            if constexpr (ELEM == MXQ_ELEM_INT8) {
                constexpr float kMagic = 12582912.0f;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    uint32_t b[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float t = fmaf(__uint_as_float(w[4 * i + j]), inv, kMagic);
                        t = fminf(fmaxf(t, kMagic - 127.0f), kMagic + 127.0f);
                        b[j] = __float_as_uint(t);
                    }
                    out[i] = __byte_perm(__byte_perm(b[0], b[1], 0x0040), __byte_perm(b[2], b[3], 0x0040), 0x5410);
                }
            } else if constexpr (ELEM == MXQ_ELEM_E2M1) {
#pragma unroll
                for (int i = 0; i < 2; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        out[i] |= cvt_e2m1_byte(__uint_as_float(w[8 * i + 2 * j]) * inv, __uint_as_float(w[8 * i + 2 * j + 1]) * inv) << (8 * j);
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t p0 = cvt_pair<ELEM>(__uint_as_float(w[4 * i]) * inv, __uint_as_float(w[4 * i + 1]) * inv);
                    const uint32_t p1 = cvt_pair<ELEM>(__uint_as_float(w[4 * i + 2]) * inv, __uint_as_float(w[4 * i + 3]) * inv);
                    out[i] = p0 | (p1 << 16);
                }
            }
        }
        if (live) {
            if constexpr (ELEM == MXQ_ELEM_E2M1) stg64_stream(codes + c * 8, make_uint2(out[0], out[1]));
            else stg128_stream(codes + c * 16, make_uint4(out[0], out[1], out[2], out[3]));
            if ((threadIdx.x & 1) == 0) scales[c >> 1] = (uint8_t)s;
        }
    }
}

// ---- generic path: any block size, bf16 or fp32 input; two tiny passes, correctness first ----------
template <typename T> __device__ __forceinline__ int exp_field(T v);
template <> __device__ __forceinline__ int exp_field<uint16_t>(uint16_t v) { return (v >> 7) & 0xFF; }
template <> __device__ __forceinline__ int exp_field<float>(float v) { return (__float_as_uint(v) >> 23) & 0xFF; }
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<uint16_t>(uint16_t v) { return __uint_as_float((uint32_t)v << 16); }
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }

template <int ELEM, typename T>
__global__ void scales_generic_kernel(const T* __restrict__ src, uint8_t* __restrict__ scales, int64_t n_blocks, int block_size) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const T* p = src + b * block_size;
    int mx = 0;
    for (int i = 0; i < block_size; ++i) mx = max(mx, exp_field<T>(p[i]));
    scales[b] = (uint8_t)shared_exp_from_maxE<ELEM>(mx);
}

template <int ELEM, typename T>
__device__ __forceinline__ uint32_t code_generic(T v, int s, bool hw_exact) {
    if (s == 255) {
        if constexpr (ELEM != MXQ_ELEM_INT8 && ELEM != MXQ_ELEM_E5M2 && sizeof(T) == 2) {
            if (hw_exact) return hw_exact_nanblock_code<ELEM>((uint32_t)v);
        }
        return 0;
    }
    return quantize_one<ELEM>(to_f32<T>(v), s);
}

template <int ELEM, typename T>
__global__ void codes_generic_kernel(const T* __restrict__ src, const uint8_t* __restrict__ scales, uint8_t* __restrict__ codes,
                                     int64_t n_elems, int block_size, uint32_t flags) {
    const bool hw_exact = (flags & MXQ_FLAG_HW_EXACT) != 0;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if constexpr (ELEM == MXQ_ELEM_E2M1) {
        // one thread per output byte; the two nibbles may belong to different blocks (odd block sizes:
        // pack_uint4 runs over the flattened tensor, utils.py:144-145)
        if (2 * i + 1 >= n_elems + 1) return;
        const int64_t e0 = 2 * i, e1 = 2 * i + 1;
        const uint32_t hi = code_generic<ELEM, T>(src[e0], scales[e0 / block_size], hw_exact);
        const uint32_t lo = code_generic<ELEM, T>(src[e1], scales[e1 / block_size], hw_exact);
        codes[i] = (uint8_t)((hi << 4) | lo);
    } else {
        if (i >= n_elems) return;
        codes[i] = (uint8_t)code_generic<ELEM, T>(src[i], scales[i / block_size], hw_exact);
    }
}

// ---- launchers ---------------------------------------------------------------------------------
template <int ELEM, int EPT>
static void launch_b32_bf16(int64_t l2_bytes, int grid, cudaStream_t stream, const uint16_t* src, uint8_t* codes, uint8_t* scales, int64_t n_blocks,
                            unsigned flags) {
    constexpr int64_t kCodeBytes = (ELEM == MXQ_ELEM_E2M1) ? 16 : 32;  // per block
    if (n_blocks * (64 + kCodeBytes) > l2_bytes) {                     // bf16 input + codes
        const int64_t window = l2_handoff_window(l2_bytes) / kCodeBytes * (32 / EPT);  // chunks of the last window of codes
        const int64_t hint_from = n_blocks * (32 / EPT) - window;
        quantize_b32_bf16_kernel<ELEM, EPT, 32, false, true><<<grid, kQuantThreads, 0, stream>>>(src, codes, scales, n_blocks, flags, hint_from);
    } else {
        quantize_b32_bf16_kernel<ELEM, EPT><<<grid, kQuantThreads, 0, stream>>>(src, codes, scales, n_blocks, flags);
    }
}

template <int ELEM>
static cudaError_t launch_quantize_elem(const void* src, int src_dtype, int64_t n_blocks, int block_size, unsigned flags, void* codes,
                                        uint8_t* scales, int sm_count, int64_t l2_bytes, int ept_override, int waves, cudaStream_t stream) {
    if (n_blocks == 0) return cudaSuccess;
    const uintptr_t a_src = (uintptr_t)src, a_codes = (uintptr_t)codes;
    if (flags & MXQ_FLAG_OPERAND_LAYOUT) {
        if constexpr (ELEM == MXQ_ELEM_E2M1 || ELEM == MXQ_ELEM_E3M2 || ELEM == MXQ_ELEM_E2M3) {
            if (block_size != 32 || src_dtype != MXQ_HP_BF16 || (a_src % 32) || (a_codes % 32)) return cudaErrorNotSupported;
            const int64_t want = (n_blocks + kQuantThreads - 1) / kQuantThreads;
            const int grid = (int)(want < 0x7FFFFFFF ? want : 0x7FFFFFFF);
            quantize_b32_bf16_kernel<ELEM, 32, 32, true><<<grid, kQuantThreads, 0, stream>>>((const uint16_t*)src, (uint8_t*)codes, scales, n_blocks, flags);
            return cudaGetLastError();
        } else {
            return cudaErrorNotSupported;
        }
    }
    if (block_size == 32 && src_dtype == MXQ_HP_BF16 && (a_src % 32) == 0 && (a_codes % 32) == 0) {
        int ept = ept_override ? ept_override : 32;
        const int lpb = 32 / ept;
        const int64_t n_chunks = n_blocks * lpb;
        const int64_t want = (n_chunks + kQuantThreads - 1) / kQuantThreads;
        // one chunk per thread measured fastest on B200 (6.7 TB/s vs 6.6 with a 4-wave grid-stride cap); MXQ_WAVES caps the grid
        const int64_t cap = waves > 0 ? (int64_t)sm_count * 8 * waves : (int64_t)0x7FFFFFFF;
        const int grid = (int)(want < cap ? want : cap);
        const uint16_t* s16 = (const uint16_t*)src;
        uint8_t* c8 = (uint8_t*)codes;
        if (ept == 8) launch_b32_bf16<ELEM, 8>(l2_bytes, grid, stream, s16, c8, scales, n_blocks, flags);
        else if (ept == 32) launch_b32_bf16<ELEM, 32>(l2_bytes, grid, stream, s16, c8, scales, n_blocks, flags);
        else launch_b32_bf16<ELEM, 16>(l2_bytes, grid, stream, s16, c8, scales, n_blocks, flags);
        return cudaGetLastError();
    }
    if (src_dtype == MXQ_HP_BF16 && (a_src % 32) == 0 && (a_codes % 32) == 0 && (block_size == 8 || block_size == 16 || block_size == 64 || block_size == 128)) {
        // the same kernel with 1, 2 or 4 lanes per block (every access stays a whole, aligned vector)
        const int lpb = block_size <= 32 ? 1 : block_size / 32;
        const int64_t n_chunks = n_blocks * lpb;
        const int64_t want = (n_chunks + kQuantThreads - 1) / kQuantThreads;
        const int grid = (int)(want < 0x7FFFFFFF ? want : 0x7FFFFFFF);
        const uint16_t* s16 = (const uint16_t*)src;
        uint8_t* c8 = (uint8_t*)codes;
        if (block_size == 8) quantize_b32_bf16_kernel<ELEM, 8, 8><<<grid, kQuantThreads, 0, stream>>>(s16, c8, scales, n_blocks, flags);
        else if (block_size == 16) quantize_b32_bf16_kernel<ELEM, 16, 16><<<grid, kQuantThreads, 0, stream>>>(s16, c8, scales, n_blocks, flags);
        else if (block_size == 64) quantize_b32_bf16_kernel<ELEM, 32, 64><<<grid, kQuantThreads, 0, stream>>>(s16, c8, scales, n_blocks, flags);
        else quantize_b32_bf16_kernel<ELEM, 32, 128><<<grid, kQuantThreads, 0, stream>>>(s16, c8, scales, n_blocks, flags);
        return cudaGetLastError();
    }
    if (block_size == 32 && src_dtype == MXQ_HP_F32 && (a_src % 32) == 0 && (a_codes % 16) == 0) {
        const int64_t want = (n_blocks * 2 + kQuantThreads - 1) / kQuantThreads;
        const int grid = (int)(want < 0x7FFFFFFF ? want : 0x7FFFFFFF);
        quantize_b32_f32_kernel<ELEM><<<grid, kQuantThreads, 0, stream>>>((const float*)src, (uint8_t*)codes, scales, n_blocks);
        return cudaGetLastError();
    }
    const int64_t n_elems = n_blocks * block_size;
    const int threads = 256;
    const int64_t n_out = (ELEM == MXQ_ELEM_E2M1) ? n_elems / 2 : n_elems;
    const unsigned g1 = (unsigned)((n_blocks + threads - 1) / threads), g2 = (unsigned)((n_out + threads - 1) / threads);
    if (src_dtype == MXQ_HP_BF16) {
        scales_generic_kernel<ELEM, uint16_t><<<g1, threads, 0, stream>>>((const uint16_t*)src, scales, n_blocks, block_size);
        codes_generic_kernel<ELEM, uint16_t><<<g2, threads, 0, stream>>>((const uint16_t*)src, scales, (uint8_t*)codes, n_elems, block_size, flags);
    } else {
        scales_generic_kernel<ELEM, float><<<g1, threads, 0, stream>>>((const float*)src, scales, n_blocks, block_size);
        codes_generic_kernel<ELEM, float><<<g2, threads, 0, stream>>>((const float*)src, scales, (uint8_t*)codes, n_elems, block_size, flags);
    }
    return cudaGetLastError();
}

cudaError_t launch_quantize(const void* src, int src_dtype, int64_t n_blocks, int block_size, int elem, unsigned flags, void* codes,
                            uint8_t* scales, int sm_count, int64_t l2_bytes, int ept_override, int waves, cudaStream_t stream) {
#define CALL(E) launch_quantize_elem<E>(src, src_dtype, n_blocks, block_size, flags, codes, scales, sm_count, l2_bytes, ept_override, waves, stream)
    switch (elem) {
    case MXQ_ELEM_E4M3: return CALL(MXQ_ELEM_E4M3);
    case MXQ_ELEM_E3M2: return CALL(MXQ_ELEM_E3M2);
    case MXQ_ELEM_E2M3: return CALL(MXQ_ELEM_E2M3);
    case MXQ_ELEM_E2M1: return CALL(MXQ_ELEM_E2M1);
    case MXQ_ELEM_INT8: return CALL(MXQ_ELEM_INT8);
    case MXQ_ELEM_E5M2: return CALL(MXQ_ELEM_E5M2);
    default: return cudaErrorInvalidValue;
    }
#undef CALL
}

}  // namespace mxq
