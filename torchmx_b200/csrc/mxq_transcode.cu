// Exact re-encoding of reference-layout element codes (fp6 in bits [5:0] of a byte, fp4 two per
// byte with the even element in the high nibble) as E4M3 bytes.  Every e3m2 / e2m3 / e2m1 value is
// an e4m3 value, so the block-scaled tensor-core path can consume all FP element types as
// kind::mxf8f6f4 E4M3 operands without touching the reference's persisted storage layout.
#include "mxq_transcode_core.cuh"

namespace mxq {

template <int ELEM>
__global__ void __launch_bounds__(256) transcode_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int64_t n_in_bytes) {
    // 16 input bytes per thread when aligned; scalar tail
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_vec = n_in_bytes / 16;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
        const uint4 v = ldg128_stream(in + i * 16);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        if constexpr (ELEM == MXQ_ELEM_E2M1) {
            uint32_t o[8];
            transcode_words_to_e4m3<ELEM, 4>(w, o);
            u32x8 r;
#pragma unroll
            for (int k = 0; k < 8; ++k) r.v[k] = o[k];
            stg256_stream(out + i * 32, r);
        } else {
            uint32_t o[4];
            transcode_words_to_e4m3<ELEM, 4>(w, o);
            stg128_stream(out + i * 16, make_uint4(o[0], o[1], o[2], o[3]));
        }
    }
    // tail bytes
    for (int64_t b = n_vec * 16 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < n_in_bytes; b += stride) {
        const uint32_t c = in[b];
        if constexpr (ELEM == MXQ_ELEM_E2M1) {
            const uint32_t p = e4m3_pair_from_fp4_byte(c);
            out[2 * b] = (uint8_t)p;
            out[2 * b + 1] = (uint8_t)(p >> 8);
        } else {
            out[b] = (uint8_t)to_e4m3_pair(decode_pair_f16x2<ELEM>(c));
        }
    }
}

cudaError_t launch_transcode(const void* codes, int elem, int64_t n_elements, void* out, int sm_count, cudaStream_t stream) {
    if (elem == MXQ_ELEM_E4M3) return cudaMemcpyAsync(out, codes, (size_t)n_elements, cudaMemcpyDeviceToDevice, stream);
    const int64_t n_in = elem == MXQ_ELEM_E2M1 ? n_elements / 2 : n_elements;
    if (((uintptr_t)codes % 16) || ((uintptr_t)out % 32)) return cudaErrorMisalignedAddress;
    const int64_t want = (n_in / 16 + 255) / 256 + 1;
    const int64_t cap = (int64_t)sm_count * 32;
    const int grid = (int)(want < cap ? want : cap);
    const uint8_t* in = (const uint8_t*)codes;
    uint8_t* o = (uint8_t*)out;
    if (elem == MXQ_ELEM_E3M2) transcode_kernel<MXQ_ELEM_E3M2><<<grid, 256, 0, stream>>>(in, o, n_in);
    else if (elem == MXQ_ELEM_E2M3) transcode_kernel<MXQ_ELEM_E2M3><<<grid, 256, 0, stream>>>(in, o, n_in);
    else transcode_kernel<MXQ_ELEM_E2M1><<<grid, 256, 0, stream>>>(in, o, n_in);
    return cudaGetLastError();
}

// ---- hardware-packed operand formats (include/mxq.h: MXQ_OPERAND_*_PACKED) -------------------------------------
// fp4: swap the nibbles of every byte (reference: even element high; TMA / UMMA: element 2i low).  16 bytes per thread.
__global__ void __launch_bounds__(256) pack_fp4_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int64_t n_bytes) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_vec = n_bytes / 16;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
        const uint4 v = ldg128_stream(in + i * 16);
        auto sw = [](uint32_t w) { return ((w & 0x0F0F0F0Fu) << 4) | ((w >> 4) & 0x0F0F0F0Fu); };
        stg128_stream(out + i * 16, make_uint4(sw(v.x), sw(v.y), sw(v.z), sw(v.w)));
    }
    for (int64_t b = n_vec * 16 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < n_bytes; b += stride) {
        const uint32_t c = in[b];
        out[b] = (uint8_t)((c << 4) | (c >> 4));
    }
}

// fp6: 16 one-byte codes (bits [5:0]) -> 12 bytes, element i in bits [6i, 6i+6) of the group
__global__ void __launch_bounds__(256) pack_fp6_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int64_t n_groups) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_groups; i += stride) {
        const uint4 v = ldg128_stream(in + i * 16);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        uint32_t t[4];  // 24 packed bits per input word (4 codes)
#pragma unroll
        for (int j = 0; j < 4; ++j) t[j] = (w[j] & 0x3F) | ((w[j] >> 2) & 0xFC0) | ((w[j] >> 4) & 0x3F000) | ((w[j] >> 6) & 0xFC0000);
        uint32_t* o = reinterpret_cast<uint32_t*>(out + i * 12);  // 12-byte groups: 4-byte aligned
        o[0] = t[0] | (t[1] << 24);
        o[1] = (t[1] >> 8) | (t[2] << 16);
        o[2] = (t[2] >> 16) | (t[3] << 8);
    }
}

// fp6 inverse: 12 packed bytes -> 16 one-byte codes (bits [5:0]; bits [7:6] zero, as the reference quantizer writes them)
__global__ void __launch_bounds__(256) unpack_fp6_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int64_t n_groups) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_groups; i += stride) {
        const uint32_t* s = reinterpret_cast<const uint32_t*>(in + i * 12);
        const uint32_t a = s[0], b = s[1], c = s[2];
        const uint32_t t[4] = {a & 0xFFFFFFu, (a >> 24) | ((b & 0xFFFFu) << 8), (b >> 16) | ((c & 0xFFu) << 16), c >> 8};
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) w[j] = (t[j] & 0x3F) | ((t[j] & 0xFC0) << 2) | ((t[j] & 0x3F000) << 4) | ((t[j] & 0xFC0000) << 6);
        stg128_stream(out + i * 16, make_uint4(w[0], w[1], w[2], w[3]));
    }
}

cudaError_t launch_unpack_operand(const void* packed, int elem, int64_t n_elements, void* out, int sm_count, cudaStream_t stream) {
    if (((uintptr_t)packed % 16) || ((uintptr_t)out % 16)) return cudaErrorMisalignedAddress;
    const int64_t cap = (int64_t)sm_count * 32;
    if (elem == MXQ_ELEM_E2M1) {  // the nibble swap is its own inverse
        const int64_t n_bytes = n_elements / 2;
        const int64_t want = (n_bytes / 16 + 255) / 256 + 1;
        pack_fp4_kernel<<<(int)(want < cap ? want : cap), 256, 0, stream>>>((const uint8_t*)packed, (uint8_t*)out, n_bytes);
    } else {
        const int64_t n_groups = n_elements / 16;
        const int64_t want = (n_groups + 255) / 256 + 1;
        unpack_fp6_kernel<<<(int)(want < cap ? want : cap), 256, 0, stream>>>((const uint8_t*)packed, (uint8_t*)out, n_groups);
    }
    return cudaGetLastError();
}

cudaError_t launch_pack_operand(const void* codes, int elem, int64_t n_elements, void* out, int sm_count, cudaStream_t stream) {
    if (((uintptr_t)codes % 16) || ((uintptr_t)out % 16)) return cudaErrorMisalignedAddress;
    const int64_t cap = (int64_t)sm_count * 32;
    if (elem == MXQ_ELEM_E2M1) {
        const int64_t n_bytes = n_elements / 2;
        const int64_t want = (n_bytes / 16 + 255) / 256 + 1;
        pack_fp4_kernel<<<(int)(want < cap ? want : cap), 256, 0, stream>>>((const uint8_t*)codes, (uint8_t*)out, n_bytes);
    } else {
        const int64_t n_groups = n_elements / 16;
        const int64_t want = (n_groups + 255) / 256 + 1;
        pack_fp6_kernel<<<(int)(want < cap ? want : cap), 256, 0, stream>>>((const uint8_t*)codes, (uint8_t*)out, n_groups);
    }
    return cudaGetLastError();
}

}  // namespace mxq
