// K5e rope_quantize_kv_kernel: one launch per attention layer and forward that takes the q / k / v projection outputs to the MX
// operands of the attention kernel (K4b) with the KV cache held as MX codes.  It replaces rotary (K5b), the bf16 cache write, the
// quantization of Q, the re-quantization of the whole key cache and K5d over the whole value cache: per step only the blocks
// the new tokens touch are computed.
//
// Layout: one thread per 32-element MX block, the blocks of Q, K and V in one flat index space (Q, then K, then V).
//  * A Q / K block is 32 channels of one (batch, head, token).  Its rotate_half partner is the block 64 channels away, so the
//    thread reads both (plus cos / sin of its own channels), rotates with K5b's rounding sequence (mxq_rope_core.cuh) and
//    quantizes with K1's arithmetic (mxq_quant_core.cuh).  Threads run in output order, so code and scale stores are contiguous.
//  * A V block is 32 consecutive positions of one (batch, kv head, channel), as K5d blocks V.  Consecutive threads take
//    consecutive channels: each of the 32 position loads of a warp is one 64-byte row segment.  Positions below L come from
//    v_open (only the block holding L has any), positions in [L, L + T) from v, the rest are zero.
//  * v_open is re-written with the block holding L + T by the thread that read the block holding L for the same channel -- the
//    only thread that reads that column -- after its reads, so no other thread's read can race with the write.
// The grid covers the largest number of V blocks T tokens can touch (ceil(T / 32) + 1); L lives on the device, and the threads
// past the blocks [L, L + T) actually touches leave at once.
#include <cstdio>

#include "mxq_quant_core.cuh"
#include "mxq_rope_core.cuh"
#include "mxq_transcode_core.cuh"

namespace mxq {
namespace glue {

struct RopeKVParams {
    const uint16_t* in[2]; int64_t in_tok_stride[2], in_batch_stride[2]; int heads[2];  // q, k
    const uint16_t* v; int64_t v_tok_stride, v_batch_stride;
    const uint16_t* cos; const uint16_t* sin; int64_t cs_batch_stride, cs_tok_stride;
    int64_t batch, tokens;
    int elem[3]; unsigned flags;  // q, k, v
    uint8_t* q_codes; uint8_t* q_scales;
    uint8_t* k_codes; uint8_t* k_scales;
    uint8_t* vt_codes; uint8_t* vt_scales;
    uint16_t* v_open;
    int64_t capacity; const int64_t* position;
    int64_t n_q, n_k, n_v, v_blocks;  // thread counts of the three sections; V blocks per (batch, kv head, channel) in the grid
};

// one block -> its scale and 32 one-byte codes in the form K4b reads: e4m3 / e5m2 as they are, fp6 / fp4 re-encoded as E4M3
template <int ELEM>
__device__ __forceinline__ int quantize_block_bytes(const uint32_t (&w)[16], bool hw_exact, uint32_t (&out)[8]) {
    if constexpr (ELEM == MXQ_ELEM_E4M3 || ELEM == MXQ_ELEM_E5M2) {
        return quantize_block32<ELEM>(w, hw_exact, out);
    } else {
        constexpr int NC = ELEM == MXQ_ELEM_E2M1 ? 4 : 8;
        uint32_t c[NC];
        const int s = quantize_block32<ELEM>(w, hw_exact, c);
        transcode_words_to_e4m3<ELEM, NC>(c, out);
        return s;
    }
}

__device__ __forceinline__ int quantize_block_bytes(int elem, const uint32_t (&w)[16], bool hw_exact, uint32_t (&out)[8]) {
    switch (elem) {
    case MXQ_ELEM_E4M3: return quantize_block_bytes<MXQ_ELEM_E4M3>(w, hw_exact, out);
    case MXQ_ELEM_E3M2: return quantize_block_bytes<MXQ_ELEM_E3M2>(w, hw_exact, out);
    case MXQ_ELEM_E2M3: return quantize_block_bytes<MXQ_ELEM_E2M3>(w, hw_exact, out);
    case MXQ_ELEM_E2M1: return quantize_block_bytes<MXQ_ELEM_E2M1>(w, hw_exact, out);
    default: return quantize_block_bytes<MXQ_ELEM_E5M2>(w, hw_exact, out);
    }
}

__device__ __forceinline__ void store_block(uint8_t* dst, const uint32_t (&o)[8]) {
    *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<uint4*>(dst + 16) = make_uint4(o[4], o[5], o[6], o[7]);
}

// 32 positions p0 .. p0 + 31 of value channel c as 16 bf16 pairs: v_open below L, v in [L, L + T), zero past it
__device__ __forceinline__ void gather_v(const RopeKVParams& p, int64_t b, int h, int c, int64_t p0, int64_t L, uint32_t (&w)[16]) {
    const uint16_t* open = p.v_open + ((b * p.heads[1] + h) * 32) * 128 + c;
    const uint16_t* src = p.v + b * p.v_batch_stride + (int64_t)h * 128 + c;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        uint32_t e[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int64_t pos = p0 + 2 * i + k;
            e[k] = pos < L ? open[(2 * i + k) * 128] : (pos < L + p.tokens ? src[(pos - L) * p.v_tok_stride] : 0);
        }
        w[i] = e[0] | (e[1] << 16);
    }
}

__global__ void __launch_bounds__(256) rope_quantize_kv_kernel(const RopeKVParams p) {
    pdl_launch_dependents();
    pdl_wait();  // (launched with programmatic serialization: nothing the predecessor wrote is read before this)
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= p.n_q + p.n_k + p.n_v) return;
    const int64_t L = *p.position;
    const bool hw_exact = (p.flags & MXQ_FLAG_HW_EXACT) != 0;
    uint32_t w[16], out[8];
    if (i < p.n_q + p.n_k) {  // a Q or K block: ((b * heads + h) * T + t) * 4 + j
        const int which = i >= p.n_q;
        int64_t r = which ? i - p.n_q : i;
        const int j = (int)(r & 3); r >>= 2;
        const int64_t t = r % p.tokens; r /= p.tokens;
        const int h = (int)(r % p.heads[which]);
        const int64_t b = r / p.heads[which];
        if (which && L + t >= p.capacity) return;
        const uint16_t* x = p.in[which] + b * p.in_batch_stride[which] + t * p.in_tok_stride[which] + (int64_t)h * 128;
        const uint16_t* pc = p.cos + b * p.cs_batch_stride + t * p.cs_tok_stride;
        const uint16_t* ps = p.sin + b * p.cs_batch_stride + t * p.cs_tok_stride;
        const int d0 = 32 * j, dp = j < 2 ? d0 + 64 : d0 - 64;  // this block's channels, its rotate_half partner's
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint4 xa = *reinterpret_cast<const uint4*>(x + d0 + 8 * u), xb = *reinterpret_cast<const uint4*>(x + dp + 8 * u);
            const uint4 ca = *reinterpret_cast<const uint4*>(pc + d0 + 8 * u), sa = *reinterpret_cast<const uint4*>(ps + d0 + 8 * u);
            const uint32_t a[4] = {xa.x, xa.y, xa.z, xa.w}, q[4] = {xb.x, xb.y, xb.z, xb.w};
            const uint32_t c[4] = {ca.x, ca.y, ca.z, ca.w}, s[4] = {sa.x, sa.y, sa.z, sa.w};
#pragma unroll
            for (int m = 0; m < 4; ++m) w[4 * u + m] = j < 2 ? rope_first_half(a[m], q[m], c[m], s[m]) : rope_second_half(a[m], q[m], c[m], s[m]);
        }
        const int sc = quantize_block_bytes(p.elem[which], w, hw_exact, out);
        if (which == 0) {
            store_block(p.q_codes + i * 32, out);
            p.q_scales[i] = (uint8_t)sc;
        } else {
            const int64_t row = (b * p.heads[1] + h) * p.capacity + L + t;
            store_block(p.k_codes + row * 128 + 32 * j, out);
            p.k_scales[row * 4 + j] = (uint8_t)sc;
        }
        return;
    }
    // a V block: ((b * kv_heads + h) * v_blocks + kb) * 128 + c, block index L / 32 + kb
    int64_t r = i - p.n_q - p.n_k;
    const int c = (int)(r & 127); r >>= 7;
    const int64_t kb = r % p.v_blocks; r /= p.v_blocks;
    const int h = (int)(r % p.heads[1]);
    const int64_t b = r / p.heads[1];
    const int64_t vb = L / 32 + kb, p0 = 32 * vb;
    if (p0 >= L + p.tokens || p0 >= p.capacity) return;
    gather_v(p, b, h, c, p0, L, w);
    const int sc = quantize_block_bytes(p.elem[2], w, hw_exact, out);
    const int64_t blk = ((b * p.heads[1] + h) * 128 + c) * (p.capacity / 32) + vb;
    store_block(p.vt_codes + blk * 32, out);
    p.vt_scales[blk] = (uint8_t)sc;
    if (kb == 0) {  // the block holding L + T becomes the open block
        const int64_t nb = (L + p.tokens) / 32;
        if (nb != vb) gather_v(p, b, h, c, 32 * nb, L, w);  // (positions >= 32 * nb > L: from v or zero, v_open not read)
        uint16_t* open = p.v_open + ((b * p.heads[1] + h) * 32) * 128 + c;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            open[(2 * k) * 128] = (uint16_t)(w[k] & 0xFFFF);
            open[(2 * k + 1) * 128] = (uint16_t)(w[k] >> 16);
        }
    }
}

}  // namespace glue

int launch_rope_quantize_kv(const mxq_rope_quantize_kv_args_t* a, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace glue;
    auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
    if (!al16(a->q) || !al16(a->k) || !al16(a->v) || !al16(a->cos) || !al16(a->sin) || (a->q_tok_stride % 8) || (a->k_tok_stride % 8) || (a->v_tok_stride % 8) ||
        (a->q_batch_stride % 8) || (a->k_batch_stride % 8) || (a->v_batch_stride % 8) || (a->cs_tok_stride % 8) || (a->cs_batch_stride % 8) ||
        !al16(a->q_codes) || !al16(a->k_codes) || !al16(a->vt_codes) || ((uintptr_t)a->v_open % 2)) {
        snprintf(msg, msg_len, "needs 16-byte aligned heads and code buffers (strides multiples of 8 elements)");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    RopeKVParams p;
    p.in[0] = (const uint16_t*)a->q; p.in[1] = (const uint16_t*)a->k; p.v = (const uint16_t*)a->v;
    p.in_tok_stride[0] = a->q_tok_stride; p.in_tok_stride[1] = a->k_tok_stride; p.v_tok_stride = a->v_tok_stride;
    p.in_batch_stride[0] = a->q_batch_stride; p.in_batch_stride[1] = a->k_batch_stride; p.v_batch_stride = a->v_batch_stride;
    p.heads[0] = a->q_heads; p.heads[1] = a->kv_heads;
    p.cos = (const uint16_t*)a->cos; p.sin = (const uint16_t*)a->sin;
    p.cs_batch_stride = a->cs_batch_stride; p.cs_tok_stride = a->cs_tok_stride;
    p.batch = a->batch; p.tokens = a->tokens;
    p.elem[0] = a->q_elem; p.elem[1] = a->k_elem; p.elem[2] = a->v_elem; p.flags = a->flags;
    p.q_codes = (uint8_t*)a->q_codes; p.q_scales = a->q_scales;
    p.k_codes = (uint8_t*)a->k_codes; p.k_scales = a->k_scales;
    p.vt_codes = (uint8_t*)a->vt_codes; p.vt_scales = a->vt_scales;
    p.v_open = (uint16_t*)a->v_open;
    p.capacity = a->capacity; p.position = a->position;
    p.v_blocks = (a->tokens + 31) / 32 + 1;
    p.n_q = a->batch * a->q_heads * a->tokens * 4;
    p.n_k = a->batch * a->kv_heads * a->tokens * 4;
    p.n_v = a->batch * a->kv_heads * p.v_blocks * 128;
    const int64_t grid = (p.n_q + p.n_k + p.n_v + 255) / 256;
    if (grid > 0x7FFFFFFF) { snprintf(msg, msg_len, "too many blocks"); return MXQ_ERR_UNSUPPORTED_SHAPE; }
    launch_pdl(rope_quantize_kv_kernel, dim3((unsigned)grid), dim3(256), 0, stream, p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

}  // namespace mxq
