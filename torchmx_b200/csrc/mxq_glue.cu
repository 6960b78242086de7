// K5: the two elementwise / row-wise steps that sit between the MX linears of a Llama / Qwen2 decoder layer and decide, at
// decode sizes, how many launches a layer costs.
//
// K5a rmsnorm_kernel: (residual add +) RMSNorm (+ MX quantization of the result).  The norm output feeds only MX linears, and the
// reference quantizes it on entry to each of them (torchmx/layers/mx_linear.py:63-66: q/k/v and gate/up quantize the SAME tensor
// three / two times); here the row is normalised and quantized in one pass -- x never makes a round trip through HBM as bf16
// between the norm and the quantizer.  Arithmetic = transformers' LlamaRMSNorm / Qwen2RMSNorm (fp32 statistics, the normalised row
// rounded to bf16 BEFORE the bf16 multiply by the weight), then K1's block quantizer (mxq_quant_core.cuh).
//
// K5b rope_kernel: rotary position embedding of the query and key heads, transformers' apply_rotary_pos_emb arithmetic with every
// bf16 rounding of its five elementwise launches per tensor reproduced (bit-identical), reading the [batch, tokens, heads, dim]
// projection output in place and writing [batch, heads, tokens, dim].
#include <cstdio>

#include "mxq_quant_core.cuh"
#include "mxq_rope_core.cuh"

namespace mxq {
namespace glue {

constexpr int kNormThreads = 256;
constexpr int MAX_CHUNKS = 4;  // 16-element chunks per thread: hidden <= 16 * 256 * 4 = 16384

struct NormParams {
    const uint16_t* x; int64_t ldx;
    const uint16_t* res; int64_t ld_res;
    uint16_t* res_out; int64_t ld_res_out;
    const uint16_t* w;
    float eps;
    int64_t rows; int hidden;
    uint16_t* y; int64_t ldy;
    uint8_t* codes; uint8_t* scales; unsigned flags;
};

// one CTA per row; thread t owns the 16-element chunks t, t + 256, ... (two 128-bit loads each)
template <int ELEM, bool QUANT>
__global__ void __launch_bounds__(kNormThreads) rmsnorm_kernel(const NormParams p) {
    pdl_launch_dependents();
    pdl_wait();  // (launched with programmatic serialization: nothing the predecessor wrote is read before this)
    __shared__ float warp_sums[kNormThreads / 32];
    const int64_t row = blockIdx.x;
    const int n_chunks = p.hidden / 16;
    uint32_t v[MAX_CHUNKS][8];
    float ss = 0.0f;
#pragma unroll
    for (int i = 0; i < MAX_CHUNKS; ++i) {
        const int c = threadIdx.x + i * kNormThreads;
        if (c < n_chunks) {
            const uint4* px = reinterpret_cast<const uint4*>(p.x + row * p.ldx + c * 16);
            const uint4 a = px[0], b = px[1];
            v[i][0] = a.x; v[i][1] = a.y; v[i][2] = a.z; v[i][3] = a.w; v[i][4] = b.x; v[i][5] = b.y; v[i][6] = b.z; v[i][7] = b.w;
            if (p.res != nullptr) {  // h = bf16(x + residual): the residual stream the decoder layer carries on
                const uint4* pr = reinterpret_cast<const uint4*>(p.res + row * p.ld_res + c * 16);
                const uint4 ra = pr[0], rb = pr[1];
                const uint32_t r[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) v[i][j] = pack_bf16x2(bf16lo(v[i][j]) + bf16lo(r[j]), bf16hi(v[i][j]) + bf16hi(r[j]));
                if (p.res_out != nullptr) {
                    uint4* po = reinterpret_cast<uint4*>(p.res_out + row * p.ld_res_out + c * 16);
                    po[0] = make_uint4(v[i][0], v[i][1], v[i][2], v[i][3]);
                    po[1] = make_uint4(v[i][4], v[i][5], v[i][6], v[i][7]);
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float lo = bf16lo(v[i][j]), hi = bf16hi(v[i][j]);
                ss = fmaf(lo, lo, ss);
                ss = fmaf(hi, hi, ss);
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) ss += __shfl_xor_sync(0xFFFFFFFFu, ss, d);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = ss;
    __syncthreads();
    float total = 0.0f;
#pragma unroll
    for (int w = 0; w < kNormThreads / 32; ++w) total += warp_sums[w];
    const float rs = rsqrtf(total / (float)p.hidden + p.eps);
#pragma unroll
    for (int i = 0; i < MAX_CHUNKS; ++i) {
        const int c = threadIdx.x + i * kNormThreads;
        const bool live = c < n_chunks;
        uint32_t o[8];
        if (live) {
            const uint4* pw = reinterpret_cast<const uint4*>(p.w + c * 16);
            const uint4 wa = pw[0], wb = pw[1];
            const uint32_t wt[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
            for (int j = 0; j < 8; ++j)  // weight * bf16(x * rsqrt(var + eps)), the product rounded to bf16 again
                o[j] = pack_bf16x2(bf16lo(wt[j]) * round_bf16(bf16lo(v[i][j]) * rs), bf16hi(wt[j]) * round_bf16(bf16hi(v[i][j]) * rs));
            if (p.y != nullptr) {
                uint4* py = reinterpret_cast<uint4*>(p.y + row * p.ldy + c * 16);
                py[0] = make_uint4(o[0], o[1], o[2], o[3]);
                py[1] = make_uint4(o[4], o[5], o[6], o[7]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = 0;
        }
        if constexpr (QUANT) {
            if (i * kNormThreads >= n_chunks) break;  // (uniform over the CTA)
            // K1 with 16 elements per thread: the two lanes of an MX block (consecutive chunks) share the block maximum; every
            // lane of the warp takes part in the shuffle, chunks past the row end carry zeros and store nothing
            uint32_t m = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) m = umax16x2(m, o[j] & 0x7FFF7FFFu);
            m = max(m & 0xFFFFu, m >> 16);
            m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, 1));
            const int s = shared_exp_from_maxE<ELEM>((int)(m >> 7));
            constexpr int NO = (ELEM == MXQ_ELEM_E2M1) ? 2 : 4;
            uint32_t q[NO];
            if (s != 255) convert_words<ELEM, 8>(o, s, q);
            else nanblock_words<ELEM, 8>(o, (p.flags & MXQ_FLAG_HW_EXACT) != 0, q);
            if (live) {
                const int64_t row_codes = (ELEM == MXQ_ELEM_E2M1) ? p.hidden / 2 : p.hidden;
                uint8_t* pc = p.codes + row * row_codes + (int64_t)c * (NO * 4);
                if constexpr (NO == 2) *reinterpret_cast<uint2*>(pc) = make_uint2(q[0], q[1]);
                else *reinterpret_cast<uint4*>(pc) = make_uint4(q[0], q[1], q[2], q[3]);
                if ((c & 1) == 0) p.scales[row * (p.hidden / 32) + (c >> 1)] = (uint8_t)s;
            }
        }
    }
}

struct RopeParams {
    const uint16_t* in[3]; uint16_t* out[3];  // q, k and (optional, unrotated) v
    int64_t in_tok_stride[3], in_batch_stride[3];
    int64_t out_batch_stride[3], out_head_stride[3], out_tok_stride[3];
    int heads[3];
    const uint16_t* cos; const uint16_t* sin;
    int64_t cs_batch_stride, cs_tok_stride;
    int64_t batch, tokens; int head_dim;
};

// one thread = 8 elements of the first half of a head and their 8 partners in the second half
__global__ void __launch_bounds__(256) rope_kernel(const RopeParams p) {
    pdl_launch_dependents();
    pdl_wait();  // (launched with programmatic serialization: nothing the predecessor wrote is read before this)
    const int half_chunks = p.head_dim / 16;  // 8-element chunks per half head
    const int64_t n0 = p.batch * p.tokens * p.heads[0] * half_chunks, n1 = p.batch * p.tokens * p.heads[1] * half_chunks;
    const int64_t n2 = p.in[2] != nullptr ? p.batch * p.tokens * p.heads[2] * half_chunks : 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n0 + n1 + n2; i += (int64_t)gridDim.x * blockDim.x) {
        const int which = i >= n0 + n1 ? 2 : (i >= n0 ? 1 : 0);
        int64_t r = which == 2 ? i - n0 - n1 : (which ? i - n0 : i);
        const int c = (int)(r % half_chunks); r /= half_chunks;
        const int h = (int)(r % p.heads[which]); r /= p.heads[which];
        const int64_t t = r % p.tokens, b = r / p.tokens;
        const uint16_t* src = p.in[which] + b * p.in_batch_stride[which] + t * p.in_tok_stride[which] + (int64_t)h * p.head_dim + c * 8;
        const uint16_t* pc = p.cos + b * p.cs_batch_stride + t * p.cs_tok_stride + c * 8;
        const uint16_t* ps = p.sin + b * p.cs_batch_stride + t * p.cs_tok_stride + c * 8;
        const int hd2 = p.head_dim / 2;
        uint16_t* dst = p.out[which] + b * p.out_batch_stride[which] + (int64_t)h * p.out_head_stride[which] + t * p.out_tok_stride[which] + c * 8;
        if (which == 2) {  // the value heads: a plain copy into their (cache) layout
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
            *reinterpret_cast<uint4*>(dst + hd2) = *reinterpret_cast<const uint4*>(src + hd2);
            continue;
        }
        const uint4 x1 = *reinterpret_cast<const uint4*>(src), x2 = *reinterpret_cast<const uint4*>(src + hd2);
        const uint4 c1 = *reinterpret_cast<const uint4*>(pc), c2 = *reinterpret_cast<const uint4*>(pc + hd2);
        const uint4 s1 = *reinterpret_cast<const uint4*>(ps), s2 = *reinterpret_cast<const uint4*>(ps + hd2);
        const uint32_t a1[4] = {x1.x, x1.y, x1.z, x1.w}, a2[4] = {x2.x, x2.y, x2.z, x2.w};
        const uint32_t k1[4] = {c1.x, c1.y, c1.z, c1.w}, k2[4] = {c2.x, c2.y, c2.z, c2.w};
        const uint32_t z1[4] = {s1.x, s1.y, s1.z, s1.w}, z2[4] = {s2.x, s2.y, s2.z, s2.w};
        uint32_t o1[4], o2[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            o1[j] = rope_first_half(a1[j], a2[j], k1[j], z1[j]);
            o2[j] = rope_second_half(a2[j], a1[j], k2[j], z2[j]);
        }
        *reinterpret_cast<uint4*>(dst) = make_uint4(o1[0], o1[1], o1[2], o1[3]);
        *reinterpret_cast<uint4*>(dst + hd2) = make_uint4(o2[0], o2[1], o2[2], o2[3]);
    }
}

// K5c heads_quantize_kernel: the attention output as the MX activation of o_proj.  The attention kernel leaves [batch, heads, tokens,
// head_dim]; the reference transposes to [batch, tokens, heads * head_dim] (a copy, torchmx/layers/mx_llama_attention.py:245-247) and
// o_proj quantizes on entry (mx_linear.py:63-66).  An MX block (32 consecutive channels) lies inside one head, so the codes can be
// produced straight from the [b, h, t, d] layout: one thread per block, K1's arithmetic, stores in [b, t, h * d] order.
template <int ELEM>
__global__ void __launch_bounds__(256) heads_quantize_kernel(const uint16_t* __restrict__ src, uint8_t* __restrict__ codes, uint8_t* __restrict__ scales,
                                                             int64_t n_blocks, int heads, int64_t tokens, int dblocks, uint32_t flags) {
    pdl_launch_dependents();
    pdl_wait();  // (launched with programmatic serialization: nothing the predecessor wrote is read before this)
    const int64_t o = (int64_t)blockIdx.x * 256 + threadIdx.x;  // block index in output order: ((b * T + t) * H + h) * dblocks + db
    if (o >= n_blocks) return;
    const int db = (int)(o % dblocks);
    int64_t r = o / dblocks;
    const int h = (int)(r % heads); r /= heads;
    const int64_t t = r % tokens, b = r / tokens;
    const uint8_t* p = reinterpret_cast<const uint8_t*>(src) + ((((b * heads + h) * tokens + t) * dblocks + db) * 64);
    uint32_t w[16];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const u32x8 v = ldg256_stream(p + 32 * j);
#pragma unroll
        for (int k = 0; k < 8; ++k) w[8 * j + k] = v.v[k];
    }
    constexpr int NO = (ELEM == MXQ_ELEM_E2M1) ? 4 : 8;
    uint32_t out[NO];
    const int sc = quantize_block32<ELEM>(w, (flags & MXQ_FLAG_HW_EXACT) != 0, out);
    uint8_t* dst = codes + o * (NO * 4);
    if constexpr (NO == 4) stg128_stream(dst, make_uint4(out[0], out[1], out[2], out[3]));
    else {
        u32x8 q;
#pragma unroll
        for (int k = 0; k < 8; ++k) q.v[k] = out[k];
        stg256_stream(dst, q);
    }
    scales[o] = (uint8_t)sc;
}

// K5d transposed_quantize_kernel: the value heads as the MX operand of P.V.  The reference quantizes V along the SEQUENCE axis
// (torchmx/layers/mx_llama_attention.py:205-212: value_states.transpose(-2, -1) -> to_mx -> transpose back), i.e. an MX block is
// 32 consecutive key positions of one (head, channel); as aten ops that is a strided copy of the whole value cache
// ([b, h, kv, d] -> [b, h, d, kv], 38 us per layer at batch 32 x 256 keys) followed by K1.  Here a CTA loads a 128-key x 64-channel
// tile with coalesced 16-byte loads, and each thread then quantizes ONE block -- 32 keys of one channel, gathered from shared
// memory -- with K1's arithmetic and stores its 32 codes contiguously in the [b, h, d, kv] layout: the transposed bf16 tensor is
// never written.  Same codes and scales as the two-step path, bit for bit.
struct TransposedQuantParams {
    const uint16_t* x; int64_t s0, s1, sr;  // x[i0][i1][r][c] at x + i0 * s0 + i1 * s1 + r * sr + c (elements)
    int64_t n1, rows, cols;
    uint8_t* codes; uint8_t* scales; unsigned flags;
};

template <int ELEM>
__global__ void __launch_bounds__(256) transposed_quantize_kernel(const TransposedQuantParams p) {
    pdl_launch_dependents();
    pdl_wait();  // (launched with programmatic serialization: nothing the predecessor wrote is read before this)
    constexpr int TR = 128, TC = 64;
    __shared__ __align__(16) uint16_t tile[TR][TC + 8];  // (+8: rows stay 16-byte aligned, column reads of a warp hit 16 distinct words)
    const int64_t slice = blockIdx.z;
    const int64_t i0 = slice / p.n1, i1 = slice % p.n1;
    const int64_t r0 = (int64_t)blockIdx.y * TR, c0 = (int64_t)blockIdx.x * TC;
    const uint16_t* src = p.x + i0 * p.s0 + i1 * p.s1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int v = threadIdx.x + i * 256;  // 16-byte vector: row v / 8, columns 8 * (v % 8) ..
        const int r = v >> 3, c8 = (v & 7) * 8;
        uint4 val = make_uint4(0, 0, 0, 0);
        if (r0 + r < p.rows && c0 + c8 < p.cols) val = *reinterpret_cast<const uint4*>(src + (r0 + r) * p.sr + c0 + c8);
        *reinterpret_cast<uint4*>(&tile[r][c8]) = val;
    }
    __syncthreads();
    const int c = threadIdx.x & (TC - 1), rb = threadIdx.x >> 6;  // channel, 32-key block within the tile
    if (c0 + c >= p.cols || r0 + rb * 32 >= p.rows) return;
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) w[i] = (uint32_t)tile[rb * 32 + 2 * i][c] | ((uint32_t)tile[rb * 32 + 2 * i + 1][c] << 16);
    constexpr int NO = (ELEM == MXQ_ELEM_E2M1) ? 4 : 8;
    uint32_t out[NO];
    const int sc = quantize_block32<ELEM>(w, (p.flags & MXQ_FLAG_HW_EXACT) != 0, out);
    const int64_t blk = (slice * p.cols + c0 + c) * (p.rows / 32) + (r0 / 32 + rb);  // block index in [.., channel, key block] order
    uint8_t* dst = p.codes + blk * (NO * 4);
    if constexpr (NO == 4) *reinterpret_cast<uint4*>(dst) = make_uint4(out[0], out[1], out[2], out[3]);
    else {
        *reinterpret_cast<uint4*>(dst) = make_uint4(out[0], out[1], out[2], out[3]);
        *reinterpret_cast<uint4*>(dst + 16) = make_uint4(out[4], out[5], out[6], out[7]);
    }
    p.scales[blk] = (uint8_t)sc;
}

}  // namespace glue

int launch_heads_quantize(const void* src, int64_t batch, int64_t heads, int64_t tokens, int64_t head_dim, int elem, unsigned flags, void* codes,
                          uint8_t* scales, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace glue;
    if (head_dim % 32 || ((uintptr_t)src % 32) || ((uintptr_t)codes % 32) || heads > 0x7FFFFFFF) {
        snprintf(msg, msg_len, "needs head_dim %% 32 == 0 and 32-byte aligned tensors");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    const int64_t n_blocks = batch * heads * tokens * (head_dim / 32);
    const int64_t grid = (n_blocks + 255) / 256;
    if (grid > 0x7FFFFFFF) { snprintf(msg, msg_len, "too many blocks"); return MXQ_ERR_UNSUPPORTED_SHAPE; }
#define MXQ_HQ_CASE(E) case E: launch_pdl(heads_quantize_kernel<E>, dim3((unsigned)grid), dim3(256), 0, stream, (const uint16_t*)src, (uint8_t*)codes, scales, n_blocks, (int)heads, tokens, (int)(head_dim / 32), (uint32_t)flags); break;
    switch (elem) {
        MXQ_HQ_CASE(MXQ_ELEM_E4M3) MXQ_HQ_CASE(MXQ_ELEM_E3M2) MXQ_HQ_CASE(MXQ_ELEM_E2M3) MXQ_HQ_CASE(MXQ_ELEM_E2M1) MXQ_HQ_CASE(MXQ_ELEM_INT8) MXQ_HQ_CASE(MXQ_ELEM_E5M2)
    default: snprintf(msg, msg_len, "unknown element type %d", elem); return MXQ_ERR_INVALID;
    }
#undef MXQ_HQ_CASE
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

int launch_rmsnorm(const mxq_rmsnorm_args_t* a, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace glue;
    const bool quant = a->codes != nullptr;
    auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
    if (a->hidden % 32 || a->hidden > 16 * kNormThreads * MAX_CHUNKS || !al16(a->x) || (a->ldx % 8) || !al16(a->weight) ||
        (a->residual && (!al16(a->residual) || (a->ld_res % 8))) || (a->residual_out && (!al16(a->residual_out) || (a->ld_res_out % 8))) ||
        (a->y && (!al16(a->y) || (a->ldy % 8))) || (quant && !al16(a->codes))) {
        snprintf(msg, msg_len, "needs hidden %% 32 == 0, hidden <= %d and 16-byte aligned rows", 16 * kNormThreads * MAX_CHUNKS);
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    if (a->rows > 0x7FFFFFFF) { snprintf(msg, msg_len, "too many rows"); return MXQ_ERR_UNSUPPORTED_SHAPE; }
    NormParams p;
    p.x = (const uint16_t*)a->x; p.ldx = a->ldx;
    p.res = (const uint16_t*)a->residual; p.ld_res = a->ld_res;
    p.res_out = (uint16_t*)a->residual_out; p.ld_res_out = a->ld_res_out;
    p.w = (const uint16_t*)a->weight; p.eps = a->eps; p.rows = a->rows; p.hidden = (int)a->hidden;
    p.y = (uint16_t*)a->y; p.ldy = a->ldy;
    p.codes = (uint8_t*)a->codes; p.scales = a->scales; p.flags = a->flags;
    const unsigned grid = (unsigned)a->rows;
#define MXQ_NORM_CASE(E) case E: launch_pdl(rmsnorm_kernel<E, true>, dim3(grid), dim3(kNormThreads), 0, stream, p); break;
    if (!quant) {
        launch_pdl(rmsnorm_kernel<MXQ_ELEM_E4M3, false>, dim3(grid), dim3(kNormThreads), 0, stream, p);
    } else {
        switch (a->elem) {
            MXQ_NORM_CASE(MXQ_ELEM_E4M3) MXQ_NORM_CASE(MXQ_ELEM_E3M2) MXQ_NORM_CASE(MXQ_ELEM_E2M3) MXQ_NORM_CASE(MXQ_ELEM_E2M1) MXQ_NORM_CASE(MXQ_ELEM_INT8)
            MXQ_NORM_CASE(MXQ_ELEM_E5M2)
        default: snprintf(msg, msg_len, "unknown element type %d", a->elem); return MXQ_ERR_INVALID;
        }
    }
#undef MXQ_NORM_CASE
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

int launch_rope(const mxq_rope_args_t* a, int sm_count, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace glue;
    auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
    if (a->head_dim % 16 || a->head_dim <= 0 || !al16(a->q) || !al16(a->k) || !al16(a->q_out) || !al16(a->k_out) || !al16(a->cos) || !al16(a->sin) ||
        (a->q_tok_stride % 8) || (a->k_tok_stride % 8) || (a->q_batch_stride % 8) || (a->k_batch_stride % 8) || (a->cs_tok_stride % 8) || (a->cs_batch_stride % 8)) {
        snprintf(msg, msg_len, "needs head_dim %% 16 == 0 and 16-byte aligned heads");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    const bool has_v = a->v != nullptr;
    const int64_t out_strides[9] = {a->q_out_batch_stride, a->q_out_head_stride, a->q_out_tok_stride, a->k_out_batch_stride, a->k_out_head_stride,
                                    a->k_out_tok_stride, a->v_out_batch_stride, a->v_out_head_stride, a->v_out_tok_stride};
    for (int i = 0; i < 9; ++i)
        if (out_strides[i] % 8) { snprintf(msg, msg_len, "output strides must be multiples of 8 elements"); return MXQ_ERR_UNSUPPORTED_SHAPE; }
    if (has_v && (!a->v_out || !al16(a->v) || !al16(a->v_out) || (a->v_tok_stride % 8) || (a->v_batch_stride % 8))) {
        snprintf(msg, msg_len, "v needs v_out and 16-byte aligned heads");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    RopeParams p;
    p.in[0] = (const uint16_t*)a->q; p.in[1] = (const uint16_t*)a->k; p.in[2] = (const uint16_t*)a->v;
    p.out[0] = (uint16_t*)a->q_out; p.out[1] = (uint16_t*)a->k_out; p.out[2] = (uint16_t*)a->v_out;
    p.in_tok_stride[0] = a->q_tok_stride; p.in_tok_stride[1] = a->k_tok_stride; p.in_tok_stride[2] = a->v_tok_stride;
    p.in_batch_stride[0] = a->q_batch_stride; p.in_batch_stride[1] = a->k_batch_stride; p.in_batch_stride[2] = a->v_batch_stride;
    p.heads[0] = a->q_heads; p.heads[1] = a->k_heads; p.heads[2] = a->k_heads;
    for (int w = 0; w < 3; ++w) {  // 0 / 0 / 0 = contiguous [batch, heads, tokens, head_dim]
        const int64_t bs = out_strides[3 * w], hs = out_strides[3 * w + 1], ts = out_strides[3 * w + 2];
        const bool contiguous = bs == 0 && hs == 0 && ts == 0;
        p.out_tok_stride[w] = contiguous ? a->head_dim : ts;
        p.out_head_stride[w] = contiguous ? a->tokens * a->head_dim : hs;
        p.out_batch_stride[w] = contiguous ? (int64_t)p.heads[w] * a->tokens * a->head_dim : bs;
    }
    p.cos = (const uint16_t*)a->cos; p.sin = (const uint16_t*)a->sin;
    p.cs_batch_stride = a->cs_batch_stride; p.cs_tok_stride = a->cs_tok_stride;
    p.batch = a->batch; p.tokens = a->tokens; p.head_dim = a->head_dim;
    const int64_t n = a->batch * a->tokens * (int64_t)(a->q_heads + a->k_heads * (has_v ? 2 : 1)) * (a->head_dim / 16);
    // one item per thread up to 64 CTAs per SM (a 2048-token prefill of Llama-8B is 2560 CTAs: capped at 16 per SM some threads took
    // two items and the launch lasted as long as two)
    const int64_t want = (n + 255) / 256, cap = (int64_t)sm_count * 64;
    launch_pdl(rope_kernel, dim3((unsigned)(want < cap ? want : cap)), dim3(256), 0, stream, p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

int launch_transposed_quantize(const mxq_transposed_quantize_args_t* a, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace glue;
    if (a->rows % 32 || a->cols % 8 || ((uintptr_t)a->x % 16) || (a->s0 % 8) || (a->s1 % 8) || (a->row_stride % 8) || ((uintptr_t)a->codes % 16)) {
        snprintf(msg, msg_len, "needs rows %% 32 == 0, cols %% 8 == 0 and 16-byte aligned rows");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    const int64_t slices = a->n0 * a->n1, gy = (a->rows + 127) / 128, gx = (a->cols + 63) / 64;
    if (slices == 0 || a->rows == 0 || a->cols == 0) return MXQ_OK;
    if (slices > 65535 || gy > 65535 || gx > 0x7FFFFFFF) { snprintf(msg, msg_len, "too many slices / rows"); return MXQ_ERR_UNSUPPORTED_SHAPE; }
    TransposedQuantParams p;
    p.x = (const uint16_t*)a->x; p.s0 = a->s0; p.s1 = a->s1; p.sr = a->row_stride;
    p.n1 = a->n1; p.rows = a->rows; p.cols = a->cols;
    p.codes = (uint8_t*)a->codes; p.scales = a->scales; p.flags = a->flags;
    const dim3 grid((unsigned)gx, (unsigned)gy, (unsigned)slices);
#define MXQ_TQ_CASE(E) case E: launch_pdl(transposed_quantize_kernel<E>, grid, dim3(256), 0, stream, p); break;
    switch (a->elem) {
        MXQ_TQ_CASE(MXQ_ELEM_E4M3) MXQ_TQ_CASE(MXQ_ELEM_E3M2) MXQ_TQ_CASE(MXQ_ELEM_E2M3) MXQ_TQ_CASE(MXQ_ELEM_E2M1) MXQ_TQ_CASE(MXQ_ELEM_INT8) MXQ_TQ_CASE(MXQ_ELEM_E5M2)
    default: snprintf(msg, msg_len, "unknown element type %d", a->elem); return MXQ_ERR_INVALID;
    }
#undef MXQ_TQ_CASE
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

}  // namespace mxq
