/*
 * mxq.h -- C ABI of the B200-native MX quantize / dequantize / block-scaled GEMM library
 *          (libmxq.so, built from torchmx_b200/csrc by `python -m torchmx_b200.build`).
 *
 * This is the drop-in boundary for torchmx's hot path.  The reference implements the path as
 * two Python `torch.library.custom_op`s plus an aten override table; the entry points below are
 * what those op bodies bind to (see INTEGRATION.md for the ctypes stub a maintainer would add to
 * the reference).  Citations are relative to the reference repository root.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary;
 *   - all pointers are DEVICE pointers on `device` unless the name says `host`;
 *   - nothing is allocated or owned by the library: outputs are caller-allocated;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *     stream) and the call returns without synchronising;
 *   - `device` is the CUDA device ordinal the pointers live on (-1 = the calling thread's
 *     current device); the library saves/restores the thread's current device around the call,
 *     it never changes it for the caller (the reference is called from arbitrary Python
 *     threads: examples/quantized_llama_chat.py:123-129);
 *   - return value 0 = success; non-zero = error, message from mxq_last_error() (thread-local).
 *     The library never throws, aborts or exits.
 */
#ifndef MXQ_H_
#define MXQ_H_

#include <stdint.h>

#if defined(__GNUC__)
#define MXQ_API __attribute__((visibility("default")))
#else
#define MXQ_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* Element formats: torchmx/dtypes.py:34-92, looked up by name through
 * dtypes.STR_TO_SUPPORTED_ELEM_DTYPE (dtypes.py:161) because the op schemas carry a string
 * (torchmx/mx_tensor.py:39,52).  MXQ_E5M2 is an extension the reference does not have. */
typedef enum {
    MXQ_ELEM_E4M3 = 0, /* float8_e4m3  1 byte / element                                  */
    MXQ_ELEM_E3M2 = 1, /* float6_e3m2  1 byte / element, code in bits [5:0]               */
    MXQ_ELEM_E2M3 = 2, /* float6_e2m3  1 byte / element, code in bits [5:0]               */
    MXQ_ELEM_E2M1 = 3, /* float4_e2m1  2 elements / byte, even element in the HIGH nibble
                          (torchmx/utils.py:120-145)                                     */
    MXQ_ELEM_INT8 = 4, /* int8         1 byte / element, two's complement                 */
    MXQ_ELEM_E5M2 = 5  /* float8_e5m2  extension, parity unpinned                         */
} mxq_elem_t;

typedef enum {
    MXQ_HP_BF16 = 0, /* the only input dtype the reference accepts (mx_tensor.py:59-61)      */
    MXQ_HP_F32 = 1   /* dequantize target (mx_tensor.py:456-472); quantize input = extension */
} mxq_hp_t;

/* flags for mxq_quantize */
#define MXQ_FLAG_HW_EXACT 1u /* env MX_HARDWARE_EXACT_QUANTIZATION == "True"
                                (torchmx/env_variables.py:16, mx_tensor.py:80-90).  Only
                                observable in NaN-scale blocks: see DESIGN.md "hw_exact quirk" */
#define MXQ_FLAG_OPERAND_LAYOUT 2u /* mxq_quantize only; float4_e2m1 / float6_* elements, block 32, bf16 source, 32-byte aligned
                                      pointers (else MXQ_ERR_UNSUPPORTED_SHAPE): `codes` receives the packed tensor-core operand
                                      stream (MXQ_OPERAND_E2M1_PACKED / MXQ_OPERAND_E3M2_PACKED / MXQ_OPERAND_E2M3_PACKED, what
                                      mxq_pack_operand makes of the reference-layout codes: n/2 or 3n/4 bytes) -- the form
                                      mxq_gemm consumes -- so an activation quantized on entry to a linear
                                      (torchmx/layers/mx_linear.py:63-66) needs no second launch */

/*
 * quantize  <->  torchmx::quantize_mx  (torchmx/mx_tensor.py:36-96)
 *   + get_e8m0_shared_exponent                          (torchmx/mx_quantization_utils.py:502-558)
 *   + quantize_mx_with_e8m0_shared_exponent_{simulated,hw_exact}   (:435-499, :253-412)
 *   + pack_uint4 for float4_e2m1                        (torchmx/utils.py:120-145)
 *
 * src    : n_blocks * block_size contiguous high-precision elements, blocks along the
 *          innermost (contiguous) axis -- the reference requires a contiguous tensor whose last
 *          dim is a multiple of block_size (mx_tensor.py:62, 68-70), so the tensor is a flat
 *          run of blocks.
 * codes  : n_blocks*block_size bytes (n_blocks*block_size/2 for MXQ_ELEM_E2M1; the total element
 *          count must then be even, utils.py:143).  int8 codes are two's complement bytes.
 * scales : n_blocks E8M0 bytes; 255 = NaN (dtypes.py:183).
 */
MXQ_API int mxq_quantize(const void *src, int src_dtype /* mxq_hp_t */, int64_t n_blocks, int block_size,
                 int elem /* mxq_elem_t */, unsigned flags, void *codes, uint8_t *scales,
                 int device, void *stream);

/*
 * dequantize (flat)  <->  torchmx::dequantize_mx with block_dim == last dim and contiguous
 * operands (torchmx/mx_tensor.py:123-164; decode mx_quantization_utils.py:93-146; scale
 * :415-432).  dst: n_blocks*block_size elements of dst_dtype.
 */
MXQ_API int mxq_dequantize(const void *codes, const uint8_t *scales, int64_t n_blocks, int block_size,
                   int elem, int dst_dtype /* mxq_hp_t */, void *dst, int device, void *stream);

/*
 * dequantize (strided)  <->  the same op for every other case the reference accepts: `data_lp`
 * a permuted / expanded view, `block_dim` != last (mx_tensor.py:157-162; exercised by
 * tests/test_mx_tensor.py:195-356).
 *   ndim          : 1..MXQ_MAX_DIMS
 *   sizes         : LOGICAL (unpacked) element counts per dim
 *   code_strides  : strides of data_lp in BYTES-OF-CODE units per dim; for MXQ_ELEM_E2M1 the
 *                   blocked dim is packed, i.e. logical index i along block_dim lives in byte
 *                   i/2 (high nibble when i is even)
 *   scale_strides : strides of shared_exp_e8m0 per dim (its size along block_dim is
 *                   sizes[block_dim]/block_size)
 *   dst           : C-contiguous in the logical shape (what FromMXConstrFunc returns,
 *                   mx_tensor.py:323)
 */
#define MXQ_MAX_DIMS 6
MXQ_API int mxq_dequantize_strided(const void *codes, const uint8_t *scales, int ndim, const int64_t *sizes,
                           const int64_t *code_strides, const int64_t *scale_strides, int block_dim,
                           int block_size, int elem, int dst_dtype, void *dst, int device,
                           void *stream);

/*
 * MX matmul  <->  the aten overrides torchmx/ops.py:29-41 (linear), :60-68 (mm / matmul),
 * :99-107 (bmm), :110-119 (addmm): D[b] = A[b] * B[b]^T (+ bias), A: [M,K] codes, B: [N,K]
 * codes, both blocked along K with block_size 32 and E8M0 scales [M,K/32] / [N,K/32];
 * D: [M,N] bf16.  The reference dequantizes both operands and calls a bf16 GEMM; this entry
 * point runs a tcgen05 block-scaled MMA (kind::mxf8f6f4) instead.
 *   a_codes / b_codes : K-major, one byte per element holding an E4M3-container code (fp6 / fp4
 *                       reference codes are transcoded exactly with mxq_transcode_to_e4m3)
 *   lda / ldb         : row strides in bytes (multiples of 16); batch strides in bytes
 *   sfa / sfb         : row-major [rows, K/32] E8M0, row stride ld_sf, batch stride given
 *   bias              : NULL or N bf16 values added to every row (aten.addmm / linear bias)
 *   d                 : bf16 [M,N], row stride ldd elements, batch stride in elements
 * Returns MXQ_ERR_UNSUPPORTED_SHAPE (2) when the shape cannot run on the tensor-core path
 * (K % 128 != 0, misaligned strides); the caller then uses the dequantize path.
 */
typedef struct {
    const void *a_codes; const uint8_t *sfa; int64_t lda, ld_sfa, a_batch_stride, sfa_batch_stride;
    const void *b_codes; const uint8_t *sfb; int64_t ldb, ld_sfb, b_batch_stride, sfb_batch_stride;
    const void *bias;
    void *d; int64_t ldd, d_batch_stride;
    int64_t batch, M, N, K;
    int a_format, b_format; /* MXQ_OPERAND_*: how a_codes / b_codes are stored (0 = E4M3 container bytes) */
    /* Fused row-parallel all-reduce (tensor parallelism over NVLink / NVSwitch): when non-NULL, `d_multicast` is the
     * MULTICAST address of a symmetric [M, N] bf16 buffer mapped on every rank of the group (ldd / d_batch_stride describe
     * it; `d` is ignored).  The epilogue does not store: it adds this rank's bf16 partial tile into the buffer of EVERY
     * rank with multimem.red (the reduction happens in the switch), so after all ranks' launches have completed and a
     * cross-rank barrier has passed, each rank's copy holds the sum.  The buffer must be zero on every rank before the
     * first launch that targets it; needs N % 8 == 0, a 16-byte aligned buffer and batch == 1. */
    void *d_multicast;
    /* Fused activation quantization (MXInferenceLinear.forward, torchmx/layers/mx_linear.py:63-94): when non-NULL, `x_bf16`
     * is the HIGH-PRECISION activation [M, K] (bf16, row stride ldx elements, 16-byte aligned rows) and a_codes / sfa are
     * ignored: the kernel computes quantize_mx(x, float8_e4m3, 32) itself, block by block, on its way into shared memory
     * (same arithmetic as mxq_quantize, bit-identical), so the activation never makes a round trip through HBM as codes and
     * the separate quantize launch disappears.  x_quant_flags = MXQ_FLAG_* of mxq_quantize.  Decode shapes only
     * (M <= 64, batch == 1); otherwise MXQ_ERR_UNSUPPORTED_SHAPE and the caller quantizes first. */
    const void *x_bf16; int64_t ldx; int x_quant_flags;
    /* MXQ_GEMM_* bits below (0 = defaults) */
    unsigned flags;
    /* decode kernel only: number of K splits per 128-row weight tile (a cluster of that many CTAs, <= 8); 0 = chosen by the
     * library.  Exposed so that tests can pin every split count; results are bit-reproducible per value. */
    int split_k;
} mxq_gemm_args_t;
/* The B operand (b_codes, sfb) is long-lived: nothing enqueued earlier on `stream` (or still running on the device) writes it.
 * True for a layer's pre-quantized weight and its cached operand shadow (torchmx/layers/mx_linear.py:21-59), false for
 * F.linear(to_mx(x), to_mx(w)) or a weight quantized on the fly (:68-92).  Only with this bit set may the decode kernel, which
 * is launched with programmatic stream serialization, request weight tiles before the preceding kernel has finished. */
#define MXQ_GEMM_B_STATIC 1u
/* keep the 256x256 CTA-pair tiles even when they would under-fill the GPU (the library otherwise prefers 128x128 tiles there) */
#define MXQ_GEMM_WIDE_TILES 2u
/* launch without programmatic stream serialization */
#define MXQ_GEMM_NO_PDL 4u
/* fp4 x fp4 (both operands MXQ_OPERAND_E2M1_PACKED): stay on kind::mxf8f6f4 instead of the double-rate kind::mxf4 kernel */
#define MXQ_GEMM_NO_MXF4 8u
MXQ_API int mxq_gemm(const mxq_gemm_args_t *args, int device, void *stream);

/*
 * MX matmul, general operands  <->  the same aten overrides (torchmx/ops.py:29-41, 60-68, 99-119) for every operand pair
 * mxq_gemm cannot take: int8 elements (examples/quantized_llama_chat.py:41-71), block sizes other than 32
 * (tests/layers/test_mx_linear.py:64-114 uses 2), blocks that do not run along the contraction (Readme.md:32-44: B blocked
 * along N), padded tensors, K % 128 != 0, arbitrary strides / expanded batches.  It is the reference's own recipe --
 * dequantize both operands to bf16 exactly as mxq_dequantize does, bf16 x bf16 products, fp32 accumulation, one rounding to
 * bf16 -- fused into one kernel (tcgen05.mma kind::f16 on tiles dequantized into shared memory), so only the accumulation
 * order differs from dequantize-then-matmul.
 *
 * An operand is the LOGICAL matrix X[batch][rows][K] (A: rows = M; B: rows = N, i.e. D = A * B^T) addressed through strides:
 *   element (r, k) has its code byte at  codes + b*batch_stride + r*row_stride + k*k_stride ;
 *   MXQ_ELEM_E2M1 is packed two per byte along the BLOCKED axis (high nibble = even index, torchmx/utils.py:145): the index
 *   along that axis is halved (k >> 1 when blocked_along_k, else r >> 1) before the stride is applied;
 *   its scale byte is at  scales + b*sbatch_stride + r*srow_stride + (k / block_size)*sk_stride  when blocked_along_k,
 *   else at  scales + b*sbatch_stride + (r / block_size)*srow_stride + k*sk_stride.
 * Any stride may be 0 (expanded dims) or describe a transposed view.  K is the logical extent (padding excluded).
 * bias: NULL or N bf16; d: bf16 [batch][M][N], row stride ldd, batch stride d_batch_stride (elements).
 */
typedef struct {
    const void *codes; const uint8_t *scales;
    int64_t row_stride, k_stride, batch_stride;
    int64_t srow_stride, sk_stride, sbatch_stride;
    int elem /* mxq_elem_t */; int block_size; int blocked_along_k;
} mxq_operand_t;
typedef struct {
    mxq_operand_t a, b;
    const void *bias;
    void *d; int64_t ldd, d_batch_stride;
    int64_t batch, M, N, K;
} mxq_gemm_dequant_args_t;
MXQ_API int mxq_gemm_dequant(const mxq_gemm_dequant_args_t *args, int device, void *stream);

/* Operand storage formats of mxq_gemm.  The packed formats are what the sm_100a TMA unit expands on the fly
 * (CU_TENSOR_MAP_DATA_TYPE_16U4_ALIGN16B / 16U6_ALIGN16B) and kind::mxf8f6f4 consumes natively, so a 4-bit operand
 * costs 0.5 B and a 6-bit operand 0.75 B of HBM traffic per element instead of 1 B:
 *   MXQ_OPERAND_E4M3_BYTES  : one E4M3 byte per element, row stride lda/ldb bytes (multiple of 16)
 *   MXQ_OPERAND_E2M1_PACKED : two e2m1 codes per byte, element 2i in the LOW nibble (the reference keeps the even
 *                             element in the HIGH nibble, torchmx/utils.py:145 -- mxq_pack_operand swaps them)
 *   MXQ_OPERAND_E3M2_PACKED / MXQ_OPERAND_E2M3_PACKED : 6-bit codes as a little-endian bit stream, element i in bits
 *                             [6i, 6i+6) of its row
 * Packed operands need a 32-byte aligned base, row / batch strides that are multiples of 32 bytes and K % 128 == 0. */
#define MXQ_OPERAND_E4M3_BYTES 0
#define MXQ_OPERAND_E2M1_PACKED 1
#define MXQ_OPERAND_E3M2_PACKED 2
#define MXQ_OPERAND_E2M3_PACKED 3
#define MXQ_OPERAND_E5M2_BYTES 4 /* one E5M2 byte per element (the float8_e5m2 extension element type) */

/* reference-layout element codes (MXQ_ELEM_E3M2 / E2M3: one byte each; MXQ_ELEM_E2M1: packed, even element high) ->
 * the packed operand format above for that element type; n elements in, n*bits/8 bytes out.  Exact (a permutation of
 * bits).  n_elements must be a multiple of 16. */
MXQ_API int mxq_pack_operand(const void *codes, int elem, int64_t n_elements, void *out_packed, int device, void *stream);

/* the inverse: packed operand stream -> reference-layout element codes (what MXTensor._data and a reference state_dict hold,
 * torchmx/mx_tensor.py:495-520), so a weight can live in HBM / on disk ONLY in its dense 4 / 6-bit form (0.5 / 0.75 B per
 * element instead of the reference's 0.5 / 1 B) and still be handed back to the reference bit-for-bit. */
MXQ_API int mxq_unpack_operand(const void *packed, int elem, int64_t n_elements, void *out_codes, int device, void *stream);

/* exact re-encoding of reference-layout element codes as E4M3 bytes (every e3m2 / e2m3 / e2m1
 * value is representable in e4m3): n elements in, n bytes out; MXQ_ELEM_E2M1 input is packed. */
MXQ_API int mxq_transcode_to_e4m3(const void *codes, int elem, int64_t n_elements, void *out_e4m3,
                          int device, void *stream);

/*
 * attention probabilities  <->  torchmx/layers/mx_llama_attention.py:214-239: the chain between the two MX matmuls of
 * MXInferenceLlamaAttention (and its Qwen2 twin),
 *     w = scores / sqrt(head_dim);  w = w + mask;  w = softmax(w, -1, dtype=float32).to(bfloat16);  to_mx(w, elem, 32)
 * as ONE pass over the scores.  `scores` is the contiguous bf16 [batch, heads, q_len, kv_len] output of the Q.K^T matmul;
 * every bf16 rounding of the chain is reproduced, the quantization is mxq_quantize's.
 *   scaling     : the fp32 factor the chain multiplies by (CUDA evaluates `x / sqrt(d)` as x * (1.0f / sqrtf(d)))
 *   mask        : NULL or an additive bf16 mask, element strides over (batch, head, query row) given, kv stride 1;
 *                 stride 0 broadcasts
 *   causal      : non-zero also hides kv index j > q + (kv_len - q_len) (what sdpa's is_causal does when no mask is given)
 *   codes/scales: [rows, kv_len] (kv_len/2 for MXQ_ELEM_E2M1) / [rows, kv_len/32], rows = batch*heads*q_len
 * kv_len must be a multiple of 32 and <= 32768; scores and codes 32-byte aligned; else MXQ_ERR_UNSUPPORTED_SHAPE.
 */
typedef struct {
    const void *scores;
    int64_t batch, heads, q_len, kv_len;
    float scaling;
    const void *mask; int64_t mask_stride_b, mask_stride_h, mask_stride_q;
    int causal;
    int elem /* mxq_elem_t */; unsigned flags /* MXQ_FLAG_* */;
    void *codes; uint8_t *scales;
} mxq_softmax_args_t;
MXQ_API int mxq_softmax_quantize(const mxq_softmax_args_t *args, int device, void *stream);

/*
 * bf16 GEMM on the tensor cores (tcgen05 kind::f16), D[b] = A[b] B[b]^T (+ bias): the second half of the reference's own recipe --
 * dequantize both operands, then a bf16 matmul (torchmx/ops.py:29-41, 60-68, 99-119) -- for LARGE contractions of operand pairs the
 * block-scaled MMA cannot take.  mxq_gemm_dequant dequantizes inside the GEMM, i.e. once per output tile; above a few hundred
 * rows and columns it is cheaper to dequantize each operand once (mxq_dequantize / mxq_dequantize_strided into scratch) and multiply
 * the bf16 matrices with the same MMA loop and epilogue fed by TMA.  No library GEMM is involved.
 *   a : bf16 [batch, M, K], K contiguous, row stride lda and batch stride in ELEMENTS (multiples of 8), 16-byte aligned
 *   b : bf16 [batch, N, K] likewise;  bias: NULL or N bf16;  d: bf16 [batch, M, N], ldd / d_batch_stride in elements
 *   K % 8 == 0, else MXQ_ERR_UNSUPPORTED_SHAPE (the caller uses mxq_gemm_dequant)
 */
MXQ_API int mxq_gemm_bf16(const void *a, int64_t lda, int64_t a_batch_stride, const void *b, int64_t ldb, int64_t b_batch_stride, const void *bias,
                  void *d, int64_t ldd, int64_t d_batch_stride, int64_t batch, int64_t M, int64_t N, int64_t K, int device, void *stream);

/*
 * MX attention as one kernel  <->  the attention of the reference's MX blocks (torchmx/layers/mx_llama_attention.py:195-243,
 * mx_qwen2_attention.py): scores = Q_mx K_mx^T, P = quantize_mx(softmax(scores * scaling + mask)), out = P_mx V_mx -- with
 * neither the scores nor the codes of P written to device memory.  Both contractions run as tcgen05 block-scaled MMAs; every
 * rounding step between them is mxq_softmax_quantize's, so P's codes and scales are the ones that entry point produces from
 * the bf16 scores, bit for bit (`p_codes` / `p_scales`, when given, receive them: the block's attention weights).
 *   q_codes  : [batch, heads, q_len, 128] one byte per element (MXQ_OPERAND_E4M3_BYTES or _E5M2_BYTES; fp6 / fp4 reference codes
 *              transcoded exactly with mxq_transcode_to_e4m3), contiguous; q_scales: [batch, heads, q_len, 4] E8M0
 *   k_codes  : [batch, kv_heads, kv_len, 128], k_scales [batch, kv_heads, kv_len, 4]; query head h reads key / value head
 *              h / (heads / kv_heads) (grouped-query attention: no repeated copies)
 *   vt_codes : [batch, kv_heads, 128, kv_len] -- V quantized along the key axis, as the reference does it (quantize the
 *              transpose, :209-213); vt_scales [batch, kv_heads, 128, kv_len / 32]
 *   mask     : NULL or additive bf16, element (b, h, q, j) at mask + b*stride_b + h*stride_h + q*stride_q + j (0 strides broadcast)
 *   causal   : additionally hide key j > q + (kv_len - q_len); key chunks no row of a tile can see are skipped
 *   out      : bf16, element (b, h, q, d) at out + b*out_batch_stride + h*out_head_stride + q*out_row_stride + d (so the caller
 *              picks [b, h, q, d] or the transposed [b, q, h, d] the reference produces next, :245)
 *   p_elem   : element type of P (any floating-point mxq_elem_t), flags: MXQ_FLAG_*
 * MXQ_ERR_UNSUPPORTED_SHAPE unless head_dim == 128, kv_len % 32 == 0, q_len <= kv_len <= MXQ_FLASH_MAX_KV (masked or not).  Rows
 * of any length add their block sums in mxq_softmax_quantize's order, including the lengths that entry point itself refuses.
 *   kv_pitch : 0, or the key capacity of K / V buffers of which only the first kv_len keys exist (a KV cache read in place):
 *              k_codes [batch, kv_heads, kv_pitch, 128], k_scales [.., kv_pitch, 4], vt_codes [batch, kv_heads, 128, kv_pitch],
 *              vt_scales [.., kv_pitch / 32]; 1 <= q_len <= kv_len <= kv_pitch <= MXQ_FLASH_MAX_KV and kv_pitch % 128 == 0, else
 *              MXQ_ERR_INVALID.  kv_len may be any value.  With n = kv_len rounded up to a multiple of 128, the result is, bit
 *              for bit, that of kv_pitch 0 on contiguous copies of the first n keys (zero codes past kv_len) with causal 0 and the
 *              mask mask' = the given mask (or zeros) with -inf on every key the causal rule hides and on every key >= kv_len
 *              (no mask at all when none is given, causal is 0 and kv_len == n).  p_codes / p_scales are then [.., n] /
 *              [.., n / 32].  No K code, K scale or V code at a position >= kv_len is read, nor the V scale of a block wholly
 *              past it.
 */
#define MXQ_FLASH_MAX_KV 131072
typedef struct {
    const void *q_codes; const uint8_t *q_scales; int q_format;
    const void *k_codes; const uint8_t *k_scales; int k_format;
    const void *vt_codes; const uint8_t *vt_scales; int v_format;
    int64_t batch, heads, kv_heads, q_len, kv_len; int head_dim;
    float scaling;
    const void *mask; int64_t mask_stride_b, mask_stride_h, mask_stride_q;
    int causal;
    int p_elem /* mxq_elem_t */; unsigned flags /* MXQ_FLAG_* */;
    void *out; int64_t out_batch_stride, out_head_stride, out_row_stride;
    void *p_codes; uint8_t *p_scales;
    int64_t kv_pitch;
} mxq_attention_args_t;
MXQ_API int mxq_flash_attention(const mxq_attention_args_t *args, int device, void *stream);

/*
 * SwiGLU gating + quantization  <->  the MLP block of the reference (torchmx/layers/mx_llama_attention.py:19-59 around
 * transformers' `down_proj(act_fn(gate_proj(x)) * up_proj(x))`) followed by the activation quantization on entry to down_proj
 * (torchmx/layers/mx_linear.py:63-66): codes, scales = quantize_mx(bf16(bf16(silu(gate)) * up), elem, 32) in one pass,
 * bit-identical to aten silu + aten mul + mxq_quantize.
 *   gate / up : bf16 [rows, cols], row strides ld_gate / ld_up in elements (>= cols, multiples of 16), 32-byte aligned bases;
 *               they may be column slices of one stacked gate+up projection output
 *   codes     : [rows, cols] (cols/2 for MXQ_ELEM_E2M1), scales: [rows, cols/32]; cols % 32 == 0
 */
MXQ_API int mxq_silu_mul_quantize(const void *gate, const void *up, int64_t rows, int64_t cols, int64_t ld_gate, int64_t ld_up,
                          int elem /* mxq_elem_t */, unsigned flags /* MXQ_FLAG_* */, void *codes, uint8_t *scales, int device, void *stream);

/*
 * (residual add +) RMSNorm (+ MX quantization)  <->  the activation every MX linear of a decoder layer receives: transformers'
 * LlamaRMSNorm / Qwen2RMSNorm output, which the reference quantizes on entry to q/k/v and to gate/up
 * (torchmx/layers/mx_linear.py:63-66) -- once per consuming layer; here once, inside the pass that normalises the row.
 *     h = x (+ residual, rounded to bf16; written to residual_out);  n = bf16(h * rsqrt(mean(h^2) + eps));  y = weight * n  (bf16)
 *     codes, scales = quantize_mx(y, elem, 32)        (same arithmetic as mxq_quantize, bit-identical given y)
 *   x, residual, residual_out, y : bf16 [rows, hidden], row strides in elements (multiples of 8), 16-byte aligned bases
 *   y may be NULL when only the quantized form is wanted; codes / scales may be NULL when only y is wanted
 *   hidden % 32 == 0 and hidden <= 16384, else MXQ_ERR_UNSUPPORTED_SHAPE (the caller runs the module and mxq_quantize)
 */
typedef struct {
    const void *x; int64_t ldx;
    const void *residual; int64_t ld_res;
    void *residual_out; int64_t ld_res_out;
    const void *weight; float eps;
    int64_t rows, hidden;
    void *y; int64_t ldy;
    void *codes; uint8_t *scales; int elem /* mxq_elem_t */; unsigned flags /* MXQ_FLAG_* */;
} mxq_rmsnorm_args_t;
MXQ_API int mxq_rmsnorm(const mxq_rmsnorm_args_t *args, int device, void *stream);

/*
 * rotary position embedding of the query and key heads between the q/k projections and the attention contraction
 * (torchmx/layers/mx_llama_attention.py:171-187 calls transformers' apply_rotary_pos_emb: five elementwise launches per tensor):
 *     out = (x * cos) + (rotate_half(x) * sin), every product and the sum rounded to bf16 as the tensor ops round them
 *   q / k   : bf16, element (b, t, h, d) at  base + b*batch_stride + t*tok_stride + h*head_dim + d  (the projection output, read in place)
 *   cos/sin : bf16 [batch | 1, tokens, head_dim] (batch stride 0 broadcasts)
 *   q_out / k_out : bf16 [batch, heads, tokens, head_dim], contiguous when the three *_out_*_stride fields are 0, else element
 *             (b, h, t, d) at  base + b*out_batch_stride + h*out_head_stride + t*out_tok_stride + d  -- the rotated keys can land in
 *             place in a KV cache (the cache update of the reference's call site, mx_llama_attention.py:189-193, folded in)
 *   v / v_out : optional (NULL): a third tensor with k's geometry, copied unrotated with the same addressing (the value heads on
 *             their way from the projection output into the cache)
 */
typedef struct {
    const void *q; int64_t q_tok_stride, q_batch_stride; int q_heads;
    const void *k; int64_t k_tok_stride, k_batch_stride; int k_heads;
    const void *cos; const void *sin; int64_t cs_tok_stride, cs_batch_stride;
    int64_t batch, tokens; int head_dim;
    void *q_out; void *k_out;
    int64_t q_out_batch_stride, q_out_head_stride, q_out_tok_stride;
    int64_t k_out_batch_stride, k_out_head_stride, k_out_tok_stride;
    const void *v; int64_t v_tok_stride, v_batch_stride;
    void *v_out; int64_t v_out_batch_stride, v_out_head_stride, v_out_tok_stride;
} mxq_rope_args_t;
MXQ_API int mxq_rope(const mxq_rope_args_t *args, int device, void *stream);

/*
 * the attention output as o_proj's MX activation  <->  `attn_output.transpose(1, 2).contiguous().reshape(b, q, h * d)`
 * (torchmx/layers/mx_llama_attention.py:245-247) followed by the quantization on entry to o_proj (torchmx/layers/mx_linear.py:63-66):
 *     codes, scales = quantize_mx(transpose(src), elem, 32)     with the transposed bf16 tensor never written
 *   src    : bf16 [batch, heads, tokens, head_dim] contiguous (what the attention kernel leaves), head_dim % 32 == 0
 *   codes  : [batch, tokens, heads * head_dim] (float4_e2m1: half), scales [batch, tokens, heads * head_dim / 32]
 */
MXQ_API int mxq_quantize_heads(const void *src, int64_t batch, int64_t heads, int64_t tokens, int64_t head_dim, int elem /* mxq_elem_t */,
                       unsigned flags /* MXQ_FLAG_* */, void *codes, uint8_t *scales, int device, void *stream);

/*
 * the value heads as the MX operand of P.V  <->  `MXTensor.to_mx(value_states.transpose(-2, -1), elem, 32)`
 * (torchmx/layers/mx_llama_attention.py:205-212: V is quantized along the SEQUENCE axis, 32 consecutive key positions of one
 * (head, channel) per block) without the strided copy that materialises the transposed bf16 tensor:
 *     codes, scales = quantize_mx(transpose(x, -2, -1), elem, 32)
 *   x      : bf16 [n0, n1, rows, cols], element (i0, i1, r, c) at x + i0 * s0 + i1 * s1 + r * row_stride + c (strides in elements,
 *            multiples of 8; base 16-byte aligned; cols contiguous): a [batch, heads, keys, head_dim] value tensor or cache slice
 *   codes  : [n0, n1, cols, rows] contiguous (float4_e2m1: rows / 2 bytes per channel), scales [n0, n1, cols, rows / 32]
 *   rows % 32 == 0, cols % 8 == 0, n0 * n1 <= 65535, else MXQ_ERR_UNSUPPORTED_SHAPE (the caller transposes and calls mxq_quantize)
 */
typedef struct {
    const void *x; int64_t n0, n1, rows, cols, s0, s1, row_stride;
    int elem /* mxq_elem_t */; unsigned flags /* MXQ_FLAG_HW_EXACT */;
    void *codes; uint8_t *scales;
} mxq_transposed_quantize_args_t;
MXQ_API int mxq_quantize_transposed(const mxq_transposed_quantize_args_t *args, int device, void *stream);

/*
 * rotary embedding + append to an MX-quantized static KV cache + quantization of Q, as ONE launch  <->  the MX attention block's
 *     q, k = apply_rotary_pos_emb(q, k, cos, sin);  keys, values = StaticCache.update(k, v)       (bf16 cache of capacity C)
 *     Q = to_mx(q);  K = to_mx(keys);  Vt = to_mx(transpose(values, -2, -1))                      (mxq_rope + mxq_quantize + mxq_quantize_transposed)
 * where only the new tokens' blocks are computed: K is blocked along head_dim, so a key row's codes depend on that row alone;
 * V is blocked along 32 consecutive positions, and every V block that [L, L + tokens) touches is re-derived from v_open (the bf16
 * positions of the block holding L below L), the new values, and zeros at and past L + tokens -- the same bytes the whole-cache
 * quantization of a zero-initialised bf16 cache gives.  Rotary arithmetic = mxq_rope's, block arithmetic = mxq_quantize's.
 *   q / k / v : bf16, element (b, t, h, d) at  base + b*batch_stride + t*tok_stride + h*head_dim + d  (projection outputs, possibly
 *               column slices of one stacked q/k/v output, read in place); strides multiples of 8 elements, 16-byte aligned bases
 *   cos/sin   : bf16 [batch | 1, tokens, head_dim] (cs_batch_stride 0 broadcasts)
 *   q_elem, k_elem, v_elem : any floating-point mxq_elem_t (MXQ_ELEM_INT8 -> MXQ_ERR_INVALID); flags: MXQ_FLAG_HW_EXACT
 * Storage, one byte per element in the form mxq_flash_attention reads: e4m3 / e5m2 codes as they are, fp6 / fp4 codes re-encoded
 * exactly as E4M3 (what mxq_transcode_to_e4m3 produces); 32-byte aligned bases:
 *   q_codes  : [batch, q_heads, tokens, 128], q_scales [batch, q_heads, tokens, 4]          (written)
 *   k_codes  : [batch, kv_heads, C, 128],     k_scales [batch, kv_heads, C, 4]              (rows L .. L + tokens - 1 written)
 *   vt_codes : [batch, kv_heads, 128, C],     vt_scales [batch, kv_heads, 128, C / 32]      (blocks touched by [L, L + tokens))
 *   v_open   : bf16 [batch, kv_heads, 32, 128]: read as the block holding L, left holding the block holding L + tokens
 *   position : DEVICE pointer to the int64 write position L (read, not advanced: a captured step replays as the caller advances it)
 * Positions at or past C are dropped.  head_dim must be 128 (MXQ_ERR_UNSUPPORTED_SHAPE otherwise, and for misaligned operands);
 * C % 32 != 0, tokens > C or a NULL pointer is MXQ_ERR_INVALID.
 */
typedef struct {
    const void *q; int64_t q_tok_stride, q_batch_stride; int q_heads;
    const void *k; int64_t k_tok_stride, k_batch_stride;
    const void *v; int64_t v_tok_stride, v_batch_stride; int kv_heads;
    const void *cos; const void *sin; int64_t cs_tok_stride, cs_batch_stride;
    int64_t batch, tokens; int head_dim;
    int q_elem, k_elem, v_elem /* mxq_elem_t */; unsigned flags /* MXQ_FLAG_HW_EXACT */;
    void *q_codes; uint8_t *q_scales;
    void *k_codes; uint8_t *k_scales;
    void *vt_codes; uint8_t *vt_scales;
    void *v_open;
    int64_t capacity; const int64_t *position;
} mxq_rope_quantize_kv_args_t;
MXQ_API int mxq_rope_quantize_kv(const mxq_rope_quantize_kv_args_t *args, int device, void *stream);

/*
 * Mixture-of-experts layer (K6)  <->  transformers' expert loop over a fused expert bank (MixtralExperts.forward and its Qwen2-MoE /
 * Qwen3-MoE / OLMoE twins: gate_up_proj [E, 2I, H], down_proj [E, H, I], SiLU gating) with every F.linear an MX matmul.  Three
 * entries; none reads a device value on the host, so a step built from them can be captured in a CUDA graph.
 *
 * mxq_moe_route: top_k_index [tokens, top_k] int64 -> a stable counting sort of the (token, slot) pairs by expert.  Slots whose
 * expert is outside [0, num_experts) are dropped (the loop skips them too).
 *   offsets      : int32 [num_experts + 1]: the routed rows of expert e are offsets[e] .. offsets[e + 1] - 1, ordered by
 *                  (token, slot); offsets[num_experts] = number of routed rows R <= tokens * top_k
 *   row_of_slot  : int32 [tokens * top_k]: routed row of (t, s) at t * top_k + s, -1 for a dropped slot
 *   token_of_row : int32 [tokens * top_k]: token of each routed row (entries >= R are not written)
 *   x / codes / scales : optional (all NULL or none): x bf16 [tokens, hidden] (row stride ldx elements, a multiple of 8, 16-byte
 *                  aligned base); routed row r of codes [tokens * top_k, hidden] (hidden / 2 bytes for MXQ_ELEM_E2M1) and scales
 *                  [tokens * top_k, hidden / 32] receives quantize_mx(x[token_of_row[r]], elem, 32) (mxq_quantize's arithmetic)
 * MXQ_ERR_INVALID: a NULL pointer, top_k outside 1..8, num_experts outside 1..256, tokens outside 0..16384, an unknown element type;
 * MXQ_ERR_UNSUPPORTED_SHAPE: hidden % 32 != 0 or a misaligned x / codes (16 bytes) when quantizing.
 */
#define MXQ_MOE_MAX_EXPERTS 256
#define MXQ_MOE_MAX_TOP_K 8
#define MXQ_MOE_MAX_TOKENS 16384
typedef struct {
    const int64_t *top_k_index; int64_t tokens; int top_k; int num_experts;
    int32_t *offsets; int32_t *row_of_slot; int32_t *token_of_row;
    const void *x; int64_t ldx; int64_t hidden;
    int elem /* mxq_elem_t */; unsigned flags /* MXQ_FLAG_HW_EXACT */;
    void *codes; uint8_t *scales;
} mxq_moe_route_args_t;
MXQ_API int mxq_moe_route(const mxq_moe_route_args_t *args, int device, void *stream);

/*
 * mxq_moe_gemm: D[r, :] = X[r, :] . W[e(r)]^T for every routed row r < offsets[num_experts], where e(r) is the expert whose
 * segment holds r -- one launch for all experts, the offsets read on the device.  Experts without rows cost no weight bytes.
 *   w_codes  : [num_experts * N, K] in operand format w_format (MXQ_OPERAND_*), rows compact (K * bits / 8 bytes);
 *   w_scales : [num_experts * N, K / 32] E8M0
 *   x_codes  : [rows, K] in x_format, compact rows; x_scales [rows, K / 32]; rows = the capacity the offsets index into
 *   d        : bf16 [rows, N]; only rows < offsets[num_experts] are written
 * MXQ_ERR_INVALID: a NULL pointer, num_experts outside 1..256, an unknown operand format;
 * MXQ_ERR_UNSUPPORTED_SHAPE: K % 128 != 0, N % 128 != 0, code pointers not 32-byte aligned, d or scales not 16-byte aligned.
 */
typedef struct {
    const void *w_codes; const uint8_t *w_scales; int w_format;
    const void *x_codes; const uint8_t *x_scales; int x_format;
    const int32_t *offsets;
    void *d;
    int64_t rows, num_experts, N, K;
} mxq_moe_gemm_args_t;
MXQ_API int mxq_moe_gemm(const mxq_moe_gemm_args_t *args, int device, void *stream);

/*
 * mxq_moe_combine: out[t, :] = the loop's successive index_add_ calls: starting from +0, for the token's slots in ascending
 * expert order, out = bf16(out + bf16(fp32(y[row_of_slot[t, s], :]) * w[t, s])).  One write per output element, no atomics.
 *   y : bf16 [*, hidden] routed rows (mxq_moe_gemm's D), top_k_index / row_of_slot as mxq_moe_route's,
 *   top_k_weights : [tokens, top_k] of weights_dtype (MXQ_HP_F32 or MXQ_HP_BF16), out : bf16 [tokens, hidden]
 * MXQ_ERR_INVALID as mxq_moe_route; MXQ_ERR_UNSUPPORTED_SHAPE: hidden % 8 != 0, y / out not 16-byte aligned.
 */
typedef struct {
    const void *y; const int64_t *top_k_index; const void *top_k_weights; int weights_dtype /* mxq_hp_t */;
    const int32_t *row_of_slot;
    int64_t tokens; int top_k; int num_experts; int64_t hidden;
    void *out;
} mxq_moe_combine_args_t;
MXQ_API int mxq_moe_combine(const mxq_moe_combine_args_t *args, int device, void *stream);

#define MXQ_OK 0
#define MXQ_ERR_INVALID 1
#define MXQ_ERR_UNSUPPORTED_SHAPE 2
#define MXQ_ERR_CUDA 3

MXQ_API const char *mxq_last_error(void);
/* ABI version: 6 (the mxq_moe_* entries) */
MXQ_API int mxq_version(void);
/* compiled-for architecture as an integer (1000 for sm_100a) -- lets the host refuse to run a
 * library that was built for something else instead of failing inside a launch. */
MXQ_API int mxq_arch(void);

#ifdef __cplusplus
}
#endif
#endif /* MXQ_H_ */
