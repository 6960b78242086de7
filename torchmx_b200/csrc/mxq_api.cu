// extern "C" surface of libmxq.so (declared in include/mxq.h).  Validates arguments, pins the CUDA
// device for the duration of the call, launches on the caller's stream, never synchronises.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "mxq_common.cuh"

namespace mxq {
cudaError_t launch_quantize(const void*, int, int64_t, int, int, unsigned, void*, uint8_t*, int, int64_t, int, int, cudaStream_t);
cudaError_t launch_dequantize(const void*, const uint8_t*, int64_t, int, int, int, void*, int, int64_t, int, int, cudaStream_t);
cudaError_t launch_dequantize_strided(const void*, const uint8_t*, int, const int64_t*, const int64_t*, const int64_t*, int, int, int, int,
                                      void*, cudaStream_t);
cudaError_t launch_transcode(const void*, int, int64_t, void*, int, cudaStream_t);
cudaError_t launch_pack_operand(const void*, int, int64_t, void*, int, cudaStream_t);
cudaError_t launch_unpack_operand(const void*, int, int64_t, void*, int, cudaStream_t);
int launch_gemm(const mxq_gemm_args_t*, int, int, cudaStream_t, char*, size_t);
namespace gemm { int launch_gemm_dequant(const mxq_gemm_dequant_args_t*, int, cudaStream_t, char*, size_t); }
namespace gemm { int launch_gemm_bf16(const void*, int64_t, int64_t, const void*, int64_t, int64_t, const void*, void*, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int,
                                       cudaStream_t, char*, size_t); }
namespace gemm { int launch_flash_attention(const mxq_attention_args_t*, int, cudaStream_t, char*, size_t); }
cudaError_t launch_silu_mul_quantize(const void*, const void*, int64_t, int64_t, int64_t, int64_t, int, unsigned, void*, uint8_t*, int, cudaStream_t);
int launch_softmax_quantize(const mxq_softmax_args_t*, cudaStream_t, char*, size_t);
int launch_rmsnorm(const mxq_rmsnorm_args_t*, cudaStream_t, char*, size_t);
int launch_rope(const mxq_rope_args_t*, int, cudaStream_t, char*, size_t);
int launch_heads_quantize(const void*, int64_t, int64_t, int64_t, int64_t, int, unsigned, void*, uint8_t*, cudaStream_t, char*, size_t);
int launch_transposed_quantize(const mxq_transposed_quantize_args_t*, cudaStream_t, char*, size_t);
int launch_rope_quantize_kv(const mxq_rope_quantize_kv_args_t*, cudaStream_t, char*, size_t);
int launch_moe_route(const mxq_moe_route_args_t*, cudaStream_t, char*, size_t);
int launch_moe_gemm(const mxq_moe_gemm_args_t*, int, cudaStream_t, char*, size_t);
int launch_moe_combine(const mxq_moe_combine_args_t*, cudaStream_t, char*, size_t);
}  // namespace mxq

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int fail_cuda(cudaError_t e, const char* what) {
    return fail(MXQ_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}

// Pins `device` as the calling thread's current device for the scope, restores the previous one.
struct DeviceScope {
    int prev = -1, cur = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceScope(int device) {
        err = cudaGetDevice(&prev);
        if (err != cudaSuccess) return;
        cur = device < 0 ? prev : device;
        if (cur != prev) err = cudaSetDevice(cur);
    }
    ~DeviceScope() {
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

int sm_count_of(int device) {
    static int cache[64];
    if (device >= 0 && device < 64 && cache[device]) return cache[device];
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0) n = 148;
    if (device >= 0 && device < 64) cache[device] = n;
    return n;
}

// L2 bytes of `device`: K1 / K2 launches that stream more than this take their L2 evict-first, back-to-front variants
int64_t l2_bytes_of(int device) {
    static int cache[64];
    if (device >= 0 && device < 64 && cache[device]) return cache[device];
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrL2CacheSize, device) != cudaSuccess || n <= 0) n = 126 << 20;
    if (device >= 0 && device < 64) cache[device] = n;
    return n;
}

bool valid_elem(int e) { return e >= MXQ_ELEM_E4M3 && e <= MXQ_ELEM_E5M2; }

// developer knobs (not part of the reference-facing contract), read once:
//   MXQ_QUANT_EPT = 8 | 16 | 32   elements per thread of the quantize fast path
//   MXQ_DEQ_CB    = 16 | 32       code bytes per thread of the dequantize fast path
//   MXQ_WAVES     = n             grid cap = SMs * 8 * n CTAs (grid-stride beyond that)
int env_int(const char* name) {
    const char* s = getenv(name);
    return s ? atoi(s) : 0;
}
int quant_ept_override() { static int v = env_int("MXQ_QUANT_EPT"); return (v == 8 || v == 16 || v == 32) ? v : 0; }
int deq_cb_override() { static int v = env_int("MXQ_DEQ_CB"); return (v == 16 || v == 32) ? v : 0; }
int waves_override() { static int v = env_int("MXQ_WAVES"); return v > 0 ? v : 0; }

}  // namespace

extern "C" {

const char* mxq_last_error(void) { return g_err; }
int mxq_version(void) { return 6; }
int mxq_arch(void) { return 1000; }

int mxq_quantize(const void* src, int src_dtype, int64_t n_blocks, int block_size, int elem, unsigned flags, void* codes, uint8_t* scales,
                 int device, void* stream) {
    if (!valid_elem(elem)) return fail(MXQ_ERR_INVALID, "mxq_quantize: unknown element type %d", elem);
    if (src_dtype != MXQ_HP_BF16 && src_dtype != MXQ_HP_F32) return fail(MXQ_ERR_INVALID, "mxq_quantize: unsupported source dtype %d", src_dtype);
    if (n_blocks < 0 || block_size < 1) return fail(MXQ_ERR_INVALID, "mxq_quantize: bad n_blocks=%lld block_size=%d", (long long)n_blocks, block_size);
    if (n_blocks == 0) return MXQ_OK;
    if (!src || !codes || !scales) return fail(MXQ_ERR_INVALID, "mxq_quantize: null pointer");
    if (elem == MXQ_ELEM_E2M1 && ((n_blocks * block_size) & 1))
        return fail(MXQ_ERR_INVALID, "mxq_quantize: float4_e2m1 needs an even element count (got %lld)", (long long)(n_blocks * block_size));
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_quantize: selecting device");
    const cudaError_t e = mxq::launch_quantize(src, src_dtype, n_blocks, block_size, elem, flags, codes, scales, sm_count_of(scope.cur),
                                               l2_bytes_of(scope.cur), quant_ept_override(), waves_override(), (cudaStream_t)stream);
    if (e == cudaErrorNotSupported && (flags & MXQ_FLAG_OPERAND_LAYOUT))
        return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_quantize: MXQ_FLAG_OPERAND_LAYOUT needs a 4 / 6-bit element type, block 32, bf16 source and 32-byte aligned pointers");
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_quantize: launch");
}

int mxq_dequantize(const void* codes, const uint8_t* scales, int64_t n_blocks, int block_size, int elem, int dst_dtype, void* dst, int device,
                   void* stream) {
    if (!valid_elem(elem)) return fail(MXQ_ERR_INVALID, "mxq_dequantize: unknown element type %d", elem);
    if (dst_dtype != MXQ_HP_BF16 && dst_dtype != MXQ_HP_F32) return fail(MXQ_ERR_INVALID, "mxq_dequantize: unsupported target dtype %d", dst_dtype);
    if (n_blocks < 0 || block_size < 1) return fail(MXQ_ERR_INVALID, "mxq_dequantize: bad n_blocks=%lld block_size=%d", (long long)n_blocks, block_size);
    if (n_blocks == 0) return MXQ_OK;
    if (!codes || !scales || !dst) return fail(MXQ_ERR_INVALID, "mxq_dequantize: null pointer");
    if (elem == MXQ_ELEM_E2M1 && ((n_blocks * block_size) & 1)) return fail(MXQ_ERR_INVALID, "mxq_dequantize: float4_e2m1 needs an even element count");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_dequantize: selecting device");
    const cudaError_t e = mxq::launch_dequantize(codes, scales, n_blocks, block_size, elem, dst_dtype, dst, sm_count_of(scope.cur), l2_bytes_of(scope.cur),
                                                 deq_cb_override(), waves_override(),
                                                 (cudaStream_t)stream);
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_dequantize: launch");
}

int mxq_dequantize_strided(const void* codes, const uint8_t* scales, int ndim, const int64_t* sizes, const int64_t* code_strides,
                           const int64_t* scale_strides, int block_dim, int block_size, int elem, int dst_dtype, void* dst, int device,
                           void* stream) {
    if (!valid_elem(elem)) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: unknown element type %d", elem);
    if (dst_dtype != MXQ_HP_BF16 && dst_dtype != MXQ_HP_F32) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: unsupported target dtype %d", dst_dtype);
    if (ndim < 1 || ndim > MXQ_MAX_DIMS) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: ndim %d outside 1..%d", ndim, MXQ_MAX_DIMS);
    if (block_dim < 0 || block_dim >= ndim || block_size < 1) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: bad block_dim=%d block_size=%d", block_dim, block_size);
    if (!sizes || !code_strides || !scale_strides) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: null shape pointer");
    int64_t total = 1;
    for (int d = 0; d < ndim; ++d) {
        if (sizes[d] < 0) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: negative size");
        total *= sizes[d];
    }
    if (sizes[block_dim] % block_size) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: size %lld along the blocked dim is not a multiple of %d", (long long)sizes[block_dim], block_size);
    if (elem == MXQ_ELEM_E2M1 && (sizes[block_dim] & 1)) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: float4_e2m1 needs an even blocked dim");
    if (total == 0) return MXQ_OK;
    if (!codes || !scales || !dst) return fail(MXQ_ERR_INVALID, "mxq_dequantize_strided: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_dequantize_strided: selecting device");
    const cudaError_t e = mxq::launch_dequantize_strided(codes, scales, ndim, sizes, code_strides, scale_strides, block_dim, block_size, elem, dst_dtype, dst, (cudaStream_t)stream);
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_dequantize_strided: launch");
}

int mxq_transcode_to_e4m3(const void* codes, int elem, int64_t n_elements, void* out, int device, void* stream) {
    if (elem < MXQ_ELEM_E4M3 || elem > MXQ_ELEM_E2M1) return fail(MXQ_ERR_INVALID, "mxq_transcode_to_e4m3: element type %d has no e4m3 container form", elem);
    if (n_elements < 0) return fail(MXQ_ERR_INVALID, "mxq_transcode_to_e4m3: negative count");
    if (n_elements == 0) return MXQ_OK;
    if (!codes || !out) return fail(MXQ_ERR_INVALID, "mxq_transcode_to_e4m3: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_transcode_to_e4m3: selecting device");
    const cudaError_t e = mxq::launch_transcode(codes, elem, n_elements, out, sm_count_of(scope.cur), (cudaStream_t)stream);
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_transcode_to_e4m3: launch");
}

int mxq_pack_operand(const void* codes, int elem, int64_t n_elements, void* out, int device, void* stream) {
    if (elem != MXQ_ELEM_E3M2 && elem != MXQ_ELEM_E2M3 && elem != MXQ_ELEM_E2M1) return fail(MXQ_ERR_INVALID, "mxq_pack_operand: element type %d has no packed operand form", elem);
    if (n_elements < 0 || n_elements % 16) return fail(MXQ_ERR_INVALID, "mxq_pack_operand: element count must be a non-negative multiple of 16");
    if (n_elements == 0) return MXQ_OK;
    if (!codes || !out) return fail(MXQ_ERR_INVALID, "mxq_pack_operand: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_pack_operand: selecting device");
    const cudaError_t e = mxq::launch_pack_operand(codes, elem, n_elements, out, sm_count_of(scope.cur), (cudaStream_t)stream);
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_pack_operand: launch");
}

int mxq_unpack_operand(const void* packed, int elem, int64_t n_elements, void* out, int device, void* stream) {
    if (elem != MXQ_ELEM_E3M2 && elem != MXQ_ELEM_E2M3 && elem != MXQ_ELEM_E2M1) return fail(MXQ_ERR_INVALID, "mxq_unpack_operand: element type %d has no packed operand form", elem);
    if (n_elements < 0 || n_elements % 16) return fail(MXQ_ERR_INVALID, "mxq_unpack_operand: element count must be a non-negative multiple of 16");
    if (n_elements == 0) return MXQ_OK;
    if (!packed || !out) return fail(MXQ_ERR_INVALID, "mxq_unpack_operand: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_unpack_operand: selecting device");
    const cudaError_t e = mxq::launch_unpack_operand(packed, elem, n_elements, out, sm_count_of(scope.cur), (cudaStream_t)stream);
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_unpack_operand: launch");
}

int mxq_gemm(const mxq_gemm_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_gemm: null args");
    if (a->batch < 0 || a->M < 0 || a->N < 0 || a->K < 0) return fail(MXQ_ERR_INVALID, "mxq_gemm: negative extent");
    if (a->batch == 0 || a->M == 0 || a->N == 0) return MXQ_OK;
    const bool xq = a->x_bf16 != nullptr;
    if ((!xq && (!a->a_codes || !a->sfa)) || !a->b_codes || !a->sfb || (!a->d && !a->d_multicast)) return fail(MXQ_ERR_INVALID, "mxq_gemm: null pointer");
    if (xq && (a->M > 64 || a->batch != 1)) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_gemm: fused activation quantization handles M <= 64, batch == 1");
    if (a->a_format < 0 || a->a_format > MXQ_OPERAND_E5M2_BYTES || a->b_format < 0 || a->b_format > MXQ_OPERAND_E5M2_BYTES)
        return fail(MXQ_ERR_INVALID, "mxq_gemm: unknown operand format %d / %d", a->a_format, a->b_format);
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_gemm: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_gemm(a, sm_count_of(scope.cur), scope.cur, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_gemm: %s", msg);
}

int mxq_gemm_dequant(const mxq_gemm_dequant_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_gemm_dequant: null args");
    if (a->batch < 0 || a->M < 0 || a->N < 0 || a->K < 0) return fail(MXQ_ERR_INVALID, "mxq_gemm_dequant: negative extent");
    if (a->batch == 0 || a->M == 0 || a->N == 0) return MXQ_OK;
    if (!a->d) return fail(MXQ_ERR_INVALID, "mxq_gemm_dequant: null output");
    for (int side = 0; side < 2; ++side) {
        const mxq_operand_t& o = side ? a->b : a->a;
        if (!valid_elem(o.elem)) return fail(MXQ_ERR_INVALID, "mxq_gemm_dequant: unknown element type %d", o.elem);
        if (o.block_size < 1) return fail(MXQ_ERR_INVALID, "mxq_gemm_dequant: bad block size %d", o.block_size);
        if (a->K > 0 && (!o.codes || !o.scales)) return fail(MXQ_ERR_INVALID, "mxq_gemm_dequant: null operand pointer");
    }
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_gemm_dequant: selecting device");
    char msg[400] = "";
    const int rc = mxq::gemm::launch_gemm_dequant(a, scope.cur, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_gemm_dequant: %s", msg);
}

int mxq_silu_mul_quantize(const void* gate, const void* up, int64_t rows, int64_t cols, int64_t ld_gate, int64_t ld_up, int elem, unsigned flags,
                          void* codes, uint8_t* scales, int device, void* stream) {
    if (!valid_elem(elem)) return fail(MXQ_ERR_INVALID, "mxq_silu_mul_quantize: unknown element type %d", elem);
    if (rows < 0 || cols < 0) return fail(MXQ_ERR_INVALID, "mxq_silu_mul_quantize: negative extent");
    if (rows == 0 || cols == 0) return MXQ_OK;
    if (!gate || !up || !codes || !scales) return fail(MXQ_ERR_INVALID, "mxq_silu_mul_quantize: null pointer");
    if (cols % 32 || ld_gate < cols || ld_up < cols || (ld_gate % 16) || (ld_up % 16) || ((uintptr_t)gate % 32) || ((uintptr_t)up % 32) || ((uintptr_t)codes % 32))
        return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_silu_mul_quantize: needs cols %% 32 == 0 and 32-byte aligned rows (base pointers, row strides %% 16 elements)");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_silu_mul_quantize: selecting device");
    const cudaError_t e = mxq::launch_silu_mul_quantize(gate, up, rows, cols, ld_gate, ld_up, elem, flags, codes, scales, sm_count_of(scope.cur), (cudaStream_t)stream);
    return e == cudaSuccess ? MXQ_OK : fail_cuda(e, "mxq_silu_mul_quantize: launch");
}

int mxq_rmsnorm(const mxq_rmsnorm_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_rmsnorm: null args");
    if (a->rows < 0 || a->hidden < 0) return fail(MXQ_ERR_INVALID, "mxq_rmsnorm: negative extent");
    if (a->rows == 0 || a->hidden == 0) return MXQ_OK;
    if (!a->x || !a->weight || (!a->y && !a->codes)) return fail(MXQ_ERR_INVALID, "mxq_rmsnorm: null pointer");
    if ((a->codes == nullptr) != (a->scales == nullptr)) return fail(MXQ_ERR_INVALID, "mxq_rmsnorm: codes and scales go together");
    if (a->codes && !valid_elem(a->elem)) return fail(MXQ_ERR_INVALID, "mxq_rmsnorm: unknown element type %d", a->elem);
    if (a->residual_out && !a->residual) return fail(MXQ_ERR_INVALID, "mxq_rmsnorm: residual_out without residual");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_rmsnorm: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_rmsnorm(a, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_rmsnorm: %s", msg);
}

int mxq_quantize_heads(const void* src, int64_t batch, int64_t heads, int64_t tokens, int64_t head_dim, int elem, unsigned flags, void* codes,
                       uint8_t* scales, int device, void* stream) {
    if (!valid_elem(elem)) return fail(MXQ_ERR_INVALID, "mxq_quantize_heads: unknown element type %d", elem);
    if (batch < 0 || heads < 0 || tokens < 0 || head_dim < 0) return fail(MXQ_ERR_INVALID, "mxq_quantize_heads: negative extent");
    if (batch == 0 || heads == 0 || tokens == 0 || head_dim == 0) return MXQ_OK;
    if (!src || !codes || !scales) return fail(MXQ_ERR_INVALID, "mxq_quantize_heads: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_quantize_heads: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_heads_quantize(src, batch, heads, tokens, head_dim, elem, flags, codes, scales, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_quantize_heads: %s", msg);
}

int mxq_quantize_transposed(const mxq_transposed_quantize_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_quantize_transposed: null args");
    if (!valid_elem(a->elem)) return fail(MXQ_ERR_INVALID, "mxq_quantize_transposed: unknown element type %d", a->elem);
    if (a->n0 < 0 || a->n1 < 0 || a->rows < 0 || a->cols < 0) return fail(MXQ_ERR_INVALID, "mxq_quantize_transposed: negative extent");
    if (a->n0 == 0 || a->n1 == 0 || a->rows == 0 || a->cols == 0) return MXQ_OK;
    if (!a->x || !a->codes || !a->scales) return fail(MXQ_ERR_INVALID, "mxq_quantize_transposed: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_quantize_transposed: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_transposed_quantize(a, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_quantize_transposed: %s", msg);
}

int mxq_rope(const mxq_rope_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_rope: null args");
    if (a->batch < 0 || a->tokens < 0 || a->q_heads < 0 || a->k_heads < 0) return fail(MXQ_ERR_INVALID, "mxq_rope: negative extent");
    if (a->batch == 0 || a->tokens == 0 || a->q_heads + a->k_heads == 0) return MXQ_OK;
    if ((a->q_heads && (!a->q || !a->q_out)) || (a->k_heads && (!a->k || !a->k_out)) || !a->cos || !a->sin) return fail(MXQ_ERR_INVALID, "mxq_rope: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_rope: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_rope(a, sm_count_of(scope.cur), (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_rope: %s", msg);
}

int mxq_gemm_bf16(const void* a, int64_t lda, int64_t a_batch_stride, const void* b, int64_t ldb, int64_t b_batch_stride, const void* bias, void* d,
                  int64_t ldd, int64_t d_batch_stride, int64_t batch, int64_t M, int64_t N, int64_t K, int device, void* stream) {
    if (batch < 0 || M < 0 || N < 0 || K < 0) return fail(MXQ_ERR_INVALID, "mxq_gemm_bf16: negative extent");
    if (batch == 0 || M == 0 || N == 0) return MXQ_OK;
    if (!a || !b || !d) return fail(MXQ_ERR_INVALID, "mxq_gemm_bf16: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_gemm_bf16: selecting device");
    char msg[400] = "";
    const int rc = mxq::gemm::launch_gemm_bf16(a, lda, a_batch_stride, b, ldb, b_batch_stride, bias, d, ldd, d_batch_stride, batch, M, N, K, scope.cur,
                                               (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_gemm_bf16: %s", msg);
}

int mxq_flash_attention(const mxq_attention_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_flash_attention: null args");
    if (!valid_elem(a->p_elem)) return fail(MXQ_ERR_INVALID, "mxq_flash_attention: unknown element type %d", a->p_elem);
    if (a->batch < 0 || a->heads < 0 || a->kv_heads < 0 || a->q_len < 0 || a->kv_len < 0) return fail(MXQ_ERR_INVALID, "mxq_flash_attention: negative extent");
    if (a->batch == 0 || a->heads == 0 || a->q_len == 0) return MXQ_OK;
    if (a->kv_heads == 0 || a->kv_len == 0) return fail(MXQ_ERR_INVALID, "mxq_flash_attention: no keys");
    if (!a->q_codes || !a->q_scales || !a->k_codes || !a->k_scales || !a->vt_codes || !a->vt_scales || !a->out)
        return fail(MXQ_ERR_INVALID, "mxq_flash_attention: null pointer");
    if ((a->p_codes == nullptr) != (a->p_scales == nullptr)) return fail(MXQ_ERR_INVALID, "mxq_flash_attention: p_codes and p_scales go together");
    if (a->kv_pitch < 0 || (a->kv_pitch > 0 && (a->kv_pitch % 128 || a->kv_pitch > MXQ_FLASH_MAX_KV || a->kv_len > a->kv_pitch || a->q_len > a->kv_len)))
        return fail(MXQ_ERR_INVALID, "mxq_flash_attention: kv_pitch %lld must be 0 or a multiple of 128 with q_len %lld <= kv_len %lld <= kv_pitch <= %d",
                    (long long)a->kv_pitch, (long long)a->q_len, (long long)a->kv_len, MXQ_FLASH_MAX_KV);
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_flash_attention: selecting device");
    char msg[400] = "";
    const int rc = mxq::gemm::launch_flash_attention(a, scope.cur, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_flash_attention: %s", msg);
}

int mxq_softmax_quantize(const mxq_softmax_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_softmax_quantize: null args");
    if (!valid_elem(a->elem)) return fail(MXQ_ERR_INVALID, "mxq_softmax_quantize: unknown element type %d", a->elem);
    if (a->batch < 0 || a->heads < 0 || a->q_len < 0 || a->kv_len < 0) return fail(MXQ_ERR_INVALID, "mxq_softmax_quantize: negative extent");
    if (a->batch == 0 || a->heads == 0 || a->q_len == 0 || a->kv_len == 0) return MXQ_OK;
    if (!a->scores || !a->codes || !a->scales) return fail(MXQ_ERR_INVALID, "mxq_softmax_quantize: null pointer");
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_softmax_quantize: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_softmax_quantize(a, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_softmax_quantize: %s", msg);
}

int mxq_rope_quantize_kv(const mxq_rope_quantize_kv_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_rope_quantize_kv: null args");
    for (int e : {a->q_elem, a->k_elem, a->v_elem})
        if (!valid_elem(e) || e == MXQ_ELEM_INT8) return fail(MXQ_ERR_INVALID, "mxq_rope_quantize_kv: element type %d has no one-byte attention operand", e);
    if (a->batch < 0 || a->tokens < 0 || a->q_heads < 0 || a->kv_heads < 0) return fail(MXQ_ERR_INVALID, "mxq_rope_quantize_kv: negative extent");
    if (a->capacity <= 0 || a->capacity % 32 || a->tokens > a->capacity)
        return fail(MXQ_ERR_INVALID, "mxq_rope_quantize_kv: capacity %lld must be a positive multiple of 32 and hold %lld tokens", (long long)a->capacity, (long long)a->tokens);
    if (a->batch == 0 || a->tokens == 0) return MXQ_OK;
    if (a->q_heads == 0 || a->kv_heads == 0) return fail(MXQ_ERR_INVALID, "mxq_rope_quantize_kv: no heads");
    if (!a->q || !a->k || !a->v || !a->cos || !a->sin || !a->q_codes || !a->q_scales || !a->k_codes || !a->k_scales || !a->vt_codes || !a->vt_scales ||
        !a->v_open || !a->position)
        return fail(MXQ_ERR_INVALID, "mxq_rope_quantize_kv: null pointer");
    if (a->head_dim != 128) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_rope_quantize_kv: needs head_dim == 128 (got %d)", a->head_dim);
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_rope_quantize_kv: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_rope_quantize_kv(a, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_rope_quantize_kv: %s", msg);
}

// shared by the three mxq_moe_* entries: the routing table's extents
static int moe_check_routing(const char* who, int64_t tokens, int top_k, int num_experts) {
    if (top_k < 1 || top_k > MXQ_MOE_MAX_TOP_K) return fail(MXQ_ERR_INVALID, "%s: top_k %d outside 1..%d", who, top_k, MXQ_MOE_MAX_TOP_K);
    if (num_experts < 1 || num_experts > MXQ_MOE_MAX_EXPERTS) return fail(MXQ_ERR_INVALID, "%s: num_experts %d outside 1..%d", who, num_experts, MXQ_MOE_MAX_EXPERTS);
    if (tokens < 0 || tokens > MXQ_MOE_MAX_TOKENS) return fail(MXQ_ERR_INVALID, "%s: tokens %lld outside 0..%d", who, (long long)tokens, MXQ_MOE_MAX_TOKENS);
    return MXQ_OK;
}

int mxq_moe_route(const mxq_moe_route_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null args");
    if (const int rc = moe_check_routing("mxq_moe_route", a->tokens, a->top_k, a->num_experts)) return rc;
    if (!a->top_k_index) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null top_k_index");
    if (!a->offsets) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null offsets");
    if (!a->row_of_slot) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null row_of_slot");
    if (!a->token_of_row) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null token_of_row");
    const bool quant = a->codes || a->scales || a->x;
    if (quant) {
        if (!a->x) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null x (codes / scales given)");
        if (!a->codes) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null codes (x given)");
        if (!a->scales) return fail(MXQ_ERR_INVALID, "mxq_moe_route: null scales (x given)");
        if (!valid_elem(a->elem)) return fail(MXQ_ERR_INVALID, "mxq_moe_route: unknown element type %d", a->elem);
        if (a->hidden <= 0 || a->hidden % 32) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_route: hidden %lld is not a positive multiple of 32", (long long)a->hidden);
        if (a->ldx < a->hidden || a->ldx % 8) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_route: ldx %lld must be >= hidden and a multiple of 8", (long long)a->ldx);
        if ((uintptr_t)a->x % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_route: x is not 16-byte aligned");
        if ((uintptr_t)a->codes % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_route: codes are not 16-byte aligned");
    }
    if (a->tokens == 0) return MXQ_OK;
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_moe_route: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_moe_route(a, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_moe_route: %s", msg);
}

int mxq_moe_gemm(const mxq_moe_gemm_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null args");
    if (a->num_experts < 1 || a->num_experts > MXQ_MOE_MAX_EXPERTS)
        return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: num_experts %lld outside 1..%d", (long long)a->num_experts, MXQ_MOE_MAX_EXPERTS);
    if (a->rows < 0 || a->N < 0 || a->K < 0) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: negative extent");
    if (a->rows > (int64_t)MXQ_MOE_MAX_TOKENS * MXQ_MOE_MAX_TOP_K) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: rows %lld exceed %d", (long long)a->rows, MXQ_MOE_MAX_TOKENS * MXQ_MOE_MAX_TOP_K);
    if (!a->w_codes) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null w_codes");
    if (!a->w_scales) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null w_scales");
    if (!a->x_codes) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null x_codes");
    if (!a->x_scales) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null x_scales");
    if (!a->offsets) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null offsets");
    if (!a->d) return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: null d");
    if (a->w_format < 0 || a->w_format > MXQ_OPERAND_E5M2_BYTES || a->x_format < 0 || a->x_format > MXQ_OPERAND_E5M2_BYTES)
        return fail(MXQ_ERR_INVALID, "mxq_moe_gemm: unknown operand format %d / %d", a->w_format, a->x_format);
    if (a->K == 0 || a->K % 128) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: K %lld is not a positive multiple of 128", (long long)a->K);
    if (a->N == 0 || a->N % 128) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: N %lld is not a positive multiple of 128", (long long)a->N);
    if ((uintptr_t)a->w_codes % 32) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: w_codes is not 32-byte aligned");
    if ((uintptr_t)a->x_codes % 32) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: x_codes is not 32-byte aligned");
    if ((uintptr_t)a->w_scales % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: w_scales is not 16-byte aligned");
    if ((uintptr_t)a->x_scales % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: x_scales is not 16-byte aligned");
    if ((uintptr_t)a->d % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_gemm: d is not 16-byte aligned");
    if (a->rows == 0) return MXQ_OK;
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_moe_gemm: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_moe_gemm(a, scope.cur, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_moe_gemm: %s", msg);
}

int mxq_moe_combine(const mxq_moe_combine_args_t* a, int device, void* stream) {
    if (!a) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: null args");
    if (const int rc = moe_check_routing("mxq_moe_combine", a->tokens, a->top_k, a->num_experts)) return rc;
    if (a->weights_dtype != MXQ_HP_F32 && a->weights_dtype != MXQ_HP_BF16) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: weights_dtype %d", a->weights_dtype);
    if (!a->y) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: null y");
    if (!a->top_k_index) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: null top_k_index");
    if (!a->top_k_weights) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: null top_k_weights");
    if (!a->row_of_slot) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: null row_of_slot");
    if (!a->out) return fail(MXQ_ERR_INVALID, "mxq_moe_combine: null out");
    if (a->hidden <= 0 || a->hidden % 8) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_combine: hidden %lld is not a positive multiple of 8", (long long)a->hidden);
    if ((uintptr_t)a->y % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_combine: y is not 16-byte aligned");
    if ((uintptr_t)a->out % 16) return fail(MXQ_ERR_UNSUPPORTED_SHAPE, "mxq_moe_combine: out is not 16-byte aligned");
    if (a->tokens == 0) return MXQ_OK;
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail_cuda(scope.err, "mxq_moe_combine: selecting device");
    char msg[400] = "";
    const int rc = mxq::launch_moe_combine(a, (cudaStream_t)stream, msg, sizeof(msg));
    return rc == MXQ_OK ? MXQ_OK : fail(rc, "mxq_moe_combine: %s", msg);
}

}  // extern "C"
