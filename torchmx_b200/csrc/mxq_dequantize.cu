// K2: fused MX dequantize (element codes + E8M0 scales -> bf16 / fp32), one pass over HBM.
//
// Replaces torchmx/mx_tensor.py:145-164 -> mx_quantization_utils.py:93-146 (decode), :415-432
// (scale), utils.py:96-117 (fp4 unpack) and the repeat_interleave that materialises a full-size
// scale tensor (13-37 aten launches on a GPU).
//
// out = RNE_target( decode(code) * 2^(s-127) ): decode is exact (F2FP to f16x2, or the integer
// itself), the fp32 product is exact (<= 8 significant bits times a power of two, fp32
// subnormals kept), so the single rounding happens in the final fp32 -> bf16 pack -- the same
// value the reference's bf16 x bf16 -> bf16 product yields.
//
// Fast path (block 32, blocked axis innermost and contiguous): flat run of blocks, a thread owns
// 16 codes (one 128-bit load; fp4: 16 bytes = one whole block) and writes 32/64 B (bf16) or
// 64/128 B (fp32) with 256-bit stores.
#include <type_traits>

#include "mxq_common.cuh"

namespace mxq {

constexpr int kDequantThreads = 256;

template <int ELEM>
__device__ __forceinline__ void decode4(uint32_t word, float sc, float (&f)[4]) {
    // four 1-byte codes in `word` (byte 0 = first element)
    if constexpr (ELEM == MXQ_ELEM_INT8) {
#pragma unroll
        for (int j = 0; j < 4; ++j) f[j] = (float)(int)(int8_t)(word >> (8 * j)) * sc;
    } else {
        const uint32_t h0 = decode_pair_f16x2<ELEM>(word & 0xFFFF), h1 = decode_pair_f16x2<ELEM>(word >> 16);
        f[0] = f16lo_to_f32(h0) * sc; f[1] = f16hi_to_f32(h0) * sc;
        f[2] = f16lo_to_f32(h1) * sc; f[3] = f16hi_to_f32(h1) * sc;
    }
}

// four packed fp4 bytes -> 8 elements; byte's HIGH nibble is the earlier element (utils.py:96-117)
__device__ __forceinline__ void decode8_e2m1(uint32_t word, float sc, float (&f)[8]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t h = decode_e2m1_byte_f16x2((word >> (8 * j)) & 0xFF);
        f[2 * j] = f16hi_to_f32(h) * sc;
        f[2 * j + 1] = f16lo_to_f32(h) * sc;
    }
}

template <int N, bool F32, bool OVER_L2 = false>
__device__ __forceinline__ void store_run(void* dst, int64_t first_elem, const float (&f)[N], uint64_t pol = 0) {
    // N consecutive outputs starting at element `first_elem`; N*sizeof(T) is a multiple of 32 and aligned
    if constexpr (F32) {
        uint8_t* p = reinterpret_cast<uint8_t*>(dst) + first_elem * 4;
#pragma unroll
        for (int j = 0; j < N / 8; ++j) {
            u32x8 o;
#pragma unroll
            for (int k = 0; k < 8; ++k) o.v[k] = __float_as_uint(f[8 * j + k]);
            stg256_stream(p + 32 * j, o);
        }
    } else {
        uint8_t* p = reinterpret_cast<uint8_t*>(dst) + first_elem * 2;
#pragma unroll
        for (int j = 0; j < N / 16; ++j) {
            u32x8 o;
#pragma unroll
            for (int k = 0; k < 8; ++k) o.v[k] = pack_bf16x2(f[16 * j + 2 * k], f[16 * j + 2 * k + 1]);
            if constexpr (OVER_L2) stg256_evict_first(p + 32 * j, o, pol);
            else stg256_stream(p + 32 * j, o);
        }
    }
}

// One thread's chunk c of CB code bytes: decode with the block scales, store the values.
template <int ELEM, bool F32, int CB, bool OVER_L2>
__device__ __forceinline__ void dequantize_b32_chunk(const uint8_t* __restrict__ codes, const uint8_t* __restrict__ scales, void* __restrict__ dst,
                                                     int64_t c, uint64_t pol) {
    // a thread owns CB = 16 or 32 consecutive code bytes; each 16-byte half is half a block (1-byte
    // codes) or a whole block (fp4) and carries its own scale byte
    constexpr int PER = (ELEM == MXQ_ELEM_E2M1) ? 2 : 1;  // elements per code byte
    constexpr int NH = CB / 16;
    uint32_t w[CB / 4];
    if constexpr (CB == 32) {
        const u32x8 v = OVER_L2 ? ldg256_evict_first(codes + c * 32, pol) : ldg256_stream(codes + c * 32);
#pragma unroll
        for (int k = 0; k < 8; ++k) w[k] = v.v[k];
    } else {
        const uint4 v = OVER_L2 ? ldg128_evict_first(codes + c * 16, pol) : ldg128_stream(codes + c * 16);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    }
    int s[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) {
        const uint8_t* sp = scales + ((c * CB + 16 * h) * PER) / 32;
        if constexpr (OVER_L2) s[h] = (int)ldg8_evict_first(sp, pol);
        else s[h] = __ldg(sp);
    }
#pragma unroll
    for (int h = 0; h < NH; ++h) {
        const float sc = scale_f32(s[h]);
        const int64_t e0 = (c * CB + 16 * h) * PER;
        if constexpr (ELEM == MXQ_ELEM_E2M1) {
            float f[32];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float t[8];
                decode8_e2m1(w[4 * h + i], sc, t);
#pragma unroll
                for (int k = 0; k < 8; ++k) f[8 * i + k] = t[k];
            }
            store_run<32, F32, OVER_L2>(dst, e0, f, pol);
        } else {
            float f[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float t[4];
                decode4<ELEM>(w[4 * h + i], sc, t);
#pragma unroll
                for (int k = 0; k < 4; ++k) f[4 * i + k] = t[k];
            }
            store_run<16, F32, OVER_L2>(dst, e0, f, pol);
        }
    }
}

// OVER_L2 (bf16 target, code + output bytes exceed L2): the CTAs walk the data back to front -- virtual CTA v
// (v = blockIdx.x + k * gridDim.x) owns tile n_tiles - 1 - v, lanes ascending inside it -- so the first CTAs read the codes a
// preceding K1 wrote last, which are still in L2.  In the first `hint_tiles` tiles (l2_handoff_window() bytes of codes) code, scale and
// output accesses are evict-first, so consumed codes and the output are replaced before the codes still ahead of the walk;
// past them there is nothing left in L2 to protect and the tiles stream as in the plain kernel.
template <int ELEM, bool F32, int CB, bool OVER_L2 = false>
__global__ void __launch_bounds__(kDequantThreads) dequantize_b32_kernel(const uint8_t* __restrict__ codes, const uint8_t* __restrict__ scales,
                                                                         void* __restrict__ dst, int64_t n_code_bytes, int64_t hint_tiles = 0) {
    const int64_t n_chunks = n_code_bytes / CB;
    if constexpr (OVER_L2) {
        const uint64_t pol = l2_evict_first_policy();
        const int64_t n_tiles = (n_chunks + kDequantThreads - 1) / kDequantThreads;
        for (int64_t v = blockIdx.x; v < n_tiles; v += gridDim.x) {
            const int64_t c = (n_tiles - 1 - v) * kDequantThreads + threadIdx.x;
            if (c >= n_chunks) continue;
            if (v < hint_tiles) dequantize_b32_chunk<ELEM, F32, CB, true>(codes, scales, dst, c, pol);
            else dequantize_b32_chunk<ELEM, F32, CB, false>(codes, scales, dst, c, 0);
        }
    } else {
        const int64_t stride = (int64_t)gridDim.x * kDequantThreads;
        for (int64_t c = (int64_t)blockIdx.x * kDequantThreads + threadIdx.x; c < n_chunks; c += stride)
            dequantize_b32_chunk<ELEM, F32, CB, false>(codes, scales, dst, c, 0);
    }
}

// ---- generic strided path ------------------------------------------------------------------------
// One thread per output element; dst is C-contiguous in the logical shape, codes / scales are
// arbitrary views (permuted, expanded, ...).  Covers every block size and every block_dim.
struct StridedArgs {
    int ndim, block_dim, block_size;
    int64_t sizes[MXQ_MAX_DIMS], code_strides[MXQ_MAX_DIMS], scale_strides[MXQ_MAX_DIMS];
    int64_t total;
};

template <int ELEM, bool F32>
__global__ void dequantize_strided_kernel(const uint8_t* __restrict__ codes, const uint8_t* __restrict__ scales, void* __restrict__ dst,
                                          StridedArgs a) {
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= a.total) return;
    int64_t rem = o, coff = 0, soff = 0;
    int nib = 0;
#pragma unroll
    for (int d = MXQ_MAX_DIMS - 1; d >= 0; --d) {
        if (d < a.ndim) {
            const int64_t idx = rem % a.sizes[d];
            rem /= a.sizes[d];
            if (d == a.block_dim) {
                soff += (idx / a.block_size) * a.scale_strides[d];
                if constexpr (ELEM == MXQ_ELEM_E2M1) { coff += (idx >> 1) * a.code_strides[d]; nib = (int)(idx & 1); }
                else coff += idx * a.code_strides[d];
            } else {
                coff += idx * a.code_strides[d];
                soff += idx * a.scale_strides[d];
            }
        }
    }
    uint32_t c = codes[coff];
    if constexpr (ELEM == MXQ_ELEM_E2M1) c = nib ? (c & 0xF) : (c >> 4);
    const float v = decode_one<ELEM>(c) * scale_f32(scales[soff]);
    if constexpr (F32) reinterpret_cast<float*>(dst)[o] = v;
    else reinterpret_cast<uint16_t*>(dst)[o] = (uint16_t)pack_bf16x2(v, 0.0f);
}

// ---- transposing path: blocked axis is second-to-last logically, but innermost physically --------
// (what aten.t / transpose(-2,-1) of a quantized tensor produces: ops.py:122-158).  A 64x64 logical
// tile is read along the physically contiguous (blocked) axis, decoded, transposed through shared
// memory and written along the logically contiguous axis.
template <int ELEM, bool F32>
__global__ void __launch_bounds__(256) dequantize_transposed_kernel(const uint8_t* __restrict__ codes, const uint8_t* __restrict__ scales,
                                                                    void* __restrict__ dst, int64_t batch, int64_t K, int64_t N,
                                                                    int64_t code_batch_stride, int64_t code_row_stride,
                                                                    int64_t scale_batch_stride, int64_t scale_row_stride, int block_size) {
    // logical [batch, K, N] (K blocked); physical codes [batch][N rows][K contiguous]
    __shared__ float tile[64][65];
    const int64_t b = blockIdx.z;
    const int64_t k0 = (int64_t)blockIdx.x * 64, n0 = (int64_t)blockIdx.y * 64;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
    for (int r = ty; r < 64; r += 4) {
        const int64_t n = n0 + r, k = k0 + tx;
        float v = 0.0f;
        if (n < N && k < K) {
            uint32_t c;
            if constexpr (ELEM == MXQ_ELEM_E2M1) {
                c = codes[b * code_batch_stride + n * code_row_stride + (k >> 1)];
                c = (k & 1) ? (c & 0xF) : (c >> 4);
            } else {
                c = codes[b * code_batch_stride + n * code_row_stride + k];
            }
            const int s = scales[b * scale_batch_stride + n * scale_row_stride + k / block_size];
            v = decode_one<ELEM>(c) * scale_f32(s);
        }
        tile[r][tx] = v;
    }
    __syncthreads();
    for (int r = ty; r < 64; r += 4) {
        const int64_t k = k0 + r, n = n0 + tx;
        if (k < K && n < N) {
            const float v = tile[tx][r];
            const int64_t o = (b * K + k) * N + n;
            if constexpr (F32) reinterpret_cast<float*>(dst)[o] = v;
            else reinterpret_cast<uint16_t*>(dst)[o] = (uint16_t)pack_bf16x2(v, 0.0f);
        }
    }
}

// ---- transposing path, block size 32, vectorised --------------------------------------------------------------------------
// The same mapping as dequantize_transposed_kernel with 128-bit accesses on both sides: a CTA owns 64 physical rows (logical
// columns n) x KT logical rows k (KT = 64 elements; 128 for fp4, whose 16-byte load holds a whole block).  Thread (row, q) loads
// 16 code bytes of its row, decodes them with the block's scale (K2's arithmetic: exact decode, exact fp32 product, one
// rounding) and scatters the values into a shared-memory tile laid out [k][n]; thread (k, q) then stores 16 consecutive n
// of one k: 32 B (bf16) / 64 B (fp32) per thread, 128 / 256 B contiguous per k row.
// Algorithmic traffic = the flat kernel's (1 + 1/32 B in, 2 / 4 B out per element).
template <int ELEM, bool F32>
__global__ void __launch_bounds__(256) dequantize_transposed_b32_kernel(const uint8_t* __restrict__ codes, const uint8_t* __restrict__ scales,
                                                                        void* __restrict__ dst, int64_t K, int64_t N, int64_t code_batch_stride,
                                                                        int64_t code_row_stride, int64_t scale_batch_stride, int64_t scale_row_stride) {
    constexpr bool FP4 = ELEM == MXQ_ELEM_E2M1;
    constexpr int EPL = FP4 ? 32 : 16;        // elements per 16-byte load
    constexpr int KT = 128;                   // logical rows k per CTA: a whole 128-byte line of every physical row (fp4: 64 bytes)
    constexpr int LOADS = KT / (4 * EPL);     // 16-byte loads per thread
    constexpr int PITCH = 64 + (F32 ? 4 : 8); // elements per tile row: 16-byte aligned rows, consecutive rows 4 banks apart
    constexpr int CH = F32 ? 4 : 8;           // elements per 16-byte chunk
    using T = typename std::conditional<F32, float, uint16_t>::type;
    __shared__ __align__(16) T tile[KT][PITCH];
    const int64_t b = blockIdx.z;
    // consecutive CTAs walk the logical columns n: their 128-byte output segments of one k row are neighbours in DRAM (the
    // output is twice the bytes of the input, so the stores get the locality)
    const int64_t n0 = (int64_t)blockIdx.x * 64, k0 = (int64_t)blockIdx.y * KT;
#pragma unroll
    for (int h = 0; h < LOADS; ++h) {
        const int row = threadIdx.x >> 2, q = threadIdx.x & 3, grp = 4 * h + q;  // grp: which EPL-wide slice of the tile's k range
        const int64_t n = n0 + row, k = k0 + grp * EPL;
        float f[EPL];
        if (n < N && k < K) {  // (K is a multiple of 32 and of EPL: a load never straddles the end of a row)
            const uint8_t* src = codes + b * code_batch_stride + n * code_row_stride + (FP4 ? (k >> 1) : k);
            const uint4 v = ldg128_stream(src);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            const float sc = scale_f32(__ldg(scales + b * scale_batch_stride + n * scale_row_stride + (k >> 5)));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if constexpr (FP4) {
                    float t[8];
                    decode8_e2m1(w[i], sc, t);
#pragma unroll
                    for (int j = 0; j < 8; ++j) f[8 * i + j] = t[j];
                } else {
                    float t[4];
                    decode4<ELEM>(w[i], sc, t);
#pragma unroll
                    for (int j = 0; j < 4; ++j) f[4 * i + j] = t[j];
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < EPL; ++i) f[i] = 0.0f;
        }
        // 16-byte chunks of a tile row are XOR-permuted with the row's load group (mod 4 = q of the thread that writes it), so the
        // four q lanes of a warp, whose rows lie a multiple of 32 banks apart, hit different banks
#pragma unroll
        for (int i = 0; i < EPL; ++i) {
            const int col = (((row / CH) ^ (F32 ? 2 * q : q)) * CH) + (row % CH);
            if constexpr (F32) tile[grp * EPL + i][col] = f[i];
            else tile[grp * EPL + i][col] = (uint16_t)pack_bf16x2(f[i], 0.0f);
        }
    }
    __syncthreads();
    constexpr int PER = 16;  // n per thread and k row
#pragma unroll
    for (int it = 0; it < KT / 64; ++it) {
        const int kk = it * 64 + (threadIdx.x >> 2), q = threadIdx.x & 3;
        const int g = (kk / EPL) & 3;
        const int64_t k = k0 + kk, n = n0 + q * PER;
        if (k >= K || n >= N) continue;
        T* out = reinterpret_cast<T*>(dst) + (b * K + k) * N + n;
        const bool vec_out = n + PER <= N && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
#pragma unroll
        for (int j = 0; j < PER / CH; ++j) {
            const int chunk = ((q * PER) / CH + j) ^ (F32 ? 2 * g : g);
            const uint4 v = *reinterpret_cast<const uint4*>(&tile[kk][chunk * CH]);
            if (vec_out) {
                stg128_stream(out + j * CH, v);
            } else {
                const T* e = reinterpret_cast<const T*>(&v);
                for (int u = 0; u < CH; ++u)
                    if (n + j * CH + u < N) out[j * CH + u] = e[u];
            }
        }
    }
}

// ---- launchers -----------------------------------------------------------------------------------
// The OVER_L2 variant for bf16 targets.  fp4 walks back to front without hints: its output is four times its code bytes and
// the evict-first streams measured slower than the handoff saves (B200, 1000 W, 16384^2 after its K1: 104.5 -> 106.9 us with
// all hints, 104.8 us without).  fp32 targets (output four / eight times the codes) keep the forward kernel.
template <int ELEM, bool F32, int CB>
static void launch_b32(int64_t l2_bytes, int grid, cudaStream_t stream, const uint8_t* codes, const uint8_t* scales, void* dst, int64_t n_code_bytes) {
    if constexpr (!F32) {
        if (n_code_bytes + n_code_bytes * (ELEM == MXQ_ELEM_E2M1 ? 4 : 2) > l2_bytes) {  // codes + bf16 output
            const int64_t hint_tiles = ELEM == MXQ_ELEM_E2M1 ? 0 : l2_handoff_window(l2_bytes) / ((int64_t)kDequantThreads * CB);
            dequantize_b32_kernel<ELEM, F32, CB, true><<<grid, kDequantThreads, 0, stream>>>(codes, scales, dst, n_code_bytes, hint_tiles);
            return;
        }
    }
    dequantize_b32_kernel<ELEM, F32, CB><<<grid, kDequantThreads, 0, stream>>>(codes, scales, dst, n_code_bytes);
}

template <int ELEM, bool F32>
static cudaError_t launch_flat(const void* codes, const uint8_t* scales, int64_t n_blocks, int block_size, void* dst, int sm_count,
                               int64_t l2_bytes, int cb, int waves, cudaStream_t stream) {
    if (n_blocks == 0) return cudaSuccess;
    if (block_size == 32 && ((uintptr_t)codes % 32) == 0 && ((uintptr_t)dst % 32) == 0) {
        const int64_t n_code_bytes = n_blocks * ((ELEM == MXQ_ELEM_E2M1) ? 16 : 32);
        // measured on B200 (tools/quick_bench.py sweep): 32 code bytes per thread is best for 1-byte codes -> bf16
        // (6.6 TB/s), 16 for fp4 and for every fp32 target (more store bytes per thread already)
        if (cb != 16 && cb != 32) cb = (!F32 && ELEM != MXQ_ELEM_E2M1) ? 32 : 16;
        if (n_code_bytes % cb) cb = 16;
        const int64_t n_chunks = n_code_bytes / cb;
        const int64_t want = (n_chunks + kDequantThreads - 1) / kDequantThreads;
        const int64_t cap = waves > 0 ? (int64_t)sm_count * 8 * waves : (int64_t)0x7FFFFFFF;
        const int grid = (int)(want < cap ? want : cap);
        if (cb == 32) launch_b32<ELEM, F32, 32>(l2_bytes, grid, stream, (const uint8_t*)codes, scales, dst, n_code_bytes);
        else launch_b32<ELEM, F32, 16>(l2_bytes, grid, stream, (const uint8_t*)codes, scales, dst, n_code_bytes);
        return cudaGetLastError();
    }
    // any other block size / alignment: the strided kernel on a 1-D view
    StridedArgs a{};
    a.ndim = 1; a.block_dim = 0; a.block_size = block_size;
    a.sizes[0] = n_blocks * block_size; a.code_strides[0] = 1; a.scale_strides[0] = 1;
    a.total = a.sizes[0];
    const unsigned grid = (unsigned)((a.total + 255) / 256);
    dequantize_strided_kernel<ELEM, F32><<<grid, 256, 0, stream>>>((const uint8_t*)codes, scales, dst, a);
    return cudaGetLastError();
}

template <int ELEM, bool F32>
static cudaError_t launch_strided(const void* codes, const uint8_t* scales, int ndim, const int64_t* sizes, const int64_t* cs,
                                  const int64_t* ss, int block_dim, int block_size, void* dst, cudaStream_t stream) {
    StridedArgs a{};
    a.ndim = ndim; a.block_dim = block_dim; a.block_size = block_size;
    a.total = 1;
    for (int d = 0; d < ndim; ++d) { a.sizes[d] = sizes[d]; a.code_strides[d] = cs[d]; a.scale_strides[d] = ss[d]; a.total *= sizes[d]; }
    if (a.total == 0) return cudaSuccess;
    // transposing fast case: logical [..., K, N], blocked dim K = ndim-2 with unit code stride, rows (N) strided,
    // leading dims collapsible into one batch index with uniform strides
    if (ndim >= 2 && block_dim == ndim - 2 && cs[ndim - 2] == 1 && ss[ndim - 2] == 1) {
        bool ok = true;
        int64_t batch = 1, cbs = 0, sbs = 0;
        // collapse leading dims right-to-left: stride[d] must equal stride[d+1]*size[d+1]
        int64_t exp_c = 0, exp_s = 0;
        bool first = true;
        for (int d = ndim - 3; d >= 0; --d) {
            if (sizes[d] == 1) continue;
            if (first) { cbs = cs[d]; sbs = ss[d]; exp_c = cs[d] * sizes[d]; exp_s = ss[d] * sizes[d]; first = false; }
            else { if (cs[d] != exp_c || ss[d] != exp_s) { ok = false; break; } exp_c *= sizes[d]; exp_s *= sizes[d]; }
            batch *= sizes[d];
        }
        const int64_t K = sizes[ndim - 2], N = sizes[ndim - 1];
        constexpr int KT = 128;
        const bool vec = block_size == 32 && K % 32 == 0 && ((uintptr_t)codes % 16) == 0 && cs[ndim - 1] % 16 == 0 && cbs % 16 == 0 &&
                         (ELEM != MXQ_ELEM_E2M1 || K % 64 == 0);
        if (ok && vec && batch <= 65535 && (K + KT - 1) / KT <= 65535) {
            dim3 grid((unsigned)((N + 63) / 64), (unsigned)((K + KT - 1) / KT), (unsigned)batch);
            dequantize_transposed_b32_kernel<ELEM, F32><<<grid, 256, 0, stream>>>((const uint8_t*)codes, scales, dst, K, N, cbs, cs[ndim - 1], sbs, ss[ndim - 1]);
            return cudaGetLastError();
        }
        if (ok && batch <= 65535 && (N + 63) / 64 <= 65535) {
            dim3 grid((unsigned)((K + 63) / 64), (unsigned)((N + 63) / 64), (unsigned)batch);
            dequantize_transposed_kernel<ELEM, F32><<<grid, 256, 0, stream>>>((const uint8_t*)codes, scales, dst, batch, K, N, cbs, cs[ndim - 1], sbs,
                                                                              ss[ndim - 1], block_size);
            return cudaGetLastError();
        }
    }
    const unsigned grid = (unsigned)((a.total + 255) / 256);
    dequantize_strided_kernel<ELEM, F32><<<grid, 256, 0, stream>>>((const uint8_t*)codes, scales, dst, a);
    return cudaGetLastError();
}

#define MXQ_DISPATCH_ELEM_DT(elem, f32, CALL)                                                    \
    switch (elem) {                                                                              \
    case MXQ_ELEM_E4M3: return f32 ? CALL(MXQ_ELEM_E4M3, true) : CALL(MXQ_ELEM_E4M3, false);     \
    case MXQ_ELEM_E3M2: return f32 ? CALL(MXQ_ELEM_E3M2, true) : CALL(MXQ_ELEM_E3M2, false);     \
    case MXQ_ELEM_E2M3: return f32 ? CALL(MXQ_ELEM_E2M3, true) : CALL(MXQ_ELEM_E2M3, false);     \
    case MXQ_ELEM_E2M1: return f32 ? CALL(MXQ_ELEM_E2M1, true) : CALL(MXQ_ELEM_E2M1, false);     \
    case MXQ_ELEM_INT8: return f32 ? CALL(MXQ_ELEM_INT8, true) : CALL(MXQ_ELEM_INT8, false);     \
    case MXQ_ELEM_E5M2: return f32 ? CALL(MXQ_ELEM_E5M2, true) : CALL(MXQ_ELEM_E5M2, false);     \
    default: return cudaErrorInvalidValue;                                                       \
    }

cudaError_t launch_dequantize(const void* codes, const uint8_t* scales, int64_t n_blocks, int block_size, int elem, int dst_dtype, void* dst,
                              int sm_count, int64_t l2_bytes, int cb, int waves, cudaStream_t stream) {
    const bool f32 = dst_dtype == MXQ_HP_F32;
#define CALL(E, F) launch_flat<E, F>(codes, scales, n_blocks, block_size, dst, sm_count, l2_bytes, cb, waves, stream)
    MXQ_DISPATCH_ELEM_DT(elem, f32, CALL)
#undef CALL
}

cudaError_t launch_dequantize_strided(const void* codes, const uint8_t* scales, int ndim, const int64_t* sizes, const int64_t* cs,
                                      const int64_t* ss, int block_dim, int block_size, int elem, int dst_dtype, void* dst,
                                      cudaStream_t stream) {
    const bool f32 = dst_dtype == MXQ_HP_F32;
#define CALL(E, F) launch_strided<E, F>(codes, scales, ndim, sizes, cs, ss, block_dim, block_size, dst, stream)
    MXQ_DISPATCH_ELEM_DT(elem, f32, CALL)
#undef CALL
}

}  // namespace mxq
