// Device-side building blocks shared by the quantize / dequantize / GEMM kernels (sm_100a only).
//
// Arithmetic contract (distilled from the reference, see DESIGN.md "element-cast spec"):
//   quantize:   s = 255 if any exponent field in the block is 255, else clamp(maxE - max_pow2, 0, 254)
//               code = RNE_satfinite( x * 2^(127-s) )          (x*2^k is exact in fp32)
//   dequantize: out = RNE_target( decode(code) * 2^(s-127) )   (product exact in fp32)
// No fast-math, no FTZ: fp32 subnormals carry real values at the ends of the E8M0 range.
#pragma once
#include <cstdlib>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/mxq.h"

namespace mxq {

// ---- format table: torchmx/dtypes.py:34-92 -------------------------------------------
template <int ELEM> struct Fmt;
template <> struct Fmt<MXQ_ELEM_E4M3> { static constexpr int ebits = 4, mbits = 3, bias = 7, max_pow2 = 8; };
template <> struct Fmt<MXQ_ELEM_E3M2> { static constexpr int ebits = 3, mbits = 2, bias = 3, max_pow2 = 4; };
template <> struct Fmt<MXQ_ELEM_E2M3> { static constexpr int ebits = 2, mbits = 3, bias = 1, max_pow2 = 2; };
template <> struct Fmt<MXQ_ELEM_E2M1> { static constexpr int ebits = 2, mbits = 1, bias = 1, max_pow2 = 2; };
template <> struct Fmt<MXQ_ELEM_INT8> { static constexpr int ebits = 0, mbits = 7, bias = 0, max_pow2 = 6; };
template <> struct Fmt<MXQ_ELEM_E5M2> { static constexpr int ebits = 5, mbits = 2, bias = 15, max_pow2 = 15; };

// ---- 128/256-bit streaming global accesses (L1 no-allocate: every byte is touched once) ----
struct alignas(32) u32x8 { uint32_t v[8]; };

__device__ __forceinline__ u32x8 ldg256_stream(const void* p) {
    u32x8 r;
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg128_stream(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg64_stream(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg256_stream(void* p, const u32x8& r) {
    asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r.v[0]), "r"(r.v[1]), "r"(r.v[2]),
                 "r"(r.v[3]), "r"(r.v[4]), "r"(r.v[5]), "r"(r.v[6]), "r"(r.v[7])
                 : "memory");
}
__device__ __forceinline__ void stg128_stream(void* p, uint4 r) {
    asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(r.x), "r"(r.y), "r"(r.z), "r"(r.w) : "memory");
}
__device__ __forceinline__ void stg64_stream(void* p, uint2 r) {
    asm volatile("st.global.L1::no_allocate.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(r.x), "r"(r.y) : "memory");
}

// ---- the same accesses with an L2 evict-first policy (launches that stream more bytes than L2 holds) --------------------
// A line touched this way is among the first L2 replaces, so the read-once streams of a large launch do not push out the lines
// written at normal priority -- the codes a following dequantize reads back.  The policy is a per-instruction operand: no
// device or stream state outlives the kernel.
// Code bytes at the end of a large K1's output (and at the start of K2's back-to-front walk) that take the hints: 3/5 of L2.
// Beyond them the codes cannot be in L2 and the hints only cost.  B200, 1000 W, bench.py's sweep: a window of 1 / 0.6 / 0.4 /
// 0.25 L2 gave 1.170 / 1.166 / 1.171 / 1.183 ms per step (parent 1.208).
inline int64_t l2_handoff_window(int64_t l2_bytes) { return l2_bytes * 3 / 5; }

__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ u32x8 ldg256_evict_first(const void* p, uint64_t pol) {
    u32x8 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint4 ldg128_evict_first(const void* p, uint64_t pol) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.b32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
    return r;
}
// one byte through the read-only path (what __ldg does), L1 allocating: the neighbouring lanes read the neighbouring bytes
__device__ __forceinline__ uint32_t ldg8_evict_first(const uint8_t* p, uint64_t pol) {
    uint32_t r;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ void stg256_evict_first(void* p, const u32x8& r, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8}, %9;" ::"l"(p), "r"(r.v[0]), "r"(r.v[1]),
                 "r"(r.v[2]), "r"(r.v[3]), "r"(r.v[4]), "r"(r.v[5]), "r"(r.v[6]), "r"(r.v[7]), "l"(pol)
                 : "memory");
}

// ---- E8M0 helpers -------------------------------------------------------------------------
// shared exponent from the max of |bits| over the block (bf16: exponent field = bits >> 7)
template <int ELEM>
__device__ __forceinline__ int shared_exp_from_maxE(int maxE) {
    int s = maxE - Fmt<ELEM>::max_pow2;
    s = max(s, 0);
    s = min(s, 254);
    return maxE == 255 ? 255 : s;
}
// 2^(127-s) as fp32 for s in [0,254]; s == 254 needs the subnormal 2^-127
__device__ __forceinline__ float inv_scale_f32(int s) {
    return __uint_as_float(s <= 253 ? (uint32_t)(254 - s) << 23 : 0x00400000u);
}
// 2^(s-127) as fp32; s == 0 is the subnormal 2^-127, s == 255 is NaN (get_fp_scale, mx_quantization_utils.py:415-432)
__device__ __forceinline__ float scale_f32(int s) {
    return __uint_as_float(s == 0 ? 0x00400000u : (s == 255 ? 0x7FC00000u : (uint32_t)s << 23));
}

// ---- packed hardware conversions (F2FP) ------------------------------------------------------
// two fp32 -> two codes in one 16-bit value: low byte = first argument
template <int ELEM>
__device__ __forceinline__ uint32_t cvt_pair(float first, float second) {
    uint16_t r;
    if constexpr (ELEM == MXQ_ELEM_E4M3) asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(second), "f"(first));
    else if constexpr (ELEM == MXQ_ELEM_E5M2) asm("cvt.rn.satfinite.e5m2x2.f32 %0, %1, %2;" : "=h"(r) : "f"(second), "f"(first));
    else if constexpr (ELEM == MXQ_ELEM_E3M2) asm("cvt.rn.satfinite.e3m2x2.f32 %0, %1, %2;" : "=h"(r) : "f"(second), "f"(first));
    else if constexpr (ELEM == MXQ_ELEM_E2M3) asm("cvt.rn.satfinite.e2m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(second), "f"(first));
    else static_assert(ELEM < 0, "no pair conversion for this element type");
    return r;
}
// two fp32 -> one byte of two e2m1 codes, `first` in the HIGH nibble (torchmx/utils.py:145)
__device__ __forceinline__ uint32_t cvt_e2m1_byte(float first, float second) {
    uint32_t r;
    asm("{ .reg .b8 t; cvt.rn.satfinite.e2m1x2.f32 t, %1, %2; cvt.u32.u8 %0, t; }" : "=r"(r) : "f"(first), "f"(second));
    return r;
}
// two codes (low 16 bits of `pair`) -> f16x2 (exact)
template <int ELEM>
__device__ __forceinline__ uint32_t decode_pair_f16x2(uint32_t pair) {
    uint32_t r;
    uint16_t p = (uint16_t)pair;
    if constexpr (ELEM == MXQ_ELEM_E4M3) asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(r) : "h"(p));
    else if constexpr (ELEM == MXQ_ELEM_E5M2) asm("cvt.rn.f16x2.e5m2x2 %0, %1;" : "=r"(r) : "h"(p));
    else if constexpr (ELEM == MXQ_ELEM_E3M2) asm("cvt.rn.f16x2.e3m2x2 %0, %1;" : "=r"(r) : "h"(p));
    else if constexpr (ELEM == MXQ_ELEM_E2M3) asm("cvt.rn.f16x2.e2m3x2 %0, %1;" : "=r"(r) : "h"(p));
    else static_assert(ELEM < 0, "no pair decode for this element type");
    return r;
}
// one byte of two e2m1 codes -> f16x2; low half = LOW nibble (the odd element), high half = HIGH nibble
__device__ __forceinline__ uint32_t decode_e2m1_byte_f16x2(uint32_t byte) {
    uint32_t r;
    asm("{ .reg .b8 t; cvt.u8.u32 t, %1; cvt.rn.f16x2.e2m1x2 %0, t; }" : "=r"(r) : "r"(byte));
    return r;
}
__device__ __forceinline__ float f16lo_to_f32(uint32_t h2) {
    float f;
    asm("{ .reg .b16 lo, hi; mov.b32 {lo, hi}, %1; cvt.f32.f16 %0, lo; }" : "=f"(f) : "r"(h2));
    return f;
}
__device__ __forceinline__ float f16hi_to_f32(uint32_t h2) {
    float f;
    asm("{ .reg .b16 lo, hi; mov.b32 {lo, hi}, %1; cvt.f32.f16 %0, hi; }" : "=f"(f) : "r"(h2));
    return f;
}
// two fp32 -> bf16x2 (RNE, subnormals kept): low half = first
// Programmatic dependent launch (sm_90+): a grid launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// while its predecessor in the stream is still running; it must execute pdl_wait() before touching anything the predecessor
// wrote (or may still read).  pdl_launch_dependents() lets a following such grid be scheduled early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Host side: launch `kernel` with the programmatic-serialization attribute (it starts while its predecessor in the stream drains
// and must call pdl_wait() before touching global memory).  The small row-wise / elementwise kernels between the MX linears of a
// decoder layer last 3-6 us at decode sizes, of which the launch itself is a good part: started early, their set-up overlaps the
// predecessor's tail.  MXQ_GLUE_PDL=0 (read once) launches them the ordinary way.
inline bool glue_pdl_enabled() {
    static const bool on = [] { const char* v = getenv("MXQ_GLUE_PDL"); return !(v && v[0] == '0'); }();
    return on;
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = glue_pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float first, float second) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(second), "f"(first));
    return r;
}

// ---- hw_exact NaN-block quirk (mx_quantization_utils.py:331-349, 367-372, 387) --------------------
// In a block whose scale is 255 the reference's integer path still writes the *subnormal* code
// of finite elements whose exponent field lies in [255-bias-mbits, 255-bias]; sign is forced to 0.
template <int ELEM>
__device__ __forceinline__ uint32_t hw_exact_nanblock_code(uint32_t h) {
    constexpr int mbits = Fmt<ELEM>::mbits, bias = Fmt<ELEM>::bias;
    const int E = (h >> 7) & 0xFF, m = h & 0x7F;
    const int ne = E - 255 + bias;
    if (E == 0 || E == 255 || ne > 0 || ne < -mbits) return 0;
    const int subman = 64 | ((m >> 4) << 3) | (((m & 0xF) != 0) << 2);
    const int shift = 7 - mbits - ne;  // 7-mbits .. 7
    const int reduced = subman >> shift;
    const int rem = subman & ((1 << shift) - 1);
    const int half = 1 << (shift - 1);
    const int up = (rem & half) && ((reduced & 1) || (rem & (half - 1)));
    const int r = reduced + up;
    return r > (1 << mbits) - 1 ? 0 : r;
}

// ---- scalar reference-free element cast used by the generic (any block size) kernels -----------
template <int ELEM>
__device__ __forceinline__ uint32_t quantize_one(float x, int s) {
    const float y = x * inv_scale_f32(s);
    if constexpr (ELEM == MXQ_ELEM_INT8) {
        float t = fmaf(x, inv_scale_f32(s), 12582912.0f);
        t = fminf(fmaxf(t, 12582912.0f - 127.0f), 12582912.0f + 127.0f);
        return __float_as_uint(t) & 0xFF;
    } else if constexpr (ELEM == MXQ_ELEM_E2M1) {
        return cvt_e2m1_byte(0.0f, y) & 0xF;
    } else {
        return cvt_pair<ELEM>(y, 0.0f) & 0xFF;
    }
}

template <int ELEM>
__device__ __forceinline__ float decode_one(uint32_t c) {
    if constexpr (ELEM == MXQ_ELEM_INT8) return (float)(int)(int8_t)c;
    else if constexpr (ELEM == MXQ_ELEM_E2M1) return f16lo_to_f32(decode_e2m1_byte_f16x2(c & 0xF));
    else return f16lo_to_f32(decode_pair_f16x2<ELEM>(c & 0xFF));
}

}  // namespace mxq
