/*
 * mx_oracle.c -- CPU restatement of torchmx's MX quantize / dequantize arithmetic.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under torchmx_b200/ may import, link or
 * execute this file; it exists so that tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs have an independent checker.
 *
 * Parity status: PINNED.  oracle/gen_golden.py imports the real reference from
 * /root/reference (through oracle/_shim/torchao) and checks this file against it
 * bit-for-bit on the exhaustive grid (every bf16 pattern under every block
 * exponent, every (code, scale) pair) for all element types and both values of
 * MX_HARDWARE_EXACT_QUANTIZATION; the digests are committed in
 * tests/golden/digests.json and re-checked by tests/test_oracle_golden.py.
 * Exception: float8_e5m2 and fp32 input are not torchmx features at all
 * (torchmx/dtypes.py:143-149, torchmx/mx_tensor.py:59-61), so there is no
 * reference output to pin them to.  The e5m2 path is pinned instead against a
 * restatement built on torch's own float8_e5m2 cast (tests/test_e5m2_reference.py);
 * fp32 input stays "parity unpinned" (header of DESIGN.md).
 *
 * Every function cites the reference lines (relative to /root/reference) it follows.
 * Plain C99, no dependencies beyond libm / pthreads.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ---------- element format table: torchmx/dtypes.py:34-92 ---------------- */
enum { MXO_E4M3 = 0, MXO_E3M2 = 1, MXO_E2M3 = 2, MXO_E2M1 = 3, MXO_INT8 = 4, MXO_E5M2 = 5, MXO_NELEM = 6 };

typedef struct {
    int ebits, mbits, bias, max_pow2;
    float max;
} fmt_t;

static const fmt_t FMT[MXO_NELEM] = {
    /* e4m3 dtypes.py:34-44 */ {4, 3, 7, 8, 448.0f},
    /* e3m2 dtypes.py:46-56 */ {3, 2, 3, 4, 28.0f},
    /* e2m3 dtypes.py:58-68 */ {2, 3, 1, 2, 7.5f},
    /* e2m1 dtypes.py:70-80 */ {2, 1, 1, 2, 6.0f},
    /* int8 dtypes.py:82-92 */ {0, 7, 0, 6, 127.0f},
    /* e5m2: extension, not in the reference; constants analogous to dtypes.py:34-44 */ {5, 2, 15, 15, 57344.0f},
};

static inline float bits_f32(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f32_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline float bf16_to_f32(uint16_t h) { return bits_f32((uint32_t)h << 16); }

/* fp32 -> bf16, round to nearest even, NaN kept quiet (what torch's .to(bfloat16) does). */
static inline uint16_t f32_to_bf16_rne(float f) {
    uint32_t u = f32_bits(f);
    if ((u & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((u >> 16) | 0x0040u);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}

/* ---------- shared exponent: torchmx/mx_quantization_utils.py:502-558 ---- */
/* exp_field[i] is the 8-bit exponent field of element i (bf16: bits>>7, fp32: bits>>23). */
static inline uint8_t shared_exponent(const int *exp_field, int n, int elem) {
    int mx = 0;
    for (int i = 0; i < n; ++i) if (exp_field[i] > mx) mx = exp_field[i];       /* :542 amax */
    if (mx == 255) return 255;                                                   /* :552-556 */
    int s = mx - FMT[elem].max_pow2;                                             /* :546 */
    if (s < 0) s = 0;
    if (s > 254) s = 254;                                                        /* :545-549 */
    return (uint8_t)s;
}

/* ---------- round_to_even: torchmx/mx_quantization_utils.py:149-215 ------ */
static inline int rte_shift(int mantissa, int shift) {
    /* callers guarantee 1 <= shift <= 14; the reference evaluates it on every lane
       and masks afterwards, we only evaluate it where the mask selects it. */
    int reduced = mantissa >> shift;                                             /* :184 */
    int rem = mantissa & ((1 << shift) - 1);                                     /* :187-189 */
    int round_bit = rem >> (shift - 1);                                          /* :192-194 */
    int odd = reduced & 1;                                                       /* :200 */
    int rest = (rem & ((1 << (shift - 1)) - 1)) != 0;                            /* :201-203 */
    return reduced + ((round_bit > 0) && (odd || rest));                         /* :206-213 */
}

/* ---------- hw_exact element cast: mx_quantization_utils.py:253-412 ------ */
static inline uint8_t cast_hw_exact(uint16_t h, int s, int elem) {
    const int ebits = FMT[elem].ebits, mbits = FMT[elem].mbits, bias = FMT[elem].bias;
    int sign = h >> 15, exp = (h >> 7) & 0xFF, man = h & 0x7F;                   /* :285-287, :16-48 */
    if (s == 255) sign = 0;                                                      /* :289-291 */
    const int is_zero = (h & 0x7FFF) == 0;                                       /* :293 (x == 0 is true for +-0, false for NaN) */
    if (exp == 0 && !is_zero) {                                                  /* :295 bf16 subnormal input */
        int lead = 6;
        while (!((man >> lead) & 1)) --lead;                                     /* :227-250 leading one, 6..0 */
        man = (man << (7 - lead)) & 0x7F;                                        /* :302,306 */
        exp = -(6 - lead);                                                       /* :303,310 */
    }
    int new_exp = exp - s + bias;                                                /* :313-315 */
    int rounded = 0;                                                             /* :319 */
    if (new_exp > 0) rounded = rte_shift(man, 7 - mbits);                        /* :322-328 */
    int sub = (new_exp <= 0) && (new_exp >= -mbits) && !is_zero;                 /* :331-333 */
    if (sub) {
        int sticky = (man & 0xF) != 0;                                           /* :336-338 */
        int subman = (1 << 6) | ((man >> 4) << 3) | (sticky << 2);               /* :339 */
        rounded = rte_shift(subman, 7 - mbits - new_exp);                        /* :341-349 */
    }
    if (rounded > (1 << mbits) - 1) { rounded = 0; new_exp += 1; }               /* :352-356 */
    sub = (new_exp <= 0) && (new_exp >= -mbits) && !is_zero;                     /* :359-361 */
    const int underflow = (new_exp < -mbits) || (s == 255) || is_zero;           /* :367-371 */
    int sat = new_exp > (1 << ebits) - 1;                                        /* :375 */
    int maxmag = (1 << (mbits + ebits)) - 1;                                     /* :376 */
    if (elem == MXO_E4M3) {                                                      /* :377-382 */
        sat = sat || (new_exp == 15 && rounded == 7);
        maxmag = 0x7E;
    }
    int z = 0;
    if (underflow) z = 0;                                                        /* :372 */
    if (sat) z = maxmag;                                                         /* :384 */
    if (sub) z = rounded;                                                        /* :387 -- written AFTER the underflow mask: in a
                                                                                    NaN-scale block this re-emits a subnormal code */
    if (!(sat || underflow || sub)) {                                            /* :390-397 */
        int e = new_exp < 1 ? 1 : new_exp;
        if (e > (1 << ebits) - 1) e = (1 << ebits) - 1;
        z = (e << mbits) | rounded;
    }
    return (uint8_t)((sign << (mbits + ebits)) | (z & 0xFF));                    /* :400-402 */
}

/* ---------- simulated element casts: mx_quantization_utils.py:435-499 ---- */

/* torch's float32 -> float8_e4m3fn conversion (c10/util/Float8_e4m3fn.h, PyTorch 2.x), the
   cast used at mx_quantization_utils.py:481.  Published algorithm: >= 480 -> NaN code;
   below the smallest normal (2^-6) add a magic float so the FPU does the RNE;
   otherwise rebias + integer RNE on the 20 dropped bits. */
static inline uint8_t f32_to_e4m3fn(float f) {
    uint32_t u = f32_bits(f);
    const uint32_t sign = u & 0x80000000u;
    u ^= sign;
    uint8_t r;
    if (u >= (1087u << 20)) {
        r = 0x7F;
    } else if (u < (121u << 23)) {
        const uint32_t magic = 141u << 23;
        r = (uint8_t)(f32_bits(bits_f32(u) + bits_f32(magic)) - magic);
    } else {
        const uint32_t odd = (u >> 20) & 1u;
        u += ((uint32_t)(7 - 127) << 23) + 0x7FFFFu;
        u += odd;
        r = (uint8_t)(u >> 20);
    }
    return (uint8_t)(r | (sign >> 24));
}

/* torch's float32 -> float8_e5m2 (c10/util/Float8_e5m2.h): fp32 -> fp16-style RNE on the top
   byte.  Extension only (the reference has no e5m2 element type). */
static inline uint8_t f32_to_e5m2(float f) {
    uint32_t u = f32_bits(f);
    const uint32_t sign = u & 0x80000000u;
    u ^= sign;
    uint8_t r;
    if (u >= (143u << 23)) {                 /* >= 65536: inf / nan */
        r = (u > 0x7F800000u) ? 0x7F : 0x7C;
    } else if (u < (113u << 23)) {           /* below 2^-14: subnormal target */
        const uint32_t magic = 134u << 23;
        r = (uint8_t)(f32_bits(bits_f32(u) + bits_f32(magic)) - magic);
    } else {
        const uint32_t odd = (u >> 21) & 1u;
        u += ((uint32_t)(15 - 127) << 23) + 0xFFFFFu;
        u += odd;
        r = (uint8_t)(u >> 21);
    }
    return (uint8_t)(r | (sign >> 24));
}

/* torchao 0.6.1 prototype/mx_formats/custom_cast.py `_f32_to_f4_or_f6_unpacked` (third-party,
   not under /root/reference; pinned version pyproject.toml:23).  Call sites:
   mx_quantization_utils.py:483,485,487.  Published algorithm: saturate at max_normal;
   below min_normal add a magic float; else rebias + integer RNE; re-attach sign. */
static inline uint8_t f32_to_fx_unpacked(float f, int ebits, int mbits) {
    const int bias = (1 << (ebits - 1)) - 1;
    const int drop = 23 - mbits;
    const float max_normal = ldexpf(2.0f - ldexpf(1.0f, -mbits), (1 << ebits) - 1 - bias);
    const float min_normal = ldexpf(1.0f, 1 - bias);
    uint32_t u = f32_bits(f);
    const uint32_t sign = u & 0x80000000u;
    u ^= sign;
    const float a = bits_f32(u);
    uint32_t r;
    if (a >= max_normal) {
        r = (1u << (ebits + mbits)) - 1u;
    } else if (a < min_normal) {
        const uint32_t magic = (uint32_t)((127 - bias) + (23 - mbits) + 1) << 23;
        r = f32_bits(a + bits_f32(magic)) - magic;
    } else {
        const uint32_t odd = (u >> drop) & 1u;
        uint32_t v = u + ((uint32_t)(bias - 127) << 23) + ((1u << (drop - 1)) - 1u) + odd;
        r = v >> drop;
    }
    return (uint8_t)(r | ((sign >> (31 - mbits - ebits)) & (1u << (ebits + mbits))));
}

/* get_fp_scale: mx_quantization_utils.py:415-432 (fp32 2^(s-127), NaN for s == 255). */
static inline float fp_scale(int s) { return s == 255 ? NAN : ldexpf(1.0f, s - 127); }

static inline uint8_t cast_simulated(float x, int s, int elem) {
    const float mx = FMT[elem].max;
    float y = x / fp_scale(s);                                                   /* :469-471 fp32 divide */
    if (!(y != y)) { if (y < -mx) y = -mx; if (y > mx) y = mx; }                 /* torch.clamp keeps NaN */
    if (y != y) y = 0.0f;                                                        /* :473 NaN -> +0 */
    switch (elem) {
    case MXO_E4M3: return f32_to_e4m3fn(y);                                      /* :479-481 */
    case MXO_E2M3: return f32_to_fx_unpacked(y, 2, 3);                           /* :482-483 */
    case MXO_E3M2: return f32_to_fx_unpacked(y, 3, 2);                           /* :484-485 */
    case MXO_E2M1: return f32_to_fx_unpacked(y, 2, 1);                           /* :486-487 */
    case MXO_INT8: return (uint8_t)(int8_t)nearbyintf(y);                        /* :489-496 torch.round = RNE */
    default:       return f32_to_e5m2(y);                                        /* extension */
    }
}

/* ---------- quantize_mx: torchmx/mx_tensor.py:36-96 ---------------------- */
/*
 * src      : n_blocks * block_size elements, bf16 bit patterns (src_is_f32 == 0) or fp32
 * scales   : n_blocks bytes (E8M0)
 * codes    : one byte per element; for MXO_E2M1 packed two per byte, element 2i in the HIGH
 *            nibble (torchmx/utils.py:120-145), i.e. n_blocks*block_size/2 bytes
 * hw_exact : env.MX_EXACT_QUANTIZATION == "True" (mx_tensor.py:80-90); ignored for int8
 */
static int quantize_range(const void *src, int src_is_f32, int64_t b0, int64_t b1, int block_size,
                          int elem, int hw_exact, uint8_t *scales, uint8_t *codes) {
    int *ef = (int *)malloc(sizeof(int) * (size_t)block_size);
    uint8_t *tmp = (uint8_t *)malloc((size_t)block_size);
    if (!ef || !tmp) { free(ef); free(tmp); return -1; }
    const int use_exact = hw_exact && elem != MXO_INT8 && elem != MXO_E5M2 && !src_is_f32;
    for (int64_t b = b0; b < b1; ++b) {
        const uint16_t *h = (const uint16_t *)src + b * block_size;
        const float *f = (const float *)src + b * block_size;
        for (int i = 0; i < block_size; ++i)
            ef[i] = src_is_f32 ? (int)((f32_bits(f[i]) >> 23) & 0xFF) : ((h[i] >> 7) & 0xFF);
        const int s = shared_exponent(ef, block_size, elem);
        scales[b] = (uint8_t)s;
        for (int i = 0; i < block_size; ++i) {
            if (use_exact) tmp[i] = cast_hw_exact(h[i], s, elem);
            else tmp[i] = cast_simulated(src_is_f32 ? f[i] : bf16_to_f32(h[i]), s, elem);
        }
        if (elem == MXO_E2M1) {
            /* pack_uint4 works on the flattened tensor (utils.py:144-145); block_size*n_blocks is
               even, and we require an even block_size so pairs never straddle a block here.  Odd
               block sizes are handled by the caller through mxo_pack_uint4. */
            uint8_t *out = codes + (b * block_size) / 2;
            for (int i = 0; i < block_size / 2; ++i) out[i] = (uint8_t)((tmp[2 * i] << 4) | (tmp[2 * i + 1] & 0xF));
        } else {
            memcpy(codes + b * block_size, tmp, (size_t)block_size);
        }
    }
    free(ef); free(tmp);
    return 0;
}

typedef struct {
    const void *src; int src_is_f32; int64_t b0, b1; int block_size, elem, hw_exact;
    uint8_t *scales, *codes; int rc;
} qjob_t;

static void *qjob_main(void *p) {
    qjob_t *j = (qjob_t *)p;
    j->rc = quantize_range(j->src, j->src_is_f32, j->b0, j->b1, j->block_size, j->elem, j->hw_exact, j->scales, j->codes);
    return NULL;
}

int mxo_quantize(const void *src, int src_is_f32, int64_t n_blocks, int block_size, int elem,
                 int hw_exact, uint8_t *scales, uint8_t *codes, int n_threads) {
    if (elem < 0 || elem >= MXO_NELEM || block_size < 1) return -2;
    if (elem == MXO_E2M1 && (block_size & 1)) return -3;
    if (n_threads < 1) n_threads = 1;
    if (n_threads == 1 || n_blocks < 4 * n_threads)
        return quantize_range(src, src_is_f32, 0, n_blocks, block_size, elem, hw_exact, scales, codes);
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)n_threads);
    qjob_t *jobs = (qjob_t *)malloc(sizeof(qjob_t) * (size_t)n_threads);
    int rc = 0;
    for (int t = 0; t < n_threads; ++t) {
        jobs[t] = (qjob_t){src, src_is_f32, n_blocks * t / n_threads, n_blocks * (t + 1) / n_threads,
                           block_size, elem, hw_exact, scales, codes, 0};
        pthread_create(&th[t], NULL, qjob_main, &jobs[t]);
    }
    for (int t = 0; t < n_threads; ++t) { pthread_join(th[t], NULL); if (jobs[t].rc) rc = jobs[t].rc; }
    free(th); free(jobs);
    return rc;
}

/* ---------- dequantize_mx: torchmx/mx_tensor.py:123-164 ------------------ */

/* decode one element code to its exact value: mx_quantization_utils.py:93-146
   (e4m3: reinterpret as float8_e4m3fn :119-120; fp6/fp4: bit-field decode :125-144;
   int8: the integer itself, mx_tensor.py:152-153). */
static inline float decode_elem(uint8_t c, int elem) {
    if (elem == MXO_INT8) return (float)(int8_t)c;
    const int ebits = FMT[elem].ebits, mbits = FMT[elem].mbits, bias = FMT[elem].bias;
    if (elem == MXO_E4M3 && (c & 0x7F) == 0x7F) return NAN;
    if (elem == MXO_E5M2 && (c & 0x7F) > 0x7C) return NAN;
    if (elem == MXO_E5M2 && (c & 0x7F) == 0x7C) return (c & 0x80) ? -INFINITY : INFINITY;
    const int e = (c >> mbits) & ((1 << ebits) - 1);                             /* :125-127 */
    const int m = c & ((1 << mbits) - 1);                                        /* :129 */
    const int sgn = (c >> (mbits + ebits)) & 1;                                  /* :131 (valid codes only) */
    float frac = (float)m / (float)(1 << mbits);                                 /* :136 */
    if (e != 0) frac += 1.0f;                                                    /* :137-139 */
    const float v = ldexpf(frac, (e == 0 ? 1 : e) - bias);                       /* :140-144 */
    return sgn ? -v : v;
}

/*
 * codes/scales laid out as produced by mxo_quantize (blocks contiguous, fp4 packed).
 * target_is_f32 == 0: dst is bf16 bit patterns; arithmetic is a bf16 x bf16 -> bf16 product
 * (mx_tensor.py:157-162: both factors are cast to target_dtype first), which is the exact
 * product rounded once.  target_is_f32 == 1: fp32 product.
 */
static void dequantize_range(const uint8_t *codes, const uint8_t *scales, int64_t b0, int64_t b1, int block_size,
                             int elem, int target_is_f32, void *dst) {
    for (int64_t b = b0; b < b1; ++b) {
        const float sc = fp_scale(scales[b]);
        for (int i = 0; i < block_size; ++i) {
            const int64_t idx = b * block_size + i;
            uint8_t c;
            if (elem == MXO_E2M1) {
                const uint8_t byte = codes[idx >> 1];
                c = (idx & 1) ? (byte & 0xF) : (byte >> 4);                      /* utils.py:96-117 */
            } else {
                c = codes[idx];
            }
            /* decode(c) has <= 8 significant bits and sc is a power of two: the fp32 product is
               exact (fp32 subnormals included), so one rounding to the target remains. */
            const float v = decode_elem(c, elem) * sc;
            if (target_is_f32) ((float *)dst)[idx] = v;
            else ((uint16_t *)dst)[idx] = f32_to_bf16_rne(v);
        }
    }
}

typedef struct {
    const uint8_t *codes, *scales; int64_t b0, b1; int block_size, elem, target_is_f32; void *dst;
} djob_t;

static void *djob_main(void *p) {
    djob_t *j = (djob_t *)p;
    dequantize_range(j->codes, j->scales, j->b0, j->b1, j->block_size, j->elem, j->target_is_f32, j->dst);
    return NULL;
}

int mxo_dequantize_mt(const uint8_t *codes, const uint8_t *scales, int64_t n_blocks, int block_size,
                      int elem, int target_is_f32, void *dst, int n_threads) {
    if (elem < 0 || elem >= MXO_NELEM || block_size < 1) return -2;
    if (elem == MXO_E2M1 && (block_size & 1)) return -3;
    if (n_threads < 1) n_threads = 1;
    if (n_threads == 1 || n_blocks < 4 * n_threads) {
        dequantize_range(codes, scales, 0, n_blocks, block_size, elem, target_is_f32, dst);
        return 0;
    }
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)n_threads);
    djob_t *jobs = (djob_t *)malloc(sizeof(djob_t) * (size_t)n_threads);
    for (int t = 0; t < n_threads; ++t) {
        jobs[t] = (djob_t){codes, scales, n_blocks * t / n_threads, n_blocks * (t + 1) / n_threads,
                           block_size, elem, target_is_f32, dst};
        pthread_create(&th[t], NULL, djob_main, &jobs[t]);
    }
    for (int t = 0; t < n_threads; ++t) pthread_join(th[t], NULL);
    free(th); free(jobs);
    return 0;
}

int mxo_dequantize(const uint8_t *codes, const uint8_t *scales, int64_t n_blocks, int block_size,
                   int elem, int target_is_f32, void *dst) {
    return mxo_dequantize_mt(codes, scales, n_blocks, block_size, elem, target_is_f32, dst, 1);
}

/* pack/unpack helpers: torchmx/utils.py:96-145 (flattened tensor, even element -> high nibble) */
void mxo_pack_uint4(const uint8_t *in, int64_t n, uint8_t *out) {
    for (int64_t i = 0; i < n / 2; ++i) out[i] = (uint8_t)((in[2 * i] << 4) | (in[2 * i + 1] & 0xF));
}
void mxo_unpack_uint4(const uint8_t *in, int64_t n_bytes, uint8_t *out) {
    for (int64_t i = 0; i < n_bytes; ++i) { out[2 * i] = in[i] >> 4; out[2 * i + 1] = in[i] & 0xF; }
}

/*
 * MX matmul reference: torchmx/ops.py:29-41, 60-68, 99-119 -- dequantize both operands to bf16
 * (exact), multiply-accumulate, round the result to bf16.  The reference accumulates in fp32 in
 * cuBLAS/MKL order; this restatement accumulates in double so that it is the order-free target
 * the GPU kernel's tolerance is measured from.  a: [M,K] bf16 bits, b: [N,K] bf16 bits (K-major
 * both), out: [M,N] fp32 (un-rounded, caller rounds / compares).
 */
int mxo_gemm_nt_bf16(const uint16_t *a, const uint16_t *b, int64_t M, int64_t N, int64_t K, float *out) {
    for (int64_t m = 0; m < M; ++m)
        for (int64_t n = 0; n < N; ++n) {
            double acc = 0.0;
            const uint16_t *ar = a + m * K, *br = b + n * K;
            for (int64_t k = 0; k < K; ++k) acc += (double)bf16_to_f32(ar[k]) * (double)bf16_to_f32(br[k]);
            out[m * N + n] = (float)acc;
        }
    return 0;
}

int mxo_version(void) { return 1; }
