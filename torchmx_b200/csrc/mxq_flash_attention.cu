// K4b: the MX attention block of the reference as ONE kernel (torchmx/layers/mx_llama_attention.py:195-243):
//
//     scores = matmul(Q_mx, K_mx^T)                  (MX operands blocked along head_dim; bf16 result)
//     P      = to_mx(softmax(scores * scaling + mask, fp32).to(bf16), attention_weights_config)   (blocked along the kv axis)
//     out    = matmul(P_mx, V_mx)                    (V quantized along the kv axis)
//
// The unfused path (K3 bmm -> K4a -> K3 bmm) writes the [b, h, q, kv] scores (268 MB per Llama-8B layer at 2048 tokens) and the
// codes of P to HBM and reads them back.  Here neither exists in HBM: both contractions run on tcgen05 block-scaled MMAs
// (kind::mxf8f6f4, E8M0 scale factors in TMEM), the accumulator of the first is read by the softmax threads straight from TMEM,
// and the codes + scales of P go through shared memory into the second.
//
// The reference quantizes the NORMALISED probabilities, so the row maximum and the row sum must be final before the first code
// of a row exists: an online (rescaling) softmax cannot reproduce the codes.  The kernel therefore makes three passes over the
// key tiles of a query tile -- (A) row maximum, (B) row sum of expf(x - max), (C) P, its MX quantization and P @ V -- and
// recomputes Q K^T in each (the tensor core has the time: the kernel is bound by the fp32 softmax arithmetic).  Every rounding
// step is K4a's (mxq_softmax_core.cuh), and the per-block sums are added in K4a's order, so the codes of P are K4a's bit for bit.
//
// CTA = 256 query rows of one (batch, head) = two query tiles of 128 rows, each with its own 128 x 64 score tile and 128 x 128
// output accumulator in TMEM, sharing the K / V tiles the TMA warp streams in.
//   warps 0..15  softmax: query tile (warp >> 3) x MX block of the score tile (sub = (warp >> 2) & 1) x TMEM lane quadrant.  TWO
//                threads per query row, one per 32-column block of every 64-column score tile: tcgen05.ld the block, K4a's
//                arithmetic, P codes -> swizzled shared-memory tile + scale bytes in the tcgen05.cp layout; finally drain half
//                of the row's output accumulator each.  What the two threads of a row must agree on goes through shared memory
//                behind a 256-thread named barrier per query tile.
//   warp 16      TMA producer: Q tiles once, then per pass the K tiles (128 keys x 128 B) and, in pass C, the V^T tiles
//                (128 channels x 128 keys)
//   warp 17      MMA issuer (one elected lane): S = Q K^T as two N = 64 halves per 128-key chunk, O += P V per chunk
//   warp 18      scale-factor loader: Q / K / V E8M0 scales from their reference layout into the tcgen05.cp chunk layout
// (At most 128 query rows per (batch, head) -- decode -- run a one-tile variant: eight softmax warps, two CTAs per SM; see Cfg.)
// Causal attention without an explicit mask skips the key chunks a query tile's rows cannot see; with an explicit additive mask
// pass A records the largest score of every (row, slot) and passes B / C skip the slots that are dead for a whole tile.  A slot
// is 2^slot_shift consecutive chunks, as few as keep a row at 64 slots (one chunk per slot up to 8192 keys).
// The key axis may be any multiple of 32 up to MXQ_FLASH_MAX_KV (a ragged last chunk is zero-filled by TMA and hidden).
// RAGGED instantiations (kv_pitch > 0) read the first kv_valid keys of K / V buffers pitched for kv_pitch keys -- a KV cache read
// in place at whatever length it has.  They compute exactly what the kernel computes on contiguous copies of the first
// n = ceil128(kv_valid) keys (zero codes in the tail) with causal off and the mask mask' = caller's mask (or zeros), -inf on every
// key the causal rule hides and on every key >= kv_valid: here kv_len is n, and the -inf keys are added in scores_of.  Nothing at
// or past kv_valid is read: the tensor maps end there (TMA zero-fills), and the scale loader feeds the neutral scale 127.
#include <cstring>

#include "mxq_softmax_core.cuh"
#include "mxq_tc.cuh"

namespace mxq {
namespace gemm {
namespace fa {

constexpr int QT = 128;     // query rows per warpgroup
constexpr int KC = 128;     // keys per chunk: four MX blocks of P = one 32-bit scale word per row
constexpr int HD = 128;     // head_dim
constexpr int kWgThreads = 256;  // softmax threads per query tile: two per row
constexpr int TILE_BYTES = 128 * 128;

// TILES = query tiles (of 128 rows) per CTA.  2: the prefill configuration described above, one CTA per SM.  1: queries of at most
// 128 rows per (batch, head) -- decode, where the grouped query heads of a key / value head are the rows -- with eight softmax
// warps, shallower K / V rings and half the tensor memory, so that TWO CTAs share an SM: a decode step is hundreds of small CTAs
// whose time is a chain of barrier round trips, not bandwidth.
template <int TILES>
struct Cfg {
    static constexpr int K_STAGES = TILES == 2 ? 3 : 2, V_STAGES = TILES == 2 ? 2 : 1;
    static constexpr int kSoftmaxWarps = 8 * TILES;
    static constexpr int kThreads = kSoftmaxWarps * 32 + 96;
    // TMEM columns
    static constexpr uint32_t TM_S = 0;                       // + 64 * wg
    static constexpr uint32_t TM_O = 64 * TILES;              // + 128 * wg
    static constexpr uint32_t TM_SFQ = TM_O + 128 * TILES;    // + 4 * wg
    static constexpr uint32_t TM_SFK = TM_SFQ + 4 * TILES;    // + 8 * (chunk & 1) + 4 * half
    static constexpr uint32_t TM_SFP = TM_SFK + 16;           // + 4 * wg
    static constexpr uint32_t TM_SFV = TM_SFP + 4 * TILES;    // + 4 * (chunk & 1)
    static constexpr int TMEM_COLS = TILES == 2 ? 512 : 256;
    static_assert(TM_SFV + 8 <= TMEM_COLS, "tensor memory budget");
};

template <int TILES>
struct SmemT {
    static constexpr int K_STAGES = Cfg<TILES>::K_STAGES, V_STAGES = Cfg<TILES>::V_STAGES;
    static constexpr int OFF_Q = 0;
    static constexpr int OFF_K = OFF_Q + TILES * TILE_BYTES;
    static constexpr int OFF_V = OFF_K + K_STAGES * TILE_BYTES;
    static constexpr int OFF_P = OFF_V + V_STAGES * TILE_BYTES;
    static constexpr int OFF_SFQ = OFF_P + TILES * TILE_BYTES;
    static constexpr int OFF_SFK = OFF_SFQ + TILES * 512;             // per stage: two 512-byte chunks (keys 0..63, 64..127)
    static constexpr int OFF_SFV = OFF_SFK + K_STAGES * 1024;
    static constexpr int OFF_SFP = OFF_SFV + V_STAGES * 512;
    static constexpr int OFF_CMAX = OFF_SFP + TILES * 512;            // [wg][slot < 64][row] bf16: largest score of the slot's chunks, from pass A
    static constexpr int OFF_LIVE = OFF_CMAX + TILES * 64 * 128 * 2;  // [wg][2] words: slots with a row that still counts after the row maximum is known
    static constexpr int OFF_XCH = OFF_LIVE + 16;                     // [wg][parity 2][sub 2][value 2][row 128] fp32: what a row's two threads exchange per chunk
    static constexpr int OFF_XMAX = OFF_XCH + TILES * 1024 * 4;       // [wg][sub][row] fp32: partial row maxima
    static constexpr int OFF_BAR = OFF_XMAX + TILES * 256 * 4;
    // q_full, qsf_full, k_full/ksf_full/k_empty[K_STAGES], v_full/vsf_full/v_empty[V_STAGES], sa_full/sa_free[2][2],
    // sc_full/sc_free/p_full/p_free/o_full[2]
    static constexpr int NUM_BARS = 2 + 3 * K_STAGES + 3 * V_STAGES + 18 + 2;
    static constexpr int OFF_TMEM_PTR = OFF_BAR + NUM_BARS * 8;
    static constexpr int TOTAL = OFF_TMEM_PTR + 16;
    static constexpr int DYN_BYTES = TOTAL + 1024;
    static_assert(DYN_BYTES <= (TILES == 2 ? 227 : 113) * 1024, "shared memory budget");
};

struct Params {
    const uint8_t* q_sf; const uint8_t* k_sf; const uint8_t* v_sf;
    const uint16_t* mask; int64_t mask_sb, mask_sh, mask_sq; int mask_vec;
    uint16_t* out; int64_t out_sb, out_sh, out_sq;
    uint8_t* p_codes; uint8_t* p_scales;
    int batch, heads, kv_heads, q_len, kv_len;
    int causal, causal_offset, skip_hidden_chunks;
    int layout;  // sm::sum_layout of a row of kv_len / 32 blocks
    int slot_shift;  // a live-chunk slot is 2^slot_shift chunks: the smallest that gives a row at most 64 slots
    float scaling;
    uint32_t idesc_qk, idesc_pv;
    uint32_t flags;
    int q_tiles;
    int kv_valid, hide_offset, kv_pitch;  // RAGGED: keys that exist; a row q sees keys < min(kv_valid, q + hide_offset + 1); key pitch
};

__device__ __forceinline__ uint32_t to_e4m3_pair(uint32_t h2) {  // f16x2 -> two e4m3 bytes (exact for every fp6 / fp4 value)
    uint16_t r;
    asm("cvt.rn.satfinite.e4m3x2.f16x2 %0, %1;" : "=h"(r) : "r"(h2));
    return r;
}

// the 32 codes of a block as the tensor core wants them: one byte per element in an 8-bit container (e5m2 as it is, every other
// element type as the E4M3 byte of the same value -- exact)
template <int ELEM>
__device__ __forceinline__ void container_bytes(const uint32_t (&out)[(ELEM == MXQ_ELEM_E2M1) ? 4 : 8], uint32_t (&c)[8]) {
    if constexpr (ELEM == MXQ_ELEM_E4M3 || ELEM == MXQ_ELEM_E5M2) {
#pragma unroll
        for (int i = 0; i < 8; ++i) c[i] = out[i];
    } else if constexpr (ELEM == MXQ_ELEM_E2M1) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const uint32_t b0 = (out[i] >> (16 * k)) & 0xFF, b1 = (out[i] >> (16 * k + 8)) & 0xFF;
                // the earlier element sits in the HIGH nibble = high f16 half: swap the halves
                const uint32_t p0 = to_e4m3_pair(__byte_perm(decode_e2m1_byte_f16x2(b0), 0, 0x1032));
                const uint32_t p1 = to_e4m3_pair(__byte_perm(decode_e2m1_byte_f16x2(b1), 0, 0x1032));
                c[2 * i + k] = p0 | (p1 << 16);
            }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            c[i] = to_e4m3_pair(decode_pair_f16x2<ELEM>(out[i] & 0xFFFF)) | (to_e4m3_pair(decode_pair_f16x2<ELEM>(out[i] >> 16)) << 16);
    }
}

template <int ELEM, bool TABLE, int TILES, bool RAGGED>
__global__ void __launch_bounds__(Cfg<TILES>::kThreads, TILES == 2 ? 1 : 2)
mx_flash_attention_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v, const Params p) {
    using C = Cfg<TILES>;
    using Smem = SmemT<TILES>;
    constexpr int K_STAGES = C::K_STAGES, V_STAGES = C::V_STAGES, kSoftmaxWarps = C::kSoftmaxWarps;
    constexpr uint32_t TM_S = C::TM_S, TM_O = C::TM_O, TM_SFQ = C::TM_SFQ, TM_SFK = C::TM_SFK, TM_SFP = C::TM_SFP, TM_SFV = C::TM_SFV;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::OFF_BAR);
    uint64_t* q_full = bars;                       // both Q tiles landed (count 1 + tx)
    uint64_t* qsf_full = bars + 1;                 // Q scales in shared memory (count 1)
    uint64_t* k_full = bars + 2;                   // K tile landed (count 1 + tx)
    uint64_t* ksf_full = k_full + K_STAGES;        // its scales (count 1)
    uint64_t* k_empty = ksf_full + K_STAGES;       // MMAs reading the stage retired (count 1, commit)
    uint64_t* v_full = k_empty + K_STAGES;
    uint64_t* vsf_full = v_full + V_STAGES;
    uint64_t* v_empty = vsf_full + V_STAGES;
    uint64_t* sa_full = v_empty + V_STAGES;        // [wg][buf] passes A, B: score tile complete (count 1, commit)
    uint64_t* sa_free = sa_full + 4;               // [wg][buf] passes A, B: score tile read into registers (count 128)
    uint64_t* sc_full = sa_free + 4;               // [wg] pass C: score tile complete (count 1, commit)
    uint64_t* sc_free = sc_full + 2;               // [wg] pass C: score tile read into registers (count 128)
    uint64_t* p_full = sc_free + 2;                // [wg] codes + scales of a chunk of P in shared memory (count 128)
    uint64_t* p_free = p_full + 2;                 // [wg] MMAs reading them retired (count 1, commit)
    uint64_t* o_full = p_free + 2;                 // [wg] output accumulator complete (count 1, commit)
    uint64_t* scan_done = o_full + 2;              // [wg] pass A finished, live-chunk words final (count 128)
    uint32_t* live_words = reinterpret_cast<uint32_t*>(smem + Smem::OFF_LIVE);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + Smem::OFF_TMEM_PTR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bh_count = p.batch * p.heads;
    const int qt = p.q_tiles - 1 - (int)(blockIdx.x / bh_count);  // the tiles with the most visible keys first
    const int bh = (int)(blockIdx.x % bh_count);
    const int b = bh / p.heads, h = bh - b * p.heads;
    const int bhk = b * p.kv_heads + h / (p.heads / p.kv_heads);  // grouped-query attention: the key / value head of this query head
    const int n_total = (p.kv_len + KC - 1) / KC;  // (kv_len % 32 == 0; the last chunk may hold 1..3 blocks: the rest reads as zero and is hidden)
    int nv[2] = {0, 0};
    bool active[2] = {false, false};
#pragma unroll
    for (int wg = 0; wg < TILES; ++wg) {
        const int q0 = qt * TILES * QT + wg * QT;
        active[wg] = q0 < p.q_len;
        const int last_row = min(q0 + QT - 1, p.q_len - 1);
        nv[wg] = !active[wg] ? 0 : (p.skip_hidden_chunks ? min(n_total, (last_row + p.causal_offset) / KC + 1) : n_total);
    }
    const int n_cta = max(nv[0], nv[1]);

    if (warp == kSoftmaxWarps && elect_one()) {
        tma_prefetch_desc(&map_q);
        tma_prefetch_desc(&map_k);
        tma_prefetch_desc(&map_v);
    }
    if (warp == kSoftmaxWarps + 1 && elect_one()) {
        mbar_init(q_full, 1);
        mbar_init(qsf_full, 1);
        for (int i = 0; i < K_STAGES; ++i) { mbar_init(&k_full[i], 1); mbar_init(&ksf_full[i], 1); mbar_init(&k_empty[i], 1); }
        for (int i = 0; i < V_STAGES; ++i) { mbar_init(&v_full[i], 1); mbar_init(&vsf_full[i], 1); mbar_init(&v_empty[i], 1); }
        for (int i = 0; i < 4; ++i) { mbar_init(&sa_full[i], 1); mbar_init(&sa_free[i], kWgThreads); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&sc_full[i], 1); mbar_init(&sc_free[i], kWgThreads); mbar_init(&p_full[i], kWgThreads); mbar_init(&p_free[i], 1); mbar_init(&o_full[i], 1);
            mbar_init(&scan_done[i], kWgThreads);
        }
        for (int i = 0; i < 4; ++i) live_words[i] = 0;
        fence_barrier_init();
    }
    if (warp == kSoftmaxWarps + 2) tmem_alloc<C::TMEM_COLS>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // With an explicit additive mask the kernel cannot know which key chunks a tile's rows see without looking.  Pass A looks at
    // everything anyway; it leaves the largest score of every (row, chunk) behind, and once a row's maximum is final a chunk whose
    // largest score lies more than 110 below it is +0 in every probability (sm::block_dead).  Chunks that are dead for all 128
    // rows of a warpgroup are skipped by passes B and C -- by the softmax threads, the tensor core and the loaders alike.
    // The table and the live words hold one entry per SLOT of 2^slot_shift chunks (the slot's largest score; live if any of its
    // chunks is).  A coarser slot only walks more chunks that turn out dead; a dead chunk adds +0 sums and +0 codes either way,
    // so the slot width never changes a result.  Without a table every slot is live and only j < nv[wg] limits the walk.
    constexpr bool use_table = TABLE;  // (launched with TABLE == (mask != nullptr): the implied-causal path carries none of this)
    auto live_chunks = [&](uint64_t (&live)[2]) {  // (callers other than the softmax threads: waits for pass A of both warpgroups)
        live[0] = live[1] = 0;
#pragma unroll
        for (int wg = 0; wg < TILES; ++wg) {
            if (!active[wg]) { live[wg] = 0; continue; }
            if (use_table) {
                mbar_wait(&scan_done[wg], 0);
                live[wg] = (uint64_t)live_words[2 * wg] | ((uint64_t)live_words[2 * wg + 1] << 32);
            } else {
                live[wg] = ~0ull;
            }
        }
    };
    auto chunk_on = [&](uint64_t live, int j) { return ((live >> (j >> p.slot_shift)) & 1) != 0; };

    if (warp < kSoftmaxWarps) {
        // ================= softmax warpgroups =================
        // 16 warps: query tile wg (0 / 1) x sub (0 / 1) x TMEM lane quadrant.  Thread = (query row, sub): of every 64-column score
        // tile the sub-0 thread of a row owns the first MX block (columns 0..31), the sub-1 thread the second -- four softmax warps
        // per scheduler instead of two (the arithmetic is latency-bound per warp).  What a row's two threads must agree on -- the
        // row maximum, the per-block sums in K4a's order, the chunk maxima -- goes through a few KB of shared memory and a named
        // barrier of the 256 threads of the query tile.
        const int wg = warp >> 3, sub = (warp >> 2) & 1, quad = warp & 3;
        const int r = quad * 32 + lane;                 // row inside the warpgroup's tile = TMEM lane
        const int q = qt * TILES * QT + wg * QT + r;        // query row
        const bool row_live = active[wg] && q < p.q_len;
        const int my_n = nv[wg];
        const uint32_t tm_lane = tmem_base + ((uint32_t)(quad * 32) << 16);
        const uint16_t* mrow = (TABLE && p.mask != nullptr && row_live) ? p.mask + (int64_t)b * p.mask_sb + (int64_t)h * p.mask_sh + (int64_t)q * p.mask_sq : nullptr;
        const int row_lim = RAGGED ? min(p.kv_valid, q + p.hide_offset + 1) : 0;  // RAGGED: the keys of mask' that are not -inf
        const int tpr = p.kv_len / 32;
        const bool hw_exact = (p.flags & MXQ_FLAG_HW_EXACT) != 0;
        uint8_t* p_tile = smem + Smem::OFF_P + wg * TILE_BYTES + r * 128;
        uint8_t* sfp_bytes = smem + Smem::OFF_SFP + wg * 512 + 16 * (r & 31) + 4 * (r >> 5);
        constexpr int NO = (ELEM == MXQ_ELEM_E2M1) ? 4 : 8;
        uint8_t* dump_codes = (p.p_codes != nullptr && row_live) ? p.p_codes + ((int64_t)bh * p.q_len + q) * tpr * (NO * 4) : nullptr;
        uint8_t* dump_scales = (p.p_codes != nullptr && row_live) ? p.p_scales + ((int64_t)bh * p.q_len + q) * tpr : nullptr;
        float* xch = reinterpret_cast<float*>(smem + Smem::OFF_XCH) + wg * 1024;  // [parity 2][sub 2][value 2][row 128]
        auto wg_sync = [&]() { asm volatile("bar.sync %0, 256;" ::"r"(1 + wg) : "memory"); };
        auto dump_zero = [&](int t, int sc) {
            if (t >= tpr) return;  // (a block past the end of a ragged last chunk)
            if constexpr (NO == 4) *reinterpret_cast<uint4*>(dump_codes + t * 16) = make_uint4(0, 0, 0, 0);
            else { *reinterpret_cast<uint4*>(dump_codes + t * 32) = make_uint4(0, 0, 0, 0); *reinterpret_cast<uint4*>(dump_codes + t * 32 + 16) = make_uint4(0, 0, 0, 0); }
            dump_scales[t] = (uint8_t)sc;
        };

        float row_max = -INFINITY, row_sum = 0.0f;
        // passes A and B keep TWO 64-column score tiles per warpgroup inside its (still unused) output accumulator, so the tensor
        // core works one tile ahead of the softmax threads; pass C has the accumulator in use and a single tile
        const uint32_t tm_sa = tm_lane + TM_O + wg * 128 + sub * 32, tm_sc = tm_lane + TM_S + wg * 64 + sub * 32;
        uint32_t ab_item = 0, c_par = 0, pfree_par = 0;
        auto take_tile = [&](uint32_t taddr, uint64_t* full, uint32_t parity, uint64_t* free_bar, uint32_t (&v)[32]) {
            mbar_wait(full, parity);
            tc_fence_after();
            tmem_ld_32x32b_x32(taddr, v);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(free_bar);  // the tensor core may overwrite the tile while we compute
        };
        auto take_ab = [&](uint32_t (&v)[32]) {
            const uint32_t buf = ab_item & 1;
            take_tile(tm_sa + buf * 64, &sa_full[wg * 2 + buf], (ab_item >> 1) & 1, &sa_free[wg * 2 + buf], v);
            ++ab_item;
        };
        auto visible = [&](int t) {  // how many of block t's 32 keys this query row may see
            int vis = (row_live && t < tpr) ? 32 : 0;
            if (p.causal && row_live) vis = min(32, max(0, q + p.causal_offset + 1 - t * 32));
            return vis;
        };
        // the 32 scores of a block as the softmax sees them: bf16 matmul result, * scaling, + mask, causal rule (mxq_softmax_core.cuh)
        auto scores_of = [&](const uint32_t (&raw)[32], int t, int vis, float (&x)[32]) {
            uint32_t w[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) w[i] = pack_bf16x2(__uint_as_float(raw[2 * i]), __uint_as_float(raw[2 * i + 1]));
            sm::scale_round(w, p.scaling, x);
            if constexpr (RAGGED) {  // + mask': the caller's mask is read only at the keys it does not replace by -inf
                const int hv = row_lim - t * 32;
                if (mrow != nullptr || hv < 32) {
                    uint32_t mw[16];
                    if (mrow != nullptr && hv >= 32) {
                        sm::load_mask(mrow + t * 32, p.mask_vec != 0, mw);
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const uint32_t m0 = 2 * i < hv ? (mrow != nullptr ? mrow[t * 32 + 2 * i] : 0u) : 0xFF80u;  // bf16 -inf
                            const uint32_t m1 = 2 * i + 1 < hv ? (mrow != nullptr ? mrow[t * 32 + 2 * i + 1] : 0u) : 0xFF80u;
                            mw[i] = m0 | (m1 << 16);
                        }
                    }
                    sm::add_mask(x, mw);
                }
            } else if (mrow != nullptr) {
                uint32_t mw[16];
                sm::load_mask(mrow + t * 32, p.mask_vec != 0, mw);
                sm::add_mask(x, mw);
            }
            if (vis < 32) sm::hide_from(x, vis);
        };
        if (active[wg]) {
            // ---- pass A: row maximum.  Without an additive mask the map score -> bf16(bf16(score) * scaling) is monotone
            // (scaling > 0), so the maximum of the mapped scores is the map of the maximum raw score: one max per element.
            const bool fast_max = !TABLE && p.scaling > 0.0f;
            float part_max = -INFINITY, chunk_max = -INFINITY;
            uint16_t* cmax = reinterpret_cast<uint16_t*>(smem + Smem::OFF_CMAX) + wg * 64 * 128 + r;
            for (int j = 0; j < my_n; ++j) {
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[32];
                    take_ab(v);
                    const int t = 4 * j + 2 * hf + sub;
                    const int vis = visible(t);
                    if (vis > 0) {
                        float m;
                        if (fast_max) {
                            if (vis == 32) {
                                m = __uint_as_float(v[0]);
#pragma unroll
                                for (int i = 1; i < 31; i += 2) m = sm::max_nan3(m, __uint_as_float(v[i]), __uint_as_float(v[i + 1]));
                                m = sm::max_nan(m, __uint_as_float(v[31]));
                            } else {
                                m = -INFINITY;
#pragma unroll
                                for (int i = 0; i < 32; ++i) m = sm::max_nan(m, i < vis ? __uint_as_float(v[i]) : -INFINITY);
                            }
                        } else {
                            float x[32];
                            scores_of(v, t, vis, x);
                            m = sm::block_max_only(x);
                        }
                        part_max = sm::max_nan(part_max, m);
                        chunk_max = sm::max_nan(chunk_max, m);
                    }
                    if (use_table && hf == 1) {  // the chunk's largest score over both threads of the row (the scores are bf16 values: exact)
                        float* slot = xch + (j & 1) * 512;
                        slot[sub * 256 + r] = chunk_max;
                        wg_sync();
                        if (sub == 0) {
                            uint16_t* e = cmax + (j >> p.slot_shift) * 128;
                            float cm = sm::max_nan(chunk_max, slot[256 + r]);
                            if ((j & ((1 << p.slot_shift) - 1)) != 0) cm = sm::max_nan(cm, __uint_as_float((uint32_t)*e << 16));
                            *e = (uint16_t)pack_bf16x2(cm, 0.0f);
                        }
                        chunk_max = -INFINITY;
                    }
                }
            }
            {
                float* slot = reinterpret_cast<float*>(smem + Smem::OFF_XMAX) + wg * 256;
                slot[sub * 128 + r] = part_max;
                wg_sync();  // (also: every chunk maximum of this query tile is in the table)
                row_max = sm::max_nan(part_max, slot[(sub ^ 1) * 128 + r]);
            }
            if (fast_max) {
                const uint32_t r1 = pack_bf16x2(row_max, 0.0f);
                const uint32_t r2 = pack_bf16x2(__uint_as_float(r1 << 16) * p.scaling, 0.0f);
                row_max = __uint_as_float(r2 << 16);
            }
            uint64_t my_live = ~0ull;
            if (use_table) {
                const int n_slots = ((my_n - 1) >> p.slot_shift) + 1;
                for (int s = 0; s < n_slots; ++s) {
                    const float cm = __uint_as_float((uint32_t)cmax[s * 128] << 16);
                    const bool counts = row_live && !(cm - row_max < -110.0f);
                    const unsigned any = __ballot_sync(0xFFFFFFFFu, counts);
                    if (lane == 0 && any) atomicOr(&live_words[2 * wg + (s >> 5)], 1u << (s & 31));
                }
                if (r == 0) atomicOr(&live_words[2 * wg], 1u);  // (a warpgroup always walks its first chunk: the output accumulator gets written)
                mbar_arrive(&scan_done[wg]);
                mbar_wait(&scan_done[wg], 0);
                my_live = (uint64_t)live_words[2 * wg] | ((uint64_t)live_words[2 * wg + 1] << 32);
            }
            // ---- pass B: row sum of expf(x - max), the per-block sums added in K4a's order (sm::sum_layout): blocks in order, or
            // butterfly-reduced groups of 8 or 32 added in order.  Layouts 0 / 1: both threads of a row add all four sums of a
            // chunk, in the same order.  Layout 2: a group of 32 blocks is E + O (mxq_softmax_core.cuh), and the sub-0 thread owns
            // exactly the even blocks of a row, the sub-1 thread the odd ones -- each builds its half alone, and the two threads
            // exchange only the halves, once per group.
            {
                float acc = 0.0f, a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
                float n[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};  // layout 2: this thread's first tree level of the open group
                bool have_acc = false;
                auto add_block = [&](int t, float s) {
                    if (p.layout == 0) {
                        acc = acc + s;
                    } else {
                        const int k8 = t & 7;
                        if (k8 == 0) a0 = s;
                        else if (k8 == 1) a1 = s;
                        else if (k8 == 2) a2 = s;
                        else if (k8 == 3) a3 = s;
                        else if (k8 == 4) a0 = a0 + s;
                        else if (k8 == 5) a1 = a1 + s;
                        else if (k8 == 6) a2 = a2 + s;
                        else {
                            const float g = (a0 + a2) + (a1 + (a3 + s));
                            acc = have_acc ? acc + g : g;
                            have_acc = true;
                        }
                    }
                };
                for (int j = 0; j < my_n; ++j) {
                    const bool walked = chunk_on(my_live, j);
                    if (!walked && p.layout != 2) {  // every block of the chunk sums to +0 for every row of the warpgroup
#pragma unroll
                        for (int bl = 0; bl < 4; ++bl) add_block(4 * j + bl, 0.0f);
                        continue;
                    }
                    float mine[2] = {0.0f, 0.0f};
#pragma unroll 1
                    for (int hf = 0; hf < 2 && walked; ++hf) {
                        uint32_t v[32];
                        take_ab(v);
                        const int t = 4 * j + 2 * hf + sub;
                        const int vis = visible(t);
                        float s = 0.0f;
                        if (vis > 0) {
                            float x[32];
                            scores_of(v, t, vis, x);
                            if (!sm::block_dead(vis, sm::block_max_only(x), row_max)) s = sm::exp_sum(x, row_max);
                        }
                        mine[hf] = s;
                    }
                    if (p.layout == 2) {
                        // blocks 4c + 2 hf + sub of the group (c = j & 7) are leaves 2c + hf of this thread's half; the first tree
                        // level adds leaves i and i + 8.  Unvisited leaves (skipped chunks, the ragged tail, a half-filled last
                        // group) stay +0, and every sum is >= +0, so adding them is exact.
                        const int c4 = j & 3;
                        n[0] += c4 == 0 ? mine[0] : 0.0f; n[1] += c4 == 0 ? mine[1] : 0.0f;
                        n[2] += c4 == 1 ? mine[0] : 0.0f; n[3] += c4 == 1 ? mine[1] : 0.0f;
                        n[4] += c4 == 2 ? mine[0] : 0.0f; n[5] += c4 == 2 ? mine[1] : 0.0f;
                        n[6] += c4 == 3 ? mine[0] : 0.0f; n[7] += c4 == 3 ? mine[1] : 0.0f;
                        if ((j & 7) == 7 || j == my_n - 1) {
                            const float half = sm::butterfly8(n[0], n[1], n[2], n[3], n[4], n[5], n[6], n[7]);
                            float* slot = xch + ((j >> 3) & 1) * 512;
                            slot[sub * 256 + r] = half;
                            wg_sync();
                            acc = acc + (half + slot[(sub ^ 1) * 256 + r]);  // E + O; (acc starts at +0: exact for group 0)
#pragma unroll
                            for (int i = 0; i < 8; ++i) n[i] = 0.0f;
                        }
                        continue;
                    }
                    float* slot = xch + (j & 1) * 512;
                    slot[sub * 256 + r] = mine[0];
                    slot[sub * 256 + 128 + r] = mine[1];
                    wg_sync();
                    const float o0 = slot[(sub ^ 1) * 256 + r], o1 = slot[(sub ^ 1) * 256 + 128 + r];
                    add_block(4 * j + 0, sub ? o0 : mine[0]);
                    add_block(4 * j + 1, sub ? mine[0] : o0);
                    add_block(4 * j + 2, sub ? o1 : mine[1]);
                    add_block(4 * j + 3, sub ? mine[1] : o1);
                }
                if (p.layout == 1 && ((4 * my_n) & 7) != 0) {  // a half-filled last group (the rest of it: hidden blocks, sum 0)
                    const float g = ((a0 + 0.0f) + (a2 + 0.0f)) + ((a1 + 0.0f) + (a3 + 0.0f));
                    acc = have_acc ? acc + g : g;
                }
                row_sum = acc;
            }
            // ---- pass C: the codes and scales of P, into the operand tile of the second contraction
            bool p_started = false;
            for (int j = 0; j < my_n; ++j) {
                if (!chunk_on(my_live, j)) {  // +0 codes for the whole chunk: nothing for the tensor core to add
                    if (dump_codes != nullptr) {
                        const int sc = sm::dead_block_scale<ELEM>(row_max, row_sum);
                        dump_zero(4 * j + sub, sc);
                        dump_zero(4 * j + 2 + sub, sc);
                    }
                    continue;
                }
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[32];
                    take_tile(tm_sc, &sc_full[wg], c_par, &sc_free[wg], v);
                    c_par ^= 1;
                    const int bl = 2 * hf + sub;   // block inside the chunk
                    const int t = 4 * j + bl;      // block inside the row
                    const int vis = visible(t);
                    float x[32];
                    float m = -INFINITY, lo = INFINITY;
                    if (vis > 0) {
                        scores_of(v, t, vis, x);
                        sm::block_max(x, m, lo);
                    }
                    uint32_t c[8];
                    int sc;
                    if (sm::block_dead(vis, m, row_max)) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) c[i] = 0;
                        sc = (row_live && t < tpr) ? sm::dead_block_scale<ELEM>(row_max, row_sum) : 127;
                        if (dump_codes != nullptr) dump_zero(t, sc);
                    } else {
                        sm::exp_sum(x, row_max);
                        uint32_t w[16];
                        sm::normalize(x, lo, row_max, row_sum, w);
                        uint32_t out[NO];
                        sc = quantize_block32<ELEM>(w, hw_exact, out);
                        if (dump_codes != nullptr) {
                            if constexpr (NO == 4) *reinterpret_cast<uint4*>(dump_codes + t * 16) = make_uint4(out[0], out[1], out[2], out[3]);
                            else {
                                *reinterpret_cast<uint4*>(dump_codes + t * 32) = make_uint4(out[0], out[1], out[2], out[3]);
                                *reinterpret_cast<uint4*>(dump_codes + t * 32 + 16) = make_uint4(out[4], out[5], out[6], out[7]);
                            }
                            dump_scales[t] = (uint8_t)sc;
                        }
                        container_bytes<ELEM>(out, c);
                    }
                    if (hf == 0) {
                        if (p_started) {  // the tensor core must be done with the previous chunk's codes before they are overwritten
                            mbar_wait(&p_free[wg], pfree_par);
                            pfree_par ^= 1;
                        }
                        p_started = true;
                    }
                    // K-major 128B-swizzled operand tile: 16-byte chunk cc of row r lives at chunk cc ^ (r & 7); the block's scale is
                    // byte bl of the row's 32-bit scale word in the tcgen05.cp layout
                    *reinterpret_cast<uint4*>(p_tile + (((2 * bl) ^ (r & 7)) << 4)) = make_uint4(c[0], c[1], c[2], c[3]);
                    *reinterpret_cast<uint4*>(p_tile + (((2 * bl + 1) ^ (r & 7)) << 4)) = make_uint4(c[4], c[5], c[6], c[7]);
                    sfp_bytes[bl] = (uint8_t)sc;
                    if (hf == 1) {
                        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core (async proxy)
                        mbar_arrive(&p_full[wg]);
                    }
                }
            }
        }
        if (active[wg]) {
            // chunks this warpgroup skipped (hidden by the causal rule): their codes are +0 and the scale is that of a zero block
            if (dump_codes != nullptr) {
                const int sc = sm::dead_block_scale<ELEM>(row_max, row_sum);
                for (int t = 4 * my_n + sub; t < tpr; t += 2) dump_zero(t, sc);
            }
            // ---- drain the output accumulator: thread = (row, column half), 64 bf16 = 128 contiguous bytes ----
            mbar_wait(&o_full[wg], 0);
            tc_fence_after();
            uint16_t* orow = p.out + (int64_t)b * p.out_sb + (int64_t)h * p.out_sh + (int64_t)q * p.out_sq + sub * 64;
#pragma unroll 1
            for (int cg = 0; cg < 2; ++cg) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(tm_lane + TM_O + wg * 128 + sub * 64 + cg * 32, v);
                tmem_ld_wait();
                if (row_live) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        uint4 o;
                        o.x = pack_bf16x2(__uint_as_float(v[8 * i + 0]), __uint_as_float(v[8 * i + 1]));
                        o.y = pack_bf16x2(__uint_as_float(v[8 * i + 2]), __uint_as_float(v[8 * i + 3]));
                        o.z = pack_bf16x2(__uint_as_float(v[8 * i + 4]), __uint_as_float(v[8 * i + 5]));
                        o.w = pack_bf16x2(__uint_as_float(v[8 * i + 6]), __uint_as_float(v[8 * i + 7]));
                        *reinterpret_cast<uint4*>(orow + cg * 32 + 8 * i) = o;
                    }
                }
            }
            tc_fence_before();
        }
    } else if (warp == kSoftmaxWarps) {
        // ================= TMA producer =================
        if (elect_one()) {
            mbar_arrive_expect_tx(q_full, (TILES == 2 && active[1] ? 2 : 1) * TILE_BYTES);
            tma_load_3d(&map_q, q_full, smem + Smem::OFF_Q, 0, qt * TILES * QT, bh);  // rows past q_len read as zero
            if (TILES == 2 && active[1]) tma_load_3d(&map_q, q_full, smem + Smem::OFF_Q + TILE_BYTES, 0, qt * TILES * QT + QT, bh);
            uint32_t ks = 0, kph = 0, vs = 0, vph = 0;
            uint64_t need = ~0ull;
            for (int pass = 0; pass < 3; ++pass) {
                if (pass == 1) {
                    uint64_t live[2];
                    live_chunks(live);
                    need = live[0] | live[1];
                }
                for (int j = 0; j < n_cta; ++j) {
                    if (!chunk_on(need, j)) continue;
                    mbar_wait(&k_empty[ks], kph ^ 1);
                    mbar_arrive_expect_tx(&k_full[ks], TILE_BYTES);
                    tma_load_3d(&map_k, &k_full[ks], smem + Smem::OFF_K + ks * TILE_BYTES, 0, j * KC, bhk);
                    if (++ks == K_STAGES) { ks = 0; kph ^= 1; }
                    if (pass == 2) {
                        mbar_wait(&v_empty[vs], vph ^ 1);
                        mbar_arrive_expect_tx(&v_full[vs], TILE_BYTES);
                        tma_load_3d(&map_v, &v_full[vs], smem + Smem::OFF_V + vs * TILE_BYTES, j * KC, 0, bhk);
                        if (++vs == V_STAGES) { vs = 0; vph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == kSoftmaxWarps + 1) {
        // ================= MMA issuer =================
        uint32_t ks = 0, kph = 0, vs = 0, vph = 0;
        uint32_t pfull_par[2] = {0, 0};
        const uint32_t q_addr = smem_u32(smem + Smem::OFF_Q), k_addr0 = smem_u32(smem + Smem::OFF_K), v_addr0 = smem_u32(smem + Smem::OFF_V);
        const uint32_t p_addr = smem_u32(smem + Smem::OFF_P);
        mbar_wait(q_full, 0);
        mbar_wait(qsf_full, 0);
        tc_fence_after();
        if (elect_one()) {
            tc_copy_sf(tmem_base + TM_SFQ, smem_desc(smem_u32(smem + Smem::OFF_SFQ), 128, kLayoutNone));
            if (TILES == 2) tc_copy_sf(tmem_base + TM_SFQ + 4, smem_desc(smem_u32(smem + Smem::OFF_SFQ + 512), 128, kLayoutNone));
        }
        __syncwarp();
        // O[wg] += P[wg] (chunk jj) x V (chunk jj)
        uint64_t live[2] = {~0ull, ~0ull};
        int last_live[2] = {-1, -1};
        bool o_started[2] = {false, false};
        uint32_t kcnt = 0, vcnt = 0;
        auto pv = [&](int jj) {
            mbar_wait(&v_full[vs], vph);
            mbar_wait(&vsf_full[vs], vph);
            tc_fence_after();
            const uint32_t tm_sfv = tmem_base + TM_SFV + 4 * (vcnt++ & 1);
            if (elect_one()) tc_copy_sf(tm_sfv, smem_desc(smem_u32(smem + Smem::OFF_SFV + vs * 512), 128, kLayoutNone));
            __syncwarp();
#pragma unroll
            for (int wg = 0; wg < TILES; ++wg) {
                if (!active[wg] || jj >= nv[wg] || !chunk_on(live[wg], jj)) continue;
                mbar_wait(&p_full[wg], pfull_par[wg]);
                pfull_par[wg] ^= 1;
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t tm_sfp = tmem_base + TM_SFP + 4 * wg;
                    tc_copy_sf(tm_sfp, smem_desc(smem_u32(smem + Smem::OFF_SFP + wg * 512), 128, kLayoutNone));
#pragma unroll
                    for (int k = 0; k < KC / UMMA_K; ++k) {
                        const uint64_t da = smem_desc(p_addr + wg * TILE_BYTES + k * UMMA_K, 1024, kLayoutSw128);
                        const uint64_t db = smem_desc(v_addr0 + vs * TILE_BYTES + k * UMMA_K, 1024, kLayoutSw128);
                        tc_mma_mx(tmem_base + TM_O + wg * 128, da, db, idesc_with_sf(p.idesc_pv, k, k), (o_started[wg] || k != 0) ? 1u : 0u, tm_sfp, tm_sfv);
                    }
                    tc_commit(&p_free[wg]);
                    if (jj == last_live[wg]) tc_commit(&o_full[wg]);
                }
                o_started[wg] = true;
                __syncwarp();
            }
            if (elect_one()) tc_commit(&v_empty[vs]);
            __syncwarp();
            if (++vs == V_STAGES) { vs = 0; vph ^= 1; }
        };
        uint32_t ab_item[2] = {0, 0}, cfree_par[2] = {0, 0};
        int prev = -1;  // pass C: the last chunk whose P @ V has not been issued yet
        for (int pass = 0; pass < 3; ++pass) {
            if (pass == 1) {
                live_chunks(live);
#pragma unroll
                for (int wg = 0; wg < TILES; ++wg) {  // the last chunk below nv[wg] of the last live slot (a live slot holds one)
                    const int s = live[wg] ? 63 - __clzll((long long)live[wg]) : -1;
                    last_live[wg] = s < 0 ? -1 : min(nv[wg] - 1, ((s + 1) << p.slot_shift) - 1);
                }
            }
            for (int j = 0; j < n_cta; ++j) {
                if (pass > 0 && !chunk_on(live[0] | live[1], j)) continue;
                mbar_wait(&k_full[ks], kph);
                mbar_wait(&ksf_full[ks], kph);
                tc_fence_after();
                const uint32_t tm_sfk = tmem_base + TM_SFK + 8 * (kcnt++ & 1);
                if (elect_one()) {
                    tc_copy_sf(tm_sfk, smem_desc(smem_u32(smem + Smem::OFF_SFK + ks * 1024), 128, kLayoutNone));
                    tc_copy_sf(tm_sfk + 4, smem_desc(smem_u32(smem + Smem::OFF_SFK + ks * 1024 + 512), 128, kLayoutNone));
                }
                __syncwarp();
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
#pragma unroll
                    for (int wg = 0; wg < TILES; ++wg) {
                        if (!active[wg] || j >= nv[wg] || (pass > 0 && !chunk_on(live[wg], j))) continue;
                        uint32_t tm_s;
                        uint64_t* full_bar;
                        if (pass < 2) {  // two tiles per warpgroup inside its output accumulator: run one tile ahead of the softmax threads
                            const uint32_t buf = ab_item[wg] & 1;
                            mbar_wait(&sa_free[wg * 2 + buf], ((ab_item[wg] >> 1) & 1) ^ 1);
                            ++ab_item[wg];
                            tm_s = tmem_base + TM_O + wg * 128 + buf * 64;
                            full_bar = &sa_full[wg * 2 + buf];
                        } else {
                            mbar_wait(&sc_free[wg], cfree_par[wg] ^ 1);
                            cfree_par[wg] ^= 1;
                            tm_s = tmem_base + TM_S + wg * 64;
                            full_bar = &sc_full[wg];
                        }
                        tc_fence_after();
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < HD / UMMA_K; ++k) {
                                const uint64_t da = smem_desc(q_addr + wg * TILE_BYTES + k * UMMA_K, 1024, kLayoutSw128);
                                const uint64_t db = smem_desc(k_addr0 + ks * TILE_BYTES + hf * (64 * 128) + k * UMMA_K, 1024, kLayoutSw128);
                                tc_mma_mx(tm_s, da, db, idesc_with_sf(p.idesc_qk, k, k), k != 0, tmem_base + TM_SFQ + 4 * wg, tm_sfk + 4 * hf);
                            }
                            tc_commit(full_bar);
                        }
                        __syncwarp();
                    }
                    // software pipeline of pass C: the P @ V of the previous chunk goes behind the first score tile of this one,
                    // so the softmax threads never wait for a score tile behind their own P @ V
                    if (pass == 2 && hf == 0 && prev >= 0) pv(prev);
                }
                if (pass == 2) prev = j;
                if (elect_one()) tc_commit(&k_empty[ks]);
                __syncwarp();
                if (++ks == K_STAGES) { ks = 0; kph ^= 1; }
            }
            if (pass == 2 && prev >= 0) pv(prev);
        }
        tc_fence_before();
    } else {
        // ================= scale-factor loader =================
        // tcgen05.cp.32x128b.warpx4 wants 32 chunks of 16 B per 128 rows: chunk i = the 32-bit scale words of rows i, i+32, i+64, i+96
        auto publish = [&](uint64_t* bar) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar);
        };
        {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(p.q_sf) + (int64_t)bh * p.q_len;
#pragma unroll
            for (int wg = 0; wg < TILES; ++wg) {
                uint32_t w[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) w[i] = src[min(qt * TILES * QT + wg * QT + i * 32 + lane, p.q_len - 1)];
                *reinterpret_cast<uint4*>(smem + Smem::OFF_SFQ + wg * 512 + 16 * lane) = make_uint4(w[0], w[1], w[2], w[3]);
            }
            publish(qsf_full);
        }
        const uint32_t* ksrc = reinterpret_cast<const uint32_t*>(p.k_sf) + (int64_t)bhk * (RAGGED ? p.kv_pitch : p.kv_len);
        const int vld = (RAGGED ? p.kv_pitch : p.kv_len) / 32;  // scale bytes per channel row of V^T
        const uint8_t* vsrc = p.v_sf + (int64_t)bhk * HD * vld;
        auto load_k = [&](int j, uint32_t (&w)[4]) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if constexpr (RAGGED) {  // keys past kv_valid: zero codes (TMA fill) times the neutral scale
                    const int key = j * KC + i * 32 + lane;
                    w[i] = key < p.kv_valid ? __ldg(ksrc + key) : 0x7F7F7F7Fu;
                } else {
                    w[i] = __ldg(ksrc + min(j * KC + i * 32 + lane, p.kv_len - 1));  // (keys past kv_len: zero codes, hidden)
                }
            }
        };
        uint32_t ks = 0, kph = 0, vs = 0, vph = 0;
        uint64_t need = ~0ull;
        for (int pass = 0; pass < 3; ++pass) {
            if (pass == 1) {
                uint64_t live[2];
                live_chunks(live);
                need = live[0] | live[1];
            }
            for (int j = 0; j < n_cta; ++j) {
                if (!chunk_on(need, j)) continue;
                uint32_t kw[4], vw[4];
                load_k(j, kw);
                if (pass == 2) {
                    const int vb = RAGGED ? (p.kv_valid + 31) / 32 : vld;  // V scale blocks that hold a key
                    if ((vld & 3) == 0 && (!RAGGED || 4 * j + 4 <= vb)) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) vw[i] = __ldg(reinterpret_cast<const uint32_t*>(vsrc + (int64_t)(i * 32 + lane) * vld + 4 * j));
                    } else {  // ragged kv_len (a channel's scale row is not a whole number of words), or the chunk reaching past kv_valid
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const uint8_t* row = vsrc + (int64_t)(i * 32 + lane) * vld;
                            uint32_t w = 0;
#pragma unroll
                            for (int bb = 0; bb < 4; ++bb) w |= (uint32_t)(4 * j + bb < vb ? __ldg(row + 4 * j + bb) : 127) << (8 * bb);
                            vw[i] = w;
                        }
                    }
                }
                mbar_wait(&k_empty[ks], kph ^ 1);
                *reinterpret_cast<uint4*>(smem + Smem::OFF_SFK + ks * 1024 + 16 * lane) = make_uint4(kw[0], kw[1], 0u, 0u);        // keys 0..63 of the chunk
                *reinterpret_cast<uint4*>(smem + Smem::OFF_SFK + ks * 1024 + 512 + 16 * lane) = make_uint4(kw[2], kw[3], 0u, 0u);  // keys 64..127
                publish(&ksf_full[ks]);
                if (++ks == K_STAGES) { ks = 0; kph ^= 1; }
                if (pass == 2) {
                    mbar_wait(&v_empty[vs], vph ^ 1);
                    *reinterpret_cast<uint4*>(smem + Smem::OFF_SFV + vs * 512 + 16 * lane) = make_uint4(vw[0], vw[1], vw[2], vw[3]);
                    publish(&vsf_full[vs]);
                    if (++vs == V_STAGES) { vs = 0; vph ^= 1; }
                }
            }
        }
    }
    __syncthreads();
    if (warp == kSoftmaxWarps + 2) {
        tc_fence_after();
        tmem_dealloc<C::TMEM_COLS>(tmem_base);
    }
}

}  // namespace fa

int launch_flash_attention(const mxq_attention_args_t* a, int device, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace fa;
    auto fmt_ok = [](int f) { return f == MXQ_OPERAND_E4M3_BYTES || f == MXQ_OPERAND_E5M2_BYTES; };
    const bool ragged = a->kv_pitch > 0;  // (the C entry checked 1 <= q_len <= kv_len <= kv_pitch <= MXQ_FLASH_MAX_KV, kv_pitch % 128 == 0)
    // the key axis the kernel walks: kv_len, or in the ragged mode n = ceil128(kv_len) keys of which the tail is hidden
    const int64_t kv_n = ragged ? (a->kv_len + KC - 1) / KC * KC : a->kv_len;
    if (a->head_dim != HD || (!ragged && (a->kv_len % 32 || a->kv_len < 32)) || a->q_len < 1 || a->kv_len < a->q_len || a->heads % a->kv_heads) {
        snprintf(msg, msg_len, "needs head_dim == 128, kv_len %% 32 == 0, kv_len >= q_len, heads %% kv_heads == 0");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    if (!fmt_ok(a->q_format) || !fmt_ok(a->k_format) || !fmt_ok(a->v_format) || a->p_elem == MXQ_ELEM_INT8) {
        snprintf(msg, msg_len, "operands must be 8-bit floating-point containers and the probabilities a floating-point element type");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    if (a->kv_len > MXQ_FLASH_MAX_KV) {
        snprintf(msg, msg_len, "kv_len %lld > %d", (long long)a->kv_len, MXQ_FLASH_MAX_KV);
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    // mask' of the ragged mode exists unless the caller gave no mask, causal is off and kv_len == n
    const bool masked = a->causal || a->mask != nullptr || kv_n != a->kv_len;
    const int tpr = (int)(kv_n / 32);
    const int layout = sm::sum_layout(tpr, masked);
    auto al16 = [](const void* ptr) { return ((uintptr_t)ptr % 16) == 0; };
    if (!al16(a->q_codes) || !al16(a->k_codes) || !al16(a->vt_codes) || ((uintptr_t)a->q_scales % 4) || ((uintptr_t)a->k_scales % 4) ||
        ((ragged || (a->kv_len % KC) == 0) && ((uintptr_t)a->vt_scales % 4)) ||
        !al16(a->out) || (a->out_batch_stride % 8) || (a->out_head_stride % 8) || (a->out_row_stride % 8) || (a->p_codes && !al16(a->p_codes))) {
        snprintf(msg, msg_len, "misaligned operand");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    const int64_t bh = a->batch * a->heads, bhk = a->batch * a->kv_heads;
    const int tiles = a->q_len <= QT ? 1 : 2;  // query tiles per CTA: one (two CTAs per SM) when a (batch, head) has at most 128 query rows
    const int64_t q_tiles = (a->q_len + tiles * QT - 1) / (tiles * QT);
    if (bh * q_tiles > 0x7FFFFFFF || a->q_len > 0x3FFFFFFF || a->kv_len > 0x3FFFFFFF) { snprintf(msg, msg_len, "extent too large"); return MXQ_ERR_UNSUPPORTED_SHAPE; }
    const int64_t pitch = ragged ? a->kv_pitch : a->kv_len;  // the maps end at kv_len: TMA zero-fills the keys past it
    CUtensorMap map_q, map_k, map_v;
    if (!cached_operand_map(&map_q, a->q_codes, HD, a->q_len, bh, HD, a->q_len * HD, 128, a->q_format, device) ||
        !cached_operand_map(&map_k, a->k_codes, HD, a->kv_len, bhk, HD, pitch * HD, 128, a->k_format, device) ||
        !cached_operand_map(&map_v, a->vt_codes, a->kv_len, HD, bhk, pitch, (int64_t)HD * pitch, 128, a->v_format, device)) {
        snprintf(msg, msg_len, "cuTensorMapEncodeTiled failed");
        return MXQ_ERR_CUDA;
    }
    fa::Params p;
    memset(&p, 0, sizeof(p));
    p.q_sf = a->q_scales; p.k_sf = a->k_scales; p.v_sf = a->vt_scales;
    p.mask = (const uint16_t*)a->mask; p.mask_sb = a->mask_stride_b; p.mask_sh = a->mask_stride_h; p.mask_sq = a->mask_stride_q;
    p.mask_vec = a->mask && ((uintptr_t)a->mask % 16 == 0) && (a->mask_stride_b % 8 == 0) && (a->mask_stride_h % 8 == 0) && (a->mask_stride_q % 8 == 0);
    p.out = (uint16_t*)a->out; p.out_sb = a->out_batch_stride; p.out_sh = a->out_head_stride; p.out_sq = a->out_row_stride;
    p.p_codes = (uint8_t*)a->p_codes; p.p_scales = a->p_scales;
    p.batch = (int)a->batch; p.heads = (int)a->heads; p.kv_heads = (int)a->kv_heads; p.q_len = (int)a->q_len; p.kv_len = (int)kv_n;
    // ragged: causal off, the causal rule and the tail folded into mask' (hide_offset: a row q sees keys <= q + hide_offset)
    p.causal = a->causal && !ragged ? 1 : 0;
    p.causal_offset = (int)(a->kv_len - a->q_len);
    p.skip_hidden_chunks = p.causal;  // (an explicit mask is data: every chunk is read)
    p.layout = layout;
    p.kv_valid = (int)a->kv_len;
    p.hide_offset = a->causal ? (int)(a->kv_len - a->q_len) : (int)a->kv_len;
    p.kv_pitch = (int)pitch;
    const int n_chunks = (int)((kv_n + KC - 1) / KC);
    while ((64 << p.slot_shift) < n_chunks) ++p.slot_shift;
    p.scaling = a->scaling;
    // the probabilities travel as E4M3 bytes (exact for every fp6 / fp4 value) unless they ARE e5m2
    const int p_format = a->p_elem == MXQ_ELEM_E5M2 ? MXQ_OPERAND_E5M2_BYTES : MXQ_OPERAND_E4M3_BYTES;
    p.idesc_qk = make_idesc(QT, 64) | idesc_formats(a->q_format, a->k_format);
    p.idesc_pv = make_idesc(QT, HD) | idesc_formats(p_format, a->v_format);
    p.flags = a->flags;
    p.q_tiles = (int)q_tiles;
    const unsigned grid = (unsigned)(bh * q_tiles);
#define MXQ_FA_LAUNCH(E, T, TL, R)                                                                                                  \
    {                                                                                                                               \
        cudaError_t e = ensure_smem_attr((const void*)mx_flash_attention_kernel<E, T, TL, R>, SmemT<TL>::DYN_BYTES, device);         \
        if (e != cudaSuccess) { snprintf(msg, msg_len, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }   \
        mx_flash_attention_kernel<E, T, TL, R><<<grid, Cfg<TL>::kThreads, SmemT<TL>::DYN_BYTES, stream>>>(map_q, map_k, map_v, p);   \
    }
    // the ragged mode runs the table (mask) variant whenever mask' exists, with or without a caller's mask
#define MXQ_FA_TILES(E, R)                                                                                                          \
    if (tiles == 1) { if (R ? masked : a->mask != nullptr) MXQ_FA_LAUNCH(E, true, 1, R) else MXQ_FA_LAUNCH(E, false, 1, R) }          \
    else { if (R ? masked : a->mask != nullptr) MXQ_FA_LAUNCH(E, true, 2, R) else MXQ_FA_LAUNCH(E, false, 2, R) }
#define MXQ_FA_CASE(E)                                                                                                              \
    case E:                                                                                                                         \
        if (ragged) { MXQ_FA_TILES(E, true) } else { MXQ_FA_TILES(E, false) }                                                       \
        break;
    switch (a->p_elem) {
        MXQ_FA_CASE(MXQ_ELEM_E4M3) MXQ_FA_CASE(MXQ_ELEM_E3M2) MXQ_FA_CASE(MXQ_ELEM_E2M3) MXQ_FA_CASE(MXQ_ELEM_E2M1) MXQ_FA_CASE(MXQ_ELEM_E5M2)
    default: snprintf(msg, msg_len, "unknown element type %d", a->p_elem); return MXQ_ERR_INVALID;
    }
#undef MXQ_FA_CASE
#undef MXQ_FA_TILES
#undef MXQ_FA_LAUNCH
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch (flash attention): %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

}  // namespace gemm
}  // namespace mxq
