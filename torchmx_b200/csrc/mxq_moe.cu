// K6: mixture-of-experts layer on MX operands (C entries mxq_moe_route / mxq_moe_gemm / mxq_moe_combine, include/mxq.h).
//
// transformers' expert loop (MixtralExperts.forward and its Qwen2-MoE / Qwen3-MoE / OLMoE twins) finds the hit experts with a
// host-synchronising nonzero() and runs ~8 launches per hit expert.  Here a layer is
//   K6a route    : stable counting sort of the (token, slot) pairs by expert + K1 quantization of the routed rows in that order
//   K6b gemm     : gate_up for every routed row in one launch
//   K1b          : SiLU gating + quantization of the two column halves (mxq_silu_mul_quantize, unchanged)
//   K6b gemm     : down for every routed row in one launch
//   K6c combine  : the index_add_ sequence of the loop, one write per output element
// and no step reads a device value on the host.
//
// K6b is the decode kernel's role swap (K3c, mxq_gemm_skinny.cu) with the activation rows grouped by expert: 128 weight rows of one
// expert are the MMA M dimension and up to N_TOK = 32 / 64 / 128 routed rows of that expert the MMA N dimension.  The grid is sized
// from what the host knows (rows, experts, N): CTA (window, tile) finds the expert whose window it is from the device offsets and
// exits before loading anything when there is none, so an expert with no rows costs no weight bytes.  Warp 0 TMA producer, warp 1
// MMA issuer, warps 2 / 3 scale-factor loaders (W / routed rows), warps 4..7 epilogue; no split-K, one accumulator.
#include "mxq_quant_core.cuh"
#include "mxq_tc.cuh"

namespace mxq {
namespace moe {

using namespace gemm;

// ================================ K6a: route ================================
constexpr int kRouteThreads = 1024;

// One CTA.  Pass 1 counts the rows of each expert (shared atomics only count; they decide no position).  Pass 2 walks the
// slots in tiles of 1024 in (token, slot) order: a slot's position is its expert's base + the slots of the same expert in
// earlier warps of the tile + its rank among the lanes of its warp that share the expert (match.any) -- deterministic.
__global__ void __launch_bounds__(kRouteThreads) route_kernel(const int64_t* __restrict__ idx, int n_slots, int top_k, int E,
                                                              int32_t* __restrict__ offsets, int32_t* __restrict__ row_of_slot,
                                                              int32_t* __restrict__ token_of_row) {
    __shared__ int cnt[MXQ_MOE_MAX_EXPERTS + 1];
    __shared__ int base[MXQ_MOE_MAX_EXPERTS];
    __shared__ int warp_cnt[kRouteThreads / 32][MXQ_MOE_MAX_EXPERTS];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_wait();
    pdl_launch_dependents();
    for (int e = tid; e < E; e += kRouteThreads) cnt[e] = 0;
    __syncthreads();
    for (int i = tid; i < n_slots; i += kRouteThreads) {
        const int64_t e = idx[i];
        if (e >= 0 && e < E) atomicAdd(&cnt[e], 1);
    }
    __syncthreads();
    if (warp == 0) {  // exclusive scan of the counts, 32 experts per step
        int carry = 0;
        for (int e0 = 0; e0 < E; e0 += 32) {
            const int e = e0 + lane;
            const int c = e < E ? cnt[e] : 0;
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += v;
            }
            if (e < E) { base[e] = carry + incl - c; offsets[e] = carry + incl - c; }
            carry += __shfl_sync(0xFFFFFFFFu, incl, 31);
        }
        if (lane == 0) offsets[E] = carry;
    }
    int* wc = &warp_cnt[0][0];
    for (int t0 = 0; t0 < n_slots; t0 += kRouteThreads) {
        for (int j = tid; j < (kRouteThreads / 32) * MXQ_MOE_MAX_EXPERTS; j += kRouteThreads) wc[j] = 0;
        __syncthreads();  // (the first pass: also publishes base[])
        const int i = t0 + tid;
        const int64_t e64 = i < n_slots ? idx[i] : -1;
        const bool valid = e64 >= 0 && e64 < E;
        const int e = valid ? (int)e64 : -1;
        const unsigned same = __match_any_sync(0xFFFFFFFFu, e);
        const int rank = __popc(same & ((1u << lane) - 1u));
        if (valid && rank == 0) warp_cnt[warp][e] = __popc(same);
        __syncthreads();
        if (valid) {
            int pos = base[e] + rank;
            for (int w = 0; w < warp; ++w) pos += warp_cnt[w][e];
            row_of_slot[i] = pos;
            token_of_row[pos] = i / top_k;
        } else if (i < n_slots) {
            row_of_slot[i] = -1;
        }
        __syncthreads();
        for (int x = tid; x < E; x += kRouteThreads) {
            int s = 0;
            for (int w = 0; w < kRouteThreads / 32; ++w) s += warp_cnt[w][x];
            base[x] += s;
        }
        __syncthreads();  // before the next tile clears warp_cnt / reads base
    }
}

// routed row r <- quantize_mx(x[token_of_row[r]], ELEM, 32): one thread per 32-element block (K1's quantize_block32)
template <int ELEM>
__global__ void __launch_bounds__(256) route_quantize_kernel(const uint16_t* __restrict__ x, int64_t ldx, int blocks_per_row,
                                                             const int32_t* __restrict__ offsets, int E, const int32_t* __restrict__ token_of_row,
                                                             int64_t n_blocks, uint8_t* __restrict__ codes, uint8_t* __restrict__ scales,
                                                             uint32_t flags) {
    constexpr int CB = ELEM == MXQ_ELEM_E2M1 ? 16 : 32;  // code bytes per block
    pdl_wait();
    pdl_launch_dependents();
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const int64_t r = b / blocks_per_row;
    const int kb = (int)(b % blocks_per_row);
    if (r >= offsets[E]) return;
    const uint4* src = reinterpret_cast<const uint4*>(x + (int64_t)token_of_row[r] * ldx + kb * 32);
    uint32_t w[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 v = src[q];
        w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
    uint32_t out[CB / 4];
    const int s = quantize_block32<ELEM>(w, (flags & MXQ_FLAG_HW_EXACT) != 0, out);
    uint4* dst = reinterpret_cast<uint4*>(codes + b * CB);
    dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
    if constexpr (CB == 32) dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
    scales[b] = (uint8_t)s;
}

// ================================ K6b: grouped GEMM ================================
constexpr int kThreadsG = 256;
constexpr int TILE_W = 128;
constexpr int SF_KB_BYTES = 512;

struct GemmParams {
    const uint8_t* sfw; const uint8_t* sfx; uint16_t* d;
    const int32_t* offsets;
    int R, N, K, E, n_tiles;
    uint32_t idesc_fmt, tx;
};

template <int N_TOK, int STAGES>
struct GSmem {
    static constexpr int W_STAGE = TILE_W * BLOCK_K;
    static constexpr int X_STAGE = N_TOK * BLOCK_K;
    static constexpr int SF_STAGE = SF_KB * SF_KB_BYTES;
    static constexpr int OFF_W = 0;
    static constexpr int OFF_X = OFF_W + STAGES * W_STAGE;
    static constexpr int OFF_SFW = OFF_X + STAGES * X_STAGE;
    static constexpr int OFF_SFX = OFF_SFW + SF_STAGES * SF_STAGE;
    static constexpr int OFF_BAR = OFF_SFX + SF_STAGES * SF_STAGE;
    static constexpr int NUM_BARS = 2 * STAGES + 2 * SF_STAGES + 1;
    static constexpr int OFF_TMEM_PTR = OFF_BAR + NUM_BARS * 8;
    static constexpr int OFF_SEG = OFF_TMEM_PTR + 16;  // expert, first row, end of the expert's segment
    static constexpr int TOTAL = OFF_SEG + 16;
    static constexpr int DYN_BYTES = TOTAL + 1024;
    static_assert(DYN_BYTES <= 227 * 1024, "shared memory budget");
};

template <int N_TOK, int STAGES>
__global__ void __launch_bounds__(kThreadsG, 1) moe_gemm_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x,
                                                              const GemmParams p) {
    using L = GSmem<N_TOK, STAGES>;
    constexpr int TMEM_NEED = N_TOK + 16;
    constexpr int TMEM_COLS = TMEM_NEED <= 64 ? 64 : (TMEM_NEED <= 128 ? 128 : 256);
    constexpr uint32_t TM_SF = N_TOK, SF_BUF_COLS = 8;  // two buffers of (4 W + 4 X) scale-factor columns

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    int* seg = reinterpret_cast<int*>(smem + L::OFF_SEG);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x % p.n_tiles, win = blockIdx.x / p.n_tiles;

    pdl_wait();  // the offsets and the routed rows are written by the preceding kernels of the stream
    if (warp == 0) {
        // window `win` of the enumeration (expert 0's windows, expert 1's, ...): which expert, which of its windows
        int acc = 0, found = -1, j = 0;
        for (int e0 = 0; e0 < p.E && found < 0; e0 += 32) {
            const int e = e0 + lane;
            const int c = e < p.E ? p.offsets[e + 1] - p.offsets[e] : 0;
            const int w = (c + N_TOK - 1) / N_TOK;
            int incl = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned hit = __ballot_sync(0xFFFFFFFFu, win >= acc + incl - w && win < acc + incl);
            if (hit) {
                const int src = __ffs(hit) - 1;
                found = e0 + src;
                j = win - acc - __shfl_sync(0xFFFFFFFFu, incl - w, src);
            }
            acc += __shfl_sync(0xFFFFFFFFu, incl, 31);
        }
        if (lane == 0) {
            seg[0] = found;
            if (found >= 0) { seg[1] = p.offsets[found] + j * N_TOK; seg[2] = p.offsets[found + 1]; }
        }
    }
    __syncthreads();
    const int expert = seg[0];
    if (expert < 0) return;  // no window here: nothing loaded, nothing stored
    const int row0 = seg[1], row_end = seg[2];
    const int w_row0 = expert * p.N + tile * TILE_W;

    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::OFF_BAR);
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;
    uint64_t* sf_full = bars + 2 * STAGES;
    uint64_t* sf_empty = sf_full + SF_STAGES;
    uint64_t* tmem_full = sf_empty + SF_STAGES;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L::OFF_TMEM_PTR);
    const int k_blocks = p.K / BLOCK_K;

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_w);
        tma_prefetch_desc(&map_x);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < SF_STAGES; ++i) { mbar_init(&sf_full[i], 2); mbar_init(&sf_empty[i], 1); }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
    }
    __syncwarp();
    if (warp == 3) tmem_alloc<TMEM_COLS>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    pdl_launch_dependents();

    if (warp == 0) {
        // ================= TMA producer =================
        if (elect_one()) {
            uint32_t stage = 0, phase = 0;
            for (int kb = 0; kb < k_blocks; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                mbar_arrive_expect_tx(&full[stage], p.tx);
                tma_load_3d(&map_w, &full[stage], smem + L::OFF_W + stage * L::W_STAGE, kb * BLOCK_K, w_row0, 0);
                tma_load_3d(&map_x, &full[stage], smem + L::OFF_X + stage * L::X_STAGE, kb * BLOCK_K, row0, 0);  // (rows past R read as 0)
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        const uint32_t idesc = make_idesc(TILE_W, N_TOK) | p.idesc_fmt;
        constexpr uint64_t HI_OPERAND = ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)kLayoutSw128 << 61);
        constexpr uint64_t HI_SF = ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)kLayoutNone << 61);
        const uint32_t w_lo0 = smem_u32(smem + L::OFF_W) >> 4, x_lo0 = smem_u32(smem + L::OFF_X) >> 4;
        const uint32_t sfw_lo0 = smem_u32(smem + L::OFF_SFW) >> 4, sfx_lo0 = smem_u32(smem + L::OFF_SFX) >> 4;
        const uint32_t tm_sf0 = tmem_base + TM_SF;
        const int n_groups = (k_blocks + SF_KB - 1) / SF_KB;
        uint32_t sfs = 0, sf_phase = 0, sf_sel = 0;
        for (int g = 0; g < n_groups; ++g) {
            mbar_wait(&sf_full[sfs], sf_phase);
#pragma unroll
            for (int j = 0; j < SF_KB; ++j) {
                const int kb = g * SF_KB + j;
                if (kb < k_blocks) {
                    const uint32_t stage = (uint32_t)(kb % STAGES), phase = (uint32_t)((kb / STAGES) & 1);
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t w_lo = w_lo0 + stage * (L::W_STAGE >> 4), x_lo = x_lo0 + stage * (L::X_STAGE >> 4);
                        const uint32_t sf_off = sfs * (L::SF_STAGE >> 4) + j * (SF_KB_BYTES >> 4);
                        const uint32_t tm_sfw = tm_sf0 + sf_sel * SF_BUF_COLS, tm_sfx = tm_sfw + 4;
                        tc_copy_sf(tm_sfw, HI_SF | (sfw_lo0 + sf_off));
                        tc_copy_sf(tm_sfx, HI_SF | (sfx_lo0 + sf_off));
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                            tc_mma_mx(tmem_base, HI_OPERAND | (w_lo + k * (UMMA_K >> 4)), HI_OPERAND | (x_lo + k * (UMMA_K >> 4)), idesc_with_sf(idesc, k, k),
                                      !(kb == 0 && k == 0), tm_sfw, tm_sfx);
                        tc_commit(&empty[stage]);
                    }
                    __syncwarp();
                    sf_sel ^= 1;
                }
            }
            if (elect_one()) tc_commit(&sf_empty[sfs]);
            __syncwarp();
            if (++sfs == SF_STAGES) { sfs = 0; sf_phase ^= 1; }
        }
        if (elect_one()) tc_commit(tmem_full);
        __syncwarp();
    } else if (warp == 2 || warp == 3) {
        // ================= scale-factor loaders (warp 2: the 128 weight rows, warp 3: the routed rows) =================
        uint32_t sfs = 0, sf_phase = 0;
        auto arrive = [&](uint32_t st) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sf_full[st]);
        };
        const int64_t ld_sf = p.K / 32;
        if (warp == 2)
            sf_load_tile4<1>(p.sfw, ld_sf, w_row0, p.E * p.N, k_blocks, smem + L::OFF_SFW, SF_KB_BYTES, sf_empty, sfs, sf_phase, lane, arrive);
        else
            sf_load_tile4<1>(p.sfx, ld_sf, row0, p.R, k_blocks, smem + L::OFF_SFX, SF_KB_BYTES, sf_empty, sfs, sf_phase, lane, arrive);
    } else {
        // ================= epilogue: accumulator lane = weight row, column = routed row; rows outside the segment are not stored =====
        const int quad = warp & 3;
        const int n = tile * TILE_W + quad * 32 + lane;
        mbar_wait(tmem_full, 0);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < N_TOK / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quad * 32) << 16) + c * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int r = row0 + c * 32 + i;
                if (r < row_end) p.d[(int64_t)r * p.N + n] = (uint16_t)pack_bf16x2(__uint_as_float(v[i]), 0.0f);
            }
        }
        tc_fence_before();
    }
    __syncwarp();
    __syncthreads();
    if (warp == 3) {
        tc_fence_after();
        tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

template <int N_TOK, int STAGES>
static int launch_gemm_t(const mxq_moe_gemm_args_t* a, int device, cudaStream_t stream, char* msg, size_t msg_len) {
    using L = GSmem<N_TOK, STAGES>;
    const int64_t ldw = a->K * operand_bits(a->w_format) / 8, ldx = a->K * operand_bits(a->x_format) / 8;
    CUtensorMap mw, mx;
    if (!cached_operand_map(&mw, a->w_codes, a->K, a->num_experts * a->N, 1, ldw, 0, TILE_W, a->w_format, device) ||
        !cached_operand_map(&mx, a->x_codes, a->K, a->rows, 1, ldx, 0, N_TOK, a->x_format, device)) {
        snprintf(msg, msg_len, "cuTensorMapEncodeTiled failed (driver entry point missing or invalid strides)");
        return MXQ_ERR_UNSUPPORTED_SHAPE;
    }
    auto kernel = moe_gemm_kernel<N_TOK, STAGES>;
    cudaError_t e = ensure_smem_attr((const void*)kernel, L::DYN_BYTES, device);
    if (e != cudaSuccess) { snprintf(msg, msg_len, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    GemmParams p;
    p.sfw = a->w_scales; p.sfx = a->x_scales; p.d = (uint16_t*)a->d; p.offsets = a->offsets;
    p.R = (int)a->rows; p.N = (int)a->N; p.K = (int)a->K; p.E = (int)a->num_experts;
    p.n_tiles = (int)(a->N / TILE_W);
    p.idesc_fmt = idesc_formats(a->w_format, a->x_format);  // the weights are the MMA A operand, the routed rows the B operand
    p.tx = (uint32_t)((TILE_W * operand_bits(a->w_format) + N_TOK * operand_bits(a->x_format)) * BLOCK_K / 8);
    // sum over experts of ceil(rows_e / N_TOK) <= (experts with rows) + rows / N_TOK
    const int64_t windows = (a->num_experts < a->rows ? a->num_experts : a->rows) + (a->rows + N_TOK - 1) / N_TOK;
    e = launch_pdl(kernel, dim3((unsigned)(windows * p.n_tiles)), dim3(kThreadsG), L::DYN_BYTES, stream, mw, mx, p);
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

// ================================ K6c: combine ================================
// one thread per (token, 8 channels): the token's slots sorted by expert (ties by slot), products and sums rounded as the loop rounds
template <bool BF16_W>
__global__ void __launch_bounds__(256) combine_kernel(const uint16_t* __restrict__ y, const int64_t* __restrict__ idx, const void* __restrict__ wts,
                                                      const int32_t* __restrict__ row_of_slot, int64_t tokens, int top_k, int E, int64_t hidden,
                                                      uint16_t* __restrict__ out) {
    pdl_wait();
    pdl_launch_dependents();
    const int64_t chunks = hidden / 8;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= tokens * chunks) return;
    const int64_t t = i / chunks, c0 = (i % chunks) * 8;
    int ex[MXQ_MOE_MAX_TOP_K], sl[MXQ_MOE_MAX_TOP_K];
    int n = 0;
    for (int s = 0; s < top_k; ++s) {  // insertion by (expert, slot)
        const int64_t e64 = idx[t * top_k + s];
        if (e64 < 0 || e64 >= E) continue;
        const int e = (int)e64;
        int j = n++;
        while (j > 0 && ex[j - 1] > e) { ex[j] = ex[j - 1]; sl[j] = sl[j - 1]; --j; }
        ex[j] = e; sl[j] = s;
    }
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.0f;
    for (int j = 0; j < n; ++j) {
        const int s = sl[j];
        const float w = BF16_W ? __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(wts)[t * top_k + s] << 16)
                               : reinterpret_cast<const float*>(wts)[t * top_k + s];
        const uint4 v = *reinterpret_cast<const uint4*>(y + (int64_t)row_of_slot[t * top_k + s] * hidden + c0);
        const uint32_t vw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float yv = __uint_as_float(q & 1 ? (vw[q / 2] & 0xFFFF0000u) : (vw[q / 2] << 16));
            const float contrib = __uint_as_float(pack_bf16x2(__fmul_rn(yv, w), 0.0f) << 16);
            acc[q] = __uint_as_float(pack_bf16x2(__fadd_rn(acc[q], contrib), 0.0f) << 16);
        }
    }
    uint32_t o[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = pack_bf16x2(acc[2 * q], acc[2 * q + 1]);
    *reinterpret_cast<uint4*>(out + t * hidden + c0) = make_uint4(o[0], o[1], o[2], o[3]);
}

}  // namespace moe

int launch_moe_route(const mxq_moe_route_args_t* a, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace moe;
    const int n_slots = (int)(a->tokens * a->top_k);
    cudaError_t e = launch_pdl(route_kernel, dim3(1), dim3(kRouteThreads), 0, stream, a->top_k_index, n_slots, a->top_k, a->num_experts,
                               a->offsets, a->row_of_slot, a->token_of_row);
    if (e != cudaSuccess) { snprintf(msg, msg_len, "route launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    if (a->codes == nullptr) return MXQ_OK;
    const int bpr = (int)(a->hidden / 32);
    const int64_t n_blocks = (int64_t)n_slots * bpr;
    const dim3 grid((unsigned)((n_blocks + 255) / 256));
    const uint16_t* x = (const uint16_t*)a->x;
    uint8_t* c8 = (uint8_t*)a->codes;
    const uint32_t fl = (uint32_t)a->flags;
    switch (a->elem) {
    case MXQ_ELEM_E4M3: e = launch_pdl(route_quantize_kernel<MXQ_ELEM_E4M3>, grid, dim3(256), 0, stream, x, a->ldx, bpr, a->offsets, a->num_experts, a->token_of_row, n_blocks, c8, a->scales, fl); break;
    case MXQ_ELEM_E3M2: e = launch_pdl(route_quantize_kernel<MXQ_ELEM_E3M2>, grid, dim3(256), 0, stream, x, a->ldx, bpr, a->offsets, a->num_experts, a->token_of_row, n_blocks, c8, a->scales, fl); break;
    case MXQ_ELEM_E2M3: e = launch_pdl(route_quantize_kernel<MXQ_ELEM_E2M3>, grid, dim3(256), 0, stream, x, a->ldx, bpr, a->offsets, a->num_experts, a->token_of_row, n_blocks, c8, a->scales, fl); break;
    case MXQ_ELEM_E2M1: e = launch_pdl(route_quantize_kernel<MXQ_ELEM_E2M1>, grid, dim3(256), 0, stream, x, a->ldx, bpr, a->offsets, a->num_experts, a->token_of_row, n_blocks, c8, a->scales, fl); break;
    case MXQ_ELEM_INT8: e = launch_pdl(route_quantize_kernel<MXQ_ELEM_INT8>, grid, dim3(256), 0, stream, x, a->ldx, bpr, a->offsets, a->num_experts, a->token_of_row, n_blocks, c8, a->scales, fl); break;
    case MXQ_ELEM_E5M2: e = launch_pdl(route_quantize_kernel<MXQ_ELEM_E5M2>, grid, dim3(256), 0, stream, x, a->ldx, bpr, a->offsets, a->num_experts, a->token_of_row, n_blocks, c8, a->scales, fl); break;
    default: snprintf(msg, msg_len, "unknown element type %d", a->elem); return MXQ_ERR_INVALID;
    }
    if (e != cudaSuccess) { snprintf(msg, msg_len, "route quantize launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

// N_TOK from the mean rows per expert: decode (a few rows per hit expert) streams the weights once per 32 rows
int launch_moe_gemm(const mxq_moe_gemm_args_t* a, int device, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace moe;
    const int64_t mean = (a->rows + a->num_experts - 1) / a->num_experts;
    if (mean <= 32) return launch_gemm_t<32, 8>(a, device, stream, msg, msg_len);
    if (mean <= 64) return launch_gemm_t<64, 8>(a, device, stream, msg, msg_len);
    return launch_gemm_t<128, 6>(a, device, stream, msg, msg_len);
}

int launch_moe_combine(const mxq_moe_combine_args_t* a, cudaStream_t stream, char* msg, size_t msg_len) {
    using namespace moe;
    const int64_t n = a->tokens * (a->hidden / 8);
    const dim3 grid((unsigned)((n + 255) / 256));
    const cudaError_t e =
        a->weights_dtype == MXQ_HP_BF16
            ? launch_pdl(combine_kernel<true>, grid, dim3(256), 0, stream, (const uint16_t*)a->y, a->top_k_index, a->top_k_weights, a->row_of_slot, a->tokens, a->top_k,
                         a->num_experts, a->hidden, (uint16_t*)a->out)
            : launch_pdl(combine_kernel<false>, grid, dim3(256), 0, stream, (const uint16_t*)a->y, a->top_k_index, a->top_k_weights, a->row_of_slot, a->tokens, a->top_k,
                         a->num_experts, a->hidden, (uint16_t*)a->out);
    if (e != cudaSuccess) { snprintf(msg, msg_len, "launch: %s", cudaGetErrorString(e)); return MXQ_ERR_CUDA; }
    return MXQ_OK;
}

}  // namespace mxq
