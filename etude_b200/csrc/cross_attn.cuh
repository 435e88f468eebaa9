// Cross-attention of the frequency-axis decoder with its K|V projection FUSED in: per frame f (256 encoder tokens x_f),
// head h and decoder layer l,  K_h | V_h = x_f [Wk_h; Wv_h]^T + b,  out = softmax(Q_h K_h^T / 8) V_h  for the 88 note
// queries (reference amt_apc.py:159-183 with MultiHeadAttentionLayer.forward, amt_apc.py:342-368).
//
// Why: as two kernels the K|V of every encoder token (1 KB per layer) went to HBM and came back (gemm_bstat writing
// 3 KB per token for the three layers, then one attention4 launch per layer): the largest block of HBM traffic of the
// forward pass that the math does not need.  Fused, per token only x (512 B) is read, per note the context written.
//
// One CTA per SM walks frames.  x_f stays resident in smem (4 K-chunks [256 tokens x 64] SW128, 128 KB) for the four
// heads.  The projection is TRANSPOSED so that it runs at the efficient N = 256 shape:
//   D[128 x 256 tokens] = [Wk_h; Wv_h] (A: [128 x 32] SW64 chunks streamed from L2) * x_f^T (B: the resident chunks)
// so TMEM lane r is output channel r (rows 0-63 K_h, 64-127 V_h) and the bias is one scalar per thread.  The epilogue
// adds it, rounds to bf16 (the rounding point of gemm_bstat's epilogue) and writes K_h^T and V_h^T, both stored as
// [key / 64][64 channel rows][128 B of keys] SW128: K_h^T is the MN-major B operand of S = Q K^T, V_h^T the K-major B
// operand of O = P V.  The attention is attention4's math for one query tile and two 128-key blocks: S_j into a
// 128-column buffer, per-block integer log2 reference, P bf16 over S, O_j = P_j V_j (TS MMA) in the buffer's columns
// [64, 128), and the drain's exact combination of the two blocks.  Queries: the input-independent q0 table (layer 0) or
// 128-row boxes of dq at row 88 f (layers 1 and 2; rows 88-127 belong to the next frame and only reach pad rows).
//
// TMEM (512 columns): [0, 256) projection accumulator, [256, 384) / [384, 512) the S / P / O buffers of key blocks 0 / 1.
// smem: x 128 KB | W ring 2 x 8 KB | K^T 32 KB | V^T 32 KB | Q 16 KB | statistics 2 KB | barriers  (226.25 KB of 227).
// Warps (24): 0 TMA producer (x, W ring, Q), 1 projection MMA issue (+ TMEM alloc), 2 S issue, 3 P V issue, 4-11 projection
// epilogue (key block (warp - 4) >> 2, lane quarter warp & 3), 12-15 drain, 16-19 / 20-23 softmax of key block 0 / 1.
// The projection of unit u + 1 = (frame, head) runs while unit u is in softmax; its epilogue waits for P V(u) of the block.
// Rows 96-127 of a query tile are padding: their softmax warps only keep the barrier protocol.
#pragma once
#include "attention4.cuh"
#include "common.cuh"

namespace etude {

constexpr int kXaThreads = 24 * 32;
constexpr int kXaXBytes = 4 * 256 * 64 * 2;     // 128 KB: x_f, 4 K-chunks of [256 tokens x 64 channels]
constexpr int kXaXChunkBytes = 256 * 64 * 2;
constexpr int kXaWStages = 2;
constexpr int kXaWStageBytes = 128 * 32 * 2;    // [Wk_h; Wv_h] rows x 32 input channels, SW64
constexpr int kXaKVBytes = 4 * 64 * 128;        // K^T (or V^T) of 256 keys: 4 atoms of 64 keys x 64 channel rows x 128 B
constexpr int kXaQBytes = 128 * 64 * 2;
constexpr int kXaStatBytes = 2 * 2 * 128 * 4;   // m[2 blocks][128], l[2 blocks][128]
constexpr size_t kCrossAttnSmemBytes = kXaXBytes + kXaWStages * kXaWStageBytes + 2 * kXaKVBytes + kXaQBytes + kXaStatBytes + 256;
static_assert(kCrossAttnSmemBytes <= 232448, "cross_attn smem over the 227 KB opt-in limit");

struct CrossAttnParams {
    int n_frames;               // sequences of 256 encoder tokens
    int q_seq_stride;           // Q rows between frames: 88 (dq) or 0 (the shared q0 table)
    const float* bias;          // [4 heads][128]: bk_h | bv_h (the rows of the head-major weight [Wk_h; Wv_h])
    __nv_bfloat16* out;         // context [n_frames * 88, 256]
    float scale_log2e;
};

// Shared-memory descriptor of a K-major operand in 64-byte swizzled rows (8 rows x 64 B = 512 B per core group; layout 4)
__device__ __forceinline__ uint64_t make_sw64_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}

__global__ void __launch_bounds__(kXaThreads, 1)
cross_attn_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                  const __grid_constant__ CUtensorMap tmap_q, const CrossAttnParams p) {
    constexpr int BUF0_COL = 256, BUF_COLS = 128, O_COL = 64;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem_raw) & 1023u) != 0) __trap();
    uint8_t* sX = smem;
    uint8_t* sW = sX + kXaXBytes;
    uint8_t* sKT = sW + kXaWStages * kXaWStageBytes;
    uint8_t* sVT = sKT + kXaKVBytes;
    uint8_t* sQ = sVT + kXaKVBytes;
    float* s_m = reinterpret_cast<float*>(sQ + kXaQBytes);   // [2 blocks][128] block reference ceil(max * scale)
    float* s_l = s_m + 2 * 128;                                // [2 blocks][128] block sum of 2^(s * scale - m)
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_l + 2 * 128);
    uint64_t* x_full = bars;                 // [4] x chunk landed
    uint64_t* x_empty = x_full + 4;          // [4] the last head's projection MMAs have read the chunk
    uint64_t* w_full = x_empty + 4;          // [2]
    uint64_t* w_empty = w_full + 2;          // [2]
    uint64_t* q_full = w_empty + 2;
    uint64_t* q_empty = q_full + 1;          // S MMAs of both blocks complete
    uint64_t* acc_full = q_empty + 1;        // projection accumulator complete   (MMA commit -> epilogue)
    uint64_t* acc_free = acc_full + 1;       // count 8: accumulator read         (epilogue warps -> projection MMA)
    uint64_t* kv_full = acc_free + 1;        // [2] count 4: K^T / V^T of block j written (epilogue group j -> S, P V issue)
    uint64_t* kv_free = kv_full + 2;         // [2] P V_j complete: block j of K^T / V^T reusable (MMA commit -> epilogue)
    uint64_t* s_full = kv_free + 2;          // [2] S_j complete                  (MMA commit -> softmax j)
    uint64_t* p_full = s_full + 2;           // [2] count 4: P_j and statistics   (softmax j -> P V issue, drain)
    uint64_t* o_full = p_full + 2;           // [2] O_j complete                  (MMA commit -> drain)
    uint64_t* buf_free = o_full + 2;         // [2] count 4: O_j read             (drain -> S issue)
    uint32_t* tmem_base_ptr = reinterpret_cast<uint32_t*>(buf_free + 2);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int my_frames = ((int)blockIdx.x < p.n_frames) ? (p.n_frames - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int N = my_frames * 4;   // (frame, head) units

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmap_x);
        tma_prefetch_desc(&tmap_w);
        tma_prefetch_desc(&tmap_q);
        for (int i = 0; i < 4; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
        for (int i = 0; i < kXaWStages; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
        mbar_init(q_full, 1); mbar_init(q_empty, 1);
        mbar_init(acc_full, 1); mbar_init(acc_free, 8);
        for (int j = 0; j < 2; ++j) {
            mbar_init(&kv_full[j], 4); mbar_init(&kv_free[j], 1);
            mbar_init(&s_full[j], 1); mbar_init(&p_full[j], 4);
            mbar_init(&o_full[j], 1); mbar_init(&buf_free[j], 4);
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(tmem_base_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_ptr;

    if (warp < 4) {
      reg_dec<40>();
      if (warp == 0) {
        // ===================================================== TMA producer: x_f chunks, the W ring, Q of every unit
        const bool leader = elect_one();
        uint32_t wc = 0;
        auto load_w = [&](int u, int c) {
            const uint32_t s = wc % kXaWStages;
            mbar_wait_inl(&w_empty[s], ((wc / kXaWStages) & 1) ^ 1);
            if (leader) {
                mbar_expect_tx(&w_full[s], kXaWStageBytes);
                tma_load_2d(sW + s * kXaWStageBytes, &tmap_w, &w_full[s], c * 32, (u & 3) * 128);
            }
            ++wc;
        };
        for (int u = 0; u < N; ++u) {
            const int f = (int)blockIdx.x + (u >> 2) * (int)gridDim.x, h = u & 3;
            if (h == 0)
                for (int c = 0; c < 4; ++c) {
                    mbar_wait_inl(&x_empty[c], ((u >> 2) & 1) ^ 1);
                    if (leader) {
                        mbar_expect_tx(&x_full[c], kXaXChunkBytes);
                        tma_load_2d(sX + c * kXaXChunkBytes, &tmap_x, &x_full[c], c * 64, f * 256);
                    }
                }
            load_w(u, 0);
            load_w(u, 1);
            mbar_wait_inl(q_empty, (u & 1) ^ 1);
            if (leader) {
                mbar_expect_tx(q_full, kXaQBytes);
                tma_load_2d(sQ, &tmap_q, q_full, h * kHeadDim, f * p.q_seq_stride);
            }
            for (int c = 2; c < 8; ++c) load_w(u, c);
            __syncwarp();
        }
      } else if (warp == 1) {
        // ===================================================== projection MMA issue: D[128 x 256] = [Wk_h; Wv_h] x_f^T
        const bool leader = elect_one();
        constexpr uint32_t idesc_p = make_idesc_bf16(128, 256, 0, 0);
        const uint64_t x_desc0 = make_sw128_desc(smem_u32(sX));
        const uint64_t w_desc0 = make_sw64_desc(smem_u32(sW));
        uint32_t wc = 0;
        for (int u = 0; u < N; ++u) {
            const int h = u & 3;
            mbar_wait_inl(acc_free, (u & 1) ^ 1);
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < 8; ++c, ++wc) {   // 32 input channels per W chunk: x chunk c / 2, bytes [64 (c & 1), + 64) of its rows
                const uint32_t s = wc % kXaWStages;
                if (h == 0 && (c & 1) == 0) mbar_wait_inl(&x_full[c >> 1], (u >> 2) & 1);
                mbar_wait_inl(&w_full[s], (wc / kXaWStages) & 1);
                tc_fence_after();
                if (leader) {
                    const uint64_t ad = w_desc0 + (uint64_t)(s * (kXaWStageBytes >> 4));
                    const uint64_t bd = x_desc0 + (uint64_t)((c >> 1) * (kXaXChunkBytes >> 4) + (c & 1) * 4);
#pragma unroll
                    for (int k = 0; k < 2; ++k) umma_bf16_ss(tmem_base, ad + 2 * k, bd + 2 * k, idesc_p, (c | k) ? 1u : 0u);
                    tc_commit(&w_empty[s]);
                    if (h == 3 && (c & 1)) tc_commit(&x_empty[c >> 1]);
                }
                __syncwarp();
            }
            if (leader) tc_commit(acc_full);
            __syncwarp();
        }
      } else if (warp == 2) {
        // ===================================================== S_j = Q K_j^T issue (K^T block j: two 64-key atoms, MN-major)
        const bool leader = elect_one();
        constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 1);
        const uint64_t q_desc = make_sw128_desc(smem_u32(sQ));
        const uint64_t k_desc0 = make_sw128_desc(smem_u32(sKT), 8192);   // LBO = 64-key atom stride
        for (int u = 0; u < N; ++u) {
            mbar_wait_inl(q_full, u & 1);
#pragma unroll 1
            for (int j = 0; j < 2; ++j) {
                mbar_wait_inl(&kv_full[j], u & 1);
                mbar_wait_inl(&buf_free[j], (u & 1) ^ 1);
                tc_fence_after();
                if (leader) {
                    const uint64_t kd = k_desc0 + (uint64_t)(j * (16384 >> 4));
                    const uint32_t tmem_s = tmem_base + BUF0_COL + j * BUF_COLS;
#pragma unroll
                    for (int k = 0; k < 4; ++k)   // 16 channels = two 8-row core groups = 2048 B further
                        umma_bf16_ss(tmem_s, q_desc + 2 * k, kd + (uint64_t)(k * 128), idesc_s, k != 0);
                    tc_commit(&s_full[j]);
                    if (j == 1) tc_commit(q_empty);
                }
                __syncwarp();
            }
        }
      } else {
        // ===================================================== O_j = P_j V_j issue (V^T K-major: 64 keys per 128-byte row)
        const bool leader = elect_one();
        constexpr uint32_t idesc_o = make_idesc_bf16(128, kHeadDim, 0, 0);
        const uint64_t v_desc0 = make_sw128_desc(smem_u32(sVT));
        for (int u = 0; u < N; ++u) {
#pragma unroll 1
            for (int j = 0; j < 2; ++j) {
                mbar_wait_inl(&kv_full[j], u & 1);
                mbar_wait_inl(&p_full[j], u & 1);
                tc_fence_after();
                if (leader) {
                    const uint32_t tmem_buf = tmem_base + BUF0_COL + j * BUF_COLS;
#pragma unroll
                    for (int s = 0; s < 8; ++s) {   // keys 128 j + 16 s: atom 2 j + s / 4, bytes 32 (s & 3) of its rows
                        const uint64_t vd = v_desc0 + (uint64_t)((2 * j + (s >> 2)) * (8192 >> 4) + (s & 3) * 2);
                        umma_bf16_ts(tmem_buf + O_COL, tmem_buf + s * 8, vd, idesc_o, s != 0);
                    }
                    tc_commit(&o_full[j]);
                    tc_commit(&kv_free[j]);
                }
                __syncwarp();
            }
        }
      }
    } else if (warp < 12) {
        // ===================================================== projection epilogue: group j writes keys [128 j, 128 j + 128)
        reg_inc<88>();
        const int j = (warp - 4) >> 2, q = warp & 3;
        const int r = q * 32 + lane;                 // output channel = TMEM lane: K_h rows 0-63, V_h rows 64-127
        const int d = r & 63, sw = d & 7;
        const uint32_t lane_off = (uint32_t)(q * 32) << 16;
        const uint32_t dst_row = smem_u32(r < 64 ? sKT : sVT) + d * 128;
        float v[32];
        for (int u = 0; u < N; ++u) {
            const float b = __ldg(p.bias + (u & 3) * 128 + r);
            mbar_wait_inl(acc_full, u & 1);
            mbar_wait_inl(&kv_free[j], (u & 1) ^ 1);   // P V(u - 1) of this block has read K^T / V^T (and S before it)
            __syncwarp();
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {            // tokens [128 j + 32 c, + 32): atom 2 j + c / 2, 16-byte chunks 4 (c & 1) + g
                tmem_ld32(tmem_base + lane_off + j * 128 + c * 32, v);
                tc_wait_ld();
                const uint32_t row = dst_row + (uint32_t)((2 * j + (c >> 1)) * 8192);
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const uint32_t x0 = pack_bf16x2(v[8 * g + 0] + b, v[8 * g + 1] + b), x1 = pack_bf16x2(v[8 * g + 2] + b, v[8 * g + 3] + b);
                    const uint32_t x2 = pack_bf16x2(v[8 * g + 4] + b, v[8 * g + 5] + b), x3 = pack_bf16x2(v[8 * g + 6] + b, v[8 * g + 7] + b);
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + (uint32_t)((((c & 1) * 4 + g) ^ sw) << 4)), "r"(x0), "r"(x1),
                                 "r"(x2), "r"(x3) : "memory");
                }
            }
            tc_fence_before();
            fence_async_smem();                      // generic-proxy stores -> visible to the tensor core
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(acc_free);
                mbar_arrive(&kv_full[j]);
            }
        }
    } else if (warp < 16) {
        // ===================================================== drain: combine the two blocks (attention4's drain) -> bf16 -> HBM
        reg_inc<112>();
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_off = (uint32_t)(q * 32) << 16;
        float acc[64];
        float v[16];
        for (int u = 0; u < N; ++u) {
            const uint32_t ph = u & 1;
            const uint32_t tmem_o0 = tmem_base + BUF0_COL + O_COL + lane_off, tmem_o1 = tmem_o0 + BUF_COLS;
            mbar_wait_inl(&p_full[0], ph);   // block 0: straight into the accumulator registers
            mbar_wait_inl(&o_full[0], ph);
            __syncwarp();
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < 4; ++c) tmem_ld16(tmem_o0 + c * 16, acc + c * 16);
            const float m0 = s_m[row], l0 = s_l[row];
            tc_wait_ld();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&buf_free[0]);
            mbar_wait_inl(&p_full[1], ph);   // block 1: exact combination of the two independently normalised blocks
            mbar_wait_inl(&o_full[1], ph);
            __syncwarp();
            tc_fence_after();
            const float m1 = s_m[128 + row], l1 = s_l[128 + row];
            const float mm = fmaxf(m0, m1);
            const float a0 = pow2_int(m0 - mm), a1 = pow2_int(m1 - mm);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                tmem_ld16(tmem_o1 + c * 16, v);
                tc_wait_ld();
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[c * 16 + i] = fmaf(acc[c * 16 + i], a0, v[i] * a1);
            }
            const float inv = rcp_fma(fmaf(l0, a0, l1 * a1));
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&buf_free[1]);
            if (row < kNotes) {
                const int f = (int)blockIdx.x + (u >> 2) * (int)gridDim.x, h = u & 3;
                __nv_bfloat16* dst = p.out + (size_t)(f * kNotes + row) * kHid + h * kHeadDim;
#pragma unroll
                for (int gq = 0; gq < 8; ++gq) {
                    uint4 pk;
                    pk.x = pack_bf16x2(acc[gq * 8 + 0] * inv, acc[gq * 8 + 1] * inv);
                    pk.y = pack_bf16x2(acc[gq * 8 + 2] * inv, acc[gq * 8 + 3] * inv);
                    pk.z = pack_bf16x2(acc[gq * 8 + 4] * inv, acc[gq * 8 + 5] * inv);
                    pk.w = pack_bf16x2(acc[gq * 8 + 6] * inv, acc[gq * 8 + 7] * inv);
                    *reinterpret_cast<uint4*>(dst + gq * 8) = pk;
                }
            }
        }
    } else {
        // ===================================================== softmax of key block j (attention4's per-block math, 128 keys)
        reg_dec<72>();
        const int j = (warp - 16) >> 2, q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t tmem_s = tmem_base + BUF0_COL + j * BUF_COLS + ((uint32_t)(q * 32) << 16);
        const float scale = p.scale_log2e;
        float v[16];
        for (int u = 0; u < N; ++u) {
            mbar_wait_inl(&s_full[j], u & 1);
            __syncwarp();
            tc_fence_after();
            if (q * 32 < kNotes) {   // lane quarter 3 holds only pad rows (96-127)
                float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    tmem_ld16(tmem_s + c * 16, v);
                    tc_wait_ld();
#pragma unroll
                    for (int i = 0; i < 16; i += 4) {
                        m0 = fmax3(m0, v[i], v[i + 1]);
                        m1 = fmax3(m1, v[i + 2], v[i + 3]);
                    }
                }
                const float m_sc = ceilf(fmaxf(m0, m1) * scale);
                float l0 = 0.f, l1 = 0.f;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    tmem_ld16(tmem_s + c * 16, v);
                    tc_wait_ld();
                    uint32_t pk[8];
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        const float e0 = ex2_approx(fmaf(v[i], scale, -m_sc));
                        const float e1 = ex2_approx(fmaf(v[i + 1], scale, -m_sc));
                        l0 += e0; l1 += e1;
                        pk[i >> 1] = pack_bf16x2(e0, e1);
                    }
                    tmem_st8(tmem_s + c * 8, pk);
                }
                s_m[j * 128 + row] = m_sc;
                s_l[j * 128 + row] = l0 + l1;
                tc_wait_st();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_full[j]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace etude
