/* etude_b200_kernels.h -- kernel-level entry points of libetude_b200.so, used by the unit tests
 * (tests/test_kernels_gpu.py) and micro-benchmarks to exercise one kernel at a time against a torch fp32
 * reference of the same op.  Same conventions as etude_b200.h.  Not needed by an integrator. */
#ifndef ETUDE_B200_KERNELS_H
#define ETUDE_B200_KERNELS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* out = epilogue(A[M,K] * W[N,K]^T + bias), bf16 operands (K contiguous), fp32 accumulation in TMEM.
 * The product library builds epilogue 0 with K == 256, N % 256 == 0 (the B-stationary projection kernel, every bias-only
 * projection of the model); the other epilogues / shapes below run the generic tile GEMM, which only
 * libetude_b200_dev.so contains (it is no longer on the product path), and fail with an error in the product library.
 * epilogue 0: bias -> bf16 [M,N];  1: bias+ReLU -> bf16 [M,N];
 * epilogue 2 (N == 256): LayerNorm(acc + bias + resid[row]) * gamma + beta -> out_f32 and out_bf16 [M,256] (both
 *   required).  resid_mod == 0: resid is fp32 [M,256].  resid_mod > 0: resid row = row % resid_mod and resid_dev is the
 *   fp32 table [resid_mod + 32, 256] whose last 32 rows repeat its first 32 (residual boxes of 32 rows never wrap).
 * K % 64 == 0, N % 256 == 0. */
int etude_k_gemm(const void* a_bf16_dev, const void* w_bf16_dev, const float* bias_dev, int M, int N, int K, int epilogue,
                 void* out_bf16_dev, const float* resid_dev, int resid_mod, const float* gamma_dev, const float* beta_dev,
                 float* out_f32_dev, void* stream);

/* Multi-head attention, 4 heads x 64: out[seq*Lq + i, 64h..] = softmax(Q_h K_h^T / 8) V_h.
 * q_dev: bf16 [q_rows, q_ld] (head h of Q at columns q_col0 + 64h; sequence s at rows s*q_seq_stride);
 * kv_dev: bf16 [n_seq*Lk, kv_ld] (K at k_col0 + 64h, V at v_col0 + 64h).  Lk in {88, 256, 512}.
 * probs_dev (optional, Lk <= 256): fp32 [n_seq, 4, Lq, Lk]. */
int etude_k_attention(const void* q_dev, int64_t q_rows, int q_ld, int q_col0, int q_seq_stride, const void* kv_dev,
                      int kv_ld, int k_col0, int v_col0, int n_seq, int Lq, int Lk, void* out_bf16_dev, float* probs_dev,
                      void* stream);

/* Cross-attention of a frequency-axis decoder layer with its K|V projection fused in (reference amt_apc.py:342-368): frames
 * of 256 encoder tokens, 88 queries, 4 heads x 64:  out[f*88 + i, 64h..] = softmax(Q_h(f) K_h^T / 8) V_h  with
 * K_h | V_h = x_f [Wk_h; Wv_h]^T + bias.  x_dev: bf16 [n_frames * 256, 256].  w_hm_dev: bf16 [512, 256] HEAD-MAJOR -- row
 * h*128 + r holds Wk row 64h + r (r < 64) or Wv row 64h + r - 64; bias_hm_dev fp32 [512] likewise.  q_dev: bf16 [q_rows, 256]
 * with frame f's queries at rows f*q_seq_stride.. (q_seq_stride 88, or 0: one table for every frame).  out_dev: bf16
 * [n_frames * 88, 256]. */
int etude_k_cross_attn(const void* x_dev, const void* w_hm_dev, const float* bias_hm_dev, const void* q_dev, int64_t q_rows,
                       int q_seq_stride, int n_frames, void* out_dev, void* stream);

/* Self-attention of an encoder layer with the Q|K|V projection fused in (reference amt_apc.py:342-368), sequences of 256
 * tokens, 4 heads x 64:  out[s*256 + i, 64h..] = softmax((x Wq_h^T + bq_h)(x Wk_h^T + bk_h)^T / 8) (x Wv_h^T + bv_h).
 * x_dev / out_dev: bf16 [n_seq * 256, 256].  w_hm_dev: bf16 [768, 256] HEAD-MAJOR -- row h*192 + r holds fc_q row 64h + r
 * (r < 64), fc_k row 64h + r - 64 (r < 128), fc_v row 64h + r - 128 otherwise; bias_hm_dev: fp32 [768] in the same order. */
int etude_k_attn_qkv(const void* x_dev, const void* w_hm_dev, const float* bias_hm_dev, int n_seq, void* out_dev, void* stream);

/* Fused token-local chain over 128-row tiles (reference amt_apc.py:250-258 / 276-284 / 304-318 with fc_o of 371):
 *   y   = LayerNorm(ctx @ Wo^T + bo + resid) * gamma + beta
 *   out = w1 ? LayerNorm(y + relu(y @ W1^T + b1) @ W2^T + b2) * gamma + beta : y
 * ctx/out bf16 [M,256]; Wo [256,256], W1 [512,256], W2 [256,512] bf16 (K contiguous); biases / gamma / beta fp32.
 * resid_dev: bf16 [resid_rows,256]; resid_mod == 0: row == token row (resid_rows == M; out may alias it);
 * resid_mod > 0: a table whose row r holds entry r % resid_mod, with resid_rows >= resid_mod + 127.
 * Pass w1 = w2 = NULL for the y-only variant. */
int etude_k_chain(const void* ctx_bf16_dev, const void* wo_bf16_dev, const float* bo_dev, const void* w1_bf16_dev,
                  const float* b1_dev, const void* w2_bf16_dev, const float* b2_dev, const float* gamma_dev, const float* beta_dev,
                  const void* resid_bf16_dev, int resid_mod, int64_t resid_rows, void* out_bf16_dev, int M, void* stream);

/* Token embedding (folded conv o linear, reference amt_apc.py:79-109) of nw windows whose first padded feature rows are
 * win_row_host[]: out bf16 [nw * 512 * 256 tokens, 256].  variant >= 16: diagnostic masks (16 + 1 no stores, + 2 no epilogue arithmetic, + 4 no A-tile build); otherwise 0. */
int etude_k_embed(etude_handle_t* h, const float* feat_dev, const int64_t* win_row_host, int n_windows, void* out_bf16_dev, int variant,
                  void* stream);

/* Output heads of the decoder (reference amt_apc.py:186-189 / 217-220, extractor.py:239-248) on a handle's window length F:
 * logits = x W^T + bias over rows of x bf16 [n_windows * F * 88, 256]; W bf16 [144, 256] (onset, offset, mpe, velocity[128],
 * padding), bias fp32 [144].  Rows are (window, frame, note) with time_major == 0, (window, note, frame) with time_major == 1.
 * Only window frames f in [keep0, keep0 + keepn) are written, at roll row out_row_host[w] + f - keep0 (fp32 rolls[0..2] get the
 * three sigmoids, int8 rolls[3] the velocity argmax, first maximum on ties); no other roll row is touched.
 * vel_logits_dev (optional): fp32 [n_windows * F * 88, 128] in (window, frame, note) order, every frame. */
int etude_k_heads(etude_handle_t* h, const void* x_bf16_dev, const void* w_bf16_dev, const float* bias_dev, int n_windows, int time_major,
                  const int64_t* out_row_host, int keep0, int keepn, void* const rolls_dev[4], float* vel_logits_dev, void* stream);

/* Time-axis transpose of the decoder (reference amt_apc.py:203-205) on a handle's window length F:
 * out[(w * 88 + n) * F + f, :] = bf16(16 * in[(w * F + f) * 88 + n, :] + pos_embedding_time[f, :]), bf16 [n_windows * F * 88, 256]. */
int etude_k_transpose_time(etude_handle_t* h, const void* in_bf16_dev, int n_windows, void* out_bf16_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif
