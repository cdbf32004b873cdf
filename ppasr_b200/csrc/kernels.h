// Launchers of the non-GEMM hot-path kernels (defined in kernels.cu / attention.cu). All take raw
// device pointers and a stream; none allocate.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ppasr {

cudaError_t launch_layernorm(float* x, __nv_bfloat16* y, const float* g1, const float* b1, const float* g2,
                             const float* b2, const int* lens, int T, int M, int D, float eps, cudaStream_t st);

cudaError_t launch_conv1_subsample(const float* feats, const float* mean, const float* istd, const float* w,
                                   const float* bias, __nv_bfloat16* out, int B, int T, int F, int C, int T1, int F1,
                                   int Th, int FH, cudaStream_t st);

// the same on the tensor cores (conv1_tc.cu): tmap_phase = 3-D map of the phase images [4][B*Th*FH][256], box 64 x 128 x 1
cudaError_t launch_conv1_tc(const CUtensorMap& tmap_phase, const float* feats, const float* mean, const float* istd,
                            const float* w, const float* bias, int B, int T, int F, int T1, int F1, int Th, int FH,
                            int num_sms, cudaStream_t st);

// conv1 (as above) fused into the conv2 GEMM's A-operand producer: feats -> c2 [B*Tout*Fout, 256] (conv1_tc.cu)
cudaError_t launch_conv_front_tc(const CUtensorMap& tmap_w2, const float* feats, const float* mean, const float* istd,
                                 const float* w1, const float* b1, const float* b2, __nv_bfloat16* out, int B, int T, int F,
                                 int T1, int F1, int Th, int FH, int Tout, int Fout, int num_sms, cudaStream_t st);

// zero_lens (nullable): output rows t >= zero_lens[b] are written as 0 (pad frames of the conv module output)
cudaError_t launch_dwconv_norm_swish(const __nv_bfloat16* g, const float* w, const float* bias, const float* pad_left,
                                     const float* gamma, const float* beta, int use_layer_norm, __nv_bfloat16* out,
                                     int B, int Tin, int Tout, int C, int K, int lpad, float eps, const int* zero_lens,
                                     cudaStream_t st);

cudaError_t launch_glu_pad(const float* bias_il, float* pad, int C, cudaStream_t st);

cudaError_t launch_softmax_rows(const float* logits, int ldl, float* probs, int M, int V, cudaStream_t st);

cudaError_t launch_argmax_rows(const float* probs, int V, int rows, int* idx, float* maxp, cudaStream_t st);

cudaError_t launch_ctc_stats_finalize(const float* pmax, const int* parg, const float* psum, int parts, int rows,
                                      int* idx, float* maxp, cudaStream_t st);

// Streaming conv-module cache (reference: conformer/convolution.py:108-117): ycat[b] = [cache[b] ; y[b]],
// then cache[b] <- last `lorder` rows of ycat[b]. cache: bf16 [B, lorder, C]; y: [B, T, C]; ycat: [B, lorder+T, C].
cudaError_t launch_conv_cache_concat(__nv_bfloat16* cache, const __nv_bfloat16* y, __nv_bfloat16* ycat, int B, int T,
                                     int lorder, int C, cudaStream_t st, const int* slots = nullptr);
// fp32 export of the device-resident caches in the reference's layouts.
cudaError_t launch_export_att_cache(const __nv_bfloat16* kk, const __nv_bfloat16* vt, float* out, int H, int Tcap,
                                    int Tcapp, int k0, int t, cudaStream_t st);
cudaError_t launch_export_cnn_cache(const __nv_bfloat16* cache, float* out, int lorder, int C, cudaStream_t st);

cudaError_t launch_ctc_collapse(const int* idx, const float* maxp, int B, int T, const int* frame_lens, int blank,
                                int* ids_out, int ld_out, int* out_len, float* score, float* score_sum,
                                int* score_cnt, cudaStream_t st);

// Fused feed-forward block (fused_ffn.cu): x += W2s swish(W1 y + b1) + b2s with trailing LayerNorm(s); optional
// chained pre-GEMM (tm_wp != null): x += mask (Wp z + bp), y = LN(x; gp, bpn) first (tm_a is then the z tile map).
// FF must be a multiple of 128 and at least 256 (cudaErrorInvalidValue otherwise).
cudaError_t launch_fused_ffn(const CUtensorMap& tm_a, const CUtensorMap* tm_wp, const CUtensorMap& tm_w1,
                             const CUtensorMap& tm_w2, int M, int FF, float* x, __nv_bfloat16* y, const float* b1,
                             const float* b2s, const float* g1, const float* bn1, const float* g2, const float* bn2,
                             float eps, const float* bp, const float* gp, const float* bpn, const int* lens, int T,
                             cudaStream_t st, int y_affine = 0, const int* ylens = nullptr, const float* pre_ys = nullptr,
                             const float* pre_yb = nullptr);

// fused_ffn variant (process-wide; env PPASR_B200_FFN_SPLIT=1/2 or ppasr_b200_set_option(ctx, "ffn_split", v)):
//   1 (default) = 2-CTA cluster per row tile, hidden dimension split over the pair, distributed-shared-memory reduction
//                 (2 x ceil(M/128) CTAs per launch: shortest single-launch latency); FF / 128 must be even and >= 4,
//                 otherwise the launch falls back to mode 2;
//   2 = the same two-team pipeline on one CTA per row tile (least SM time per launch; the throughput pipeline uses it).
// set_ffn_split_mode returns false and keeps the current mode for any other value.
int ffn_split_mode();
bool set_ffn_split_mode(int mode);

// Fused attention out-projection + residual + norm_conv + pointwise_conv1 + GLU (fused_attn_out.cu)
cudaError_t launch_fused_attn_out(const CUtensorMap& tm_att, const CUtensorMap& tm_wo, const CUtensorMap& tm_wpw1, int M,
                                  float* x, __nv_bfloat16* g, const float* bo, const float* ln_g, const float* ln_b,
                                  const float* bpw1, const int* lens, int T, float eps, cudaStream_t st);

// Squeezeformer time reduction, depthwise part (squeezeformer/time_reduction.py:61-84 conv1d k5 s2 pad3, :183-206 stream
// k1 s2): out[b, tr, c] = bias[c] + sum_k w[c, k] * xm[b, 2 tr + k - pad, c] with xm = x zeroed at t >= lens[b] -> bf16
cudaError_t launch_time_reduce_dw(const float* x, const float* w, const float* bias, const int* lens, __nv_bfloat16* out,
                                  int B, int T, int Tr, int C, int K, int pad, cudaStream_t st);
// lens_out[b] = (lens_in[b] + 1) / 2
cudaError_t launch_halve_lens(const int* lens_in, int* lens_out, int B, cudaStream_t st);

// DeepSpeech2 (ds2.cu): fused CMVN + 2 x (Conv2d k3 s2 + ReLU) with 32 channels; recurrent half of one LSTM / GRU layer
// (persistent weight-stationary cooperative kernel, both directions concurrently); LayerNorm over wide rows
cudaError_t launch_ds2_conv(const float* feats, const float* mean, const float* istd, const float* w1, const float* b1,
                            const float* w2t, const float* b2, __nv_bfloat16* out, int B, int T, int F, int Tp, int Kpad,
                            cudaStream_t st);
cudaError_t launch_rnn_layer(const float* xg, const __nv_bfloat16* whh, const float* bhh, const int* lens, const float* h_init,
                             const float* c_init, float* h_final, float* c_final, float* out, float* hbuf, unsigned* bar,
                             int B, int T, int H, int nd, int gru, int num_sms, cudaStream_t st);
cudaError_t launch_row_layernorm(const float* x, const float* g, const float* b, __nv_bfloat16* y, int M, int N, float eps,
                                 cudaStream_t st);

// CTC prefix beam search (beam.cu)
struct BeamStateHeader {
  int nb;       // entries in the beam
  int next_id;  // next free prefix id (0 = root)
  int frames;   // frames consumed so far
  int pad;
};
struct BeamEntry {
  unsigned long long hash;  // identity of the prefix string
  int id, parent_id, last, len;
  float b_prev, nb_prev, score;
  int prev1, prev2;  // the tokens before `last` (-1 = none): n-gram context of the external scorer
  int prev3;
};
// External scorer = character-based back-off n-gram LM as an open-addressing hash table (ppasr_b200/decoders/ngram_lm.py):
// token 1 = <s>, v + 2 = vocabulary id v; key = (lo, hi): lo = the four most recent tokens packed 16 bits each (most recent in
// the low bits), hi = the oldest token of a 5-gram (0 otherwise; array may be null for order <= 4); value = (ln p, ln bo)
struct BeamLm {
  const unsigned long long* keys;  // null = no scorer
  const unsigned* keys_hi;         // null = every key has hi = 0 (order <= 4)
  const float2* vals;
  const int* in_lm;                // [V] 1 if the token has a unigram
  unsigned mask;                   // capacity - 1
  int order;                       // <= 5
  float alpha, beta;
};
size_t beam_state_stride(int node_cap);
cudaError_t launch_ctc_prune(const float* probs, int V, int rows, float cutoff_prob, int top_n, int* cnt, int* cid,
                             float* clp, cudaStream_t st);
cudaError_t launch_beam_reset(void* states, int B, int node_cap, cudaStream_t st);
cudaError_t launch_beam_advance(const int* cnt, const int* cid, const float* clp, int B, int T, const int* frame_lens,
                                int beam, int topn, int blank, int max_frames, void* states, int node_cap, cudaStream_t st,
                                const float* probs = nullptr, int V = 0, const BeamLm* lm = nullptr);
// writes the first `nbest` beam entries (best first): out_ids [B, nbest, lmax], out_lens / out_scores [B, nbest]
cudaError_t launch_beam_result(const void* states, int B, int node_cap, int nbest, int* out_ids, int lmax, int* out_lens,
                               float* out_scores, cudaStream_t st);
constexpr int BEAM_MAX_TOPN = 64;
constexpr int BEAM_MAX_BEAM = 512;

// Relative-position attention (attention.cu). Tensor maps are built by the caller.
struct AttnParams {
  int B, H;
  int T1;        // query frames per utterance
  int T2;        // key frames per utterance (cache + new)
  int q_rows_per_bh;   // rows of q2 per (b,h)  (= T1)
  int k_rows_per_bh;   // rows of kk per (b,h)
  int k_row0;    // first key row inside each (b,h) block of kk / first key column of vt (cache start)
  int pos_row0;  // first row of the positional table used for key 0
  int pos_col0;  // first column (layer * D) of this layer's slice in the positional table
  int D;         // H * 64
  const int* klens;  // per-utterance valid key count (nullable = all T2 valid)
  // ragged streaming sessions: per-utterance cache slot, first key row and first positional row (nullable = scalars above)
  const int* slots;
  const int* k_row0s;
  const int* pos_row0s;
  __nv_bfloat16* out;  // [B*T1, D]
};
cudaError_t launch_rel_attention(const CUtensorMap& tm_q, const CUtensorMap& tm_k, const CUtensorMap& tm_p,
                                 const CUtensorMap& tm_vt, const AttnParams& p, cudaStream_t st);

// QKV projection + relative-position attention in one kernel (attention.cu, offline blocks): one CTA per (head, utterance)
// projects y [B*T, D] with the head's rows of the packed wqkv and attends over the utterance's T keys. tm_y: the y map of the
// QKV GEMM (box 128 rows); tm_w: wqkv [3D, D] with a 64-row box; tm_p: the positional table (box 128 rows).
// Only D = 256, H = 4 and 1 <= T <= 256 (cudaErrorInvalidValue otherwise). Bit-identical to the QKV GEMM + rel_attention.
struct QkvAttnParams {
  int B, H, T, D;
  int pos_row0;  // positional row of key 0
  int pos_col0;  // first column (layer * D) of this layer's slice in the positional table
  const float* bqkv;   // [3D]
  const float* pos_u;  // [D] pos_bias_u
  const float* pos_v;  // [D] pos_bias_v
  const int* klens;    // per-utterance valid key count (nullable = all T valid)
  __nv_bfloat16* out;  // [B*T, D]
};
cudaError_t launch_qkv_rel_attention(const CUtensorMap& tm_y, const CUtensorMap& tm_w, const CUtensorMap& tm_p,
                                     const QkvAttnParams& p, cudaStream_t st);


// Grouped rel-pos attention of the Efficient Conformer (grouped_attention.cu)
struct GroupedAttnParams {
  int B, H;
  int T;    // query frames per utterance
  int Tg;   // query groups per utterance = ceil(T / 3); also the key groups when Tgk == 0 (offline: queries == keys)
  const int* klens;     // per-utterance valid KEY frame count (nullable)
  __nv_bfloat16* out;   // [B*T, 256]
  // chunk streaming (forward_chunk, attention.py:128-193 with a cache): the keys are the append-only grouped cache
  int Tgk = 0;          // key groups to attend (0: = Tg)
  int k_pitch = 0;      // rows of the K operand per (b, h) (0: = Tg); the cache's group capacity when streaming
};
cudaError_t launch_grouped_attention(const CUtensorMap& tm_q, const CUtensorMap& tm_k, const CUtensorMap& tm_p,
                                     const CUtensorMap& tm_vt, const GroupedAttnParams& p, cudaStream_t st);
cudaError_t launch_grouped_pos(const __nv_bfloat16* tab, int ldtab, int col0, int T, int Tpad, __nv_bfloat16* out,
                               cudaStream_t st);
cudaError_t launch_dwconv_stride(const __nv_bfloat16* g, const float* w, const float* bias, const float* pad_left,
                                 const float* ng, const float* nb, int layer_norm, __nv_bfloat16* z, int B, int T, int Tout,
                                 int C, int K, int lpad, int stride, float eps, const int* zero_lens, cudaStream_t st);
cudaError_t launch_avgpool2(const float* x, float* out, int B, int T, int Tout, int C, cudaStream_t st);

}  // namespace ppasr
