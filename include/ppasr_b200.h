/*
 * ppasr_b200 -- C-ABI of the B200-native PPASR inference hot path
 * (fbank features -> Conformer encoder -> CTC projection -> greedy / beam-search decode).
 *
 * Plain C: opaque handle, raw pointers and sizes, int status codes (0 = ok; message via
 * ppasr_b200_last_error()). No torch / C++ types cross this boundary. Each entry point cites the
 * reference interface (yeyupiaoling/PPASR @ c8bb3b96, paths under ppasr/) that it replaces; the
 * Python binding a PPASR maintainer would add is ppasr_b200/_lib.py (ctypes), see INTEGRATION.md.
 *
 * Threading: a context is not re-entrant (like the reference's InferencePredictor, which owns mutable
 * stream caches: infer_utils/inference_predictor.py:35-39); use one context per CUDA stream.
 * All `stream` arguments are a cudaStream_t passed as void* (NULL = default stream).
 */
#ifndef PPASR_B200_H_
#define PPASR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ppasr_b200_ctx ppasr_b200_ctx;

/* Model hyper-parameters = the inference-relevant keys of configs/conformer.yml / configs/squeezeformer.yml
 * (encoder_conf, streaming, preprocess_conf.n_mels) plus the vocabulary size. */
typedef struct ppasr_b200_config {
  int32_t model_type;      /* 0 = conformer, 1 = squeezeformer, 2 = deepspeech2, 3 = efficient_conformer */
  int32_t feat_dim;        /* preprocess_conf.n_mels, 80 */
  int32_t d_model;         /* encoder_conf.output_size (squeezeformer: encoder_dim), 256; deepspeech2: rnn_size (<= 1024) */
  int32_t n_heads;         /* encoder_conf.attention_heads, 4 (d_model / n_heads must be 64) */
  int32_t ffn_dim;         /* encoder_conf.linear_units, 2048 (squeezeformer: encoder_dim * feed_forward_expansion_factor) */
  int32_t n_layers;        /* encoder_conf.num_blocks, 12; deepspeech2: num_rnn_layers, 5 */
  int32_t conv_kernel;     /* encoder_conf.cnn_module_kernel, 15 (7, 15 or 31) */
  int32_t causal;          /* `streaming: True` => causal depthwise conv (conformer/model.py:35-39); deepspeech2: forward-only
                            * RNN instead of bidirectional (deepspeech2/model.py:40) */
  int32_t conv_norm;       /* 0 = layer_norm (shipped default, conformer/encoder.py:51), 1 = batch_norm */
  int32_t vocab_size;      /* CTC output size V */
  int32_t max_len;         /* positional table length, 5000 (conformer/embedding.py:30) */
  /* squeezeformer only (squeezeformer/encoder.py:33-34, model.py:35-41); ignored for model_type 0 */
  int32_t reduce_idx;          /* block before which the time-reduction layer runs (5), -1 = none */
  int32_t recover_idx;         /* block before which the sequence is recovered to full length (11), -1 = none */
  int32_t time_reduce_kernel;  /* 1 = TimeReductionLayerStream (streaming), 5 = TimeReductionLayer1D */
  int32_t use_gru;             /* deepspeech2 only: encoder_conf.use_gru (GRU instead of LSTM, deepspeech2/encoder.py:41-53) */
  /* efficient_conformer only (efficient_conformer/encoder.py:49-54; the constructor defaults 3 / 0..3 / 3 / True apply to
   * the shipped config because its `efficient_conf` block is swallowed by **kwargs) */
  int32_t stride_layer_idx;    /* block whose depthwise conv has stride 2 (3), -1 = none */
  int32_t group_layer_mask;    /* bit l set: block l uses GroupedRelPositionMultiHeadedAttention (0b1111) */
  int32_t group_size;          /* 3 */
  int32_t stride_kernel;       /* 1: depthwise kernel 15 -> 7 after the stride block */
  int32_t reserved[1];
} ppasr_b200_config;

const char* ppasr_b200_last_error(void);
int ppasr_b200_abi_version(void);
/* Number of CUDA kernels this library has launched so far in this process (bench.py "gpu_launches"). */
int64_t ppasr_b200_launch_count(void);

/* Process-wide: launch kernels with programmatic dependent launch (default 1; env PPASR_B200_PDL=0). PDL shortens the
 * single-batch critical path (-7 %); with several batches in flight the early-started CTAs only hold SMs, so the
 * throughput pipeline switches it off. */
int ppasr_b200_set_pdl(int32_t enable);

/* Process-wide: fused feed-forward kernel variant (env PPASR_B200_FFN_SPLIT). 1 (default) = each 128-row tile is
 * computed by a 2-CTA thread-block cluster, the 2048-wide hidden dimension split over the pair and the two partial
 * outputs reduced through distributed shared memory (2 x ceil(M/128) CTAs per launch: lowest latency of one launch;
 * a hidden dimension of fewer than 4 or an odd number of 128-wide chunks runs as 2);
 * 2 = the same two-team Swish pipeline on one CTA per tile (least SM time: used when several batches are in flight).
 * Any other mode returns PPASR_ERR_INVALID and keeps the current one. Replaces nothing in the reference (a tuning
 * switch of positionwise.py:30-39's kernel); results agree to fp32 summation order. */
int ppasr_b200_set_ffn_split(int32_t mode);
int ppasr_b200_get_ffn_split(void);

/* ---- life cycle ------------------------------------------------------------------------------
 * replaces: InferencePredictor.__init__ loading model.pdmodel/.pdiparams
 *           (infer_utils/inference_predictor.py:12-45). */
int ppasr_b200_create(const ppasr_b200_config* cfg, ppasr_b200_ctx** out);
int ppasr_b200_destroy(ppasr_b200_ctx* ctx);
/* Hands one parameter over by its reference (Paddle) name and layout, fp32, host memory; e.g.
 * "encoder.encoders.0.self_attn.linear_q.weight" with shape [256,256] = [in,out] (SURVEY.md App. A).
 * The data is copied. */
int ppasr_b200_load_tensor(ppasr_b200_ctx* ctx, const char* name, const float* data, int32_t ndim,
                           const int64_t* shape);
/* Packs (transposes to K-major bf16, interleaves GLU rows, folds BatchNorm), uploads, and
 * precomputes the weight-only linear_pos(pos_emb) table. Fails listing any missing parameter. */
int ppasr_b200_finalize(ppasr_b200_ctx* ctx);

/* ---- offline encoder -------------------------------------------------------------------------
 * replaces: Model.get_encoder_out up to (not including) the CTC soft-max
 *           (model_utils/conformer/model.py:148-162 -> conformer/encoder.py:164-206).
 * feats: fp32 [B, T, feat_dim] row-major, zero padded; on the device if feats_on_device != 0 else in
 * host memory (copied inside, asynchronously if pinned). lens_host: int64 [B] valid frame counts
 * (NULL = all T). Leaves the encoder output in the context for the ctc_* calls below. */
int ppasr_b200_encode(ppasr_b200_ctx* ctx, const float* feats, int32_t feats_on_device, const int64_t* lens_host,
                      int32_t B, int32_t T, void* stream);
/* T' = ((T-1)/2 - 1)/2 : output frames for T input frames (conformer/subsampling.py:96-115); efficient_conformer with a
 * stride block: ceil(T'/2) (efficient_conformer/encoder.py:255-260). */
int ppasr_b200_out_frames(const ppasr_b200_ctx* ctx, int32_t T);

/* replaces: CTCLoss.softmax (model_utils/loss/ctc.py:62-70) + copy_to_cpu
 *           (infer_utils/inference_predictor.py:143-145).
 * probs: fp32 [B, T', V] dense, device or host. */
int ppasr_b200_ctc_probs(ppasr_b200_ctx* ctx, float* probs, int32_t probs_on_device, void* stream);
/* fp32 logits [B, T', V] (before the soft-max); for parity tests (CTCLoss.ctc_lo, loss/ctc.py:27). */
int ppasr_b200_ctc_logits(ppasr_b200_ctx* ctx, float* logits, int32_t on_device, void* stream);

/* Fused CTC head + greedy decode: never materialises [B,T',V].
 * replaces: CTCLoss.softmax + greedy_decoder / greedy_decoder_batch
 *           (loss/ctc.py:62-70, decoders/ctc_greedy_decoder.py:6-49).
 * ids: int32 [B, T'] (collapsed, blank-free token ids; first out_lens[b] entries valid),
 * out_lens: int32 [B], scores: fp32 [B] = mean max-probability over non-blank frames (x100 on the
 * host gives the reference score). trim_to_lens != 0 decodes only the valid frames of each utterance;
 * 0 reproduces the reference's evaluate(), which decodes padded frames too (trainer.py:347).
 * frame_ids / frame_probs (nullable, device-or-host like the others): per-frame arg-max id and its
 * probability [B, T']. */
int ppasr_b200_ctc_greedy(ppasr_b200_ctx* ctx, int32_t* ids, int32_t* out_lens, float* scores, int32_t* frame_ids,
                          float* frame_probs, int32_t outputs_on_device, int32_t trim_to_lens, int32_t blank_id,
                          void* stream);

/* ---- chunk streaming ---------------------------------------------------------------------------
 * replaces: Model.get_encoder_out_chunk / ConformerEncoder.forward_chunk
 *           (model_utils/conformer/model.py:164-184, conformer/encoder.py:208-283) and the stream state of
 *           InferencePredictor (infer_utils/inference_predictor.py:35-39,184-220).
 * The attention K/V cache and the conv-module cache stay on the device inside the context (the reference
 * round-trips both through host NumPy every chunk). B lock-step streams are supported (reference: B=1).
 * stream_reset == InferencePredictor.reset_stream. encode_chunk consumes feats fp32 [B, t, feat_dim]
 * (t = 67 for a full window, predict.py:277-300), appends ((t-1)/2-1)/2 output frames, applies
 * required_cache_size exactly like encoder.py:255-260 (<0 keep all, 0 drop, >0 keep last n) and leaves the
 * chunk's encoder output for ppasr_b200_ctc_probs / ctc_greedy. */
int ppasr_b200_stream_reset(ppasr_b200_ctx* ctx, int32_t B);
int ppasr_b200_encode_chunk(ppasr_b200_ctx* ctx, const float* feats, int32_t feats_on_device, int32_t B, int32_t t,
                            int32_t required_cache_size, void* stream);
/* ---- ragged streaming sessions (conformer): many independent streams, each with its own position and caches, stepped
 * together in one batch -- the engine side of a continuous-batching scheduler for predict_stream traffic (the reference
 * serves one stream per process: predict.py:232-337, infer_server.py:103-156).
 * sessions_init allocates `max_sessions` cache slots; sessions_reset(slot) starts a new stream in a slot; sessions_step
 * runs one chunk [n, t, feat_dim] for the n distinct slots listed in `slots` (host int32 [n]); afterwards the ctc_* calls
 * return the n chunk results in that order. required_cache_size as in encode_chunk. */
int ppasr_b200_sessions_init(ppasr_b200_ctx* ctx, int32_t max_sessions);
int ppasr_b200_sessions_reset(ppasr_b200_ctx* ctx, int32_t slot);
int ppasr_b200_sessions_step(ppasr_b200_ctx* ctx, const float* feats, int32_t feats_on_device, const int32_t* slots, int32_t n,
                             int32_t t, int32_t required_cache_size, void* stream);

/* DeepSpeech2 streaming states after the last encode_chunk: h, c fp32 [num_rnn_layers * num_directions, B, rnn_size]
 * (either may be NULL). replaces: self.output_state_h / self.output_state_c copy_to_cpu
 * (infer_utils/inference_predictor.py:176-180). */
int ppasr_b200_ds2_states(ppasr_b200_ctx* ctx, float* h, float* c, int32_t on_device, void* stream);

/* offset = encoder frames produced so far (== self.offset of the reference), cache_t = cached keys. */
int ppasr_b200_stream_info(ppasr_b200_ctx* ctx, int32_t* offset, int32_t* cache_t);
/* fp32 copies of stream 0's caches in the reference layouts: att_cache [L, H, cache_t, 128] (k | v),
 * cnn_cache [L, 1, d_model, conv_kernel-1]; either pointer may be NULL. */
int ppasr_b200_stream_export(ppasr_b200_ctx* ctx, float* att_cache, float* cnn_cache, int32_t on_device, void* stream);

/* ---- stand-alone decoders on a probability tensor (device pointers) --------------------------
 * replaces: greedy_decoder / greedy_decoder_batch (decoders/ctc_greedy_decoder.py:6-49).
 * probs: fp32 [B, T, V] dense. frame_lens (nullable): int32 [B]. tmp_idx: int32 [B*T], tmp_maxp: fp32 [B*T]
 * scratch that afterwards holds the per-frame arg-max ids / probabilities. */
int ppasr_b200_greedy_decode(const float* probs, int32_t B, int32_t T, int32_t V, const int32_t* frame_lens,
                             int32_t blank_id, int32_t* ids, int32_t ld_ids, int32_t* out_lens, float* scores,
                             int32_t* tmp_idx, float* tmp_maxp, void* stream);

/* ---- CTC prefix beam search without external scorer (device pointers) ---------------------------
 * replaces: ctc_beam_search_decoding / ctc_beam_search_decoding_batch / CtcBeamSearchDecoderBatch.next+decode
 *           (decoders/swig_wrapper.py:35-121 -> paddlespeech_ctcdecoders, ext_scoring_func=None).
 * `states` (ppasr_b200_beam_state_bytes) holds the beam and the prefix table of B utterances across calls,
 * so advance() can be fed chunk by chunk (decode_chunk) or once (offline). probs: fp32 [B,T,V] dense
 * probabilities (not logs), like the reference. beam <= 512 (configs/conformer.yml:84 ships 300), cutoff_top_n is capped
 * at 64 (ships 40), V < 65535. advance() refuses to run past the `max_frames` the state was sized for: the state is left
 * untouched, flagged, and result() then reports out_lens = -2 for every entry.
 * result(): out_ids int32 [B, beam, lmax], out_lens int32 [B, beam] (-1 = no such entry), out_scores fp32
 * [B, beam] = log P(prefix) sorted best first (the reference returns -score to Python); result_nbest() writes only the
 * first nbest <= beam entries ([B, nbest, lmax], [B, nbest]). */
int64_t ppasr_b200_beam_state_bytes(int32_t B, int32_t max_frames, int32_t beam);
int64_t ppasr_b200_beam_workspace_bytes(int32_t B, int32_t T);
int ppasr_b200_beam_reset(void* states, int32_t B, int32_t max_frames, int32_t beam, void* stream);
int ppasr_b200_beam_advance(const float* probs, int32_t B, int32_t T, int32_t V, const int32_t* frame_lens,
                            int32_t beam, float cutoff_prob, int32_t cutoff_top_n, int32_t blank_id, void* states,
                            int32_t max_frames, void* workspace, void* stream);
/* Same with an external scorer (replaces Scorer + ext_scoring_func of swig_wrapper.py:4-19,35-64): a character-based
 * back-off n-gram LM as an open-addressing hash table on the device (built by ppasr_b200/decoders/ngram_lm.py from an ARPA
 * file): lm_keys uint64 [lm_capacity] (0 = empty; the four most recent token ids packed 16 bits each, <s> = 1, vocabulary id
 * v = v + 2, most recent token in the low bits), lm_keys_hi uint32 [lm_capacity] (the oldest token of a 5-gram, 0 for shorter
 * n-grams; may be NULL when lm_order <= 4), lm_vals float [lm_capacity][2] = (ln p, ln backoff), lm_in_vocab int32 [V]; home
 * slot = murmur3 finaliser of lo ^ hi * 0x9E3779B97F4A7C15, linear probing. lm_order <= 5 (the reference trains `-o 5`).
 * Every emitted character adds alpha * ln P(c | history) + beta; the published min_cutoff pruning is applied. */
int ppasr_b200_beam_advance_lm(const float* probs, int32_t B, int32_t T, int32_t V, const int32_t* frame_lens, int32_t beam,
                               float cutoff_prob, int32_t cutoff_top_n, int32_t blank_id, void* states, int32_t max_frames,
                               void* workspace, const uint64_t* lm_keys, const uint32_t* lm_keys_hi, const float* lm_vals,
                               const int32_t* lm_in_vocab, int64_t lm_capacity, int32_t lm_order, float alpha, float beta,
                               void* stream);
int ppasr_b200_beam_result(const void* states, int32_t B, int32_t max_frames, int32_t beam, int32_t* out_ids,
                           int32_t lmax, int32_t* out_lens, float* out_scores, void* stream);
int ppasr_b200_beam_result_nbest(const void* states, int32_t B, int32_t max_frames, int32_t beam, int32_t nbest,
                                 int32_t* out_ids, int32_t lmax, int32_t* out_lens, float* out_scores, void* stream);
/* The pruning scan of the posterior alone (decoder_utils.cpp get_pruned_log_probs), for the HBM roofline. */
int ppasr_b200_op_ctc_prune(const float* probs, int32_t rows, int32_t V, float cutoff_prob, int32_t cutoff_top_n,
                            void* workspace, void* stream);

/* ---- op-level entry points (parity tests, per-kernel roofline) ------------------------------- */
/* out = epilogue(A[M,K] bf16 * W[N,K]^T bf16 + bias). epilogue: 0 = bf16 store with act (0 none,
 * 1 relu, 2 swish); 1 = fp32 x = (residual ? x : 0) + alpha*(acc+bias) with optional pad-row mask
 * (lens int32 [M/T]); 2 = GLU over interleaved column pairs -> bf16 [M, N/2]; 3 = fp32 logits. */
int ppasr_b200_op_linear(const void* a_bf16, int64_t lda, const void* w_bf16, int64_t w_rows, const float* bias,
                         void* out, int64_t ldo, int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t act,
                         float alpha, int32_t residual, const int32_t* lens, int32_t T, int32_t block_n, void* stream);
int ppasr_b200_op_layernorm(float* x, void* y_bf16, const float* g1, const float* b1, const float* g2,
                            const float* b2, const int32_t* lens, int32_t T, int32_t M, int32_t D, float eps,
                            void* stream);
int ppasr_b200_op_dwconv(const void* g_bf16, const float* w, const float* bias, const float* pad_left,
                         const float* gamma, const float* beta, int32_t use_layer_norm, void* out_bf16, int32_t B,
                         int32_t Tin, int32_t Tout, int32_t C, int32_t K, int32_t lpad, float eps, void* stream);
int ppasr_b200_op_softmax(const float* logits, int32_t ldl, float* probs, int32_t M, int32_t V, void* stream);
/* fused feed-forward block (plain mode of fused_ffn.cu): x += W2s swish(W1 y + b1) + b2s, then LayerNorm(s).
 * y [M,256] bf16, w1 [FF,256] bf16, w2s [256,FF] bf16 (already scaled by the macaron factor), x fp32 [M,256] in place,
 * y_out bf16 [M,256]; g2/bn2 NULL = single LayerNorm. */
int ppasr_b200_op_fused_ffn(const void* y_bf16, const void* w1_bf16, const void* w2s_bf16, float* x, void* y_out,
                            const float* b1, const float* b2s, const float* g1, const float* bn1, const float* g2,
                            const float* bn2, int32_t M, int32_t FF, float eps, void* stream);
/* rel-pos attention on packed q2 [B,H,T1,128], kk [B,H,T2,64], vt [B,H,64,T2p], pos [pos_rows, pos_ld]
 * (all bf16) -> out bf16 [B*T1, H*64]; klens nullable int32 [B]. */
int ppasr_b200_op_attention(const void* q2, const void* kk, const void* vt, int32_t T2p, const void* pos,
                            int32_t pos_rows, int32_t pos_ld, int32_t pos_row0, int32_t pos_col0, void* out,
                            int32_t B, int32_t H, int32_t T1, int32_t T2, const int32_t* klens, void* stream);
/* QKV projection + rel-pos attention of one offline block (D = 256, H = 4): y [B*T,256] bf16 (the LayerNorm output),
 * wqkv [768,256] bf16 (K-major rows: q, k, v; row = h*64 + d inside each), bqkv fp32 [768], pos_u / pos_v fp32 [256],
 * pos [pos_rows, pos_ld] bf16 with key 0 at row pos_row0 and the block's columns from pos_col0 -> out bf16 [B*T,256];
 * klens nullable int32 [B]. fused != 0 runs qkv_rel_attention_kernel (1 <= T <= 256, otherwise an error), fused = 0 the
 * QKV GEMM + rel_attention_kernel pair on scratch operands; the two give the same bits. */
int ppasr_b200_op_qkv_attention(const void* y, const void* wqkv, const float* bqkv, const float* pos_u, const float* pos_v,
                                const void* pos, int32_t pos_rows, int32_t pos_ld, int32_t pos_row0, int32_t pos_col0,
                                const int32_t* klens, int32_t B, int32_t T, void* out, int32_t fused, void* stream);
/* grouped rel-pos attention of the Efficient Conformer (group size 3, 4 heads x 192) on the operand layouts the grouped QKV
 * epilogue writes: q2g [B,H,ceil(T/3),384] = [q+u | q+v], kk [B,H,k_pitch,192], vt [B,H,192,vt_pitch] (vt_pitch % 8 == 0),
 * pos [Tgk,768] (all bf16) -> out bf16 [B*T,256]. Tgk key groups (<= k_pitch, vt_pitch; any count), klens nullable int32 [B]
 * valid key FRAMES per utterance. Offline: Tgk = k_pitch = ceil(T/3); streaming: k_pitch = the cache's group capacity. */
int ppasr_b200_op_grouped_attention(const void* q2g, const void* kk, int32_t k_pitch, const void* vt, int32_t vt_pitch,
                                    const void* pos, void* out, int32_t B, int32_t H, int32_t T, int32_t Tgk,
                                    const int32_t* klens, void* stream);

/* ---- front end (the step before the hot path; SURVEY 8f rank 1) ----------------------------------------
 * replaces: AudioFeaturizer.featurize for feature_method 'fbank' (data_utils/featurizer/audio_featurizer.py:37-69,120-138):
 * optional -20 dB RMS normalisation (data_utils/audio.py:287-304), int16 scaling (audio.py:549-574), Kaldi fbank with
 * 25 ms / 10 ms frames, dither 0, n_mels bins. audio: fp32 in [-1, 1], device memory, [B, stride] with N valid samples per
 * row (n_samples: optional device int32 [B] per-utterance counts <= N). out: device fp32 [B, Tmax, n_mels], frames beyond an
 * utterance's own count are zero. gain_ws: device float [B] scratch (needed when db_normalize != 0). */
int ppasr_b200_fbank_frames(int32_t n_samples);
int ppasr_b200_fbank(const float* audio, int32_t B, int64_t stride, int32_t N, const int32_t* n_samples, int32_t n_mels,
                     int32_t sample_rate, int32_t db_normalize, float target_db, float* gain_ws, float* out, int32_t Tmax,
                     void* stream);

/* Switches: "fused_conv" (default 2) selects the subsampling front end: 2 = conv1 (split-tf32 GEMM) as the A-operand producer of the conv2 GEMM in one kernel, 0 = conv1 kernel + conv2 GEMM
 * through the stride-phase images (bit-identical to 2 with conv1_tc = 1; the only front end for feat_dim > 96); "conv1_tc" (default 1) the first
 * subsampling conv on the tensor cores (split-tf32, conv1_tc.cu; 0 = the CUDA-core kernel); "ffn_split" (1 or 2) = ppasr_b200_set_ffn_split;
 * "host_sync" (default 1): ppasr_b200_ctc_greedy with host outputs synchronises the stream before
 * returning -- 0 leaves the copies in flight (pinned host buffers; the caller synchronises), used by the
 * double-buffered serving pipeline. */
int ppasr_b200_set_option(ppasr_b200_ctx* ctx, const char* name, int32_t value);

/* ---- CUDA graph of the steady-state step ------------------------------------------------------------------------------
 * replaces nothing in the reference (SURVEY 8d "timed region: CUDA-Graph steady state"). graph_begin puts `stream` (not the
 * default stream) into capture; everything enqueued on it through this library until graph_end -- typically ppasr_b200_encode
 * with device features and ppasr_b200_ctc_greedy with device outputs -- is recorded, with its programmatic-dependent-launch
 * edges, instead of run; graph_launch replays it as ONE launch (features are re-read from the pointer given at capture time,
 * the valid lengths from the context's pinned staging buffer). Run the step once with the same shapes before capturing; no
 * host synchronisation or host-output call inside the capture. graph_kernels = kernels per replay. */
int ppasr_b200_graph_begin(ppasr_b200_ctx* ctx, void* stream);
int ppasr_b200_graph_end(ppasr_b200_ctx* ctx, void* stream);
int ppasr_b200_graph_launch(ppasr_b200_ctx* ctx, void* stream);
int32_t ppasr_b200_graph_kernels(const ppasr_b200_ctx* ctx);

/* Per-kernel-class device timing of the model-level calls (cudaEvent pairs around every launch).
 * enable, run encode/ctc_* once, then read: counts[i] launches and total_ms[i] for class i in
 * [0, ppasr_b200_profile_num_classes()). Used by bench.py for the live roofline figure. enable = 1: every class (the
 * event records between back-to-back kernels of a few microseconds inflate them); enable = 2 + class id: event pairs around
 * the launches of that class only, the rest of the step runs undisturbed. */
int ppasr_b200_profile_enable(ppasr_b200_ctx* ctx, int32_t enable);
int ppasr_b200_profile_num_classes(void);
const char* ppasr_b200_profile_class_name(int32_t cls);
int ppasr_b200_profile_read(ppasr_b200_ctx* ctx, int32_t* counts, float* total_ms);

/* Debug/inspection: copies an internal activation (fp32 residual stream x [B*T', d_model]) to the
 * device buffer `dst`. Used by the layer-wise parity tests only. */
int ppasr_b200_debug_copy_x(ppasr_b200_ctx* ctx, float* dst_device, void* stream);
/* The first subsampling conv's output (subsampling.py:84-85: Conv2d(1, D, 3, 2) + ReLU) as the four stride-phase images
 * the second conv reads: bf16 [4][B*Th*FH][D], phase = 2*(t1 & 1) + (f1 & 1), row = (b*Th + t1/2)*FH + f1/2. dims
 * receives {B, Th, FH, D}; dst_device may be null to query the dims only. Used by the front-end parity tests. */
int ppasr_b200_debug_copy_phase(ppasr_b200_ctx* ctx, void* dst_device, int32_t* dims, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PPASR_B200_H_ */
