// Model-level runtime behind the C-ABI (include/ppasr_b200.h): parameter packing, workspace,
// the Conformer / Efficient Conformer encoder launch sequence and the CTC head / greedy decode.
//
// Reference call path being replaced (yeyupiaoling/PPASR @ c8bb3b96):
//   InferencePredictor.predict (ppasr/infer_utils/inference_predictor.py:103-145)
//   -> ConformerModel.get_encoder_out (ppasr/model_utils/conformer/model.py:148-162)
//   -> ConformerEncoder.forward (ppasr/model_utils/conformer/encoder.py:164-206)
//   -> CTCLoss.softmax (ppasr/model_utils/loss/ctc.py:62-70) -> greedy_decoder (ppasr/decoders/ctc_greedy_decoder.py)
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "common.h"
#include "gemm.cuh"
#include "kernels.h"
#include "ppasr_b200.h"
#include "tmap.h"

namespace ppasr {

GemmShape make_shape(int M, int N, int K, int block_n);

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

// simple bump allocator over one cudaMalloc'ed slab (weights) / growable slab (workspace)
struct DeviceSlab {
  uint8_t* base = nullptr;
  size_t cap = 0, used = 0;
  bool overflow = false;  // a take() did not fit: it returned nullptr and every later take() does too
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (base) cudaFree(base);
    base = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&base, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void rewind() { used = 0, overflow = false; }
  template <class T>
  T* take(size_t count) {
    const size_t off = (used + 255) & ~size_t(255);
    if (overflow || off + count * sizeof(T) > cap) {
      overflow = true;
      return nullptr;
    }
    used = off + count * sizeof(T);
    return reinterpret_cast<T*>(base + off);
  }
  void release() {
    if (base) cudaFree(base);
    base = nullptr;
    cap = used = 0;
  }
};

// attention and conv-module weights of a Conformer-family block (Conformer, Efficient Conformer, Squeezeformer)
struct BlockW {
  const __nv_bfloat16 *wqkv, *wo, *pw1, *pw2;  // K-major bf16
  const float *bqkv, *bo, *pos_u, *pos_v, *pw1_b, *pw2_b, *dw_w, *dw_b, *cn_g, *cn_b, *glu_pad;
};
struct BlockMaps {  // their tensor maps (B operands)
  CUtensorMap wqkv, wo, pw1, pw2;
  CUtensorMap wqkv_h;  // the same wqkv with a 64-row box: one head's q, k or v rows (qkv_rel_attention_kernel)
};

struct LayerW : BlockW {
  // layer norms (gamma, beta) fp32 [D]
  const float *ln_ffm_g, *ln_ffm_b, *ln_mha_g, *ln_mha_b, *ln_conv_g, *ln_conv_b, *ln_ff_g, *ln_ff_b, *ln_fin_g,
      *ln_fin_b;
  // feed-forward (macaron, final): K-major bf16, *_w2s / *_b2s = 0.5 * W2 / b2 (macaron scale folded)
  const __nv_bfloat16 *ffm_w1, *ff_w1, *ffm_w2s, *ff_w2s;
  const float *ffm_b1, *ff_b1, *ffm_b2s, *ff_b2s;
};

struct Plan {  // everything that depends on (B, T)
  int B = 0, T = 0, T1 = 0, Tp = 0, Th = 0, M = 0, Mr = 0, Tkp = 0;
  // activations
  float* feats = nullptr;
  int* vlen = nullptr;
  __nv_bfloat16 *phase = nullptr, *c2 = nullptr, *y = nullptr, *q2 = nullptr, *kk = nullptr, *vt = nullptr,
                *att = nullptr, *g = nullptr, *z = nullptr;
  // view of the encoder output the CTC head reads (== M / Tp / vlen unless the model changes the frame rate)
  int Mc = 0, Tc = 0;
  int* vc = nullptr;
  // Efficient Conformer grouped attention operands
  int Tg = 0, Tgp = 0;
  __nv_bfloat16 *q2g = nullptr, *kkg = nullptr, *vtg = nullptr, *pg = nullptr;
  CUtensorMap tm_qg, tm_kg, tm_vtg, tm_pg[4];
  float *x2 = nullptr;  // Squeezeformer / Efficient Conformer: half-rate residual stream [B*ceil(Tp/2), D]
  int* vlen2 = nullptr; // ... and its valid lengths
  float *x = nullptr, *logits = nullptr, *pmax = nullptr, *psum = nullptr, *maxp = nullptr, *score = nullptr,
        *probs = nullptr;
  int *parg = nullptr, *idx = nullptr, *ids = nullptr, *out_len = nullptr;
  // streaming conv module: [cache ; chunk] rows
  int Tcat = 0, Mcat = 0;
  __nv_bfloat16 *ycat = nullptr, *gcat = nullptr;
  // tensor maps (A operands)
  CUtensorMap tm_phase, tm_c2, tm_y, tm_att, tm_g, tm_z, tm_q, tm_k, tm_vt, tm_ycat;
};

}  // namespace ppasr

using namespace ppasr;

struct ppasr_b200_ctx {
  ppasr_b200_config cfg;
  std::map<std::string, HostTensor> host;
  bool finalized = false;
  int F1 = 0, F2 = 0, FH = 0, Kemb = 0, Vpad = 0, Vld = 0, ctc_parts = 0;
  DeviceSlab wslab, aslab;
  // global weights
  const float *cmvn_mean = nullptr, *cmvn_istd = nullptr, *conv1_w = nullptr, *conv1_b = nullptr, *conv2_b = nullptr,
              *emb_b = nullptr, *after_g = nullptr, *after_b = nullptr, *ctc_b = nullptr;
  const __nv_bfloat16 *conv2_w = nullptr, *emb_w = nullptr, *ctc_w = nullptr, *pos_tab = nullptr;
  std::vector<LayerW> layers;
  // weight tensor maps (B operands); tm_pos2: every second row of the positional table (pos_emb[:, ::2])
  CUtensorMap tm_conv2_w, tm_emb_w, tm_ctc_w, tm_pos, tm_pos2;
  struct LayerMaps : BlockMaps {
    CUtensorMap ffm_w1_128, ff_w1_128, ffm_w2s, ff_w2s;
  };
  std::vector<LayerMaps> lmaps;
  cudaError_t upload_err = cudaSuccess;  // first failed weight copy of finalize
  // ---- Squeezeformer (model_type 1; squeezeformer/encoder.py) ----
  struct SqLayerW : BlockW {
    const float *ln_g[4], *ln_b[4];    // layer_norm1..4
    const float *ada_s[4], *ada_b[4];  // adaptive scale/bias of: 0 self_attn, 1 ffn1, 2 conv_module, 3 ffn2
    const __nv_bfloat16 *w1[2], *w2[2];
    const float *b1[2], *b2[2];
  };
  struct SqLayerMaps : BlockMaps {
    CUtensorMap w1_128[2], w2[2];
  };
  struct Sqz {
    std::vector<SqLayerW> layers;
    std::vector<SqLayerMaps> maps;
    const float *preln_g = nullptr, *preln_b = nullptr, *tr_dw_w = nullptr, *tr_dw_b = nullptr, *tr_pw_b = nullptr,
                *rec_b = nullptr, *ones = nullptr, *zeros = nullptr;
    const __nv_bfloat16 *tr_pw = nullptr, *rec_w = nullptr;
    CUtensorMap tm_tr_pw, tm_rec_w;
    int reduce_idx = -1, recover_idx = -1, tr_k = 1;
  } sq;
  // ---- DeepSpeech2 (model_type 2; deepspeech2/encoder.py) ----
  struct Ds2LayerW {
    const __nv_bfloat16 *wih = nullptr, *whh = nullptr;  // [nd*G*H, Kin_pad], [nd][G*H][H]
    const float *bih = nullptr, *bhh = nullptr, *ln_g = nullptr, *ln_b = nullptr;
    CUtensorMap tm_wih;
  };
  struct Ds2 {
    std::vector<Ds2LayerW> layers;
    const float* conv2_wt = nullptr;  // [cin*9 + k][cout]
    int nd = 2, gru = 0, kin0 = 0, kin0_pad = 0;
    float *xg = nullptr, *rnn_out = nullptr, *hbuf = nullptr;
    unsigned* bar = nullptr;
    CUtensorMap tm_y0;
    // streaming states [L*nd, B, H] (inference_predictor.py:157-164), device resident
    float *h_state = nullptr, *c_state = nullptr;
    int state_B = 0;
  } ds;
  int ctc_k = 0;  // input features of the CTC projection
  // ---- Efficient Conformer (model_type 3; efficient_conformer/encoder.py) ----
  int eff_stride_idx = -1;      // block with the strided depthwise conv (-1: none)
  unsigned eff_group_mask = 0;  // bit l: block l uses grouped attention
  std::vector<int> layer_k;     // depthwise kernel size per block
  Plan plan;
  int sms = 148;
  // ---- streaming state (reference: inference_predictor.py:35-39,215-220; device resident here) ----
  struct StreamState {
    int B = 0;          // lock-step streams
    int Tcap = 0;       // key capacity per (b,h)
    int kstart = 0;     // first cached key kept (required_cache_size trimming)
    int kend = 0;       // one past the last cached key
    int offset = 0;     // encoder output frames produced so far
    __nv_bfloat16* kk = nullptr;   // [L][B,H,Tcap,64]
    __nv_bfloat16* vt = nullptr;   // [L][B,H,64,Tcap]
    __nv_bfloat16* cnn = nullptr;  // [L][B,lorder,D]
    std::vector<CUtensorMap> tm_k, tm_vt;  // per layer, rebuilt every chunk (extent = kend)
    // Efficient Conformer streaming: the grouped blocks keep K [B,H,Gcap,192] / V^T [B,H,192,Gcap] in their layer slices;
    // groups at or past gdirty have been zero since the caches were last cleared (stream_reset zeroes [0, gdirty) only)
    int Gcap = 0;
    int gdirty = 0;
    // positional operands of the (<= 4) grouped blocks [4][Gcap][768], rebuilt per chunk, and the map of this chunk's
    // grouped queries
    __nv_bfloat16* pgc = nullptr;
    CUtensorMap tm_pgc[4], tm_qgc;
    // ragged sessions (ppasr_b200_sessions_*): every cache slot is an independent stream with its own positions
    bool ragged = false;                        // set for the duration of a sessions_step
    std::vector<int> s_kstart, s_kend, s_offset;  // per slot (host)
    int* d_step = nullptr;                      // device [5][B]: slots, kofs, k_row0, pos_row0, klen of the current step
    int step_T2 = 0;
  } ss;
  bool conv1_tc = true;   // conv1 on the tensor cores (conv1_tc.cu); 0 = the CUDA-core kernel (env PPASR_B200_CONV1_TC / option "conv1_tc")
  int fused_conv = 2;  // 2 (default): conv_front_tc (tensor-core conv1 producer inside the conv2 GEMM), 0: conv1 + conv2 GEMM; env PPASR_B200_FUSED_CONV
  bool host_sync = true;  // ctc_* with host outputs synchronise the stream before returning
  // valid-length staging (pinned: the H2D copy may be part of a captured CUDA graph and is re-read at every replay)
  int* h_vlen = nullptr;
  int h_vlen_cap = 0;
  int vlen_flip = 0;
  // CUDA graph of a steady-state step (ppasr_b200_graph_*): everything enqueued between begin and end, replayed as one launch
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  bool capturing = false;
  long long graph_kernels = 0, capture_count0 = 0;
  // optional per-kernel-class timing (cudaEvent pairs around every launch of the step)
  bool profiling = false;
  int prof_only = -1;  // >= 0: event pairs only around launches of this kernel class (undisturbed neighbours)
  struct ProfRec {
    int cls;
    cudaEvent_t e0, e1;
  };
  std::vector<ProfRec> prof;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_pool;
  size_t prof_used = 0;
};

namespace {

enum ProfClass : int {
  PC_CONV1 = 0, PC_CONV2, PC_EMBED, PC_LAYERNORM, PC_FFN1, PC_FFN2, PC_QKV, PC_ATTENTION, PC_OUTPROJ, PC_PW1_GLU,
  PC_DWCONV, PC_PW2, PC_CTC_STATS, PC_CTC_FINALIZE, PC_CTC_COLLAPSE, PC_CTC_LOGITS, PC_SOFTMAX, PC_FUSED_FFN, PC_FUSED_ATTN_OUT, PC_CONV_FRONT, PC_COUNT
};
const char* const kProfNames[PC_COUNT] = {"conv1_subsample", "conv2_gemm", "embed_gemm", "layernorm", "ffn1_gemm",
                                          "ffn2_gemm", "qkv_gemm", "attention", "outproj_gemm", "pw1_glu_gemm",
                                          "dwconv_norm_swish", "pw2_gemm", "ctc_stats_gemm", "ctc_finalize",
                                          "ctc_collapse", "ctc_logits_gemm", "softmax", "fused_ffn", "fused_attn_out", "conv_front"};

struct ProfScope {
  ppasr_b200_ctx* c;
  cudaStream_t st;
  cudaEvent_t e1 = nullptr;
  ProfScope(ppasr_b200_ctx* c_, int cls, cudaStream_t st_) : c(c_), st(st_) {
    if (!c->profiling || (c->prof_only >= 0 && c->prof_only != cls)) return;
    if (c->prof_used == c->prof_pool.size()) {
      cudaEvent_t a, b;
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      c->prof_pool.emplace_back(a, b);
    }
    auto& pr = c->prof_pool[c->prof_used++];
    c->prof.push_back({cls, pr.first, pr.second});
    e1 = pr.second;
    cudaEventRecord(pr.first, st);
  }
  ~ProfScope() {
    if (e1) cudaEventRecord(e1, st);
  }
};
#define PROF(cls) ProfScope _prof_scope(c, cls, st)

constexpr int BN_WIDE = 256, ST_WIDE = 4;    // N >= 512 outputs
constexpr int BN_NARROW = 128, ST_NARROW = 6;  // N = 256 outputs (fills 124 of 148 SMs at M = 7936)

const HostTensor* find(ppasr_b200_ctx* c, const std::string& name, std::string* missing) {
  auto it = c->host.find(name);
  if (it == c->host.end()) {
    if (missing) *missing += (missing->empty() ? "" : ", ") + name;
    return nullptr;
  }
  return &it->second;
}

std::vector<__nv_bfloat16> to_bf16(const std::vector<float>& v) {
  std::vector<__nv_bfloat16> o(v.size());
  for (size_t i = 0; i < v.size(); ++i) o[i] = __float2bfloat16_rn(v[i]);
  return o;
}

// Paddle Linear weight [in, out] -> K-major [rows_pad, in] (row = output feature)
std::vector<float> transpose_in_out(const HostTensor& w, int rows_pad = 0) {
  const int64_t in = w.shape[0], out = w.shape[1];
  const int64_t rows = rows_pad > out ? rows_pad : out;
  std::vector<float> o((size_t)rows * in, 0.f);
  for (int64_t i = 0; i < in; ++i)
    for (int64_t j = 0; j < out; ++j) o[(size_t)j * in + i] = w.data[(size_t)i * out + j];
  return o;
}

int finalize_squeezeformer(ppasr_b200_ctx* c);  // runtime_squeezeformer.inl
int finalize_ds2(ppasr_b200_ctx* c);            // runtime_ds2.inl

// ---- weight packing shared by the finalize of every model ------------------------------------------------------------
// An upload that does not fit the slab, or whose copy fails, returns nullptr (or an unwritten pointer) and is reported by
// check_weights(), which runs before anything launches on the slab and at the end of finalize.
template <class T>
const T* upload(ppasr_b200_ctx* c, const std::vector<T>& v) {
  T* d = c->wslab.take<T>(v.size());
  if (d && c->upload_err == cudaSuccess) c->upload_err = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  return d;
}

const float* vecf(ppasr_b200_ctx* c, const std::string& n) { return upload(c, c->host[n].data); }

int check_weights(ppasr_b200_ctx* c) {
  if (c->wslab.overflow) {
    set_last_error("internal error: weight slab too small");
    return PPASR_ERR_STATE;
  }
  PPASR_CUDA_CHECK(c->upload_err);
  return PPASR_OK;
}

int require_present(ppasr_b200_ctx* c, const std::vector<std::string>& names) {
  std::string missing;
  for (auto& n : names) find(c, n, &missing);
  if (!missing.empty()) {
    set_last_error("missing parameters: " + missing);
    return PPASR_ERR_STATE;
  }
  return PPASR_OK;
}

// parameters of block prefix p read by pack_attention / pack_conv_module
void block_names(const ppasr_b200_config& cfg, const std::string& p, bool pos_bias, std::vector<std::string>* names) {
  for (const char* s : {"linear_q", "linear_k", "linear_v", "linear_out"}) {
    names->push_back(p + "self_attn." + s + ".weight");
    names->push_back(p + "self_attn." + s + ".bias");
  }
  names->push_back(p + "self_attn.linear_pos.weight");
  if (pos_bias) names->push_back(p + "self_attn.linear_pos.bias");
  names->push_back(p + "self_attn.pos_bias_u");
  names->push_back(p + "self_attn.pos_bias_v");
  for (const char* s : {"pointwise_conv1", "depthwise_conv", "pointwise_conv2", "norm"}) {
    names->push_back(p + "conv_module." + s + ".weight");
    names->push_back(p + "conv_module." + s + ".bias");
  }
  if (cfg.conv_norm == 1) {
    names->push_back(p + "conv_module.norm._mean");
    names->push_back(p + "conv_module.norm._variance");
  }
}

// Weight slab size of the Conformer family: no packed weight is larger than its fp32 host tensor (bf16 halves it;
// transposes, the value/gate interleave and BatchNorm folding keep it), plus what finalize derives (sinusoid and
// positional tables, linear_pos biases, GLU pads, zero / one vectors, the padded CTC head) and 256 B alignment each.
size_t conformer_slab_bytes(const ppasr_b200_ctx* c) {
  const auto& cfg = c->cfg;
  const size_t D = cfg.d_model, L = cfg.n_layers, ML = cfg.max_len;
  size_t bytes = 0;
  for (auto& t : c->host) bytes += (size_t)t.second.numel() * 4;
  bytes += ML * (L + 1) * D * 2 + (3 * L * D + D + 4096 + (size_t)c->Vpad * (D + 1)) * 4;
  bytes += (c->host.size() + 8 * L + 64) * 256;
  return bytes;
}

// front end: CMVN, conv1 [D,1,3,3] (conv1_name), conv2 [D,D,3,3] (conv2_name) as K-major [D, (kh*3+kw)*D + i] and the
// embedding Linear [D*F2 (c*F2+f), D] (emb_name) as K-major [D, f*D + c]; its bias is stored times emb_b_scale
int pack_front(ppasr_b200_ctx* c, const std::string& conv1_name, const std::string& conv2_name, const std::string& emb_name,
               float emb_b_scale) {
  const int D = c->cfg.d_model;
  c->cmvn_mean = vecf(c, "encoder.global_cmvn.mean");
  c->cmvn_istd = vecf(c, "encoder.global_cmvn.istd");
  {
    const HostTensor& w = c->host[conv1_name + ".weight"];
    PPASR_REQUIRE(w.numel() == (int64_t)D * 9, conv1_name + ".weight shape");
    c->conv1_w = upload(c, w.data);
    c->conv1_b = vecf(c, conv1_name + ".bias");
  }
  {
    const HostTensor& w = c->host[conv2_name + ".weight"];
    PPASR_REQUIRE(w.numel() == (int64_t)D * D * 9, conv2_name + ".weight shape");
    std::vector<float> p((size_t)D * 9 * D);
    for (int o = 0; o < D; ++o)
      for (int i = 0; i < D; ++i)
        for (int t = 0; t < 9; ++t) p[(size_t)o * 9 * D + (size_t)t * D + i] = w.data[((size_t)o * D + i) * 9 + t];
    c->conv2_w = upload(c, to_bf16(p));
    c->conv2_b = vecf(c, conv2_name + ".bias");
  }
  {
    const HostTensor& w = c->host[emb_name + ".weight"];
    PPASR_REQUIRE(w.shape.size() == 2 && w.shape[0] == (int64_t)D * c->F2 && w.shape[1] == D, emb_name + ".weight shape");
    std::vector<float> p((size_t)D * c->Kemb);
    for (int ch = 0; ch < D; ++ch)
      for (int f = 0; f < c->F2; ++f)
        for (int o = 0; o < D; ++o) p[(size_t)o * c->Kemb + (size_t)f * D + ch] = w.data[((size_t)ch * c->F2 + f) * D + o];
    c->emb_w = upload(c, to_bf16(p));
    std::vector<float> b = c->host[emb_name + ".bias"].data;
    for (auto& v : b) v *= emb_b_scale;
    c->emb_b = upload(c, b);
  }
  if (int rc = check_weights(c)) return rc;
  std::string err;
  if (!make_tmap_2d(&c->tm_conv2_w, c->conv2_w, (uint64_t)9 * D, D, (uint64_t)9 * D * 2, BN_WIDE, &err) ||
      !make_tmap_2d(&c->tm_emb_w, c->emb_w, c->Kemb, D, (uint64_t)c->Kemb * 2, BN_WIDE, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  return PPASR_OK;
}

// CTC head: <prefix>ctc_lo.weight [K, V] -> K-major [Vpad, K] bf16, bias zero-padded to Vpad
int pack_ctc(ppasr_b200_ctx* c, const std::string& prefix, int K) {
  const int V = c->cfg.vocab_size;
  const HostTensor& w = c->host[prefix + "ctc_lo.weight"];
  PPASR_REQUIRE(w.shape.size() == 2 && w.shape[0] == K && w.shape[1] == V, prefix + "ctc_lo.weight shape");
  c->ctc_w = upload(c, to_bf16(transpose_in_out(w, c->Vpad)));
  std::vector<float> b(c->Vpad, 0.f);
  std::memcpy(b.data(), c->host[prefix + "ctc_lo.bias"].data.data(), sizeof(float) * V);
  c->ctc_b = upload(c, b);
  c->ctc_k = K;
  if (int rc = check_weights(c)) return rc;
  std::string err;
  if (!make_tmap_2d(&c->tm_ctc_w, c->ctc_w, K, c->Vpad, (uint64_t)K * 2, BN_NARROW, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  return PPASR_OK;
}

// self-attention of block l (prefix p): Q/K/V concatenated into one [3D, D] GEMM operand; linear_pos goes into the
// positional table's operands wpos_all [L*D, D] / bpos_all [L*D] (with its bias where the block has one)
int pack_attention(ppasr_b200_ctx* c, const std::string& p, int l, bool grouped, bool pos_bias, BlockW& w, BlockMaps& m,
                   std::vector<float>& wpos_all, std::vector<float>& bpos_all) {
  const int D = c->cfg.d_model;
  PPASR_REQUIRE(c->host[p + "self_attn.pos_bias_u"].numel() == (int64_t)c->cfg.n_heads * (grouped ? 192 : 64) &&
                    c->host[p + "self_attn.pos_bias_v"].numel() == (int64_t)c->cfg.n_heads * (grouped ? 192 : 64),
                "pos_bias_u / pos_bias_v shape");
  {
    std::vector<float> qkv((size_t)3 * D * D), bq((size_t)3 * D);
    const char* nm[3] = {"linear_q", "linear_k", "linear_v"};
    for (int s = 0; s < 3; ++s) {
      auto t = transpose_in_out(c->host[p + "self_attn." + nm[s] + ".weight"]);
      std::memcpy(qkv.data() + (size_t)s * D * D, t.data(), sizeof(float) * D * D);
      std::memcpy(bq.data() + (size_t)s * D, c->host[p + "self_attn." + nm[s] + ".bias"].data.data(), sizeof(float) * D);
    }
    w.wqkv = upload(c, to_bf16(qkv));
    w.bqkv = upload(c, bq);
  }
  w.wo = upload(c, to_bf16(transpose_in_out(c->host[p + "self_attn.linear_out.weight"])));
  w.bo = vecf(c, p + "self_attn.linear_out.bias");
  w.pos_u = vecf(c, p + "self_attn.pos_bias_u");
  w.pos_v = vecf(c, p + "self_attn.pos_bias_v");
  {
    auto t = transpose_in_out(c->host[p + "self_attn.linear_pos.weight"]);
    std::memcpy(wpos_all.data() + (size_t)l * D * D, t.data(), sizeof(float) * D * D);
    if (pos_bias)
      std::memcpy(bpos_all.data() + (size_t)l * D, c->host[p + "self_attn.linear_pos.bias"].data.data(), sizeof(float) * D);
  }
  if (int rc = check_weights(c)) return rc;
  std::string err;
  if (!make_tmap_2d(&m.wqkv, w.wqkv, D, 3 * D, (uint64_t)D * 2, BN_NARROW, &err) ||
      !make_tmap_2d(&m.wqkv_h, w.wqkv, D, 3 * D, (uint64_t)D * 2, 64, &err) ||
      !make_tmap_2d(&m.wo, w.wo, D, D, (uint64_t)D * 2, BN_WIDE, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  return PPASR_OK;
}

// conv module of a block (prefix p) with depthwise kernel K
int pack_conv_module(ppasr_b200_ctx* c, const std::string& p, int K, BlockW& w, BlockMaps& m) {
  const auto& cfg = c->cfg;
  const int D = cfg.d_model;
  {
    // pointwise_conv1.weight [2D, D, 1]: rows [0,D) = "a", [D,2D) = gate -> interleave (2c, 2c+1)
    const HostTensor& pw = c->host[p + "conv_module.pointwise_conv1.weight"];
    const HostTensor& pb = c->host[p + "conv_module.pointwise_conv1.bias"];
    PPASR_REQUIRE(pw.numel() == (int64_t)2 * D * D, "pointwise_conv1.weight shape");
    std::vector<float> wi((size_t)2 * D * D), bi((size_t)2 * D);
    for (int ch = 0; ch < D; ++ch) {
      std::memcpy(&wi[(size_t)(2 * ch) * D], &pw.data[(size_t)ch * D], sizeof(float) * D);
      std::memcpy(&wi[(size_t)(2 * ch + 1) * D], &pw.data[(size_t)(ch + D) * D], sizeof(float) * D);
      bi[2 * ch] = pb.data[ch];
      bi[2 * ch + 1] = pb.data[ch + D];
    }
    w.pw1 = upload(c, to_bf16(wi));
    w.pw1_b = upload(c, bi);
  }
  float* pad = c->wslab.take<float>(D);
  {
    const HostTensor& dw = c->host[p + "conv_module.depthwise_conv.weight"];  // [D,1,K]
    PPASR_REQUIRE(dw.numel() == (int64_t)D * K, "depthwise_conv.weight shape");
    w.dw_w = upload(c, dw.data);
    w.dw_b = vecf(c, p + "conv_module.depthwise_conv.bias");
  }
  if (cfg.conv_norm == 0) {
    w.cn_g = vecf(c, p + "conv_module.norm.weight");
    w.cn_b = vecf(c, p + "conv_module.norm.bias");
  } else {
    // eval-mode BatchNorm1D folded to scale/shift (epsilon 1e-5)
    const auto& g = c->host[p + "conv_module.norm.weight"].data;
    const auto& b = c->host[p + "conv_module.norm.bias"].data;
    const auto& mu = c->host[p + "conv_module.norm._mean"].data;
    const auto& var = c->host[p + "conv_module.norm._variance"].data;
    std::vector<float> sc(D), sh(D);
    for (int i = 0; i < D; ++i) {
      sc[i] = g[i] / std::sqrt(var[i] + 1e-5f);
      sh[i] = b[i] - mu[i] * sc[i];
    }
    w.cn_g = upload(c, sc);
    w.cn_b = upload(c, sh);
  }
  {
    const HostTensor& pw = c->host[p + "conv_module.pointwise_conv2.weight"];  // [D, D, 1] = [out, in]
    PPASR_REQUIRE(pw.numel() == (int64_t)D * D, "pointwise_conv2.weight shape");
    w.pw2 = upload(c, to_bf16(pw.data));
    w.pw2_b = vecf(c, p + "conv_module.pointwise_conv2.bias");
  }
  if (int rc = check_weights(c)) return rc;
  PPASR_CUDA_CHECK(launch_glu_pad(w.pw1_b, pad, D, 0));
  w.glu_pad = pad;
  std::string err;
  if (!make_tmap_2d(&m.pw1, w.pw1, D, 2 * D, (uint64_t)D * 2, BN_WIDE, &err) ||
      !make_tmap_2d(&m.pw2, w.pw2, D, D, (uint64_t)D * 2, BN_WIDE, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  return PPASR_OK;
}

// weight-only precompute: pos_tab[pos, l*D + h*64 + d] = linear_pos_l(pe[pos]) + bpos_l, and the tensor maps of all its
// rows (tm_pos) and of every second row (tm_pos2, the half-rate blocks)
// (reference: conformer/embedding.py:41-53 table, attention.py:234-236 projection; the projection of a constant table by a
//  constant matrix is folded here, like BatchNorm folding)
int pack_pos_table(ppasr_b200_ctx* c, const std::vector<float>& wpos_all, const std::vector<float>& bpos_all) {
  const int D = c->cfg.d_model, L = c->cfg.n_layers, ML = c->cfg.max_len;
  std::vector<float> pe((size_t)ML * D);
  for (int pos = 0; pos < ML; ++pos)
    for (int i = 0; i < D / 2; ++i) {
      const float div = std::exp((float)(2 * i) * -(std::log(10000.0f) / (float)D));
      pe[(size_t)pos * D + 2 * i] = std::sin((float)pos * div);
      pe[(size_t)pos * D + 2 * i + 1] = std::cos((float)pos * div);
    }
  const __nv_bfloat16* pe_d = upload(c, to_bf16(pe));
  const __nv_bfloat16* wpos_d = upload(c, to_bf16(wpos_all));
  __nv_bfloat16* tab = c->wslab.take<__nv_bfloat16>((size_t)ML * L * D);
  const float* bpos_d = upload(c, bpos_all);
  if (int rc = check_weights(c)) return rc;
  std::string err;
  CUtensorMap ta, tb;
  if (!make_tmap_2d(&ta, pe_d, D, ML, (uint64_t)D * 2, GEMM_BLOCK_M, &err) ||
      !make_tmap_2d(&tb, wpos_d, D, (uint64_t)L * D, (uint64_t)D * 2, BN_WIDE, &err) ||
      !make_tmap_2d(&c->tm_pos, tab, (uint64_t)L * D, ML, (uint64_t)L * D * 2, 128, &err) ||
      !make_tmap_2d(&c->tm_pos2, tab, (uint64_t)L * D, ML / 2, (uint64_t)2 * L * D * 2, 128, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  GemmShape s = make_shape(ML, L * D, D, BN_WIDE);
  EpiStoreBF16<BN_WIDE, ACT_NONE> epi{tab, bpos_d, L * D, ML, L * D};
  PPASR_CUDA_CHECK((launch_gemm<BN_WIDE, ST_WIDE, false>(ta, tb, s, epi, c->sms, 0)));
  c->pos_tab = tab;
  return PPASR_OK;
}

// waits for the packing kernels, reports any failed upload, and drops the host copies
int finish_finalize(ppasr_b200_ctx* c) {
  PPASR_CUDA_CHECK(cudaDeviceSynchronize());
  if (int rc = check_weights(c)) return rc;
  c->host.clear();
  c->finalized = true;
  return PPASR_OK;
}

}  // namespace

extern "C" {

int ppasr_b200_create(const ppasr_b200_config* cfg, ppasr_b200_ctx** out) {
  PPASR_REQUIRE(cfg && out, "null pointer");
  PPASR_REQUIRE(cfg->model_type >= 0 && cfg->model_type <= 3,
                "model_type must be 0 (conformer), 1 (squeezeformer), 2 (deepspeech2) or 3 (efficient_conformer)");
  PPASR_REQUIRE(cfg->feat_dim >= 7 && cfg->vocab_size > 1 && cfg->n_layers > 0, "bad config");
  if (cfg->model_type == 2) {
    PPASR_REQUIRE(cfg->d_model >= 64 && cfg->d_model <= 1024 && cfg->d_model % 64 == 0,
                  "deepspeech2: rnn_size must be a multiple of 64 and <= 1024 in this build (W_hh slices live in shared memory)");
  } else {
    PPASR_REQUIRE(cfg->d_model == 256, "d_model must be 256 in this build");
    PPASR_REQUIRE(cfg->n_heads * 64 == cfg->d_model, "head dim must be 64");
    PPASR_REQUIRE(cfg->ffn_dim % 256 == 0 && cfg->ffn_dim > 0, "ffn_dim must be a multiple of 256");
    PPASR_REQUIRE(cfg->conv_kernel == 7 || cfg->conv_kernel == 15 || cfg->conv_kernel == 31, "conv_kernel 7/15/31");
    PPASR_REQUIRE(cfg->max_len > 16, "bad config");
  }
  if (cfg->model_type == 1) {
    const int ri = cfg->reduce_idx, ci = cfg->recover_idx;
    PPASR_REQUIRE((ri < 0 && ci < 0) || (ri >= 0 && ri < ci && ci < cfg->n_layers),
                  "squeezeformer: need 0 <= reduce_idx < recover_idx < num_blocks (or neither)");
    PPASR_REQUIRE(cfg->time_reduce_kernel == 1 || cfg->time_reduce_kernel == 5, "time_reduce_kernel must be 1 (stream) or 5 (conv1d)");
  }
  if (cfg->model_type == 3) {
    PPASR_REQUIRE(cfg->group_size == 3, "efficient_conformer: group_size must be 3");
    PPASR_REQUIRE(cfg->stride_layer_idx >= -1 && cfg->stride_layer_idx < cfg->n_layers, "bad stride_layer_idx");
    PPASR_REQUIRE(cfg->n_layers <= 32, "at most 32 blocks");
    for (int l = 0; l < cfg->n_layers; ++l)
      if ((cfg->group_layer_mask >> l) & 1)
        PPASR_REQUIRE(cfg->stride_layer_idx < 0 || l <= cfg->stride_layer_idx,
                      "efficient_conformer: grouped attention is supported in blocks up to the stride block");
    int ng = 0;
    for (int l = 0; l < cfg->n_layers; ++l) ng += (cfg->group_layer_mask >> l) & 1;
    PPASR_REQUIRE(ng <= 4, "at most 4 grouped-attention blocks");
    PPASR_REQUIRE(cfg->conv_kernel == 15 || !cfg->stride_kernel, "stride_kernel needs cnn_module_kernel 15 (15 -> 7)");
  }
  auto* c = new ppasr_b200_ctx();
  c->cfg = *cfg;
  c->layer_k.assign(cfg->n_layers, cfg->conv_kernel);
  if (const char* e = std::getenv("PPASR_B200_CONV1_TC")) c->conv1_tc = std::atoi(e) != 0;
  if (const char* e = std::getenv("PPASR_B200_FUSED_CONV")) {  // an invalid value keeps the default
    const int v = std::atoi(e);
    if (v == 0 || v == 2) c->fused_conv = v;
  }
  if (cfg->model_type == 3) {
    c->eff_stride_idx = cfg->stride_layer_idx;
    c->eff_group_mask = (unsigned)cfg->group_layer_mask;
    if (cfg->stride_layer_idx >= 0 && cfg->stride_kernel)
      for (int l = cfg->stride_layer_idx + 1; l < cfg->n_layers; ++l) c->layer_k[l] = cfg->conv_kernel / 2;
  }
  c->F1 = (cfg->feat_dim - 1) / 2;
  c->F2 = (c->F1 - 1) / 2;
  c->FH = (c->F1 + 1) / 2;
  c->Kemb = c->F2 * cfg->d_model;
  if (cfg->model_type != 2 && c->Kemb % GEMM_BLOCK_K != 0) {
    delete c;
    set_last_error("subsampled feature size * d_model must be a multiple of 64");
    return PPASR_ERR_INVALID;
  }
  c->Vpad = (cfg->vocab_size + BN_NARROW - 1) / BN_NARROW * BN_NARROW;
  c->Vld = (cfg->vocab_size + 3) / 4 * 4;
  c->ctc_parts = 2 * (c->Vpad / BN_NARROW);
  *out = c;
  return PPASR_OK;
}

int ppasr_b200_destroy(ppasr_b200_ctx* ctx) {
  if (!ctx) return PPASR_OK;
  ctx->wslab.release();
  ctx->aslab.release();
  if (ctx->ss.kk) cudaFree(ctx->ss.kk);
  if (ctx->ss.vt) cudaFree(ctx->ss.vt);
  if (ctx->ss.cnn) cudaFree(ctx->ss.cnn);
  if (ctx->ss.pgc) cudaFree(ctx->ss.pgc);
  if (ctx->ss.d_step) cudaFree(ctx->ss.d_step);
  if (ctx->ds.h_state) cudaFree(ctx->ds.h_state);
  if (ctx->ds.c_state) cudaFree(ctx->ds.c_state);
  if (ctx->h_vlen) cudaFreeHost(ctx->h_vlen);
  if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
  if (ctx->graph) cudaGraphDestroy(ctx->graph);
  delete ctx;
  return PPASR_OK;
}

int ppasr_b200_load_tensor(ppasr_b200_ctx* ctx, const char* name, const float* data, int32_t ndim,
                           const int64_t* shape) {
  PPASR_REQUIRE(ctx && name && data && shape && ndim >= 1 && ndim <= 4, "bad arguments");
  if (ctx->finalized) {
    set_last_error("context already finalized");
    return PPASR_ERR_STATE;
  }
  HostTensor t;
  t.shape.assign(shape, shape + ndim);
  t.data.assign(data, data + t.numel());
  ctx->host[name] = std::move(t);
  return PPASR_OK;
}

int ppasr_b200_finalize(ppasr_b200_ctx* c) {
  PPASR_REQUIRE(c, "null ctx");
  if (c->finalized) return PPASR_OK;
  const auto& cfg = c->cfg;
  const int D = cfg.d_model, L = cfg.n_layers, FF = cfg.ffn_dim;
  int dev = 0;
  PPASR_CUDA_CHECK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  PPASR_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_last_error("ppasr_b200 requires an sm_100 (Blackwell B200) device; found sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor));
    return PPASR_ERR_CUDA;
  }
  c->sms = prop.multiProcessorCount;
  c->upload_err = cudaSuccess;
  if (cfg.model_type == 1) return finalize_squeezeformer(c);
  if (cfg.model_type == 2) return finalize_ds2(c);

  // ---- presence check first, so the error lists everything -------------------------------------
  std::vector<std::string> names = {"encoder.global_cmvn.mean", "encoder.global_cmvn.istd",
                                    "encoder.embed.conv.0.weight", "encoder.embed.conv.0.bias",
                                    "encoder.embed.conv.2.weight", "encoder.embed.conv.2.bias",
                                    "encoder.embed.out.0.weight", "encoder.embed.out.0.bias",
                                    "encoder.after_norm.weight", "encoder.after_norm.bias",
                                    "ctc.ctc_lo.weight", "ctc.ctc_lo.bias"};
  for (int l = 0; l < L; ++l) {
    const std::string p = "encoder.encoders." + std::to_string(l) + ".";
    for (const char* s : {"norm_ff_macaron", "norm_mha", "norm_conv", "norm_ff", "norm_final"}) {
      names.push_back(p + s + ".weight");
      names.push_back(p + s + ".bias");
    }
    for (const char* s : {"feed_forward_macaron", "feed_forward"})
      for (const char* t : {".w_1.weight", ".w_1.bias", ".w_2.weight", ".w_2.bias"}) names.push_back(p + s + t);
    block_names(cfg, p, (c->eff_group_mask >> l) & 1, &names);  // grouped linear_pos has a bias (efficient_conformer/attention.py:31)
  }
  if (int rc = require_present(c, names)) return rc;

  PPASR_CUDA_CHECK(c->wslab.reserve(conformer_slab_bytes(c)));
  c->wslab.rewind();
  int rc;
  if ((rc = pack_front(c, "encoder.embed.conv.0", "encoder.embed.conv.2", "encoder.embed.out.0", 1.0f))) return rc;
  c->after_g = vecf(c, "encoder.after_norm.weight");
  c->after_b = vecf(c, "encoder.after_norm.bias");
  if ((rc = pack_ctc(c, "ctc.", D))) return rc;

  // ---- encoder layers -------------------------------------------------------------------------
  c->layers.resize(L);
  c->lmaps.resize(L);
  std::vector<float> wpos_all((size_t)L * D * D), bpos_all((size_t)L * D, 0.f);  // bias: grouped blocks only
  for (int l = 0; l < L; ++l) {
    const std::string p = "encoder.encoders." + std::to_string(l) + ".";
    LayerW& w = c->layers[l];
    auto& m = c->lmaps[l];
    const bool grouped = (c->eff_group_mask >> l) & 1;
    w.ln_ffm_g = vecf(c, p + "norm_ff_macaron.weight"), w.ln_ffm_b = vecf(c, p + "norm_ff_macaron.bias");
    w.ln_mha_g = vecf(c, p + "norm_mha.weight"), w.ln_mha_b = vecf(c, p + "norm_mha.bias");
    w.ln_conv_g = vecf(c, p + "norm_conv.weight"), w.ln_conv_b = vecf(c, p + "norm_conv.bias");
    w.ln_ff_g = vecf(c, p + "norm_ff.weight"), w.ln_ff_b = vecf(c, p + "norm_ff.bias");
    w.ln_fin_g = vecf(c, p + "norm_final.weight"), w.ln_fin_b = vecf(c, p + "norm_final.bias");
    w.ffm_w1 = upload(c, to_bf16(transpose_in_out(c->host[p + "feed_forward_macaron.w_1.weight"])));
    w.ff_w1 = upload(c, to_bf16(transpose_in_out(c->host[p + "feed_forward.w_1.weight"])));
    w.ffm_b1 = vecf(c, p + "feed_forward_macaron.w_1.bias");
    w.ff_b1 = vecf(c, p + "feed_forward.w_1.bias");
    {
      // ff_scale = 0.5 (encoder.py:331-332) folded into W2 / b2 for the fused kernel (exact: power of two)
      auto scaled = [&](const std::string& wn, const std::string& bn, const __nv_bfloat16** wd, const float** bd) {
        std::vector<float> t = transpose_in_out(c->host[wn]);
        for (auto& v : t) v *= 0.5f;
        *wd = upload(c, to_bf16(t));
        std::vector<float> bv = c->host[bn].data;
        for (auto& v : bv) v *= 0.5f;
        *bd = upload(c, bv);
      };
      scaled(p + "feed_forward_macaron.w_2.weight", p + "feed_forward_macaron.w_2.bias", &w.ffm_w2s, &w.ffm_b2s);
      scaled(p + "feed_forward.w_2.weight", p + "feed_forward.w_2.bias", &w.ff_w2s, &w.ff_b2s);
    }
    if ((rc = pack_attention(c, p, l, grouped, grouped, w, m, wpos_all, bpos_all))) return rc;
    if ((rc = pack_conv_module(c, p, c->layer_k[l], w, m))) return rc;
    std::string err;
    if (!make_tmap_2d(&m.ffm_w2s, w.ffm_w2s, FF, D, (uint64_t)FF * 2, BN_WIDE, &err) ||
        !make_tmap_2d(&m.ff_w2s, w.ff_w2s, FF, D, (uint64_t)FF * 2, BN_WIDE, &err) ||
        !make_tmap_2d(&m.ffm_w1_128, w.ffm_w1, D, FF, (uint64_t)D * 2, 128, &err) ||
        !make_tmap_2d(&m.ff_w1_128, w.ff_w1, D, FF, (uint64_t)D * 2, 128, &err)) {
      set_last_error(err);
      return PPASR_ERR_CUDA;
    }
  }
  if ((rc = pack_pos_table(c, wpos_all, bpos_all))) return rc;
  return finish_finalize(c);
}

int ppasr_b200_out_frames(const ppasr_b200_ctx* c, int32_t T) {
  if (T < 7) return 0;
  const int tp = ((T - 1) / 2 - 1) / 2;
  if (c && c->cfg.model_type == 3 && c->eff_stride_idx >= 0) return (tp + 1) / 2;
  return tp;
}

}  // extern "C"

namespace {

// (re)builds the activation workspace and A-operand tensor maps for a (B, T) problem
int build_plan(ppasr_b200_ctx* c, int B, int T) {
  Plan& p = c->plan;
  if (p.B == B && p.T == T) return PPASR_OK;
  const auto& cfg = c->cfg;
  const int D = cfg.d_model, H = cfg.n_heads, F = cfg.feat_dim;
  PPASR_REQUIRE(T >= 7, "need at least 7 feature frames (subsampling right context, predict.py:288)");
  Plan n;
  n.B = B, n.T = T;
  n.T1 = (T - 1) / 2;
  n.Tp = (n.T1 - 1) / 2;
  n.Th = (n.T1 + 1) / 2;
  n.M = B * n.Tp;
  n.Mr = B * n.Th * c->FH;
  n.Tkp = (n.Tp + 63) / 64 * 64;
  n.Tcat = n.Tp + cfg.conv_kernel - 1;
  n.Mcat = B * n.Tcat;
  PPASR_REQUIRE(n.Tp >= 1 && n.Tp < cfg.max_len, "sequence too long for the positional table (embedding.py:110-112)");
  const size_t M = n.M;
  size_t bytes = 0;
  auto acc = [&](size_t b) { bytes += ((b + 255) & ~size_t(255)) + 256; };
  acc((size_t)B * T * F * 4);
  acc(B * 4);
  acc((size_t)4 * n.Mr * D * 2);
  acc(M * c->Kemb * 2);
  acc(M * D * 4);                                   // x
  acc(M * D * 2 + 1024);                            // x2 (reduced stream)
  if (cfg.model_type == 3) {
    const size_t tg = (n.Tp + 2) / 3, tgp = (tg + 63) / 64 * 64;
    acc((size_t)B * H * tg * 384 * 2 + 4096);
    acc((size_t)B * H * tg * 192 * 2 + 4096);
    acc((size_t)B * H * 192 * tgp * 2 + 4096);
    acc((size_t)4 * tg * 768 * 2 + 4096);
  }
  acc(B * 4);
  acc(M * D * 2 * 4);                               // y, att, g, z
  acc((size_t)n.Mcat * D * 2 * 2);                  // ycat, gcat
  acc((size_t)B * H * n.Tp * 128 * 2);              // q2
  acc((size_t)B * H * n.Tp * 64 * 2);               // kk
  acc((size_t)B * H * 64 * n.Tkp * 2);              // vt
  acc(M * c->Vld * 4);                              // logits
  acc(M * (size_t)cfg.vocab_size * 4);              // probs
  acc(M * c->ctc_parts * 4 * 3);                    // partial stats
  acc(M * 4 * 3 + (size_t)B * 4 * 3);
  bytes += 1u << 20;
  if (bytes > c->aslab.cap) {
    PPASR_CUDA_CHECK(cudaDeviceSynchronize());
    PPASR_CUDA_CHECK(c->aslab.reserve(bytes));
    // q2/kk/vt padding regions must be finite for masked-out MMA operands
    PPASR_CUDA_CHECK(cudaMemset(c->aslab.base, 0, c->aslab.cap));
  }
  c->aslab.rewind();
  auto& a = c->aslab;
  n.feats = a.take<float>((size_t)B * T * F);
  n.vlen = a.take<int>(B);
  n.phase = a.take<__nv_bfloat16>((size_t)4 * n.Mr * D);
  n.c2 = a.take<__nv_bfloat16>(M * c->Kemb);
  n.x = a.take<float>(M * D);
  n.x2 = a.take<float>((size_t)B * ((n.Tp + 1) / 2) * D);
  n.vlen2 = a.take<int>(B);
  if (cfg.model_type == 3) {
    n.Tg = (n.Tp + 2) / 3;
    n.Tgp = (n.Tg + 63) / 64 * 64;
    n.q2g = a.take<__nv_bfloat16>((size_t)B * H * n.Tg * 384);
    n.kkg = a.take<__nv_bfloat16>((size_t)B * H * n.Tg * 192);
    n.vtg = a.take<__nv_bfloat16>((size_t)B * H * 192 * n.Tgp);
    n.pg = a.take<__nv_bfloat16>((size_t)4 * n.Tg * 768);
  }
  n.y = a.take<__nv_bfloat16>(M * D);
  n.att = a.take<__nv_bfloat16>(M * D);
  n.g = a.take<__nv_bfloat16>(M * D);
  n.z = a.take<__nv_bfloat16>(M * D);
  n.ycat = a.take<__nv_bfloat16>((size_t)n.Mcat * D);
  n.gcat = a.take<__nv_bfloat16>((size_t)n.Mcat * D);
  n.q2 = a.take<__nv_bfloat16>((size_t)B * H * n.Tp * 128);
  n.kk = a.take<__nv_bfloat16>((size_t)B * H * n.Tp * 64);
  n.vt = a.take<__nv_bfloat16>((size_t)B * H * 64 * n.Tkp);
  n.logits = a.take<float>(M * c->Vld);
  n.probs = a.take<float>(M * (size_t)cfg.vocab_size);
  n.pmax = a.take<float>(M * c->ctc_parts);
  n.psum = a.take<float>(M * c->ctc_parts);
  n.parg = a.take<int>(M * c->ctc_parts);
  n.idx = a.take<int>(M);
  n.maxp = a.take<float>(M);
  n.ids = a.take<int>(M);
  n.out_len = a.take<int>(B);
  n.score = a.take<float>(B);
  if (a.overflow) {
    set_last_error("internal error: activation slab overflow");
    return PPASR_ERR_STATE;
  }
  std::string err;
  bool ok = make_tmap_3d(&n.tm_phase, n.phase, D, n.Mr, 4, (uint64_t)D * 2, (uint64_t)n.Mr * D * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_c2, n.c2, c->Kemb, M, (uint64_t)c->Kemb * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_y, n.y, D, M, (uint64_t)D * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_att, n.att, D, M, (uint64_t)D * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_g, n.g, D, M, (uint64_t)D * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_z, n.z, D, M, (uint64_t)D * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_ycat, n.ycat, D, n.Mcat, (uint64_t)D * 2, GEMM_BLOCK_M, &err) &&
            make_tmap_2d(&n.tm_q, n.q2, 128, (uint64_t)B * H * n.Tp, 256, 128, &err) &&
            make_tmap_2d(&n.tm_k, n.kk, 64, (uint64_t)B * H * n.Tp, 128, 128, &err) &&
            make_tmap_2d(&n.tm_vt, n.vt, n.Tp, (uint64_t)B * H * 64, (uint64_t)n.Tkp * 2, 64, &err);
  if (ok && cfg.model_type == 3) {
    ok = make_tmap_2d(&n.tm_qg, n.q2g, 384, (uint64_t)B * H * n.Tg, 384 * 2, 128, &err) &&
         make_tmap_2d(&n.tm_kg, n.kkg, 192, (uint64_t)B * H * n.Tg, 192 * 2, 64, &err) &&
         make_tmap_2d(&n.tm_vtg, n.vtg, n.Tg, (uint64_t)B * H * 192, (uint64_t)n.Tgp * 2, 192, &err);
    for (int i = 0; ok && i < 4; ++i)
      ok = make_tmap_2d(&n.tm_pg[i], n.pg + (size_t)i * n.Tg * 768, 768, n.Tg, 768 * 2, 64, &err);
  }
  if (!ok) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  n.Mc = n.M, n.Tc = n.Tp, n.vc = n.vlen;
  if (cfg.model_type == 3 && c->eff_stride_idx >= 0) {
    n.Tc = (n.Tp + 1) / 2;
    n.Mc = B * n.Tc;
    n.vc = n.vlen2;
  }
  p = n;
  return PPASR_OK;
}

// Offline plain attention: the QKV projection runs inside the attention kernel (qkv_rel_attention_kernel) when every
// utterance fits two 128-frame tiles; longer ones take the QKV GEMM + rel_attention_kernel pair.
bool fused_qkv_attention(int D, int H, int T) { return D == 256 && H == 4 && T >= 1 && T <= 256; }

template <int BN, int ST, class Epi>
cudaError_t gemm(ppasr_b200_ctx* c, const CUtensorMap& a, const CUtensorMap& b, int M, int N, int K, const Epi& epi,
                 cudaStream_t st) {
  GemmShape s = make_shape(M, N, K, BN);
  return launch_gemm<BN, ST, false>(a, b, s, epi, c->sms, st);
}

// CMVN + Conv2d(1->D,k3,s2)+ReLU + Conv2d(D->D,k3,s2)+ReLU -> c2 [M, F2*D] (conformer/subsampling.py:84-87,110-111;
// squeezeformer/subsampling.py:33-39,59-63 with dw_stride False is the same pair of convolutions)
int run_subsampling_convs(ppasr_b200_ctx* c, cudaStream_t st) {
  Plan& p = c->plan;
  const auto& cfg = c->cfg;
  const int D = cfg.d_model;
  if (c->fused_conv == 2 && D == 256 && cfg.feat_dim <= 96) {
    // CMVN + conv1 (split-tf32 GEMM) + ReLU + conv2 + ReLU in one tcgen05 kernel (conv1_tc.cu) -> c2 [M, F2*D]
    PROF(PC_CONV_FRONT);
    PPASR_CUDA_CHECK(launch_conv_front_tc(c->tm_conv2_w, p.feats, c->cmvn_mean, c->cmvn_istd, c->conv1_w, c->conv1_b, c->conv2_b,
                                          p.c2, p.B, p.T, cfg.feat_dim, p.T1, c->F1, p.Th, c->FH, p.Tp, c->F2, c->sms, st));
  } else {
    // CMVN + conv1 + ReLU -> stride-phase images
    { PROF(PC_CONV1);
    if (c->conv1_tc && D == 256 && cfg.feat_dim <= 256)
      PPASR_CUDA_CHECK(launch_conv1_tc(p.tm_phase, p.feats, c->cmvn_mean, c->cmvn_istd, c->conv1_w, c->conv1_b, p.B, p.T,
                                       cfg.feat_dim, p.T1, c->F1, p.Th, c->FH, c->sms, st));
    else
      PPASR_CUDA_CHECK(launch_conv1_subsample(p.feats, c->cmvn_mean, c->cmvn_istd, c->conv1_w, c->conv1_b, p.phase, p.B,
                                              p.T, cfg.feat_dim, D, p.T1, c->F1, p.Th, c->FH, st)); }
    // conv2 + ReLU as 9 shifted GEMM taps -> c2 [M, F2*D]
    GemmShape s = make_shape(p.Mr, D, 9 * D, BN_WIDE);
    s.conv_pitch = c->FH;
    s.conv_kc = D / GEMM_BLOCK_K;
    EpiConv2<BN_WIDE> epi{p.c2, c->conv2_b, p.Mr, D, p.Th, c->FH, p.Tp, c->F2};
    PROF(PC_CONV2);
    PPASR_CUDA_CHECK((launch_gemm<BN_WIDE, ST_WIDE, true>(p.tm_phase, c->tm_conv2_w, s, epi, c->sms, st)));
  }
  return PPASR_OK;
}

#include "runtime_squeezeformer.inl"
#include "runtime_ds2.inl"

// Conformer (model_type 0) and Efficient Conformer (model_type 3): the pre-norm macaron block on the fused kernels.
// Reference: conformer/encoder.py:164-206 (forward), :380-429 (block); efficient_conformer/encoder.py:212-264 (forward),
// :455-548 (stride block), attention.py:128-193 (grouped attention), convolution.py:80-138 (strided conv module).
// What the Efficient Conformer changes per block:
//   * grouped blocks: the QKV epilogue writes the (T/3 tokens x 4 heads x 192) views, grouped_attention_kernel;
//   * the stride block: strided depthwise conv, AvgPool1D(2, ceil) on the residual, then everything (rows, lengths,
//     positional rows) at half rate; blocks after it use depthwise kernel 7 (layer_k).
//
// chunk: forward_chunk (conformer/encoder.py:208-275, efficient_conformer/encoder.py:266-394) on the device-resident caches
// in c->ss, no padding masks. This chunk's K/V are appended to the block's cache at row kend (at the block's rate) and
// keys kstart .. kend + chunk are attended with positions offset - cache_t ... (conformer/attention.py:225-232,
// encoder.py:253). The Efficient Conformer streams with required_cache_size < 0 (PPASRPredictor, predict.py:304-306), so
// its caches are append-only (kstart = 0, offset = kend) and pad4group's re-grouping from the first cached frame
// (attention.py:153-160) is simply group = absolute_frame // 3:
//   * grouped blocks keep K as [B,H,group,192] and V^T as [B,H,192,group] (the EpiQKVGrouped operand layout) inside the
//     same per-layer cache slices the plain blocks use; a new frame f lands in group f / 3 at feature (f % 3) * 256 + c;
//     the caches start zeroed, so the missing frames of a partially filled last group read as zero (a real, unmasked key);
//   * queries are grouped from the CHUNK start (zero padded before pos_bias_u/v are added);
//   * p = linear_pos(pos_emb[0 : t_total]) zero-padded to a multiple of 3 is rebuilt per chunk (grouped_pos_kernel);
//   * blocks after the stride block run at half rate: keys at positions 2 j (tm_pos2), caches hold kend / 2 frames
//     (the reference stores them repeated x2 and reads ::2, encoder.py:351,368), conv caches of K/2 - 1 = 6 rows;
//   * the stride block's stride-2 "valid" conv over [cache 14 | chunk] is aligned with the offline run because chunks
//     start at even frames; its residual goes through AvgPool1D(2, 2, ceil).
// tests/test_effconf_chunk_layout_spec_cpu.py states this layout in NumPy and checks it against the reference code's own
// streaming outputs.
int run_encoder(ppasr_b200_ctx* c, cudaStream_t st, bool chunk) {
  Plan& p = c->plan;
  auto& ss = c->ss;
  const auto& cfg = c->cfg;
  const int D = cfg.d_model, H = cfg.n_heads, FF = cfg.ffn_dim, L = cfg.n_layers, B = p.B;
  const int lmax = cfg.conv_kernel - 1;  // conv-cache rows per (layer, stream)
  const float eps = 1e-5f;
  { int rcf = run_subsampling_convs(c, st); if (rcf) return rcf; }
  // the residual stream at the current rate: rows, frames per utterance, valid lengths, positional rows
  float* xc = p.x;
  int Tc = p.Tp, Mc = p.M, rate = 1;
  const int* vl = chunk ? nullptr : p.vlen;
  const CUtensorMap* tmpos = &c->tm_pos;
  // Linear(F2*D -> D) then x * sqrt(D) (subsampling.py:113, embedding.py:113), fused with block 0's first LayerNorm
  {
    EpiResidLN<BN_WIDE> e{p.x, c->emb_b, D, p.M, D, std::sqrt((float)D), 0, nullptr, p.Tp, 0, 0, c->layers[0].ln_ffm_g,
                          c->layers[0].ln_ffm_b, nullptr, nullptr, p.y, eps};
    PROF(PC_EMBED);
    PPASR_CUDA_CHECK((gemm<BN_WIDE, ST_WIDE>(c, p.tm_c2, c->tm_emb_w, p.M, D, c->Kemb, e, st)));
  }
  int gi = 0;  // index of the grouped block (its padded positional rows live in slot gi of p.pg / ss.pgc)
  for (int l = 0; l < L; ++l) {
    const LayerW& w = c->layers[l];
    const auto& m = c->lmaps[l];
    const int K = c->layer_k[l];
    const bool grouped = (c->eff_group_mask >> l) & 1;
    const bool strided = l == c->eff_stride_idx;
    // ---- macaron FFN: x += 0.5 * W2 swish(W1 LN(x)); then y = norm_mha(x)        (encoder.py:380-390)
    {
      PROF(PC_FUSED_FFN);
      PPASR_CUDA_CHECK(launch_fused_ffn(p.tm_y, nullptr, m.ffm_w1_128, m.ffm_w2s, Mc, FF, xc, p.y, w.ffm_b1, w.ffm_b2s, w.ln_mha_g,
                                        w.ln_mha_b, nullptr, nullptr, eps, nullptr, nullptr, nullptr, nullptr, Tc, st));
    }
    // ---- rel-pos MHA (encoder.py:389-409)
    const size_t lk = (size_t)l * ss.B * H * ss.Tcap * 64;
    const int kend = ss.kend / rate, kstart = ss.kstart / rate, cache_t = kend - kstart;  // chunk: cached keys at this rate
    if (grouped && !chunk) {
      // pad4group of p = linear_pos(pos_emb): rows >= T are zero (attention.py:73-77)
      PPASR_CUDA_CHECK(launch_grouped_pos(c->pos_tab, L * D, l * D, Tc, 3 * p.Tg, p.pg + (size_t)gi * p.Tg * 768, st));
      EpiQKVGrouped<BN_NARROW> e{p.q2g, p.kkg, p.vtg, w.bqkv, w.pos_u, w.pos_v, Mc, Tc, H, p.Tg, p.Tgp};
      { PROF(PC_QKV); PPASR_CUDA_CHECK((gemm<BN_NARROW, ST_NARROW>(c, p.tm_y, m.wqkv, Mc, 3 * D, D, e, st))); }
      GroupedAttnParams gp{B, H, Tc, p.Tg, vl, p.att};
      { PROF(PC_ATTENTION); PPASR_CUDA_CHECK(launch_grouped_attention(p.tm_qg, p.tm_kg, p.tm_pg[gi], p.tm_vtg, gp, st)); }
      ++gi;
    } else if (grouped) {
      // positional operand of the T2 keys at positions j * rate, zero beyond T2 inside the last group
      const int T2 = cache_t + Tc, G2 = (T2 + 2) / 3;
      PPASR_CUDA_CHECK(launch_grouped_pos(c->pos_tab, L * D * rate, l * D, T2, 3 * G2, ss.pgc + (size_t)gi * ss.Gcap * 768, st));
      EpiQKVGrouped<BN_NARROW> e{p.q2g, ss.kk + lk, ss.vt + lk, w.bqkv, w.pos_u, w.pos_v, Mc, Tc, H, (Tc + 2) / 3, ss.Gcap};
      e.kofs = kend, e.Tgk = ss.Gcap;
      { PROF(PC_QKV); PPASR_CUDA_CHECK((gemm<BN_NARROW, ST_NARROW>(c, p.tm_y, m.wqkv, Mc, 3 * D, D, e, st))); }
      GroupedAttnParams gp{B, H, Tc, (Tc + 2) / 3, nullptr, p.att};
      gp.Tgk = G2, gp.k_pitch = ss.Gcap;
      { PROF(PC_ATTENTION); PPASR_CUDA_CHECK(launch_grouped_attention(ss.tm_qgc, ss.tm_k[l], ss.tm_pgc[gi], ss.tm_vt[l], gp, st)); }
      ++gi;
    } else {
      AttnParams ap{};
      ap.B = B, ap.H = H, ap.T1 = Tc, ap.D = D, ap.pos_col0 = l * D, ap.out = p.att, ap.q_rows_per_bh = Tc;
      if (!chunk && fused_qkv_attention(D, H, Tc)) {
        QkvAttnParams qp{B, H, Tc, D, 0, l * D, w.bqkv, w.pos_u, w.pos_v, vl, p.att};
        { PROF(PC_ATTENTION); PPASR_CUDA_CHECK(launch_qkv_rel_attention(p.tm_y, m.wqkv_h, *tmpos, qp, st)); }
      } else if (!chunk) {
        EpiQKV<BN_NARROW> e{p.q2, p.kk, p.vt, w.bqkv, w.pos_u, w.pos_v, Mc, Tc, H, Tc, p.Tkp, 0};
        { PROF(PC_QKV); PPASR_CUDA_CHECK((gemm<BN_NARROW, ST_NARROW>(c, p.tm_y, m.wqkv, Mc, 3 * D, D, e, st))); }
        ap.T2 = Tc, ap.k_rows_per_bh = Tc, ap.k_row0 = 0, ap.pos_row0 = 0, ap.klens = vl;
        { PROF(PC_ATTENTION); PPASR_CUDA_CHECK(launch_rel_attention(p.tm_q, p.tm_k, *tmpos, p.tm_vt, ap, st)); }
      } else {
        EpiQKV<BN_NARROW> e{p.q2, ss.kk + lk, ss.vt + lk, w.bqkv, w.pos_u, w.pos_v, Mc, Tc, H, ss.Tcap, ss.Tcap, kend};
        if (ss.ragged) e.slots = ss.d_step, e.kofs_b = ss.d_step + B;
        { PROF(PC_QKV); PPASR_CUDA_CHECK((gemm<BN_NARROW, ST_NARROW>(c, p.tm_y, m.wqkv, Mc, 3 * D, D, e, st))); }
        ap.T2 = cache_t + Tc, ap.k_rows_per_bh = ss.Tcap, ap.k_row0 = kstart;
        ap.pos_row0 = (ss.offset - (ss.kend - ss.kstart)) / rate, ap.klens = nullptr;
        if (ss.ragged) {  // per-session cache slot / key range / positions
          ap.T2 = ss.step_T2;
          ap.slots = ss.d_step, ap.k_row0s = ss.d_step + 2 * B, ap.pos_row0s = ss.d_step + 3 * B, ap.klens = ss.d_step + 4 * B;
        }
        { PROF(PC_ATTENTION); PPASR_CUDA_CHECK(launch_rel_attention(p.tm_q, ss.tm_k[l], *tmpos, ss.tm_vt[l], ap, st)); }
      }
    }
    // ---- x += Wo att + bo; y = mask(norm_conv(x)); then the conv module's pw1 + GLU, depthwise conv, norm, swish -> z
    //      (encoder.py:407-421; pad frames of the conv-module input are zeroed, convolution.py:104-106)
    const __nv_bfloat16* gin = p.g;  // GLU output the depthwise conv reads
    int Tin = Tc;                    // ... and its frames per utterance
    if (!chunk) {
      PROF(PC_FUSED_ATTN_OUT);
      PPASR_CUDA_CHECK(launch_fused_attn_out(p.tm_att, m.wo, m.pw1, Mc, xc, p.g, w.bo, w.ln_conv_g, w.ln_conv_b, w.pw1_b, vl, Tc,
                                             eps, st));
    } else {
      {
        EpiResidLN<BN_WIDE> e{xc, w.bo, D, Mc, D, 1.0f, 1, nullptr, Tc, 0, 1, w.ln_conv_g, w.ln_conv_b, nullptr, nullptr, p.y, eps};
        PROF(PC_OUTPROJ);
        PPASR_CUDA_CHECK((gemm<BN_WIDE, ST_WIDE>(c, p.tm_att, m.wo, Mc, D, D, e, st)));
      }
      // [cnn_cache ; chunk] -> pw1 + GLU -> "valid" depthwise conv; cache <- last K-1 input rows (convolution.py:108-117)
      const int lorder = K - 1, Mcat = B * (lorder + Tc);
      PPASR_CUDA_CHECK(launch_conv_cache_concat(ss.cnn + (size_t)l * ss.B * lmax * D, p.y, p.ycat, B, Tc, lorder, D, st,
                                                ss.ragged ? ss.d_step : nullptr));
      EpiGLU<BN_WIDE> eg{p.gcat, w.pw1_b, D, Mcat, 2 * D};
      { PROF(PC_PW1_GLU); PPASR_CUDA_CHECK((gemm<BN_WIDE, ST_WIDE>(c, p.tm_ycat, m.pw1, Mcat, 2 * D, D, eg, st))); }
      gin = p.gcat, Tin = lorder + Tc;
    }
    // offline: 'same' padding (causal: K-1 rows on the left, read from glu_pad); chunk: the cache is the left context
    const int lpad = chunk ? 0 : cfg.causal ? K - 1 : (K - 1) / 2;
    const float* pad_left = (!chunk && cfg.causal) ? w.glu_pad : nullptr;
    if (!strided) {
      PROF(PC_DWCONV);
      PPASR_CUDA_CHECK(launch_dwconv_norm_swish(gin, w.dw_w, w.dw_b, pad_left, w.cn_g, w.cn_b, cfg.conv_norm == 0, p.z, B, Tin,
                                                Tc, D, K, lpad, eps, vl, st));
    } else {
      const int T2 = chunk ? (Tin - K) / 2 + 1 : (Tc + 1) / 2;  // == ceil(Tc / 2), the pooled residual's length
      if (!chunk) PPASR_CUDA_CHECK(launch_halve_lens(p.vlen, p.vlen2, B, st));
      { PROF(PC_DWCONV);
        PPASR_CUDA_CHECK(launch_dwconv_stride(gin, w.dw_w, w.dw_b, pad_left, w.cn_g, w.cn_b, cfg.conv_norm == 0, p.z, B, Tin, T2,
                                              D, K, lpad, 2, eps, chunk ? nullptr : p.vlen2, st)); }
      // residual through AvgPool1D(2, 2, ceil_mode) (efficient_conformer/encoder.py:523-526)
      PPASR_CUDA_CHECK(launch_avgpool2(xc, p.x2, B, Tc, T2, D, st));
      if (chunk) PPASR_CUDA_CHECK(launch_halve_lens(p.vlen, p.vlen2, B, st));  // the CTC head's lengths: every row is valid
      xc = p.x2, Tc = T2, Mc = B * T2, vl = chunk ? nullptr : p.vlen2, tmpos = &c->tm_pos2, rate = 2;
    }
    // ---- x += mask * (pw2 z + b); y = norm_ff(x); FFN: x += 0.5 * W2 swish(W1 y); x = norm_final(x);
    //      y = next block's first LayerNorm (or after_norm)                                 (encoder.py:419-429, 201-202)
    {
      const float* g2 = (l + 1 < L) ? c->layers[l + 1].ln_ffm_g : c->after_g;
      const float* b2 = (l + 1 < L) ? c->layers[l + 1].ln_ffm_b : c->after_b;
      PROF(PC_FUSED_FFN);
      // pointwise_conv2 + residual + norm_ff chained in front (z rows of pad frames are zero, bias masked)
      PPASR_CUDA_CHECK(launch_fused_ffn(p.tm_z, &m.pw2, m.ff_w1_128, m.ff_w2s, Mc, FF, xc, p.y, w.ff_b1, w.ff_b2s, w.ln_fin_g,
                                        w.ln_fin_b, g2, b2, eps, w.pw2_b, w.ln_ff_g, w.ln_ff_b, vl, Tc, st));
    }
  }
  return PPASR_OK;
}

int copy_out(void* dst, const void* src_dev, size_t bytes, int on_device, cudaStream_t st) {
  if (!dst) return PPASR_OK;
  PPASR_CUDA_CHECK(cudaMemcpyAsync(dst, src_dev, bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  return PPASR_OK;
}

}  // namespace

extern "C" {

int ppasr_b200_encode(ppasr_b200_ctx* c, const float* feats, int32_t feats_on_device, const int64_t* lens_host,
                      int32_t B, int32_t T, void* stream) {
  PPASR_REQUIRE(c && feats && B > 0 && T > 0, "bad arguments");
  if (!c->finalized) {
    set_last_error("ppasr_b200_finalize has not been called");
    return PPASR_ERR_STATE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool ds2 = c->cfg.model_type == 2;
  int rc = ds2 ? build_plan_ds2(c, B, T) : build_plan(c, B, T);
  if (rc != PPASR_OK) return rc;
  Plan& p = c->plan;
  PPASR_CUDA_CHECK(cudaMemcpyAsync(p.feats, feats, (size_t)B * T * c->cfg.feat_dim * sizeof(float),
                                   feats_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  // valid subsampled frames: mask[:, :, :-2:2][:, :, :-2:2] keeps frame j iff 4*j < len (subsampling.py:115);
  // deepspeech2 uses x_len = ((len - 1) // 2 - 1) // 2 as the RNN sequence_length (deepspeech2/conv.py:20)
  if (c->h_vlen_cap < B) {
    if (c->capturing) {
      set_last_error("batch size grew inside a graph capture: run the step once before ppasr_b200_graph_begin");
      return PPASR_ERR_STATE;
    }
    PPASR_CUDA_CHECK(cudaDeviceSynchronize());  // an earlier copy (on any stream) may still read the old staging buffer
    if (c->h_vlen) cudaFreeHost(c->h_vlen);
    c->h_vlen = nullptr;
    PPASR_CUDA_CHECK(cudaMallocHost(&c->h_vlen, sizeof(int) * (size_t)B * 2));
    c->h_vlen_cap = B;
  }
  // two halves used alternately: the copy of the previous call may still be in flight when the next lengths are written
  int* vlen = c->h_vlen + (c->capturing ? 0 : ((c->vlen_flip ^= 1) ? c->h_vlen_cap : 0));
  for (int b = 0; b < B; ++b) {
    const int64_t len = lens_host ? lens_host[b] : T;
    int64_t v = ds2 ? ((len - 1) / 2 - 1) / 2 : (len + 3) / 4;
    if (v > p.Tp) v = p.Tp;
    if (v < 0) v = 0;
    vlen[b] = (int)v;
  }
  PPASR_CUDA_CHECK(cudaMemcpyAsync(p.vlen, vlen, sizeof(int) * B, cudaMemcpyHostToDevice, st));
  if (ds2) return run_encoder_ds2(c, st, false);
  return c->cfg.model_type == 1 ? run_encoder_squeezeformer(c, st) : run_encoder(c, st, false);
}

// ---- streaming ------------------------------------------------------------------------------------
int ppasr_b200_stream_reset(ppasr_b200_ctx* c, int32_t B) {
  PPASR_REQUIRE(c && B > 0 && B <= 1024, "bad arguments");
  if (!c->finalized) {
    set_last_error("ppasr_b200_finalize has not been called");
    return PPASR_ERR_STATE;
  }
  // the memsets below run on the legacy default stream while chunks run on caller streams (PyTorch streams are
  // non-blocking): a reset is rare, so order it against everything queued before and after with device-wide syncs
  struct SyncBothSides {
    SyncBothSides() { cudaDeviceSynchronize(); }
    ~SyncBothSides() { cudaDeviceSynchronize(); }
  } sync_both_sides;
  if (c->cfg.model_type == 2) {
    // zero LSTM / GRU states [L*nd, B, H] (inference_predictor.py:157-164)
    auto& ds = c->ds;
    const size_t n = (size_t)c->cfg.n_layers * ds.nd * B * c->cfg.d_model;
    if (ds.state_B != B || !ds.h_state) {
      PPASR_CUDA_CHECK(cudaDeviceSynchronize());
      if (ds.h_state) cudaFree(ds.h_state);
      if (ds.c_state) cudaFree(ds.c_state);
      ds.h_state = ds.c_state = nullptr;
      PPASR_CUDA_CHECK(cudaMalloc(&ds.h_state, n * 4));
      PPASR_CUDA_CHECK(cudaMalloc(&ds.c_state, n * 4));
      ds.state_B = B;
    }
    PPASR_CUDA_CHECK(cudaMemset(ds.h_state, 0, n * 4));
    PPASR_CUDA_CHECK(cudaMemset(ds.c_state, 0, n * 4));
    return PPASR_OK;
  }
  if (c->cfg.model_type != 0 && c->cfg.model_type != 1 && c->cfg.model_type != 3) {
    set_last_error("chunk streaming (forward_chunk) is implemented for conformer, squeezeformer, efficient_conformer and deepspeech2");
    return PPASR_ERR_STATE;
  }
  if (!c->cfg.causal) {
    set_last_error("chunk streaming needs a streaming (causal) model");
    return PPASR_ERR_STATE;
  }
  auto& ss = c->ss;
  const auto& cfg = c->cfg;
  const int L = cfg.n_layers, H = cfg.n_heads, D = cfg.d_model, lorder = cfg.conv_kernel - 1;
  if (ss.B != B || !ss.kk) {
    PPASR_CUDA_CHECK(cudaDeviceSynchronize());
    if (ss.kk) cudaFree(ss.kk);
    if (ss.vt) cudaFree(ss.vt);
    if (ss.cnn) cudaFree(ss.cnn);
    ss.kk = ss.vt = ss.cnn = nullptr;
    ss.Tcap = (cfg.max_len + 63) / 64 * 64;
    if (cfg.model_type == 3) {
      // grouped blocks: the key groups of the longest stream (kend < max_len frames, full rate), a multiple of 8 so the
      // V^T row pitch is a multiple of 16 bytes (TMA); their K / V^T views must fit the layer's slice of B*H*Tcap*64
      ss.Gcap = ((cfg.max_len + 1) / 3 + 7) / 8 * 8;
      ss.Tcap = std::max(ss.Tcap, (3 * ss.Gcap + 63) / 64 * 64);
      PPASR_REQUIRE((size_t)ss.Gcap * 192 <= (size_t)ss.Tcap * 64 && ss.Gcap * 2 % 16 == 0 && 3 * ss.Gcap >= cfg.max_len - 1,
                    "internal error: grouped cache capacity");
    }
    ss.gdirty = 0;
    const size_t n = (size_t)L * B * H * ss.Tcap * 64;
    PPASR_CUDA_CHECK(cudaMalloc(&ss.kk, n * 2));
    PPASR_CUDA_CHECK(cudaMalloc(&ss.vt, n * 2));
    PPASR_CUDA_CHECK(cudaMalloc(&ss.cnn, (size_t)L * B * lorder * D * 2));
    PPASR_CUDA_CHECK(cudaMemset(ss.kk, 0, n * 2));
    PPASR_CUDA_CHECK(cudaMemset(ss.vt, 0, n * 2));
    ss.B = B;
    ss.tm_k.resize(L);
    ss.tm_vt.resize(L);
  }
  // empty conv cache == the reference's zero left padding of the first chunk (convolution.py:109-110)
  PPASR_CUDA_CHECK(cudaMemset(ss.cnn, 0, (size_t)L * B * lorder * D * 2));
  if (cfg.model_type == 3) {
    // grouped blocks append into zeroed caches: the missing frames of a partially filled last group must read as zero.
    // Only the grouped blocks read beyond what was written (the plain blocks are bounded by the tensor-map extents), and
    // only groups [0, gdirty) of each (b, h) have been written since the caches were last zero, so only those are cleared:
    // the leading gdirty of every Gcap-group K row block and of every V^T row
    const size_t slice = (size_t)B * H * ss.Tcap * 64;
    for (int l = 0; l < L && ss.gdirty > 0; ++l) {
      if (!((c->eff_group_mask >> l) & 1)) continue;
      PPASR_CUDA_CHECK(cudaMemset2D(ss.kk + (size_t)l * slice, (size_t)ss.Gcap * 192 * 2, 0, (size_t)ss.gdirty * 192 * 2,
                                    (size_t)B * H));
      PPASR_CUDA_CHECK(cudaMemset2D(ss.vt + (size_t)l * slice, (size_t)ss.Gcap * 2, 0, (size_t)ss.gdirty * 2, (size_t)B * H * 192));
    }
    ss.gdirty = 0;
    if (!ss.pgc) {  // rows past a chunk's keys are masked; zero them once so they hold finite values
      PPASR_CUDA_CHECK(cudaMalloc(&ss.pgc, (size_t)4 * ss.Gcap * 768 * 2));
      PPASR_CUDA_CHECK(cudaMemset(ss.pgc, 0, (size_t)4 * ss.Gcap * 768 * 2));
    }
  }
  ss.kstart = ss.kend = ss.offset = 0;
  return PPASR_OK;
}

int ppasr_b200_encode_chunk(ppasr_b200_ctx* c, const float* feats, int32_t feats_on_device, int32_t B, int32_t t,
                            int32_t required_cache_size, void* stream) {
  PPASR_REQUIRE(c && feats && B > 0 && t > 0, "bad arguments");
  if (c->cfg.model_type == 2) {
    // predict_chunk_deepspeech (inference_predictor.py:147-182): every row of the chunk is valid; states carry over
    if (c->ds.state_B != B || !c->ds.h_state) {
      int rc0 = ppasr_b200_stream_reset(c, B);
      if (rc0) return rc0;
    }
    cudaStream_t st2 = reinterpret_cast<cudaStream_t>(stream);
    int rc2 = build_plan_ds2(c, B, t);
    if (rc2 != PPASR_OK) return rc2;
    Plan& p2 = c->plan;
    PPASR_CUDA_CHECK(cudaMemcpyAsync(p2.feats, feats, (size_t)B * t * c->cfg.feat_dim * sizeof(float),
                                     feats_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st2));
    std::vector<int> vlen(B, p2.Tp);
    PPASR_CUDA_CHECK(cudaMemcpyAsync(p2.vlen, vlen.data(), sizeof(int) * B, cudaMemcpyHostToDevice, st2));
    return run_encoder_ds2(c, st2, true);
  }
  auto& ss = c->ss;
  if (ss.B != B || !ss.kk) {
    int rc = ppasr_b200_stream_reset(c, B);
    if (rc) return rc;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int rc = build_plan(c, B, t);
  if (rc != PPASR_OK) return rc;
  Plan& p = c->plan;
  const auto& cfg = c->cfg;
  const int H = cfg.n_heads, L = cfg.n_layers;
  if (ss.kend + p.Tp > ss.Tcap || ss.offset + p.Tp >= cfg.max_len) {
    set_last_error("stream longer than the positional table (max_len); call reset_stream (embedding.py:64-66)");
    return PPASR_ERR_STATE;
  }
  PPASR_CUDA_CHECK(cudaMemcpyAsync(p.feats, feats, (size_t)B * t * cfg.feat_dim * sizeof(float),
                                   feats_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  {
    std::vector<int> vlen(B, p.Tp);
    PPASR_CUDA_CHECK(cudaMemcpyAsync(p.vlen, vlen.data(), sizeof(int) * B, cudaMemcpyHostToDevice, st));
  }
  const bool sqz = cfg.model_type == 1;
  const int kend_new = ss.kend + p.Tp;
  if (sqz && c->sq.reduce_idx >= 0) {
    // the half-rate blocks address their caches / positions at half rate (runtime_squeezeformer.inl)
    // (an odd number of frames is fine for the LAST chunk of a stream: the state it leaves behind is not used again)
    PPASR_REQUIRE(ss.kend % 2 == 0 && ss.kstart % 2 == 0 && ss.offset % 2 == 0 &&
                      (required_cache_size < 0 || required_cache_size % 2 == 0),
                  "squeezeformer chunk streaming needs even chunk sizes (all but the last chunk) and an even required_cache_size");
  }
  if (cfg.model_type == 3) {
    // forward_chunk of the Efficient Conformer: append-only caches (run_encoder)
    PPASR_REQUIRE(required_cache_size < 0, "efficient_conformer streaming keeps the whole history (required_cache_size < 0, "
                                           "as PPASRPredictor passes, predict.py:304-306)");
    PPASR_REQUIRE(c->eff_stride_idx < 0 || ss.kend % 2 == 0,
                  "efficient_conformer chunk streaming needs even chunk sizes (all but the last chunk of a stream)");
    ss.gdirty = std::max(ss.gdirty, (kend_new + 2) / 3);  // groups this chunk's grouped QKV epilogues write into
  }
  // per-layer cache maps with extent = keys valid after this chunk (TMA zero-fills beyond)
  std::string err;
  int gi = 0;
  for (int l = 0; l < L; ++l) {
    const size_t lk = (size_t)l * B * H * ss.Tcap * 64;
    // half rate: the Squeezeformer's time-reduced section, the blocks after the Efficient Conformer's stride block
    const bool half = sqz ? (c->sq.reduce_idx >= 0 && l >= c->sq.reduce_idx && l < c->sq.recover_idx)
                          : (c->eff_stride_idx >= 0 && l > c->eff_stride_idx);
    const int rate = half ? 2 : 1;
    const int kv = (kend_new + rate - 1) / rate;  // keys valid after this chunk, at the block's rate
    bool ok;
    if ((c->eff_group_mask >> l) & 1) {
      ok = gi < 4 && make_tmap_2d(&ss.tm_k[l], ss.kk + lk, 192, (uint64_t)B * H * ss.Gcap, 192 * 2, 64, &err) &&
           make_tmap_2d(&ss.tm_vt[l], ss.vt + lk, (uint64_t)((kv + 2) / 3), (uint64_t)B * H * 192, (uint64_t)ss.Gcap * 2, 192, &err) &&
           make_tmap_2d(&ss.tm_pgc[gi], ss.pgc + (size_t)gi * ss.Gcap * 768, 768, ss.Gcap, 768 * 2, 64, &err);
      if (gi >= 4) err = "more than 4 grouped blocks are not supported";
      ++gi;
    } else {
      ok = make_tmap_2d(&ss.tm_k[l], ss.kk + lk, 64, (uint64_t)B * H * ss.Tcap, 128, 128, &err) &&
           make_tmap_2d(&ss.tm_vt[l], ss.vt + lk, kv, (uint64_t)B * H * 64, (uint64_t)ss.Tcap * 2, 64, &err);
    }
    if (!ok) {
      set_last_error(err);
      return PPASR_ERR_CUDA;
    }
  }
  if (c->eff_group_mask != 0 &&
      !make_tmap_2d(&ss.tm_qgc, p.q2g, 384, (uint64_t)B * H * ((p.Tp + 2) / 3), 384 * 2, 128, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  rc = sqz ? run_encoder_squeezeformer(c, st, true) : run_encoder(c, st, true);
  if (rc) return rc;
  // cache bookkeeping (encoder.py:255-260,272): keep everything (<0), nothing (0) or the last `required` keys
  ss.kend = kend_new;
  ss.offset += p.Tp;
  if (required_cache_size == 0)
    ss.kstart = ss.kend;
  else if (required_cache_size > 0 && ss.kend - ss.kstart > required_cache_size)
    ss.kstart = ss.kend - required_cache_size;
  return PPASR_OK;
}

// ---- ragged streaming sessions (SURVEY 8f rank 3: many independent streams stepped in one batch) --------------------
int ppasr_b200_sessions_init(ppasr_b200_ctx* c, int32_t max_sessions) {
  PPASR_REQUIRE(c && max_sessions > 0 && max_sessions <= 1024, "bad arguments");
  PPASR_REQUIRE(c->cfg.model_type == 0, "sessions are implemented for the conformer");
  int rc = ppasr_b200_stream_reset(c, max_sessions);  // caches for max_sessions slots, zeroed
  if (rc) return rc;
  auto& ss = c->ss;
  ss.s_kstart.assign(max_sessions, 0);
  ss.s_kend.assign(max_sessions, 0);
  ss.s_offset.assign(max_sessions, 0);
  if (ss.d_step) cudaFree(ss.d_step);
  ss.d_step = nullptr;
  PPASR_CUDA_CHECK(cudaMalloc(&ss.d_step, sizeof(int) * 5 * max_sessions));
  return PPASR_OK;
}

int ppasr_b200_sessions_reset(ppasr_b200_ctx* c, int32_t slot) {
  PPASR_REQUIRE(c && c->ss.d_step && slot >= 0 && slot < c->ss.B, "bad slot (call sessions_init first)");
  auto& ss = c->ss;
  const auto& cfg = c->cfg;
  const int lorder = cfg.conv_kernel - 1, D = cfg.d_model;
  ss.s_kstart[slot] = ss.s_kend[slot] = ss.s_offset[slot] = 0;
  // ordered against the steps queued on caller (non-blocking) streams before and after: a slot is recycled rarely
  PPASR_CUDA_CHECK(cudaDeviceSynchronize());
  for (int l = 0; l < cfg.n_layers; ++l)  // empty conv cache == zero left padding of the first chunk
    PPASR_CUDA_CHECK(cudaMemset(ss.cnn + ((size_t)l * ss.B + slot) * lorder * D, 0, (size_t)lorder * D * 2));
  PPASR_CUDA_CHECK(cudaDeviceSynchronize());
  return PPASR_OK;
}

int ppasr_b200_sessions_step(ppasr_b200_ctx* c, const float* feats, int32_t feats_on_device, const int32_t* slots, int32_t n,
                             int32_t t, int32_t required_cache_size, void* stream) {
  PPASR_REQUIRE(c && feats && slots && n > 0 && t > 0, "bad arguments");
  auto& ss = c->ss;
  PPASR_REQUIRE(ss.d_step && n <= ss.B, "call ppasr_b200_sessions_init with enough slots first");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int rc = build_plan(c, n, t);
  if (rc != PPASR_OK) return rc;
  Plan& p = c->plan;
  const auto& cfg = c->cfg;
  const int H = cfg.n_heads, L = cfg.n_layers, S = ss.B;
  std::vector<int> step(5 * n);
  int T2max = 0;
  for (int b = 0; b < n; ++b) {
    const int s = slots[b];
    PPASR_REQUIRE(s >= 0 && s < S, "slot out of range");
    for (int q = 0; q < b; ++q) PPASR_REQUIRE(slots[q] != s, "a slot may appear only once per step");
    if (ss.s_kend[s] + p.Tp > ss.Tcap || ss.s_offset[s] + p.Tp >= cfg.max_len) {
      set_last_error("session longer than the positional table (max_len); reset it");
      return PPASR_ERR_STATE;
    }
    const int cache_t = ss.s_kend[s] - ss.s_kstart[s];
    step[b] = s;
    step[n + b] = ss.s_kend[s];
    step[2 * n + b] = ss.s_kstart[s];
    step[3 * n + b] = ss.s_offset[s] - cache_t;
    step[4 * n + b] = cache_t + p.Tp;
    T2max = std::max(T2max, cache_t + p.Tp);
  }
  PPASR_CUDA_CHECK(cudaMemcpyAsync(p.feats, feats, (size_t)n * t * cfg.feat_dim * sizeof(float),
                                   feats_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  PPASR_CUDA_CHECK(cudaMemcpyAsync(ss.d_step, step.data(), sizeof(int) * 5 * n, cudaMemcpyHostToDevice, st));
  {
    std::vector<int> vlen(n, p.Tp);
    PPASR_CUDA_CHECK(cudaMemcpyAsync(p.vlen, vlen.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
  }
  std::string err;
  for (int l = 0; l < L; ++l) {  // whole-capacity maps: validity comes from the per-session key counts
    const size_t lk = (size_t)l * S * H * ss.Tcap * 64;
    if (!make_tmap_2d(&ss.tm_k[l], ss.kk + lk, 64, (uint64_t)S * H * ss.Tcap, 128, 128, &err) ||
        !make_tmap_2d(&ss.tm_vt[l], ss.vt + lk, ss.Tcap, (uint64_t)S * H * 64, (uint64_t)ss.Tcap * 2, 64, &err)) {
      set_last_error(err);
      return PPASR_ERR_CUDA;
    }
  }
  ss.ragged = true;
  ss.step_T2 = T2max;
  rc = run_encoder(c, st, true);
  ss.ragged = false;
  if (rc) return rc;
  for (int b = 0; b < n; ++b) {  // cache bookkeeping per session (encoder.py:255-260,272)
    const int s = slots[b];
    ss.s_kend[s] += p.Tp;
    ss.s_offset[s] += p.Tp;
    if (required_cache_size == 0)
      ss.s_kstart[s] = ss.s_kend[s];
    else if (required_cache_size > 0 && ss.s_kend[s] - ss.s_kstart[s] > required_cache_size)
      ss.s_kstart[s] = ss.s_kend[s] - required_cache_size;
  }
  return PPASR_OK;
}

int ppasr_b200_ds2_states(ppasr_b200_ctx* c, float* h, float* cc, int32_t on_device, void* stream) {
  PPASR_REQUIRE(c && c->cfg.model_type == 2, "deepspeech2 context required");
  PPASR_REQUIRE(c->ds.h_state, "no stream state (call stream_reset / encode_chunk first)");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t n = (size_t)c->cfg.n_layers * c->ds.nd * c->ds.state_B * c->cfg.d_model * 4;
  const cudaMemcpyKind k = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (h) PPASR_CUDA_CHECK(cudaMemcpyAsync(h, c->ds.h_state, n, k, st));
  if (cc) PPASR_CUDA_CHECK(cudaMemcpyAsync(cc, c->ds.c_state, n, k, st));
  if (!on_device) PPASR_CUDA_CHECK(cudaStreamSynchronize(st));
  return PPASR_OK;
}

int ppasr_b200_stream_info(ppasr_b200_ctx* c, int32_t* offset, int32_t* cache_t) {
  PPASR_REQUIRE(c, "null ctx");
  if (offset) *offset = c->ss.offset;
  if (cache_t) *cache_t = c->ss.kend - c->ss.kstart;
  return PPASR_OK;
}

int ppasr_b200_stream_export(ppasr_b200_ctx* c, float* att_cache, float* cnn_cache, int32_t on_device, void* stream) {
  PPASR_REQUIRE(c && c->ss.kk, "no stream state");
  PPASR_REQUIRE(c->cfg.model_type == 0, "cache export in the reference layout is implemented for the conformer only");
  auto& ss = c->ss;
  const auto& cfg = c->cfg;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int L = cfg.n_layers, H = cfg.n_heads, D = cfg.d_model, lorder = cfg.conv_kernel - 1;
  const int t = ss.kend - ss.kstart;
  float* tmp = nullptr;
  const size_t na = (size_t)L * H * t * 128, nc = (size_t)L * D * lorder;
  if (!on_device) PPASR_CUDA_CHECK(cudaMalloc(&tmp, (na + nc) * 4 + 16));
  float* da = on_device ? att_cache : tmp;
  float* dc = on_device ? cnn_cache : tmp + na;
  for (int l = 0; l < L; ++l) {
    const size_t lk = (size_t)l * ss.B * H * ss.Tcap * 64;
    if (att_cache && t > 0)
      PPASR_CUDA_CHECK(launch_export_att_cache(ss.kk + lk, ss.vt + lk, da + (size_t)l * H * t * 128, H, ss.Tcap, ss.Tcap,
                                               ss.kstart, t, st));
    if (cnn_cache)
      PPASR_CUDA_CHECK(launch_export_cnn_cache(ss.cnn + (size_t)l * ss.B * lorder * D, dc + (size_t)l * D * lorder, lorder, D, st));
  }
  if (!on_device) {
    if (att_cache && t > 0) PPASR_CUDA_CHECK(cudaMemcpyAsync(att_cache, da, na * 4, cudaMemcpyDeviceToHost, st));
    if (cnn_cache) PPASR_CUDA_CHECK(cudaMemcpyAsync(cnn_cache, dc, nc * 4, cudaMemcpyDeviceToHost, st));
    PPASR_CUDA_CHECK(cudaStreamSynchronize(st));
    cudaFree(tmp);
  }
  return PPASR_OK;
}

static int run_ctc_logits(ppasr_b200_ctx* c, cudaStream_t st) {
  Plan& p = c->plan;
  EpiLogitsF32<BN_NARROW> e{p.logits, c->ctc_b, c->Vld, p.Mc, c->cfg.vocab_size};
  PROF(PC_CTC_LOGITS);
  PPASR_CUDA_CHECK((gemm<BN_NARROW, ST_NARROW>(c, p.tm_y, c->tm_ctc_w, p.Mc, c->cfg.vocab_size, c->ctc_k, e, st)));
  return PPASR_OK;
}

int ppasr_b200_ctc_logits(ppasr_b200_ctx* c, float* logits, int32_t on_device, void* stream) {
  PPASR_REQUIRE(c && logits && c->plan.Mc > 0, "encode first");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int rc = run_ctc_logits(c, st);
  if (rc) return rc;
  Plan& p = c->plan;
  PPASR_CUDA_CHECK(cudaMemcpy2DAsync(logits, (size_t)c->cfg.vocab_size * 4, p.logits, (size_t)c->Vld * 4,
                                     (size_t)c->cfg.vocab_size * 4, p.Mc,
                                     on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  if (!on_device) PPASR_CUDA_CHECK(cudaStreamSynchronize(st));
  return PPASR_OK;
}

int ppasr_b200_ctc_probs(ppasr_b200_ctx* c, float* probs, int32_t probs_on_device, void* stream) {
  PPASR_REQUIRE(c && probs && c->plan.Mc > 0, "encode first");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int rc = run_ctc_logits(c, st);
  if (rc) return rc;
  Plan& p = c->plan;
  float* dst = probs_on_device ? probs : p.probs;
  { PROF(PC_SOFTMAX);
  PPASR_CUDA_CHECK(launch_softmax_rows(p.logits, c->Vld, dst, p.Mc, c->cfg.vocab_size, st)); }
  if (!probs_on_device) {
    PPASR_CUDA_CHECK(cudaMemcpyAsync(probs, p.probs, (size_t)p.Mc * c->cfg.vocab_size * 4, cudaMemcpyDeviceToHost, st));
    PPASR_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  return PPASR_OK;
}

int ppasr_b200_ctc_greedy(ppasr_b200_ctx* c, int32_t* ids, int32_t* out_lens, float* scores, int32_t* frame_ids,
                          float* frame_probs, int32_t outputs_on_device, int32_t trim_to_lens, int32_t blank_id,
                          void* stream) {
  PPASR_REQUIRE(c && c->plan.Mc > 0, "encode first");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  Plan& p = c->plan;
  const int V = c->cfg.vocab_size;
  EpiCtcStats<BN_NARROW> e{p.pmax, p.parg, p.psum, c->ctc_b, p.Mc, V, c->ctc_parts};
  { PROF(PC_CTC_STATS);
  PPASR_CUDA_CHECK((gemm<BN_NARROW, ST_NARROW>(c, p.tm_y, c->tm_ctc_w, p.Mc, V, c->ctc_k, e, st))); }
  { PROF(PC_CTC_FINALIZE);
  PPASR_CUDA_CHECK(launch_ctc_stats_finalize(p.pmax, p.parg, p.psum, c->ctc_parts, p.Mc, p.idx, p.maxp, st)); }
  PROF(PC_CTC_COLLAPSE);
  PPASR_CUDA_CHECK(launch_ctc_collapse(p.idx, p.maxp, p.B, p.Tc, trim_to_lens ? p.vc : nullptr, blank_id, p.ids, p.Tc,
                                       p.out_len, p.score, nullptr, nullptr, st));
  int rc;
  if ((rc = copy_out(ids, p.ids, (size_t)p.Mc * 4, outputs_on_device, st))) return rc;
  if ((rc = copy_out(out_lens, p.out_len, (size_t)p.B * 4, outputs_on_device, st))) return rc;
  if ((rc = copy_out(scores, p.score, (size_t)p.B * 4, outputs_on_device, st))) return rc;
  if ((rc = copy_out(frame_ids, p.idx, (size_t)p.Mc * 4, outputs_on_device, st))) return rc;
  if ((rc = copy_out(frame_probs, p.maxp, (size_t)p.Mc * 4, outputs_on_device, st))) return rc;
  if (!outputs_on_device && c->host_sync) PPASR_CUDA_CHECK(cudaStreamSynchronize(st));
  return PPASR_OK;
}

int ppasr_b200_greedy_decode(const float* probs, int32_t B, int32_t T, int32_t V, const int32_t* frame_lens,
                             int32_t blank_id, int32_t* ids, int32_t ld_ids, int32_t* out_lens, float* scores,
                             int32_t* tmp_idx, float* tmp_maxp, void* stream) {
  PPASR_REQUIRE(probs && ids && out_lens && scores && tmp_idx && tmp_maxp, "null pointer");
  PPASR_REQUIRE(B > 0 && T > 0 && V > 0 && ld_ids >= T, "bad sizes");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  PPASR_CUDA_CHECK(launch_argmax_rows(probs, V, B * T, tmp_idx, tmp_maxp, st));
  PPASR_CUDA_CHECK(launch_ctc_collapse(tmp_idx, tmp_maxp, B, T, frame_lens, blank_id, ids, ld_ids, out_lens, scores,
                                       nullptr, nullptr, st));
  return PPASR_OK;
}

// ---- CUDA graph of the steady-state step ------------------------------------------------------------------------------
// begin: the stream enters capture; every call made on it until end (encode, ctc_greedy with DEVICE outputs, ...) is recorded
// instead of run -- kernels with their programmatic-dependent-launch edges, the feature copy from the pointer passed at capture
// time, the valid-length copy from the context's pinned staging buffer. launch replays the whole step as one graph launch.
// The step must have run once with the same shapes before (workspace, function attributes), must not change shapes, and must not
// synchronise or copy to pageable host memory inside the capture.
int ppasr_b200_graph_begin(ppasr_b200_ctx* c, void* stream) {
  PPASR_REQUIRE(c && stream, "graph capture needs a non-default stream");
  PPASR_REQUIRE(!c->capturing && !c->profiling, "already capturing, or profiling is on");
  PPASR_REQUIRE(c->plan.M > 0 || c->plan.B > 0, "run the step once before capturing it");
  if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec), c->graph_exec = nullptr;
  if (c->graph) cudaGraphDestroy(c->graph), c->graph = nullptr;
  PPASR_CUDA_CHECK(cudaDeviceSynchronize());  // nothing in flight still reads the staging buffers the capture will rewrite
  PPASR_CUDA_CHECK(cudaStreamBeginCapture(reinterpret_cast<cudaStream_t>(stream), cudaStreamCaptureModeThreadLocal));
  c->capturing = true;
  c->capture_count0 = launch_count();
  return PPASR_OK;
}

int ppasr_b200_graph_end(ppasr_b200_ctx* c, void* stream) {
  PPASR_REQUIRE(c && c->capturing, "no capture in progress");
  c->capturing = false;
  cudaGraph_t g = nullptr;
  PPASR_CUDA_CHECK(cudaStreamEndCapture(reinterpret_cast<cudaStream_t>(stream), &g));
  c->graph = g;
  c->graph_kernels = launch_count() - c->capture_count0;
  add_launches(-c->graph_kernels);  // recorded, not run
  PPASR_CUDA_CHECK(cudaGraphInstantiate(&c->graph_exec, c->graph, 0));
  return PPASR_OK;
}

int ppasr_b200_graph_launch(ppasr_b200_ctx* c, void* stream) {
  PPASR_REQUIRE(c && c->graph_exec, "no captured graph (ppasr_b200_graph_begin / _end first)");
  PPASR_CUDA_CHECK(cudaGraphLaunch(c->graph_exec, reinterpret_cast<cudaStream_t>(stream)));
  add_launches(c->graph_kernels);
  return PPASR_OK;
}

int32_t ppasr_b200_graph_kernels(const ppasr_b200_ctx* c) { return c ? (int32_t)c->graph_kernels : 0; }

int ppasr_b200_set_option(ppasr_b200_ctx* c, const char* name, int32_t value) {
  PPASR_REQUIRE(c && name, "null pointer");
  const std::string n(name);
  if (n == "host_sync") {
    c->host_sync = value != 0;
    return PPASR_OK;
  }
  if (n == "conv1_tc") {
    c->conv1_tc = value != 0;
    return PPASR_OK;
  }
  if (n == "ffn_split") {  // process-wide: which fused_ffn kernel launch_fused_ffn dispatches to
    PPASR_REQUIRE(set_ffn_split_mode(value), "ffn_split must be 1 or 2");
    return PPASR_OK;
  }
  if (n == "fused_conv") {
    PPASR_REQUIRE(value == 0 || value == 2, "fused_conv must be 0 or 2");
    c->fused_conv = value;
    return PPASR_OK;
  }
  set_last_error("unknown option: " + n);
  return PPASR_ERR_INVALID;
}

int ppasr_b200_profile_enable(ppasr_b200_ctx* c, int32_t enable) {
  PPASR_REQUIRE(c, "null ctx");
  c->profiling = enable != 0;
  c->prof_only = enable >= 2 ? enable - 2 : -1;  // enable = 2 + class id: profile that class only
  c->prof.clear();
  c->prof_used = 0;
  return PPASR_OK;
}

int ppasr_b200_profile_num_classes(void) { return PC_COUNT; }
const char* ppasr_b200_profile_class_name(int32_t cls) { return (cls >= 0 && cls < PC_COUNT) ? kProfNames[cls] : ""; }

int ppasr_b200_profile_read(ppasr_b200_ctx* c, int32_t* counts, float* total_ms) {
  PPASR_REQUIRE(c && counts && total_ms, "null pointer");
  PPASR_CUDA_CHECK(cudaDeviceSynchronize());
  for (int i = 0; i < PC_COUNT; ++i) counts[i] = 0, total_ms[i] = 0.f;
  for (auto& r : c->prof) {
    float ms = 0.f;
    PPASR_CUDA_CHECK(cudaEventElapsedTime(&ms, r.e0, r.e1));
    counts[r.cls] += 1;
    total_ms[r.cls] += ms;
  }
  c->prof.clear();
  c->prof_used = 0;
  return PPASR_OK;
}

int ppasr_b200_debug_copy_x(ppasr_b200_ctx* c, float* dst_device, void* stream) {
  PPASR_REQUIRE(c && dst_device && c->plan.M > 0, "encode first");
  PPASR_CUDA_CHECK(cudaMemcpyAsync(dst_device, c->plan.x, (size_t)c->plan.M * c->cfg.d_model * 4,
                                   cudaMemcpyDeviceToDevice, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

int ppasr_b200_debug_copy_phase(ppasr_b200_ctx* c, void* dst_device, int32_t* dims, void* stream) {
  PPASR_REQUIRE(c && dims && c->plan.M > 0, "encode first");
  PPASR_REQUIRE(c->cfg.model_type != 4 && c->plan.phase != nullptr, "no conv2d subsampling front end in this model");
  dims[0] = c->plan.B, dims[1] = c->plan.Th, dims[2] = c->FH, dims[3] = c->cfg.d_model;
  if (dst_device)
    PPASR_CUDA_CHECK(cudaMemcpyAsync(dst_device, c->plan.phase, (size_t)4 * c->plan.Mr * c->cfg.d_model * 2,
                                     cudaMemcpyDeviceToDevice, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

// ---- op-level wrappers ------------------------------------------------------------------------
int ppasr_b200_op_layernorm(float* x, void* y_bf16, const float* g1, const float* b1, const float* g2,
                            const float* b2, const int32_t* lens, int32_t T, int32_t M, int32_t D, float eps,
                            void* stream) {
  PPASR_REQUIRE(x && y_bf16 && g1 && b1, "null pointer");
  PPASR_CUDA_CHECK(launch_layernorm(x, (__nv_bfloat16*)y_bf16, g1, b1, g2, b2, lens, T, M, D, eps,
                                    reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

int ppasr_b200_op_dwconv(const void* g_bf16, const float* w, const float* bias, const float* pad_left,
                         const float* gamma, const float* beta, int32_t use_layer_norm, void* out_bf16, int32_t B,
                         int32_t Tin, int32_t Tout, int32_t C, int32_t K, int32_t lpad, float eps, void* stream) {
  PPASR_REQUIRE(g_bf16 && w && bias && gamma && beta && out_bf16, "null pointer");
  PPASR_CUDA_CHECK(launch_dwconv_norm_swish((const __nv_bfloat16*)g_bf16, w, bias, pad_left, gamma, beta, use_layer_norm,
                                            (__nv_bfloat16*)out_bf16, B, Tin, Tout, C, K, lpad, eps, nullptr,
                                            reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

int ppasr_b200_op_softmax(const float* logits, int32_t ldl, float* probs, int32_t M, int32_t V, void* stream) {
  PPASR_REQUIRE(logits && probs, "null pointer");
  PPASR_CUDA_CHECK(launch_softmax_rows(logits, ldl, probs, M, V, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

int ppasr_b200_op_attention(const void* q2, const void* kk, const void* vt, int32_t T2p, const void* pos,
                            int32_t pos_rows, int32_t pos_ld, int32_t pos_row0, int32_t pos_col0, void* out,
                            int32_t B, int32_t H, int32_t T1, int32_t T2, const int32_t* klens, void* stream) {
  PPASR_REQUIRE(q2 && kk && vt && pos && out, "null pointer");
  PPASR_REQUIRE(T2p % 8 == 0 && T2p >= T2 && pos_ld % 8 == 0, "T2p / pos_ld must be multiples of 8");
  std::string err;
  CUtensorMap tq, tk, tp, tv;
  if (!make_tmap_2d(&tq, q2, 128, (uint64_t)B * H * T1, 256, 128, &err) ||
      !make_tmap_2d(&tk, kk, 64, (uint64_t)B * H * T2, 128, 128, &err) ||
      !make_tmap_2d(&tp, pos, pos_ld, pos_rows, (uint64_t)pos_ld * 2, 128, &err) ||
      !make_tmap_2d(&tv, vt, T2, (uint64_t)B * H * 64, (uint64_t)T2p * 2, 64, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  AttnParams ap{};
  ap.B = B, ap.H = H, ap.T1 = T1, ap.T2 = T2, ap.q_rows_per_bh = T1, ap.k_rows_per_bh = T2, ap.k_row0 = 0;
  ap.pos_row0 = pos_row0, ap.pos_col0 = pos_col0, ap.D = H * 64, ap.klens = klens, ap.out = (__nv_bfloat16*)out;
  PPASR_CUDA_CHECK(launch_rel_attention(tq, tk, tp, tv, ap, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

int ppasr_b200_op_qkv_attention(const void* y, const void* wqkv, const float* bqkv, const float* pos_u, const float* pos_v,
                                const void* pos, int32_t pos_rows, int32_t pos_ld, int32_t pos_row0, int32_t pos_col0,
                                const int32_t* klens, int32_t B, int32_t T, void* out, int32_t fused, void* stream) {
  PPASR_REQUIRE(y && wqkv && bqkv && pos_u && pos_v && pos && out, "null pointer");
  PPASR_REQUIRE(B > 0 && T > 0 && pos_ld % 8 == 0, "bad shape (pos_ld must be a multiple of 8)");
  const int D = 256, H = 4, M = B * T;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  std::string err;
  CUtensorMap ty, tp;
  if (!make_tmap_2d(&ty, y, D, M, (uint64_t)D * 2, GEMM_BLOCK_M, &err) ||
      !make_tmap_2d(&tp, pos, pos_ld, pos_rows, (uint64_t)pos_ld * 2, 128, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  if (fused) {
    CUtensorMap tw;
    if (!make_tmap_2d(&tw, wqkv, D, 3 * D, (uint64_t)D * 2, 64, &err)) {
      set_last_error(err);
      return PPASR_ERR_CUDA;
    }
    QkvAttnParams qp{B, H, T, D, pos_row0, pos_col0, bqkv, pos_u, pos_v, klens, (__nv_bfloat16*)out};
    PPASR_CUDA_CHECK(launch_qkv_rel_attention(ty, tw, tp, qp, st));
    return PPASR_OK;
  }
  // the QKV GEMM + rel_attention_kernel pair on scratch q2 / kk / vt laid out as in the offline plan
  const int Tkp = (T + 63) / 64 * 64;
  __nv_bfloat16 *q2 = nullptr, *kk = nullptr, *vt = nullptr;
  const size_t nq = (size_t)B * H * T * 128, nk = (size_t)B * H * T * 64, nv = (size_t)B * H * 64 * Tkp;
  PPASR_CUDA_CHECK(cudaMallocAsync(&q2, (nq + nk + nv) * 2, st));
  kk = q2 + nq, vt = kk + nk;
  int rc = PPASR_OK;
  CUtensorMap tw, tq, tk, tv;
  if (!make_tmap_2d(&tw, wqkv, D, 3 * D, (uint64_t)D * 2, BN_NARROW, &err) ||
      !make_tmap_2d(&tq, q2, 128, (uint64_t)B * H * T, 256, 128, &err) ||
      !make_tmap_2d(&tk, kk, 64, (uint64_t)B * H * T, 128, 128, &err) ||
      !make_tmap_2d(&tv, vt, T, (uint64_t)B * H * 64, (uint64_t)Tkp * 2, 64, &err)) {
    set_last_error(err);
    rc = PPASR_ERR_CUDA;
  } else {
    cudaError_t e = cudaMemsetAsync(vt, 0, nv * 2, st);
    EpiQKV<BN_NARROW> epi{q2, kk, vt, bqkv, pos_u, pos_v, M, T, H, T, Tkp, 0};
    if (e == cudaSuccess)
      e = launch_gemm<BN_NARROW, ST_NARROW, false>(ty, tw, make_shape(M, 3 * D, D, BN_NARROW), epi, device_sm_count(), st);
    AttnParams ap{};
    ap.B = B, ap.H = H, ap.T1 = T, ap.T2 = T, ap.q_rows_per_bh = T, ap.k_rows_per_bh = T, ap.k_row0 = 0;
    ap.pos_row0 = pos_row0, ap.pos_col0 = pos_col0, ap.D = D, ap.klens = klens, ap.out = (__nv_bfloat16*)out;
    if (e == cudaSuccess) e = launch_rel_attention(tq, tk, tp, tv, ap, st);
    if (e != cudaSuccess) {
      set_last_error(std::string("CUDA error: ") + cudaGetErrorString(e));
      rc = PPASR_ERR_CUDA;
    }
  }
  cudaFreeAsync(q2, st);
  return rc;
}

int ppasr_b200_op_grouped_attention(const void* q2g, const void* kk, int32_t k_pitch, const void* vt, int32_t vt_pitch,
                                    const void* pos, void* out, int32_t B, int32_t H, int32_t T, int32_t Tgk,
                                    const int32_t* klens, void* stream) {
  PPASR_REQUIRE(q2g && kk && vt && pos && out, "null pointer");
  PPASR_REQUIRE(B > 0 && H == 4 && T > 0 && Tgk > 0 && k_pitch >= Tgk && vt_pitch >= Tgk, "bad shape (H must be 4)");
  PPASR_REQUIRE(vt_pitch % 8 == 0, "vt_pitch must be a multiple of 8");
  const int Tg = (T + 2) / 3;
  std::string err;
  CUtensorMap tq, tk, tp, tv;
  if (!make_tmap_2d(&tq, q2g, 384, (uint64_t)B * H * Tg, 384 * 2, 128, &err) ||
      !make_tmap_2d(&tk, kk, 192, (uint64_t)B * H * k_pitch, 192 * 2, 64, &err) ||
      !make_tmap_2d(&tp, pos, 768, Tgk, 768 * 2, 64, &err) ||
      !make_tmap_2d(&tv, vt, Tgk, (uint64_t)B * H * 192, (uint64_t)vt_pitch * 2, 192, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  GroupedAttnParams gp{B, H, T, Tg, klens, (__nv_bfloat16*)out};
  gp.Tgk = Tgk, gp.k_pitch = k_pitch;
  PPASR_CUDA_CHECK(launch_grouped_attention(tq, tk, tp, tv, gp, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

}  // extern "C"
