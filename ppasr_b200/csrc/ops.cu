// Op-level C-ABI entry points: each hot-path kernel callable on raw device pointers.
// Used by the parity tests (kernel vs oracle) and by bench.py's per-kernel roofline leg.
// The model-level entry points (ppasr_b200_create / encode / decode ...) live in runtime.cu.
#include "common.h"
#include "gemm.cuh"
#include "kernels.h"
#include "ppasr_b200.h"
#include "tmap.h"

#include <atomic>
#include <cstdlib>
#include <mutex>

namespace ppasr {

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* get_last_error() { return g_last_error.c_str(); }

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }
void add_launches(long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static std::atomic<int> g_pdl{-1};
bool pdl_enabled() {
  int v = g_pdl.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("PPASR_B200_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
    g_pdl.store(v, std::memory_order_relaxed);
  }
  return v != 0;
}
void set_pdl_enabled(bool on) { g_pdl.store(on ? 1 : 0, std::memory_order_relaxed); }

int device_sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return 148;
    sms = prop.multiProcessorCount;
  }
  return sms;
}

GemmShape make_shape(int M, int N, int K, int block_n) {
  GemmShape s;
  s.M = M;
  s.N = N;
  s.num_k_blocks = K / GEMM_BLOCK_K;
  s.num_m_tiles = (M + GEMM_BLOCK_M - 1) / GEMM_BLOCK_M;
  s.num_n_tiles = (N + block_n - 1) / block_n;
  s.conv_pitch = 0;
  s.conv_kc = 1;
  return s;
}

}  // namespace ppasr

using namespace ppasr;

extern "C" {

const char* ppasr_b200_last_error(void) { return get_last_error(); }

int ppasr_b200_abi_version(void) { return 3; }

int64_t ppasr_b200_launch_count(void) { return (int64_t)launch_count(); }

int ppasr_b200_set_pdl(int32_t enable) {
  set_pdl_enabled(enable != 0);
  return PPASR_OK;
}

int ppasr_b200_set_ffn_split(int32_t mode) {
  PPASR_REQUIRE(set_ffn_split_mode(mode), "ffn_split must be 1 or 2");
  return PPASR_OK;
}
int ppasr_b200_get_ffn_split(void) { return ffn_split_mode(); }

// C = epilogue(A[M,K] * W[N,K]^T + bias).  See include/ppasr_b200.h for the epilogue codes.
int ppasr_b200_op_linear(const void* a_bf16, int64_t lda, const void* w_bf16, int64_t w_rows, const float* bias,
                         void* out, int64_t ldo, int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t act,
                         float alpha, int32_t residual, const int32_t* lens, int32_t T, int32_t block_n, void* stream) {
  PPASR_REQUIRE(a_bf16 && w_bf16 && bias && out, "null pointer");
  PPASR_REQUIRE(M > 0 && N > 0 && K > 0 && K % GEMM_BLOCK_K == 0, "K must be a positive multiple of 64");
  PPASR_REQUIRE(block_n == 128 || block_n == 256, "block_n must be 128 or 256");
  PPASR_REQUIRE(w_rows >= ((N + block_n - 1) / block_n) * (int64_t)block_n, "weight rows must be padded to block_n");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  std::string err;
  CUtensorMap ta, tb;
  if (!make_tmap_2d(&ta, a_bf16, (uint64_t)K, (uint64_t)M, (uint64_t)lda * 2, GEMM_BLOCK_M, &err) ||
      !make_tmap_2d(&tb, w_bf16, (uint64_t)K, (uint64_t)w_rows, (uint64_t)K * 2, (uint32_t)block_n, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  GemmShape s = make_shape(M, N, K, block_n);
  const int sms = device_sm_count();
  cudaError_t e = cudaSuccess;
  switch (epilogue) {
    case 0: {  // bf16 store with activation
      if (block_n == 256) {
#define LAUNCH_STORE(ACT)                                                                       \
  {                                                                                             \
    EpiStoreBF16<256, ACT> epi{(__nv_bfloat16*)out, bias, (int)ldo, M, N};                      \
    e = launch_gemm<256, 4, false>(ta, tb, s, epi, sms, st);                                    \
  }
        if (act == ACT_NONE) LAUNCH_STORE(ACT_NONE) else if (act == ACT_RELU) LAUNCH_STORE(ACT_RELU) else LAUNCH_STORE(ACT_SWISH)
#undef LAUNCH_STORE
      } else {
#define LAUNCH_STORE(ACT)                                                                       \
  {                                                                                             \
    EpiStoreBF16<128, ACT> epi{(__nv_bfloat16*)out, bias, (int)ldo, M, N};                      \
    e = launch_gemm<128, 6, false>(ta, tb, s, epi, sms, st);                                    \
  }
        if (act == ACT_NONE) LAUNCH_STORE(ACT_NONE) else if (act == ACT_RELU) LAUNCH_STORE(ACT_RELU) else LAUNCH_STORE(ACT_SWISH)
#undef LAUNCH_STORE
      }
      break;
    }
    case 1: {  // fp32 residual update
      if (block_n == 256) {
        EpiResidF32<256> epi{(float*)out, bias, (int)ldo, M, N, alpha, residual, lens, T};
        e = launch_gemm<256, 4, false>(ta, tb, s, epi, sms, st);
      } else {
        EpiResidF32<128> epi{(float*)out, bias, (int)ldo, M, N, alpha, residual, lens, T};
        e = launch_gemm<128, 6, false>(ta, tb, s, epi, sms, st);
      }
      break;
    }
    case 2: {  // GLU over interleaved columns
      if (block_n == 256) {
        EpiGLU<256> epi{(__nv_bfloat16*)out, bias, (int)ldo, M, N};
        e = launch_gemm<256, 4, false>(ta, tb, s, epi, sms, st);
      } else {
        EpiGLU<128> epi{(__nv_bfloat16*)out, bias, (int)ldo, M, N};
        e = launch_gemm<128, 6, false>(ta, tb, s, epi, sms, st);
      }
      break;
    }
    case 3: {  // fp32 logits
      PPASR_REQUIRE(ldo % 4 == 0, "ldo must be a multiple of 4 for fp32 logits");
      if (block_n == 256) {
        EpiLogitsF32<256> epi{(float*)out, bias, (int)ldo, M, N};
        e = launch_gemm<256, 4, false>(ta, tb, s, epi, sms, st);
      } else {
        EpiLogitsF32<128> epi{(float*)out, bias, (int)ldo, M, N};
        e = launch_gemm<128, 6, false>(ta, tb, s, epi, sms, st);
      }
      break;
    }
    default:
      set_last_error("unknown epilogue code");
      return PPASR_ERR_INVALID;
  }
  PPASR_CUDA_CHECK(e);
  return PPASR_OK;
}

// ---- CTC prefix beam search (no external scorer) ---------------------------------------------------
int64_t ppasr_b200_beam_state_bytes(int32_t B, int32_t max_frames, int32_t beam) {
  return (int64_t)beam_state_stride(max_frames * beam + 1) * B;
}
int64_t ppasr_b200_beam_workspace_bytes(int32_t B, int32_t T) {
  return (int64_t)B * T * (4 + 8 * BEAM_MAX_TOPN) + 1024;
}
int ppasr_b200_beam_reset(void* states, int32_t B, int32_t max_frames, int32_t beam, void* stream) {
  PPASR_REQUIRE(states && B > 0 && max_frames > 0 && beam >= 1 && beam <= BEAM_MAX_BEAM, "bad arguments");
  PPASR_CUDA_CHECK(launch_beam_reset(states, B, max_frames * beam + 1, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}
int ppasr_b200_beam_advance(const float* probs, int32_t B, int32_t T, int32_t V, const int32_t* frame_lens,
                            int32_t beam, float cutoff_prob, int32_t cutoff_top_n, int32_t blank_id, void* states,
                            int32_t max_frames, void* workspace, void* stream) {
  PPASR_REQUIRE(probs && states && workspace, "null pointer");
  PPASR_REQUIRE(B > 0 && T > 0 && V > 1, "bad sizes");
  PPASR_REQUIRE(beam >= 1 && beam <= BEAM_MAX_BEAM, "beam_size must be in [1,512] in this build");
  PPASR_REQUIRE(cutoff_top_n >= 1 && V < 65535, "cutoff_top_n must be >= 1 and the vocabulary below 65535");
  PPASR_REQUIRE(max_frames >= 1, "max_frames must be >= 1");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int top_n = cutoff_top_n < BEAM_MAX_TOPN ? cutoff_top_n : BEAM_MAX_TOPN;
  int* cnt = reinterpret_cast<int*>(workspace);
  int* cid = cnt + (((size_t)B * T + 63) & ~size_t(63));
  float* clp = reinterpret_cast<float*>(cid + (size_t)B * T * BEAM_MAX_TOPN);
  PPASR_CUDA_CHECK(launch_ctc_prune(probs, V, B * T, cutoff_prob, top_n, cnt, cid, clp, st));
  PPASR_CUDA_CHECK(launch_beam_advance(cnt, cid, clp, B, T, frame_lens, beam, top_n < V ? top_n : V, blank_id, max_frames, states,
                                       max_frames * beam + 1, st));
  return PPASR_OK;
}
int ppasr_b200_beam_advance_lm(const float* probs, int32_t B, int32_t T, int32_t V, const int32_t* frame_lens, int32_t beam,
                               float cutoff_prob, int32_t cutoff_top_n, int32_t blank_id, void* states, int32_t max_frames,
                               void* workspace, const uint64_t* lm_keys, const uint32_t* lm_keys_hi, const float* lm_vals,
                               const int32_t* lm_in_vocab, int64_t lm_capacity, int32_t lm_order, float alpha, float beta,
                               void* stream) {
  PPASR_REQUIRE(probs && states && workspace && lm_keys && lm_vals && lm_in_vocab, "null pointer");
  PPASR_REQUIRE(B > 0 && T > 0 && V > 1 && V + 2 < 65536, "bad sizes (the scorer packs token ids in 16 bits)");
  PPASR_REQUIRE(beam >= 1 && beam <= BEAM_MAX_BEAM, "beam_size must be in [1,512] in this build");
  PPASR_REQUIRE(cutoff_top_n >= 1 && max_frames >= 1, "cutoff_top_n and max_frames must be >= 1");
  PPASR_REQUIRE(lm_order >= 1 && lm_order <= 5, "the scorer supports n-gram orders 1..5");
  PPASR_REQUIRE(lm_order <= 4 || lm_keys_hi != nullptr, "order-5 tables need lm_keys_hi (the oldest token of every 5-gram)");
  PPASR_REQUIRE(lm_capacity >= 2 && (lm_capacity & (lm_capacity - 1)) == 0, "lm_capacity must be a power of two");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int top_n = cutoff_top_n < BEAM_MAX_TOPN ? cutoff_top_n : BEAM_MAX_TOPN;
  int* cnt = reinterpret_cast<int*>(workspace);
  int* cid = cnt + (((size_t)B * T + 63) & ~size_t(63));
  float* clp = reinterpret_cast<float*>(cid + (size_t)B * T * BEAM_MAX_TOPN);
  PPASR_CUDA_CHECK(launch_ctc_prune(probs, V, B * T, cutoff_prob, top_n, cnt, cid, clp, st));
  BeamLm lm;
  lm.keys = reinterpret_cast<const unsigned long long*>(lm_keys);
  lm.keys_hi = lm_keys_hi;
  lm.vals = reinterpret_cast<const float2*>(lm_vals);
  lm.in_lm = lm_in_vocab;
  lm.mask = (unsigned)(lm_capacity - 1);
  lm.order = lm_order;
  lm.alpha = alpha, lm.beta = beta;
  PPASR_CUDA_CHECK(launch_beam_advance(cnt, cid, clp, B, T, frame_lens, beam, top_n < V ? top_n : V, blank_id, max_frames, states,
                                       max_frames * beam + 1, st, probs, V, &lm));
  return PPASR_OK;
}
int ppasr_b200_beam_result(const void* states, int32_t B, int32_t max_frames, int32_t beam, int32_t* out_ids,
                           int32_t lmax, int32_t* out_lens, float* out_scores, void* stream) {
  return ppasr_b200_beam_result_nbest(states, B, max_frames, beam, beam, out_ids, lmax, out_lens, out_scores, stream);
}
int ppasr_b200_beam_result_nbest(const void* states, int32_t B, int32_t max_frames, int32_t beam, int32_t nbest,
                                 int32_t* out_ids, int32_t lmax, int32_t* out_lens, float* out_scores, void* stream) {
  PPASR_REQUIRE(states && out_ids && out_lens && out_scores && lmax > 0, "bad arguments");
  PPASR_REQUIRE(B > 0 && beam >= 1 && beam <= BEAM_MAX_BEAM && nbest >= 1 && nbest <= beam, "bad sizes");
  PPASR_CUDA_CHECK(launch_beam_result(states, B, max_frames * beam + 1, nbest, out_ids, lmax, out_lens, out_scores,
                                      reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}
// pruning scan alone (per-kernel roofline: reads B*T*V*4 bytes once)
int ppasr_b200_op_ctc_prune(const float* probs, int32_t rows, int32_t V, float cutoff_prob, int32_t cutoff_top_n,
                            void* workspace, void* stream) {
  PPASR_REQUIRE(probs && workspace && rows > 0, "bad arguments");
  const int top_n = cutoff_top_n < BEAM_MAX_TOPN ? cutoff_top_n : BEAM_MAX_TOPN;
  int* cnt = reinterpret_cast<int*>(workspace);
  int* cid = cnt + (((size_t)rows + 63) & ~size_t(63));
  float* clp = reinterpret_cast<float*>(cid + (size_t)rows * BEAM_MAX_TOPN);
  PPASR_CUDA_CHECK(launch_ctc_prune(probs, V, rows, cutoff_prob, top_n, cnt, cid, clp, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

// Fused FFN block on raw pointers (plain mode): x += W2s swish(W1 y + b1) + b2s ; y_out = LN(x; g1, bn1) [; double]
int ppasr_b200_op_fused_ffn(const void* y_bf16, const void* w1_bf16, const void* w2s_bf16, float* x, void* y_out,
                            const float* b1, const float* b2s, const float* g1, const float* bn1, const float* g2,
                            const float* bn2, int32_t M, int32_t FF, float eps, void* stream) {
  PPASR_REQUIRE(y_bf16 && w1_bf16 && w2s_bf16 && x && y_out && b1 && b2s && g1 && bn1, "null pointer");
  PPASR_REQUIRE(M > 0 && FF >= 256 && FF % 128 == 0, "FF must be a multiple of 128 and at least 256");
  std::string err;
  CUtensorMap ta, t1, t2;
  if (!make_tmap_2d(&ta, y_bf16, 256, (uint64_t)M, 512, 128, &err) ||
      !make_tmap_2d(&t1, w1_bf16, 256, (uint64_t)FF, 512, 128, &err) ||
      !make_tmap_2d(&t2, w2s_bf16, (uint64_t)FF, 256, (uint64_t)FF * 2, 256, &err)) {
    set_last_error(err);
    return PPASR_ERR_CUDA;
  }
  PPASR_CUDA_CHECK(launch_fused_ffn(ta, nullptr, t1, t2, M, FF, x, (__nv_bfloat16*)y_out, b1, b2s, g1, bn1, g2, bn2, eps,
                                    nullptr, nullptr, nullptr, nullptr, 1, reinterpret_cast<cudaStream_t>(stream)));
  return PPASR_OK;
}

}  // extern "C"
