// Fused relative-position multi-head attention for sm_100a (tcgen05 + TMEM + TMA).
//
// Reference math (ppasr/model_utils/conformer/attention.py:198-262, 86-126):
//   S = ((q + u) k^T + (q + v) p^T) / sqrt(dk)          -- rel_shift is NOT applied (attention.py:256-258)
//   S[key >= klen] = -inf ; A = softmax(S) ; A[key >= klen] = 0 ; out = A V
// Because there is no rel_shift, S is one contraction over a 128-wide head dimension:
//   S = [q+u | q+v] . [k | p]^T, with p = linear_pos(pos_emb) independent of the batch.
//
// One CTA per (128-query tile, head, utterance). Per 128-key block:
//   control thread : TMA loads K, P(pos), V^T tiles  -> tcgen05.mma S = Qu.K^T + Qv.P^T   (TMEM cols 0..127)
//   256 softmax thr: two threads per query row (TMEM lane): warps w and w + 4 share a lane quadrant, each owns 64 of the
//                    128 key columns of a block and 32 of the 64 output dims. Two passes over the S row in TMEM (max --
//                    exchanged between the two halves through shared memory -- then exp2), probabilities written as bf16
//                    into 128B-swizzled smem (K-major A operand)
//   control thread : tcgen05.mma O_blk = Prob . V   (TMEM cols 128..191)
//   128 softmax thr: o_reg = o_reg * alpha + O_blk  (online soft-max rescale in registers)
// Scores never touch HBM. smem: Q 32 KB + (K|P, reused for the probabilities) 32 KB + V^T 16 KB.
#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"

namespace ppasr {

void count_launch();

constexpr int ATT_BM = 128;
constexpr int ATT_BN = 128;
constexpr int ATT_THREADS = 288;  // warps 0..7 softmax (TMEM lane quadrant = warp & 3, column half = warp >> 2), warp 8 control
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // one [128 x 64] bf16 swizzled tile = 16 KB
constexpr int ATT_SMEM_Q = 0;
constexpr int ATT_SMEM_KP = 2 * ATT_TILE_BYTES;         // K tile, P tile (later: probabilities half 0 / half 1)
constexpr int ATT_SMEM_V = 4 * ATT_TILE_BYTES;          // two [64 d x 64 keys] tiles = 16 KB
constexpr int ATT_SMEM_BAR = 5 * ATT_TILE_BYTES;
constexpr int ATT_SMEM_XCH = ATT_SMEM_BAR + 128;        // float [2][128]: row maxima / sums exchanged between the column halves
constexpr int ATT_SMEM_TOTAL = ATT_SMEM_XCH + 1024 + 1024;
constexpr int ATT_TMEM_COLS = 256;

__global__ void __launch_bounds__(ATT_THREADS, 2)
rel_attention_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                     const __grid_constant__ CUtensorMap tm_p, const __grid_constant__ CUtensorMap tm_vt,
                     const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_q = smem + ATT_SMEM_Q;
  uint8_t* s_kp = smem + ATT_SMEM_KP;
  uint8_t* s_v = smem + ATT_SMEM_V;
  uint64_t* bar_q_full = reinterpret_cast<uint64_t*>(smem + ATT_SMEM_BAR);
  uint64_t* bar_kv_full = bar_q_full + 1;
  uint64_t* bar_s_full = bar_q_full + 2;
  uint64_t* bar_p_ready = bar_q_full + 3;
  uint64_t* bar_o_full = bar_q_full + 4;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bar_q_full + 5);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q_tile = blockIdx.x;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int bh = b * p.H + h;
  const int kbh = (p.slots ? __ldg(p.slots + b) : b) * p.H + h;  // (slot, head) of the cached K / V rows
  const int k_row0 = p.k_row0s ? __ldg(p.k_row0s + b) : p.k_row0;
  const int pos_row0 = p.pos_row0s ? __ldg(p.pos_row0s + b) : p.pos_row0;
  const int row0 = q_tile * ATT_BM;
  const int klen = p.klens ? min(p.T2, __ldg(p.klens + b)) : p.T2;
  const int nblk = (p.T2 + ATT_BN - 1) / ATT_BN;

  if (warp_idx == 8) {
    if (elect_one()) {
      tma_prefetch_desc(&tm_q);
      tma_prefetch_desc(&tm_k);
      tma_prefetch_desc(&tm_p);
      tma_prefetch_desc(&tm_vt);
      mbar_init(bar_q_full, 1);
      mbar_init(bar_kv_full, 1);
      mbar_init(bar_s_full, 1);
      mbar_init(bar_p_ready, 256);
      mbar_init(bar_o_full, 1);
      fence_barrier_init();
      fence_proxy_async_smem();
    }
    __syncwarp();
    tmem_alloc<ATT_TMEM_COLS>(tmem_ptr_smem);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tmem_s = tmem_base;        // S: columns [0,128)
  const uint32_t tmem_o = tmem_base + 128;  // O_blk: columns [128,192)

  if (warp_idx == 8) {
    // ============================ control: TMA + MMA issue ============================
    if (elect_one()) {
      constexpr uint32_t idesc_qk = umma_idesc_bf16(128, 128);
      constexpr uint32_t idesc_pv = umma_idesc_bf16(128, 64);
      mbar_arrive_expect_tx(bar_q_full, 2 * ATT_TILE_BYTES);
      tma_load_2d(s_q, &tm_q, bar_q_full, 0, bh * p.q_rows_per_bh + row0);
      tma_load_2d(s_q + ATT_TILE_BYTES, &tm_q, bar_q_full, 64, bh * p.q_rows_per_bh + row0);
      for (int j = 0; j < nblk; ++j) {
        const int k0 = j * ATT_BN;
        if (j > 0) {
          mbar_wait(bar_o_full, (j - 1) & 1);  // PV(j-1) finished: probabilities + V^T smem are free
        }
        mbar_arrive_expect_tx(bar_kv_full, 3 * ATT_TILE_BYTES);
        tma_load_2d(s_kp, &tm_k, bar_kv_full, 0, kbh * p.k_rows_per_bh + k_row0 + k0);
        tma_load_2d(s_kp + ATT_TILE_BYTES, &tm_p, bar_kv_full, p.pos_col0 + h * 64, pos_row0 + k0);
        tma_load_2d(s_v, &tm_vt, bar_kv_full, k_row0 + k0, kbh * 64);
        tma_load_2d(s_v + ATT_TILE_BYTES / 2, &tm_vt, bar_kv_full, k_row0 + k0 + 64, kbh * 64);
        if (j == 0) mbar_wait(bar_q_full, 0);
        mbar_wait(bar_kv_full, j & 1);
        tc_fence_after();
        {
          const uint32_t qa = smem_u32(s_q), ka = smem_u32(s_kp);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_s, umma_desc_k_sw128(qa + k * 32), umma_desc_k_sw128(ka + k * 32), idesc_qk, k > 0);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_s, umma_desc_k_sw128(qa + ATT_TILE_BYTES + k * 32),
                      umma_desc_k_sw128(ka + ATT_TILE_BYTES + k * 32), idesc_qk, 1u);
        }
        umma_commit(bar_s_full);
        mbar_wait(bar_p_ready, j & 1);
        tc_fence_after();
        {
          const uint32_t pa = smem_u32(s_kp), va = smem_u32(s_v);
#pragma unroll
          for (int kh = 0; kh < 2; ++kh)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_o, umma_desc_k_sw128(pa + kh * ATT_TILE_BYTES + k * 32),
                        umma_desc_k_sw128(va + kh * (ATT_TILE_BYTES / 2) + k * 32), idesc_pv, (kh | k) != 0);
        }
        umma_commit(bar_o_full);
      }
    }
  } else {
    // ============================ softmax: two threads per query row ============================
    const int quad = warp_idx & 3;   // TMEM lanes 32*quad ..
    const int ch = warp_idx >> 2;    // column half: keys [64 ch, 64 ch + 64) of a block, output dims [32 ch, 32 ch + 32)
    const int r = quad * 32 + lane;
    const uint32_t lane_base = ((uint32_t)(quad * 32)) << 16;
    float* xch = reinterpret_cast<float*>(smem + ATT_SMEM_XCH);  // [2][128]
    const float sc = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
    float m_run = -INFINITY, l_run = 0.f;            // l_run: this thread's half of the row sum
    float o[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) o[i] = 0.f;

    for (int j = 0; j < nblk; ++j) {
      const int k0 = j * ATT_BN + ch * 64;
      mbar_wait(bar_s_full, j & 1);
      tc_fence_after();
      // pass 1: maximum over this thread's 64 columns, then over the row (exchange with the other half)
      float bm = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t rr[32];
        tmem_ld_32x32b_x32(tmem_s + lane_base + ch * 64 + c * 32, rr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const bool valid = (k0 + c * 32 + i) < klen;
          bm = fmaxf(bm, valid ? __uint_as_float(rr[i]) : -INFINITY);
        }
      }
      xch[ch * 128 + r] = bm;
      named_bar_sync(1, 256);
      bm = fmaxf(bm, xch[(ch ^ 1) * 128 + r]);
      const float m_new = fmaxf(m_run, bm * sc);
      const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
      const float alpha = exp2f(m_run - m_use);  // m_run = -inf -> 0
      // pass 2: probabilities -> bf16, swizzled K-major A operand in smem: this half's 64 keys are tile `ch`
      float bsum = 0.f;
      uint8_t* tile = s_kp + ch * ATT_TILE_BYTES + r * 128;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t rr[32];
        tmem_ld_32x32b_x32(tmem_s + lane_base + ch * 64 + c * 32, rr);
        tmem_ld_wait();
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int kk0 = k0 + c * 32 + 2 * i;
          float p0 = (kk0 < klen) ? exp2f(fmaf(__uint_as_float(rr[2 * i]), sc, -m_use)) : 0.f;
          float p1 = (kk0 + 1 < klen) ? exp2f(fmaf(__uint_as_float(rr[2 * i + 1]), sc, -m_use)) : 0.f;
          // accumulate the row sum from the bf16-rounded values actually used by the P.V MMA
          const __nv_bfloat162 pb = __floats2bfloat162_rn(p0, p1);
          bsum += __low2float(pb) + __high2float(pb);
          pk[i] = *reinterpret_cast<const uint32_t*>(&pb);
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int chunk = c * 4 + q4;  // 16-byte chunk index inside the 128-byte row
          *reinterpret_cast<uint4*>(tile + ((chunk ^ (r & 7)) << 4)) =
              make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
        }
      }
      l_run = l_run * alpha + bsum;
      m_run = m_new;
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive(bar_p_ready);
      // O_blk -> registers with rescale (this thread's 32 output dims)
      mbar_wait(bar_o_full, j & 1);
      tc_fence_after();
      {
        uint32_t ro[32];
        tmem_ld_32x32b_x32(tmem_o + lane_base + ch * 32, ro);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = fmaf(o[i], alpha, __uint_as_float(ro[i]));
      }
      tc_fence_before();
      named_bar_sync(1, 256);  // the exchange slots may be rewritten by the next block
    }
    // row sum = the two halves' sums (same rescaling history: both use the row maximum)
    xch[ch * 128 + r] = l_run;
    named_bar_sync(1, 256);
    l_run += xch[(ch ^ 1) * 128 + r];
    const int t = row0 + r;
    if (t < p.T1) {
      const float inv = l_run > 0.f ? 1.0f / l_run : 0.f;
      uint32_t pk[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) pk[i] = pack_bf16x2(o[2 * i] * inv, o[2 * i + 1] * inv);
      uint4* dst = reinterpret_cast<uint4*>(p.out + ((size_t)b * p.T1 + t) * p.D + h * 64 + ch * 32);
#pragma unroll
      for (int i = 0; i < 4; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 8) {
    tc_fence_after();
    tmem_dealloc<ATT_TMEM_COLS>(tmem_base);
  }
}

cudaError_t launch_rel_attention(const CUtensorMap& tm_q, const CUtensorMap& tm_k, const CUtensorMap& tm_p,
                                 const CUtensorMap& tm_vt, const AttnParams& p, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(rel_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         ATT_SMEM_TOTAL);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  dim3 grid((p.T1 + ATT_BM - 1) / ATT_BM, p.H, p.B);
  cudaError_t le = launch_pdl(rel_attention_kernel, grid, dim3(ATT_THREADS), (size_t)ATT_SMEM_TOTAL, st, tm_q, tm_k, tm_p, tm_vt, p);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

// ================================================================================================================
// QKV projection + relative-position attention in one kernel (offline blocks, T' <= 256, D = 256, H = 4).
//
// One CTA per (head, utterance) computes the head's q / k / v for all T' frames from y (the LayerNorm output the QKV
// GEMM reads) and then runs the attention above on them, so q2 / kk / vt never go through global memory.
//   phase A  control thread: TMA W_h (the head's 64 q, 64 k and 64 v rows of wqkv, K-major, resident) and the
//            utterance's <= 2 row tiles of y through a 4-stage ring; tcgen05.mma 128 x 192 x 16 per row tile into TMEM
//            (columns 256 r ..), k order as the QKV GEMM (four 64-wide k-blocks of four k = 16 steps).
//            512 soft-max threads: drain with EpiQKV's arithmetic (acc + bqkv, q + pos_bias_u / pos_bias_v, bf16) into
//            the operand tiles of phase B, which reuse phase A's shared memory: [q+u | q+v] and K as K-major 128B-swizzled
//            tiles, V^T as two [64 d x 64 keys] K-major tiles per key block (the layout the V^T TMA load gives).
//   phase B  rel_attention_kernel's per-block math, element for element, for both query tiles at once: group g
//            (warps 8 g .. 8 g + 7) owns query tile g with its own S (TMEM 256 g ..) and O_blk (256 g + 128 ..) and is
//            organised like rel_attention_kernel's 256 soft-max threads. Group 0 writes its probabilities over the
//            block's K | P tiles once both groups' S MMAs have read them; group 1 has a buffer of its own.
// Rows of the second y tile past T' (the next utterance, or TMA zero fill past M) only reach masked keys and queries
// that are not stored. The outputs are bit-identical to the QKV GEMM + rel_attention_kernel pair.
// smem: phase A W_h 96 KB + y ring 64 KB; phase B Q 64 KB + K 32 KB + V^T 32 KB + group 1's probabilities 32 KB;
// positional tiles 32 KB in both phases (loaded at the start). TMEM: 512 columns.
// ================================================================================================================
constexpr int QA_THREADS = 544;  // warps 0..15: two soft-max groups of 8 warps, warp 16: control
constexpr int QA_W = 0;                   // phase A: W_h, 4 k-blocks of [192 rows x 64] (24 KB each)
constexpr int QA_Y = 96 * 1024;           // phase A: y ring, 4 stages of [128 rows x 64]
constexpr int QA_POS = 160 * 1024;        // positional key tiles of blocks 0, 1 (later: group 0's probabilities, half 1)
constexpr int QA_Q = 0;                   // phase B: query tile g at 32 KB g: [q+u] then [q+v]
constexpr int QA_K = 64 * 1024;           // phase B: key tiles of blocks 0, 1 (later: group 0's probabilities, half 0)
constexpr int QA_V = 96 * 1024;           // phase B: V^T of block j at 16 KB j: two [64 d x 64 keys] tiles
constexpr int QA_P1 = 128 * 1024;         // phase B: group 1's probabilities, two [128 x 64] tiles
constexpr int QA_BAR = 192 * 1024;
constexpr int QA_XCH = QA_BAR + 256;      // float [2 groups][2 halves][128]
constexpr int QA_SMEM_TOTAL = QA_XCH + 2048 + 1024;
constexpr int QA_TMEM_COLS = 512;

__global__ void __launch_bounds__(QA_THREADS, 1)
qkv_rel_attention_kernel(const __grid_constant__ CUtensorMap tm_y, const __grid_constant__ CUtensorMap tm_w,
                         const __grid_constant__ CUtensorMap tm_p, const QkvAttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(smem + QA_BAR);
  uint64_t* bar_yf = bar_w + 1;     // [4] y stage full
  uint64_t* bar_ye = bar_w + 5;     // [4] y stage consumed
  uint64_t* bar_pos = bar_w + 9;
  uint64_t* bar_acc = bar_w + 10;   // projection accumulators complete
  uint64_t* bar_qkv = bar_w + 11;   // operand tiles written (512 arrivals)
  uint64_t* bar_s = bar_w + 12;     // [2] per group
  uint64_t* bar_pr = bar_w + 14;    // [2] probabilities written (256 arrivals)
  uint64_t* bar_o = bar_w + 16;     // [2] P.V complete
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bar_w + 18);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int h = blockIdx.x;
  const int b = blockIdx.y;
  const int T = p.T;
  const int nt = (T + 127) / 128;  // row tiles == query tiles == key blocks (1 or 2)
  const int klen = p.klens ? min(T, __ldg(p.klens + b)) : T;

  if (warp_idx == 16) {
    if (elect_one()) {
      tma_prefetch_desc(&tm_y);
      tma_prefetch_desc(&tm_w);
      tma_prefetch_desc(&tm_p);
      mbar_init(bar_w, 1);
      for (int i = 0; i < 4; ++i) {
        mbar_init(bar_yf + i, 1);
        mbar_init(bar_ye + i, 1);
      }
      mbar_init(bar_pos, 1);
      mbar_init(bar_acc, 1);
      mbar_init(bar_qkv, 512);
      for (int g = 0; g < 2; ++g) {
        mbar_init(bar_s + g, 1);
        mbar_init(bar_pr + g, 256);
        mbar_init(bar_o + g, 1);
      }
      fence_barrier_init();
      fence_proxy_async_smem();
    }
    __syncwarp();
    tmem_alloc<QA_TMEM_COLS>(tmem_ptr_smem);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  if (warp_idx == 16 && elect_one()) {
    // the weights are not written by the preceding kernels: start their load before the dependency wait
    mbar_arrive_expect_tx(bar_w, 12 * 8192);
    for (int kb = 0; kb < 4; ++kb)
      for (int part = 0; part < 3; ++part)
        tma_load_2d(smem + QA_W + kb * 24576 + part * 8192, &tm_w, bar_w, kb * 64, part * p.D + h * 64);
  }
  pdl_wait();
  pdl_launch_dependents();

  if (warp_idx == 16) {
    // ============================ control: TMA + MMA issue ============================
    if (elect_one()) {
      const int row0 = b * T;
      mbar_arrive_expect_tx(bar_pos, nt * ATT_TILE_BYTES);
      for (int j = 0; j < nt; ++j)
        tma_load_2d(smem + QA_POS + j * ATT_TILE_BYTES, &tm_p, bar_pos, p.pos_col0 + h * 64, p.pos_row0 + j * 128);
      // load i = 4 r + kb of the y ring: row tile r, k-block kb, stage i % 4
      const int nload = nt * 4;
      for (int i = 0; i < 4 && i < nload; ++i) {
        mbar_arrive_expect_tx(bar_yf + i, ATT_TILE_BYTES);
        tma_load_2d(smem + QA_Y + i * ATT_TILE_BYTES, &tm_y, bar_yf + i, i * 64, row0);
      }
      constexpr uint32_t idesc_proj = umma_idesc_bf16(128, 192);
      mbar_wait(bar_w, 0);
      for (int i = 0; i < nload; ++i) {
        const int s = i & 3, kb = i & 3, r = i >> 2;
        mbar_wait(bar_yf + s, (i >> 2) & 1);
        tc_fence_after();
        const uint32_t ya = smem_u32(smem + QA_Y + s * ATT_TILE_BYTES), wa = smem_u32(smem + QA_W + kb * 24576);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_base + r * 256, umma_desc_k_sw128(ya + k * 32), umma_desc_k_sw128(wa + k * 32), idesc_proj,
                    (kb | k) != 0);
        umma_commit(bar_ye + s);
        // refill the stage of load i - 1 (its MMAs were queued before this load's) with load i + 3
        if (i >= 1 && i + 3 < nload) {
          const int ps = (i - 1) & 3, li = i + 3;
          mbar_wait(bar_ye + ps, ((i - 1) >> 2) & 1);
          mbar_arrive_expect_tx(bar_yf + ps, ATT_TILE_BYTES);
          tma_load_2d(smem + QA_Y + ps * ATT_TILE_BYTES, &tm_y, bar_yf + ps, (li & 3) * 64, row0 + (li >> 2) * 128);
        }
      }
      umma_commit(bar_acc);
      // ---- phase B: the attention MMAs, as in rel_attention_kernel, for both query tiles
      constexpr uint32_t idesc_qk = umma_idesc_bf16(128, 128);
      constexpr uint32_t idesc_pv = umma_idesc_bf16(128, 64);
      mbar_wait(bar_pos, 0);
      mbar_wait(bar_qkv, 0);
      tc_fence_after();
      for (int j = 0; j < nt; ++j) {
        for (int g = 0; g < nt; ++g) {
          if (j > 0) mbar_wait(bar_o + g, (j - 1) & 1);  // PV(g, j-1) finished: group g has read S and O_blk
          tc_fence_after();
          const uint32_t qa = smem_u32(smem + QA_Q + g * 2 * ATT_TILE_BYTES);
          const uint32_t ka = smem_u32(smem + QA_K + j * ATT_TILE_BYTES), pa = smem_u32(smem + QA_POS + j * ATT_TILE_BYTES);
          const uint32_t tmem_s = tmem_base + g * 256;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_s, umma_desc_k_sw128(qa + k * 32), umma_desc_k_sw128(ka + k * 32), idesc_qk, k > 0);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_s, umma_desc_k_sw128(qa + ATT_TILE_BYTES + k * 32), umma_desc_k_sw128(pa + k * 32), idesc_qk, 1u);
          umma_commit(bar_s + g);
        }
        for (int g = 0; g < nt; ++g) {
          mbar_wait(bar_pr + g, j & 1);
          tc_fence_after();
          const uint32_t pt0 = smem_u32(smem + (g == 0 ? QA_K + j * ATT_TILE_BYTES : QA_P1));
          const uint32_t pt1 = smem_u32(smem + (g == 0 ? QA_POS + j * ATT_TILE_BYTES : QA_P1 + ATT_TILE_BYTES));
          const uint32_t va = smem_u32(smem + QA_V + j * ATT_TILE_BYTES);
          const uint32_t tmem_o = tmem_base + g * 256 + 128;
#pragma unroll
          for (int kh = 0; kh < 2; ++kh)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_o, umma_desc_k_sw128((kh ? pt1 : pt0) + k * 32),
                        umma_desc_k_sw128(va + kh * (ATT_TILE_BYTES / 2) + k * 32), idesc_pv, (kh | k) != 0);
          umma_commit(bar_o + g);
        }
      }
    }
  } else {
    const int g = warp_idx >> 3;        // group: projection row tile and query tile g
    const int quad = warp_idx & 3;      // TMEM lanes 32*quad ..
    const int ch = (warp_idx >> 2) & 1; // column half
    const int r = quad * 32 + lane;
    const uint32_t lane_base = ((uint32_t)(quad * 32)) << 16;
    // ============================ projection drain: EpiQKV's arithmetic ============================
    if (g < nt) {
      mbar_wait(bar_acc, 0);
      tc_fence_after();
      const int hd = h * 64;
      // 32-column chunks of the [q | k | v] accumulator: half 0 takes q0 q1 k0, half 1 takes k1 v0 v1
#pragma unroll 1
      for (int c = 0; c < 3; ++c) {
        const int cc = ch * 3 + c;
        const int which = cc >> 1, d0 = (cc & 1) * 32;
        uint32_t rr[32];
        tmem_ld_32x32b_x32(tmem_base + lane_base + g * 256 + cc * 32, rr);
        tmem_ld_wait();
        float v[32];
        const float* bias = p.bqkv + which * p.D + hd + d0;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(rr[j]) + __ldg(bias + j);
        if (which == 0) {
          uint8_t* qrow = smem + QA_Q + g * 2 * ATT_TILE_BYTES + r * 128;
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            uint32_t pu[4], pv[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int e = q4 * 8 + 2 * j;
              const float2 u = __ldg(reinterpret_cast<const float2*>(p.pos_u + hd + d0 + e));
              const float2 w = __ldg(reinterpret_cast<const float2*>(p.pos_v + hd + d0 + e));
              pu[j] = pack_bf16x2(v[e] + u.x, v[e + 1] + u.y);
              pv[j] = pack_bf16x2(v[e] + w.x, v[e + 1] + w.y);
            }
            const int sw = ((d0 >> 3) + q4) ^ (r & 7);
            *reinterpret_cast<uint4*>(qrow + (sw << 4)) = make_uint4(pu[0], pu[1], pu[2], pu[3]);
            *reinterpret_cast<uint4*>(qrow + ATT_TILE_BYTES + (sw << 4)) = make_uint4(pv[0], pv[1], pv[2], pv[3]);
          }
        } else if (which == 1) {
          uint8_t* krow = smem + QA_K + g * ATT_TILE_BYTES + r * 128;
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const int e = q4 * 8;
            const int sw = ((d0 >> 3) + q4) ^ (r & 7);
            *reinterpret_cast<uint4*>(krow + (sw << 4)) =
                make_uint4(pack_bf16x2(v[e], v[e + 1]), pack_bf16x2(v[e + 2], v[e + 3]), pack_bf16x2(v[e + 4], v[e + 5]),
                           pack_bf16x2(v[e + 6], v[e + 7]));
          }
        } else {
          // V^T: key r of block g is column r % 64 of tile r / 64; row d = d0 + j
          uint8_t* vtile = smem + QA_V + g * ATT_TILE_BYTES + (r >> 6) * (ATT_TILE_BYTES / 2);
          const int kc = r & 63;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int d = d0 + j;
            *reinterpret_cast<__nv_bfloat16*>(vtile + d * 128 + ((((kc >> 3) ^ (d & 7))) << 4) + (kc & 7) * 2) =
                __float2bfloat16_rn(v[j]);
          }
        }
      }
    }
    tc_fence_before();
    fence_proxy_async_smem();
    mbar_arrive(bar_qkv);

    // ============================ soft-max: rel_attention_kernel's per-thread math ============================
    if (g < nt) {
      float* xch = reinterpret_cast<float*>(smem + QA_XCH) + g * 256;  // [2][128]
      const uint32_t tmem_s = tmem_base + g * 256, tmem_o = tmem_s + 128;
      const float sc = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
      float m_run = -INFINITY, l_run = 0.f;
      float o[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] = 0.f;

      for (int j = 0; j < nt; ++j) {
        const int k0 = j * ATT_BN + ch * 64;
        mbar_wait(bar_s + g, j & 1);
        tc_fence_after();
        float bm = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          uint32_t rr[32];
          tmem_ld_32x32b_x32(tmem_s + lane_base + ch * 64 + c * 32, rr);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const bool valid = (k0 + c * 32 + i) < klen;
            bm = fmaxf(bm, valid ? __uint_as_float(rr[i]) : -INFINITY);
          }
        }
        xch[ch * 128 + r] = bm;
        named_bar_sync(1 + g, 256);
        bm = fmaxf(bm, xch[(ch ^ 1) * 128 + r]);
        const float m_new = fmaxf(m_run, bm * sc);
        const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
        const float alpha = exp2f(m_run - m_use);
        // group 0's probabilities overwrite the block's K | P tiles: both groups' S MMAs must have read them
        if (g == 0 && nt == 2) mbar_wait(bar_s + 1, j & 1);
        float bsum = 0.f;
        uint8_t* tile = smem + (g == 0 ? (ch == 0 ? QA_K : QA_POS) + j * ATT_TILE_BYTES : QA_P1 + ch * ATT_TILE_BYTES) + r * 128;
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          uint32_t rr[32];
          tmem_ld_32x32b_x32(tmem_s + lane_base + ch * 64 + c * 32, rr);
          tmem_ld_wait();
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int kk0 = k0 + c * 32 + 2 * i;
            float p0 = (kk0 < klen) ? exp2f(fmaf(__uint_as_float(rr[2 * i]), sc, -m_use)) : 0.f;
            float p1 = (kk0 + 1 < klen) ? exp2f(fmaf(__uint_as_float(rr[2 * i + 1]), sc, -m_use)) : 0.f;
            const __nv_bfloat162 pb = __floats2bfloat162_rn(p0, p1);
            bsum += __low2float(pb) + __high2float(pb);
            pk[i] = *reinterpret_cast<const uint32_t*>(&pb);
          }
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const int chunk = c * 4 + q4;
            *reinterpret_cast<uint4*>(tile + ((chunk ^ (r & 7)) << 4)) =
                make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
          }
        }
        l_run = l_run * alpha + bsum;
        m_run = m_new;
        tc_fence_before();
        fence_proxy_async_smem();
        mbar_arrive(bar_pr + g);
        mbar_wait(bar_o + g, j & 1);
        tc_fence_after();
        {
          uint32_t ro[32];
          tmem_ld_32x32b_x32(tmem_o + lane_base + ch * 32, ro);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = fmaf(o[i], alpha, __uint_as_float(ro[i]));
        }
        tc_fence_before();
        named_bar_sync(1 + g, 256);
      }
      xch[ch * 128 + r] = l_run;
      named_bar_sync(1 + g, 256);
      l_run += xch[(ch ^ 1) * 128 + r];
      const int t = g * ATT_BM + r;
      if (t < T) {
        const float inv = l_run > 0.f ? 1.0f / l_run : 0.f;
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) pk[i] = pack_bf16x2(o[2 * i] * inv, o[2 * i + 1] * inv);
        uint4* dst = reinterpret_cast<uint4*>(p.out + ((size_t)b * T + t) * p.D + h * 64 + ch * 32);
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 16) {
    tc_fence_after();
    tmem_dealloc<QA_TMEM_COLS>(tmem_base);
  }
}

cudaError_t launch_qkv_rel_attention(const CUtensorMap& tm_y, const CUtensorMap& tm_w, const CUtensorMap& tm_p,
                                     const QkvAttnParams& p, cudaStream_t st) {
  if (p.D != 256 || p.H != 4 || p.T < 1 || p.T > 256 || p.B < 1) return cudaErrorInvalidValue;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(qkv_rel_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         QA_SMEM_TOTAL);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  cudaError_t le = launch_pdl(qkv_rel_attention_kernel, dim3(p.H, p.B), dim3(QA_THREADS), (size_t)QA_SMEM_TOTAL, st, tm_y,
                              tm_w, tm_p, p);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

}  // namespace ppasr
