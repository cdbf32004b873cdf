// Fused position-wise feed-forward block for sm_100a (tcgen05 + TMEM + TMA), 128 rows per tile.
//
//   plain  :  x <- x + W2s . swish(W1 . y + b1) + b2s                      (W2s = alpha*W2, b2s = alpha*b2)
//   chained:  x <- x + mask * (Wp . z + bp)        (conv module's pointwise_conv2 + residual, pad rows masked)
//             y  = LN(x; gp, bp_n)                 (norm_ff)             -- never leaves shared memory
//             x <- x + W2s . swish(W1 . y + b1) + b2s
//   then   single:  y_out = LN(x; g1, bn1)     or  double:  x <- LN(x; g1, bn1) ; y_out = LN(x; g2, bn2)
//
// Reference: PositionwiseFeedForward.forward (ppasr/model_utils/conformer/positionwise.py:30-39) and the
// surrounding residual / LayerNorm code of ConformerEncoderLayer.forward (conformer/encoder.py:380-386,
// 407-429); chained mode additionally covers convolution.py:133-140 (pointwise_conv2 + pad masking).
//
// fused_ffn_split_kernel<PRE, SPLIT> computes one 128-row tile (PRE = chained mode). TMEM holds the S double buffer in
// columns [0,256) and the output accumulator O in [256,512); the FF-wide hidden activation never leaves the SM:
//     GEMM1(j): S[j&1] = Y[128x256] . W1_j^T                 16 x tcgen05.mma 128x128x16
//     swish(j): TMEM -> +b1 -> swish -> bf16 -> 128B-swizzled smem H[j&1]
//     GEMM2(j): O += H[j&1][128x128] . W2s_j^T                8 x tcgen05.mma 128x256x16
//  * Swish runs on two teams of 8 warps (even / odd chunks), S is released right after the TMEM load, and GEMM1(j+2) is
//    issued BEFORE GEMM2(j): the tensor pipe always has the next GEMM1 queued while a team is still in its Swish.
//  * Weights stream through a 3 x 32 KB TMA ring; the tiles that do not depend on the predecessor kernel are requested
//    before griddepcontrol.wait.
//  * SPLIT (ffn_split mode 1): the tile is shared by a 2-CTA thread-block cluster. CTA `rank` owns hidden chunks
//    [rank*NCH/2, (rank+1)*NCH/2) and ends with a PARTIAL output tile O_rank in TMEM. The two partials are reduced through
//    distributed shared memory: each CTA stages its tile in shared memory, bulk-copies the 64 rows the PEER finalises into
//    the peer's receive buffer (cp.async.bulk.shared::cluster, completion on the peer's mbarrier) and finalises its own 64
//    rows. One launch therefore covers 2 x ceil(M/128) CTAs (124 at C2 instead of 62 on 148 SMs).
//  * !SPLIT (ffn_split mode 2): the same pipeline on one CTA per tile, all chunks, all 128 rows (least SM time per launch).
//  * The output tile is staged in fp32 shared memory and finalised warp-per-row: partial(s) + b2s [+ residual from global
//    memory] -> LayerNorm(s) -> coalesced x / y stores.
//  * plain mode: no residual preload at all -- x is added in the final pass from global memory (coalesced).
//  * chained mode: the residual tile (+ masked bp) is preloaded into O through a coalesced smem slab, the pre-GEMM
//    accumulates on top of it, and LN(x_mid) replaces z in the A tiles. Under SPLIT both CTAs run the small pre-GEMM +
//    LayerNorm redundantly (1/16 of the FLOPs); rank 1 then discards the residual by starting its GEMM2 chain with
//    accumulate = 0, so x_mid is counted once.
#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"
#include "row_tile.cuh"

#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>

namespace ppasr {

void count_launch();

constexpr int FFN_TILE = 128 * 64 * 2;       // 16 KB: [128 rows x 64 bf16] swizzled tile
constexpr int FFN_SMEM_A = 0;                // 4 tiles (Y or Z, K = 256)
constexpr int FFN_SMEM_H = 4 * FFN_TILE;     // 2 buffers x 2 tiles (also: residual preload slab)
constexpr int FFN_SMEM_W = 8 * FFN_TILE;     // ring: 3 big slots x 32 KB
constexpr int FFN_RING = 3;
constexpr int FFN_SMEM_BAR = 14 * FFN_TILE;  // 229376
constexpr int FFN_SMEM_TOTAL = FFN_SMEM_BAR + 512 + 1024;
constexpr int FFN_SLAB_PITCH = 68;           // residual preload slab [128][68] fp32 (64 columns at a time)

struct FfnParams {
  int M;             // rows
  int nchunks;       // FF / 128
  float* x;          // fp32 residual stream [M, 256]
  __nv_bfloat16* y;  // bf16 output of the trailing LayerNorm [M, 256]
  const float* b1;   // [FF]
  const float* b2s;  // [256] already scaled by alpha
  const float *g1, *bn1, *g2, *bn2;  // trailing LayerNorm params (g2 null = single)
  float eps;
  // chained pre-GEMM (null bp = plain mode)
  const float* bp;        // [256] bias of the pre-GEMM
  const float *gp, *bpn;  // LayerNorm between pre-GEMM and FFN
  const int* lens;        // valid frames per utterance (pad rows: pre-GEMM branch contributes 0)
  int T;
  // post-norm models (Squeezeformer): double mode with y_affine writes x <- LN(x; g1, bn1) and the bf16 output
  // y = g2 * x + bn2 (adaptive scale / bias of the next module); rows t >= ylens[b] of y are zeroed when ylens != null
  // (conv-module input, squeezeformer/convolution.py:119-127).
  int y_affine;
  const int* ylens;
  // post-norm chained mode (pre_ys != null): the LayerNorm after the pre-GEMM is the block's own post-norm, i.e. the
  // residual itself becomes x <- LN(x + Wp z + bp; gp, bpn) (written back into TMEM O) and the FFN input is its adaptive
  // affine pre_ys * x + pre_yb (squeezeformer/encoder.py:468-487: MHA -> layer_norm1 -> ffn1, conv -> layer_norm3 -> ffn2)
  const float *pre_ys, *pre_yb;
};

constexpr int FS_THREADS = 640;                     // warps 0..3 control, 4..11 team 0, 12..19 team 1
constexpr int FS_PITCH = 260;                       // fp32 staging pitch
constexpr int FS_SMEM_XS = 0;                       // [128][260] fp32: own partial tile
constexpr int FS_SMEM_RECV = 128 * FS_PITCH * 4;    // [64][260] fp32: peer's partial of my rows
constexpr int FS_SMEM_PRM = FS_SMEM_RECV + 64 * FS_PITCH * 4;  // [5][256] fp32 parameters
constexpr int FS_PIECE_ROWS = 16;
constexpr int FS_PIECE_BYTES = FS_PIECE_ROWS * FS_PITCH * 4;   // 16640
static_assert(FS_SMEM_PRM + 5 * 256 * 4 <= FFN_SMEM_BAR, "epilogue staging must fit below the barrier block");

template <bool PRE, bool SPLIT>
__global__ void __launch_bounds__(FS_THREADS, 1)
fused_ffn_split_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_wp,
                       const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_w2,
                       const FfnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_a = smem + FFN_SMEM_A;
  uint8_t* s_h = smem + FFN_SMEM_H;
  uint8_t* s_w = smem + FFN_SMEM_W;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + FFN_SMEM_BAR);
  uint64_t* a_full = bars;
  uint64_t* w_full = bars + 1;   // [3]
  uint64_t* w_empty = bars + 4;  // [3]
  uint64_t* s_full = bars + 7;   // [2]
  uint64_t* s_free = bars + 9;   // [2]
  uint64_t* h_full = bars + 11;  // [2]
  uint64_t* h_free = bars + 13;  // [2]
  uint64_t* o_full = bars + 15;
  uint64_t* x_loaded = bars + 16;
  uint64_t* pre_full = bars + 17;
  uint64_t* a_ready = bars + 18;
  uint64_t* peer_free = bars + 19;  // arrived REMOTELY by the peer: its staging / receive buffers are idle
  uint64_t* recv_full = bars + 20;  // [4] tx barriers: piece k of the peer's partial has landed
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 24);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // SPLIT = false: the same pipeline on one CTA per row tile (no cluster, no exchange): all chunks, all 128 rows
  const uint32_t rank = SPLIT ? cluster_ctarank() : 0u;
  const int m0 = (SPLIT ? (blockIdx.x >> 1) : blockIdx.x) * 128;
  const int NCHH = SPLIT ? (p.nchunks >> 1) : p.nchunks;  // chunks of this CTA
  const int j0 = (int)rank * NCHH;                        // first global hidden chunk

  if (warp_idx == 0 && elect_one()) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_w1);
    tma_prefetch_desc(&tm_w2);
    if (PRE) tma_prefetch_desc(&tm_wp);
  }
  if (warp_idx == 1 && elect_one()) {
    mbar_init(a_full, 1);
    for (int i = 0; i < FFN_RING; ++i) {
      mbar_init(&w_full[i], 1);
      mbar_init(&w_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 256);
      mbar_init(&h_full[i], 256);
      mbar_init(&h_free[i], 1);
    }
    mbar_init(o_full, 1);
    mbar_init(x_loaded, 256);
    mbar_init(pre_full, 1);
    mbar_init(a_ready, 256);
    mbar_init(peer_free, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&recv_full[i], 1);
    fence_barrier_init();
    if (SPLIT)
      for (int i = 0; i < 4; ++i) mbar_arrive_expect_tx(&recv_full[i], FS_PIECE_BYTES);
    fence_proxy_async_smem();
  }
  if (warp_idx == 2) tmem_alloc<512>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  if (SPLIT) cluster_sync_all();  // the peer's barriers are initialised before anything remote can reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t tmem_o = tmem_base + 256;
  pdl_launch_dependents();  // the successor may start its own prologue (it waits for this grid before reading x / y)

  if (warp_idx == 0) {
    // ============================ TMA producer ============================
    if (elect_one()) {
      int slot = 0;
      uint32_t phase = 0;
      auto load_rows256 = [&](const CUtensorMap* tm, int k0) {  // one slot: [256 rows x 64 K]
        mbar_wait(&w_empty[slot], phase ^ 1);
        mbar_arrive_expect_tx(&w_full[slot], 2 * FFN_TILE);
        tma_load_2d(s_w + slot * 2 * FFN_TILE, tm, &w_full[slot], k0, 0);
        if (++slot == FFN_RING) slot = 0, phase ^= 1;
      };
      auto load_w1_half = [&](int j, int s) {  // one slot: k-blocks (2s, 2s+1) of W1 rows [(j0+j)*128, +128)
        mbar_wait(&w_empty[slot], phase ^ 1);
        mbar_arrive_expect_tx(&w_full[slot], 2 * FFN_TILE);
        tma_load_2d(s_w + slot * 2 * FFN_TILE, &tm_w1, &w_full[slot], (2 * s) * 64, (j0 + j) * 128);
        tma_load_2d(s_w + slot * 2 * FFN_TILE + FFN_TILE, &tm_w1, &w_full[slot], (2 * s + 1) * 64, (j0 + j) * 128);
        if (++slot == FFN_RING) slot = 0, phase ^= 1;
      };
      // the first three ring slots hold weights only: request them before waiting for the predecessor kernel
      if (PRE) {
        for (int kb = 0; kb < 3; ++kb) load_rows256(&tm_wp, kb * 64);
      } else {
        load_w1_half(0, 0);
        load_w1_half(0, 1);
        load_w1_half(1, 0);
      }
      pdl_wait();
      mbar_arrive_expect_tx(a_full, 4 * FFN_TILE);
      for (int kb = 0; kb < 4; ++kb) tma_load_2d(s_a + kb * FFN_TILE, &tm_a, a_full, kb * 64, m0);
      if (PRE) {
        load_rows256(&tm_wp, 3 * 64);
        load_w1_half(0, 0);
        load_w1_half(0, 1);
        load_w1_half(1, 0);
      }
      load_w1_half(1, 1);
      for (int j = 0; j < NCHH; ++j) {
        if (j + 2 < NCHH) {
          load_w1_half(j + 2, 0);
          load_w1_half(j + 2, 1);
        }
        load_rows256(&tm_w2, (j0 + j) * 128);
        load_rows256(&tm_w2, (j0 + j) * 128 + 64);
      }
    }
  } else if (warp_idx == 1) {
    // ============================ MMA issuer ============================
    if (elect_one()) {
      constexpr uint32_t idesc_g1 = umma_idesc_bf16(128, 128);
      constexpr uint32_t idesc_g2 = umma_idesc_bf16(128, 256);
      int slot = 0;
      uint32_t phase = 0;
      const uint32_t a_addr = smem_u32(s_a);
      mbar_wait(a_full, 0);
      tc_fence_after();
      if (PRE) {
        mbar_wait(x_loaded, 0);
        tc_fence_after();
        for (int kb = 0; kb < 4; ++kb) {
          mbar_wait(&w_full[slot], phase);
          tc_fence_after();
          const uint32_t w_addr = smem_u32(s_w + slot * 2 * FFN_TILE);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_o, umma_desc_k_sw128(a_addr + kb * FFN_TILE + k * 32), umma_desc_k_sw128(w_addr + k * 32),
                      idesc_g2, 1u);
          umma_commit(&w_empty[slot]);
          if (++slot == FFN_RING) slot = 0, phase ^= 1;
        }
        umma_commit(pre_full);
        mbar_wait(a_ready, 0);
        tc_fence_after();
      }
      // O starts from the residual only where it was preloaded and must be kept (chained mode, rank 0)
      const uint32_t keep_o = (PRE && rank == 0) ? 1u : 0u;  // (non-split plain mode adds x in the final pass instead)
      auto gemm1 = [&](int j) {
        const int b = j & 1;
        if (j >= 2) {
          mbar_wait(&s_free[b], ((j >> 1) + 1) & 1);  // the team has pulled S[b] of chunk j-2 into registers
          tc_fence_after();
        }
        const uint32_t tmem_s = tmem_base + b * 128;
        for (int s = 0; s < 2; ++s) {
          mbar_wait(&w_full[slot], phase);
          tc_fence_after();
          const uint32_t w_addr = smem_u32(s_w + slot * 2 * FFN_TILE);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int kb = 2 * s + t;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_s, umma_desc_k_sw128(a_addr + kb * FFN_TILE + k * 32),
                        umma_desc_k_sw128(w_addr + t * FFN_TILE + k * 32), idesc_g1, (kb | k) != 0);
          }
          umma_commit(&w_empty[slot]);
          if (++slot == FFN_RING) slot = 0, phase ^= 1;
        }
        umma_commit(&s_full[b]);
      };
      auto gemm2 = [&](int j) {
        const int b = j & 1;
        mbar_wait(&h_full[b], (j >> 1) & 1);
        tc_fence_after();
        const uint32_t h_addr = smem_u32(s_h + b * 2 * FFN_TILE);
        for (int kb = 0; kb < 2; ++kb) {
          mbar_wait(&w_full[slot], phase);
          tc_fence_after();
          const uint32_t w_addr = smem_u32(s_w + slot * 2 * FFN_TILE);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_o, umma_desc_k_sw128(h_addr + kb * FFN_TILE + k * 32), umma_desc_k_sw128(w_addr + k * 32),
                      idesc_g2, (uint32_t)((j | kb | k) != 0) | keep_o);
          umma_commit(&w_empty[slot]);
          if (++slot == FFN_RING) slot = 0, phase ^= 1;
        }
        umma_commit(&h_free[b]);
      };
      gemm1(0);
      gemm1(1);
      for (int j = 0; j < NCHH; ++j) {
        if (j + 2 < NCHH) gemm1(j + 2);
        gemm2(j);
      }
      umma_commit(o_full);
    }
  } else if (warp_idx >= 4) {
    // ============================ compute warps (two teams) ============================
    pdl_wait();
    const int cw = warp_idx - 4;        // 0..15
    const int team = cw >> 3;
    const int ew = cw & 7;
    const int quad = ew & 3;            // == warp_idx & 3: the TMEM lane quarter this warp may touch
    const int half = ew >> 2;
    const int r = quad * 32 + lane;
    const int ct = threadIdx.x - 128 - team * 256;  // 0..255 inside the team
    const uint32_t lane_base = ((uint32_t)(quad * 32)) << 16;
    if (PRE && team == 0) {
      const int row_g = m0 + r;
      bool pad = false;
      if (p.lens != nullptr && row_g < p.M) {
        const int b = row_g / p.T;
        pad = (row_g - b * p.T) >= __ldg(p.lens + b);
      }
      // ---- residual tile (+ masked bias of the pre-GEMM) -> TMEM O through a coalesced slab in the idle H region ----
      float* slab = reinterpret_cast<float*>(s_h);
      for (int s = 0; s < 4; ++s) {
        {
          const int cq = ct & 15;
          float4 v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = (ct >> 4) + 16 * i;
            v[i] = ((m0 + rr) < p.M)
                       ? __ldcg(reinterpret_cast<const float4*>(p.x + (size_t)(m0 + rr) * 256 + s * 64) + cq)
                       : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i)
            *reinterpret_cast<float4*>(slab + ((ct >> 4) + 16 * i) * FFN_SLAB_PITCH + cq * 4) = v[i];
        }
        named_bar_sync(1, 256);
        if (half == (s >> 1)) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t v[32];
            const int col0 = s * 64 + c * 32;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 t = *reinterpret_cast<const float4*>(slab + r * FFN_SLAB_PITCH + c * 32 + 4 * j);
              if (!pad) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bp + col0) + j);
                t.x += bb.x, t.y += bb.y, t.z += bb.z, t.w += bb.w;
              }
              v[4 * j] = __float_as_uint(t.x), v[4 * j + 1] = __float_as_uint(t.y);
              v[4 * j + 2] = __float_as_uint(t.z), v[4 * j + 3] = __float_as_uint(t.w);
            }
            tmem_st_32x32b_x32(tmem_o + lane_base + col0, v);
          }
          tmem_st_wait();
        }
        named_bar_sync(1, 256);
      }
      tc_fence_before();
      mbar_arrive(x_loaded);
      // ---- y = LN(x_mid) -> A tiles (bf16, 128B swizzle); x_mid stays in TMEM O ----
      mbar_wait(pre_full, 0);
      tc_fence_after();
      float4* sc = reinterpret_cast<float4*>(s_h);
      FfnStat st{0.f, 0.f, 0.f};
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t ro[32];
        tmem_ld_32x32b_x32(tmem_o + lane_base + half * 128 + c * 32, ro);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ro[j]);
        ffn_add_chunk(st, v);
      }
      ffn_exchange(st, sc, r, half, 2);
      const float mean = st.mean;
      const float rstd = rsqrtf(st.m2 * (1.0f / 256.0f) + p.eps);
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int cc = half * 128 + c * 32;
        uint32_t ro[32];
        tmem_ld_32x32b_x32(tmem_o + lane_base + cc, ro);
        tmem_ld_wait();
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 gg = __ldg(reinterpret_cast<const float4*>(p.gp + cc) + j);
          const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bpn + cc) + j);
          float y0 = (__uint_as_float(ro[4 * j + 0]) - mean) * rstd * gg.x + bb.x;
          float y1 = (__uint_as_float(ro[4 * j + 1]) - mean) * rstd * gg.y + bb.y;
          float y2 = (__uint_as_float(ro[4 * j + 2]) - mean) * rstd * gg.z + bb.z;
          float y3 = (__uint_as_float(ro[4 * j + 3]) - mean) * rstd * gg.w + bb.w;
          if (p.pre_ys != nullptr) {
            ro[4 * j + 0] = __float_as_uint(y0), ro[4 * j + 1] = __float_as_uint(y1);
            ro[4 * j + 2] = __float_as_uint(y2), ro[4 * j + 3] = __float_as_uint(y3);
            const float4 as = __ldg(reinterpret_cast<const float4*>(p.pre_ys + cc) + j);
            const float4 ab = __ldg(reinterpret_cast<const float4*>(p.pre_yb + cc) + j);
            y0 = fmaf(as.x, y0, ab.x), y1 = fmaf(as.y, y1, ab.y), y2 = fmaf(as.z, y2, ab.z), y3 = fmaf(as.w, y3, ab.w);
          }
          pk[2 * j] = pack_bf16x2(y0, y1);
          pk[2 * j + 1] = pack_bf16x2(y2, y3);
        }
        if (p.pre_ys != nullptr) tmem_st_32x32b_x32(tmem_o + lane_base + cc, ro);
        uint8_t* atile = s_a + (cc >> 6) * FFN_TILE + r * 128;
        const int ch0 = (cc & 63) >> 3;
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4)
          *reinterpret_cast<uint4*>(atile + (((ch0 + q4) ^ (r & 7)) << 4)) =
              make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
      }
      if (p.pre_ys != nullptr) tmem_st_wait();
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive(a_ready);
    }
    // ---- Swish between the two GEMMs: team t owns local chunks j = t, t+2, ... (S[t], H[t]) ----
    for (int j = team; j < NCHH; j += 2) {
      const int b = team;
      const int it = j >> 1;
      mbar_wait(&s_full[b], it & 1);
      tc_fence_after();
      uint32_t rr2[2][32];
      tmem_ld_32x32b_x32(tmem_base + lane_base + b * 128 + half * 64, rr2[0]);
      tmem_ld_32x32b_x32(tmem_base + lane_base + b * 128 + half * 64 + 32, rr2[1]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&s_free[b]);  // S[b] is in registers: GEMM1(j+2) may overwrite it while this team computes
      if (it >= 1) mbar_wait(&h_free[b], (it + 1) & 1);  // GEMM2(j-2) has consumed H[b]
      uint8_t* htile = s_h + b * 2 * FFN_TILE + half * FFN_TILE + r * 128;
      const float* b1p = p.b1 + (j0 + j) * 128 + half * 64;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const uint32_t(&rr)[32] = rr2[c];
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 bv = __ldg(reinterpret_cast<const float4*>(b1p + c * 32) + i);
          pk[2 * i] = pack_bf16x2(swish_f(__uint_as_float(rr[4 * i]) + bv.x), swish_f(__uint_as_float(rr[4 * i + 1]) + bv.y));
          pk[2 * i + 1] =
              pack_bf16x2(swish_f(__uint_as_float(rr[4 * i + 2]) + bv.z), swish_f(__uint_as_float(rr[4 * i + 3]) + bv.w));
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int chunk = c * 4 + q4;
          *reinterpret_cast<uint4*>(htile + ((chunk ^ (r & 7)) << 4)) =
              make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
        }
      }
      fence_proxy_async_smem();
      mbar_arrive(&h_full[b]);
    }
    // ---- reduce the two partial tiles through distributed shared memory and finalise 64 rows per CTA ----
    mbar_wait(o_full, 0);
    tc_fence_after();
    const int ct16 = threadIdx.x - 128;  // 0..511
    const uint32_t peer = rank ^ 1u;
    if (SPLIT && ct16 == 0) mbar_arrive_remote(mapa_u32(smem_u32(peer_free), peer));  // all my MMAs are done: my buffers are idle
    float* xs = reinterpret_cast<float*>(smem + FS_SMEM_XS);
    float* rcv = reinterpret_cast<float*>(smem + FS_SMEM_RECV);
    float* prm = reinterpret_cast<float*>(smem + FS_SMEM_PRM);  // [5][256]: b2s, g1, bn1, g2, bn2
    {
      const int cg = cw >> 2;  // 64-column group of this warp
      float* xrow = xs + r * FS_PITCH + cg * 64;
      uint32_t ro[2][32];
      tmem_ld_32x32b_x32(tmem_o + lane_base + cg * 64, ro[0]);
      tmem_ld_32x32b_x32(tmem_o + lane_base + cg * 64 + 32, ro[1]);
      tmem_ld_wait();
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<float4*>(xrow + u * 32 + 4 * j) =
              make_float4(__uint_as_float(ro[u][4 * j]), __uint_as_float(ro[u][4 * j + 1]),
                          __uint_as_float(ro[u][4 * j + 2]), __uint_as_float(ro[u][4 * j + 3]));
    }
    if (ct16 < 256) {
      prm[ct16] = __ldg(p.b2s + ct16);
      prm[256 + ct16] = __ldg(p.g1 + ct16);
      prm[512 + ct16] = __ldg(p.bn1 + ct16);
    } else if (p.g2 != nullptr) {
      prm[768 + ct16 - 256] = __ldg(p.g2 + ct16 - 256);
      prm[1024 + ct16 - 256] = __ldg(p.bn2 + ct16 - 256);
    }
    if (SPLIT) fence_proxy_async_smem();  // the staged tile is read by the bulk-copy engine
    named_bar_sync(4, 512);
    if (SPLIT && ct16 == 0) {
      mbar_wait_cluster(peer_free, 0);  // the peer is out of its main loop: its receive buffer may be written
      const uint32_t dst = mapa_u32(smem_u32(rcv), peer);
      const uint32_t dbar = mapa_u32(smem_u32(recv_full), peer);
      const float* src = xs + (size_t)(peer * 64) * FS_PITCH;  // the 64 rows the peer finalises
#pragma unroll
      for (int k = 0; k < 4; ++k)
        bulk_copy_to_cluster(dst + k * FS_PIECE_BYTES, reinterpret_cast<const uint8_t*>(src) + k * FS_PIECE_BYTES,
                             FS_PIECE_BYTES, dbar + k * 8);
    }
    // warp-per-row finalisation of local rows i = cw + 16 k (split: piece k of the peer's partial; 4 rows per warp.
    // single CTA: all 128 rows, 8 per warp)
    constexpr int NROW = SPLIT ? 4 : 8;
    const int rbase = m0 + (int)rank * 64;
    const bool dbl = p.g2 != nullptr;
    float4 pb[2], pg1[2], pn1[2], pg2[2], pn2[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      pb[h] = *reinterpret_cast<const float4*>(prm + 4 * lane + 128 * h);
      pg1[h] = *reinterpret_cast<const float4*>(prm + 256 + 4 * lane + 128 * h);
      pn1[h] = *reinterpret_cast<const float4*>(prm + 512 + 4 * lane + 128 * h);
      if (dbl) {
        pg2[h] = *reinterpret_cast<const float4*>(prm + 768 + 4 * lane + 128 * h);
        pn2[h] = *reinterpret_cast<const float4*>(prm + 1024 + 4 * lane + 128 * h);
      } else {
        pg2[h] = pn2[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll 1
    for (int kk = 0; kk < NROW; kk += 4) {
    float4 xg[4][2];  // residual rows of this group of four, requested before the (split: peer) data is needed
    if (!PRE) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int R = rbase + cw + 16 * (kk + k);
#pragma unroll
        for (int h = 0; h < 2; ++h)
          xg[k][h] = (R < p.M) ? __ldcg(reinterpret_cast<const float4*>(p.x + (size_t)R * 256) + lane + 32 * h)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int kq = 0; kq < 4; ++kq) {
      const int k = kk + kq;
      if (SPLIT) mbar_wait(&recv_full[k], 0);
      const int i = cw + 16 * k;
      const int R = rbase + i;
      if (R >= p.M) continue;
      const float* a = xs + ((int)rank * 64 + i) * FS_PITCH;
      const float* bq = rcv + i * FS_PITCH;
      float v[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 t0 = *reinterpret_cast<const float4*>(a + 4 * lane + 128 * h);
        const float4 t1 = SPLIT ? *reinterpret_cast<const float4*>(bq + 4 * lane + 128 * h) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[4 * h + 0] = t0.x + t1.x + pb[h].x, v[4 * h + 1] = t0.y + t1.y + pb[h].y;
        v[4 * h + 2] = t0.z + t1.z + pb[h].z, v[4 * h + 3] = t0.w + t1.w + pb[h].w;
        if (!PRE) v[4 * h + 0] += xg[kq][h].x, v[4 * h + 1] += xg[kq][h].y, v[4 * h + 2] += xg[kq][h].z, v[4 * h + 3] += xg[kq][h].w;
      }
      float s = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) s += v[e];
      float mean = warp_sum(s) * (1.0f / 256.0f);
      float q = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) q += (v[e] - mean) * (v[e] - mean);
      float rstd = rsqrtf(warp_sum(q) * (1.0f / 256.0f) + p.eps);
      const float g1v[8] = {pg1[0].x, pg1[0].y, pg1[0].z, pg1[0].w, pg1[1].x, pg1[1].y, pg1[1].z, pg1[1].w};
      const float n1v[8] = {pn1[0].x, pn1[0].y, pn1[0].z, pn1[0].w, pn1[1].x, pn1[1].y, pn1[1].z, pn1[1].w};
      float y[8];
      if (dbl) {
        const float g2v[8] = {pg2[0].x, pg2[0].y, pg2[0].z, pg2[0].w, pg2[1].x, pg2[1].y, pg2[1].z, pg2[1].w};
        const float n2v[8] = {pn2[0].x, pn2[0].y, pn2[0].z, pn2[0].w, pn2[1].x, pn2[1].y, pn2[1].z, pn2[1].w};
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = (v[e] - mean) * rstd * g1v[e] + n1v[e];  // x <- LN(x; g1, bn1)
        if (p.y_affine) {
#pragma unroll
          for (int e = 0; e < 8; ++e) y[e] = v[e] * g2v[e] + n2v[e];
        } else {
          float s2 = 0.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) s2 += v[e];
          const float mean2 = warp_sum(s2) * (1.0f / 256.0f);
          float q2 = 0.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) q2 += (v[e] - mean2) * (v[e] - mean2);
          const float rstd2 = rsqrtf(warp_sum(q2) * (1.0f / 256.0f) + p.eps);
#pragma unroll
          for (int e = 0; e < 8; ++e) y[e] = (v[e] - mean2) * rstd2 * g2v[e] + n2v[e];
        }
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) y[e] = (v[e] - mean) * rstd * g1v[e] + n1v[e];
      }
      bool zero_y = false;
      if (p.ylens != nullptr) {
        const int bb = R / p.T;
        zero_y = (R - bb * p.T) >= __ldg(p.ylens + bb);
      }
      float4* dx = reinterpret_cast<float4*>(p.x + (size_t)R * 256);
      uint2* dy = reinterpret_cast<uint2*>(p.y + (size_t)R * 256);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        dx[lane + 32 * h] = make_float4(v[4 * h], v[4 * h + 1], v[4 * h + 2], v[4 * h + 3]);
        dy[lane + 32 * h] = zero_y ? make_uint2(0u, 0u)
                                   : make_uint2(pack_bf16x2(y[4 * h], y[4 * h + 1]), pack_bf16x2(y[4 * h + 2], y[4 * h + 3]));
      }
    }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (SPLIT) cluster_sync_all();  // neither CTA exits while the other's bulk copy may still read or write its shared memory
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

static std::atomic<int> g_ffn_split{-1};
int ffn_split_mode() {
  int v = g_ffn_split.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("PPASR_B200_FFN_SPLIT");
    v = (e != nullptr && std::strcmp(e, "2") == 0) ? 2 : 1;
    g_ffn_split.store(v, std::memory_order_relaxed);
  }
  return v;
}
bool set_ffn_split_mode(int mode) {
  if (mode != 1 && mode != 2) return false;
  g_ffn_split.store(mode, std::memory_order_relaxed);
  return true;
}

cudaError_t launch_fused_ffn(const CUtensorMap& tm_a, const CUtensorMap* tm_wp, const CUtensorMap& tm_w1,
                             const CUtensorMap& tm_w2, int M, int FF, float* x, __nv_bfloat16* y, const float* b1,
                             const float* b2s, const float* g1, const float* bn1, const float* g2, const float* bn2,
                             float eps, const float* bp, const float* gp, const float* bpn, const int* lens, int T,
                             cudaStream_t st, int y_affine, const int* ylens, const float* pre_ys, const float* pre_yb) {
  if (FF % 128 != 0 || FF < 256 || M <= 0) return cudaErrorInvalidValue;  // the pipeline starts with GEMM1(0) and GEMM1(1)
  static std::once_flag once;
  static cudaError_t cfg_err = cudaSuccess;
  std::call_once(once, [] {
    cudaError_t e = cudaFuncSetAttribute(fused_ffn_split_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FFN_SMEM_TOTAL);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(fused_ffn_split_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FFN_SMEM_TOTAL);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(fused_ffn_split_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FFN_SMEM_TOTAL);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(fused_ffn_split_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FFN_SMEM_TOTAL);
    cfg_err = e;
  });
  if (cfg_err != cudaSuccess) return cfg_err;
  FfnParams p;
  p.M = M, p.nchunks = FF / 128, p.x = x, p.y = y, p.b1 = b1, p.b2s = b2s;
  p.g1 = g1, p.bn1 = bn1, p.g2 = g2, p.bn2 = bn2, p.eps = eps;
  p.bp = bp, p.gp = gp, p.bpn = bpn, p.lens = lens, p.T = T;
  p.y_affine = y_affine, p.ylens = ylens, p.pre_ys = pre_ys, p.pre_yb = pre_yb;
  const int grid = (M + 127) / 128;
  cudaError_t le;
  if (ffn_split_mode() == 1 && p.nchunks >= 4 && (p.nchunks & 1) == 0) {
    // 2-CTA cluster per row tile, hidden dimension split over the pair (each half needs at least two chunks)
    if (tm_wp != nullptr)
      le = launch_pdl_cluster(fused_ffn_split_kernel<true, true>, dim3(2 * grid), dim3(FS_THREADS), (size_t)FFN_SMEM_TOTAL, st, 2u,
                              tm_a, *tm_wp, tm_w1, tm_w2, p);
    else
      le = launch_pdl_cluster(fused_ffn_split_kernel<false, true>, dim3(2 * grid), dim3(FS_THREADS), (size_t)FFN_SMEM_TOTAL, st, 2u,
                              tm_a, tm_w1, tm_w1, tm_w2, p);
  } else {
    // the two-team pipeline on one CTA per row tile (least SM time per launch: several batches in flight)
    if (tm_wp != nullptr)
      le = launch_pdl(fused_ffn_split_kernel<true, false>, dim3(grid), dim3(FS_THREADS), (size_t)FFN_SMEM_TOTAL, st, tm_a, *tm_wp,
                      tm_w1, tm_w2, p);
    else
      le = launch_pdl(fused_ffn_split_kernel<false, false>, dim3(grid), dim3(FS_THREADS), (size_t)FFN_SMEM_TOTAL, st, tm_a, tm_w1,
                      tm_w1, tm_w2, p);
  }
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

}  // namespace ppasr
