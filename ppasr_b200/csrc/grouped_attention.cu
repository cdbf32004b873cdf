// Grouped relative-position multi-head attention for sm_100a (tcgen05 + TMEM + TMA).
//
// Reference: GroupedRelPositionMultiHeadedAttention.forward / pad4group / forward_attention
// (ppasr/model_utils/efficient_conformer/attention.py:128-193, 40-79, 81-126), group size 3:
//   tokens = groups of 3 frames, 4 heads x 192 features;  S = ((q+u) k^T + (q+v) p^T) / sqrt(192)   (no rel_shift)
//   keys g with 3g >= len are masked (mask[:, ::3, ::3]);  out = softmax(S) V, re-viewed as frames and trimmed to T.
// As in attention.cu the two score terms are one contraction [q+u | q+v] . [k | p]^T, here over K = 384.
//
// One CTA per (128-query tile, head, utterance). TMEM holds four 64-column score slots in [0,256) and O in [256,448). The
// soft-max is a plain two-pass one (global row maximum, then probabilities block by block feeding P.V with accumulation in
// TMEM); no online rescaling and no 192-float output registers per thread.
//   control thread : TMA Q (6 tiles), per 64-key block K|P (6 tiles) -> 24 x tcgen05.mma 128x64x16 -> S_j
//   128 softmax thr: row max over all blocks; per block exp2 -> bf16 probabilities -> swizzled smem tile
//   control thread : TMA V^T_j [192 x 64] -> 4 x tcgen05.mma 128x192x16, O += P_j V_j
//   128 softmax thr: O / l -> bf16, stored at frame t = 3g + i/256, column i%256 (i = h*192 + d), rows t >= T dropped
// Two paths, chosen by the number of 64-key blocks nblk:
//   resident  (nblk <= 4, up to 256 key groups = 768 frames): every S_j stays in its slot and is scored once.
//   recompute (nblk > 4): pass 1 streams S_j through the slots as a ring (the softmax threads hand a slot back through
//             bar_sf once its maximum is read); pass 2 re-issues the K|P loads and S_j MMAs into the same ring, a few blocks
//             ahead of P.V. The per-block probabilities, P.V and lsum order are the resident path's, so for the same S it
//             gives what the resident path would with unbounded TMEM, at one extra QK^T (K = 384) per block.
#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"

namespace ppasr {

void count_launch();

constexpr int GA_SLOTS = 4;                    // 64-column score slots in TMEM (256 key groups resident)
constexpr int GA_THREADS = 160;
constexpr int GA_QT = 128 * 64 * 2;            // [128 x 64] tile, 16 KB
constexpr int GA_KT = 64 * 64 * 2;             // [64 x 64] tile, 8 KB
constexpr int GA_SMEM_Q = 0;                   // 6 tiles
constexpr int GA_SMEM_KP = 6 * GA_QT;          // 6 tiles of 8 KB
constexpr int GA_SMEM_V = GA_SMEM_KP + 6 * GA_KT;   // [192 x 64] = 24 KB
constexpr int GA_SMEM_P = GA_SMEM_V + 192 * 64 * 2; // probabilities [128 x 64] = 16 KB
constexpr int GA_SMEM_BAR = GA_SMEM_P + GA_QT;
constexpr int GA_SMEM_TOTAL = GA_SMEM_BAR + 128 + 1024;

__global__ void __launch_bounds__(GA_THREADS, 1)
grouped_attention_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                         const __grid_constant__ CUtensorMap tm_p, const __grid_constant__ CUtensorMap tm_vt,
                         const GroupedAttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_q = smem + GA_SMEM_Q;
  uint8_t* s_kp = smem + GA_SMEM_KP;
  uint8_t* s_v = smem + GA_SMEM_V;
  uint8_t* s_p = smem + GA_SMEM_P;
  uint64_t* bar_q = reinterpret_cast<uint64_t*>(smem + GA_SMEM_BAR);
  uint64_t* bar_kp = bar_q + 1;
  uint64_t* bar_v = bar_q + 2;
  uint64_t* bar_p = bar_q + 3;      // probabilities of block j written (128 arrivals)
  uint64_t* bar_pv = bar_q + 4;     // P.V of block j complete (P tile and V smem free)
  uint64_t* bar_s = bar_q + 5;      // [GA_SLOTS] S in slot s complete (also: K|P smem free); one phase per use of the slot
  uint64_t* bar_sf = bar_s + GA_SLOTS;  // [GA_SLOTS] recompute path: the softmax threads have read slot s (128 arrivals)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bar_sf + GA_SLOTS);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int h = blockIdx.y, b = blockIdx.z;
  const int bh = b * p.H + h;
  const int row0 = blockIdx.x * 128;
  const int Tgk = p.Tgk > 0 ? p.Tgk : p.Tg;           // key groups (streaming: the whole cache, queries: this chunk)
  const int kpitch = p.k_pitch > 0 ? p.k_pitch : p.Tg;
  const int klen = p.klens ? min(Tgk, (__ldg(p.klens + b) + 2) / 3) : Tgk;  // keys g with 3g < len
  const int nblk = (Tgk + 63) / 64;
  const bool resident = nblk <= GA_SLOTS;  // the whole score row fits the slots: each S_j is computed once

  if (warp_idx == 4) {
    if (elect_one()) {
      tma_prefetch_desc(&tm_q);
      tma_prefetch_desc(&tm_k);
      tma_prefetch_desc(&tm_p);
      tma_prefetch_desc(&tm_vt);
      mbar_init(bar_q, 1);
      mbar_init(bar_kp, 1);
      for (int i = 0; i < GA_SLOTS; ++i) mbar_init(bar_s + i, 1), mbar_init(bar_sf + i, 128);
      mbar_init(bar_v, 1);
      mbar_init(bar_p, 128);
      mbar_init(bar_pv, 1);
      fence_barrier_init();
      fence_proxy_async_smem();
    }
    __syncwarp();
    tmem_alloc<512>(tmem_ptr_smem);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tmem_s = tmem_base;
  const uint32_t tmem_o = tmem_base + 256;

  if (warp_idx == 4) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 64);
      constexpr uint32_t idesc_o = umma_idesc_bf16(128, 192);
      mbar_arrive_expect_tx(bar_q, 6 * GA_QT);
      for (int kt = 0; kt < 6; ++kt) tma_load_2d(s_q + kt * GA_QT, &tm_q, bar_q, kt * 64, bh * p.Tg + row0);
      // the n-th score issue computes S_j into slot n % GA_SLOTS (n = j in pass 1, nblk + j in pass 2)
      auto issue_s = [&](int n, int j) {
        const int slot = n % GA_SLOTS;
        if (n > 0) mbar_wait(bar_s + (n - 1) % GA_SLOTS, ((n - 1) / GA_SLOTS) & 1);  // MMAs reading K|P of issue n-1 done
        if (n >= GA_SLOTS) mbar_wait(bar_sf + slot, (n / GA_SLOTS - 1) & 1);      // the slot's previous block was read
        const int k0 = j * 64;
        mbar_arrive_expect_tx(bar_kp, 6 * GA_KT);
        for (int kt = 0; kt < 3; ++kt) {
          tma_load_2d(s_kp + kt * GA_KT, &tm_k, bar_kp, kt * 64, bh * kpitch + k0);
          tma_load_2d(s_kp + (3 + kt) * GA_KT, &tm_p, bar_kp, h * 192 + kt * 64, k0);
        }
        if (n == 0) mbar_wait(bar_q, 0);
        mbar_wait(bar_kp, n & 1);
        tc_fence_after();
        const uint32_t qa = smem_u32(s_q), ka = smem_u32(s_kp);
#pragma unroll
        for (int kt = 0; kt < 6; ++kt)
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_s + slot * 64, umma_desc_k_sw128(qa + kt * GA_QT + k * 32), umma_desc_k_sw128(ka + kt * GA_KT + k * 32),
                      idesc_s, (kt | k) != 0);
        umma_commit(bar_s + slot);
      };
      // O += P_j V_j
      auto issue_pv = [&](int j) {
        if (j > 0) mbar_wait(bar_pv, (j - 1) & 1);
        mbar_arrive_expect_tx(bar_v, 192 * 64 * 2);
        tma_load_2d(s_v, &tm_vt, bar_v, j * 64, bh * 192);
        mbar_wait(bar_v, j & 1);
        mbar_wait(bar_p, j & 1);
        tc_fence_after();
        const uint32_t pa = smem_u32(s_p), va = smem_u32(s_v);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_o, umma_desc_k_sw128(pa + k * 32), umma_desc_k_sw128(va + k * 32), idesc_o, (j | k) != 0);
        umma_commit(bar_pv);
      };
      // ---- pass 1: scores (kept in their slots when resident, streamed through the ring for the row maximum otherwise)
      for (int j = 0; j < nblk; ++j) issue_s(j, j);
      // ---- pass 2: P.V (recompute: S_j re-issued up to GA_SLOTS - 1 blocks ahead of the P.V that consumes it)
      if (resident) {
        for (int j = 0; j < nblk; ++j) issue_pv(j);
      } else {
        int n = nblk;
        for (int j = 0; j < nblk; ++j) {
          for (; n < 2 * nblk && n - nblk < j + GA_SLOTS; ++n) issue_s(n, n - nblk);
          issue_pv(j);
        }
      }
    }
  } else {
    const int quad = warp_idx;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = ((uint32_t)(quad * 32)) << 16;
    const float sc = 0.07216878364870322f * 1.4426950408889634f;  // 1/sqrt(192) * log2(e)
    // ---- pass 1: row maximum over all key blocks
    float mx = -INFINITY;
    for (int j = 0; j < nblk; ++j) {
      const int slot = j % GA_SLOTS;
      mbar_wait(bar_s + slot, (j / GA_SLOTS) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t rr[32];
        tmem_ld_32x32b_x32(tmem_s + lane_base + slot * 64 + c * 32, rr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) mx = fmaxf(mx, (j * 64 + c * 32 + i) < klen ? __uint_as_float(rr[i]) : -INFINITY);
      }
      if (!resident) {
        tc_fence_before();
        mbar_arrive(bar_sf + slot);
      }
    }
    const float m_use = (mx == -INFINITY) ? 0.f : mx * sc;
    // ---- pass 2: probabilities block by block, in key order
    float lsum = 0.f;
    for (int j = 0; j < nblk; ++j) {
      if (j > 0) mbar_wait(bar_pv, (j - 1) & 1);  // the probability tile is free again
      int slot = j;
      if (!resident) {
        slot = (nblk + j) % GA_SLOTS;
        mbar_wait(bar_s + slot, ((nblk + j) / GA_SLOTS) & 1);
        tc_fence_after();
      }
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t rr[32];
        tmem_ld_32x32b_x32(tmem_s + lane_base + slot * 64 + c * 32, rr);
        tmem_ld_wait();
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int kk0 = j * 64 + c * 32 + 2 * i;
          const float p0 = (kk0 < klen) ? exp2f(fmaf(__uint_as_float(rr[2 * i]), sc, -m_use)) : 0.f;
          const float p1 = (kk0 + 1 < klen) ? exp2f(fmaf(__uint_as_float(rr[2 * i + 1]), sc, -m_use)) : 0.f;
          const __nv_bfloat162 pb = __floats2bfloat162_rn(p0, p1);
          lsum += __low2float(pb) + __high2float(pb);
          pk[i] = *reinterpret_cast<const uint32_t*>(&pb);
        }
        uint8_t* tile = s_p + r * 128;
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int chunk = c * 4 + q4;
          *reinterpret_cast<uint4*>(tile + ((chunk ^ (r & 7)) << 4)) =
              make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
        }
      }
      tc_fence_before();
      if (!resident) mbar_arrive(bar_sf + slot);  // slot read (tmem_ld_wait above): pass 2 may overwrite it
      fence_proxy_async_smem();
      mbar_arrive(bar_p);
    }
    mbar_wait(bar_pv, (nblk - 1) & 1);
    tc_fence_after();
    const int g = row0 + r;
    const float inv = lsum > 0.f ? 1.0f / lsum : 0.f;
#pragma unroll 1
    for (int c = 0; c < 6; ++c) {
      uint32_t rr[32];
      tmem_ld_32x32b_x32(tmem_o + lane_base + c * 32, rr);
      tmem_ld_wait();
      if (g < p.Tg) {
        const int i0 = h * 192 + c * 32;       // position inside the 768-wide group token
        const int t = 3 * g + i0 / 256;
        if (t < p.T) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i)
            pk[i] = pack_bf16x2(__uint_as_float(rr[2 * i]) * inv, __uint_as_float(rr[2 * i + 1]) * inv);
          uint4* dst = reinterpret_cast<uint4*>(p.out + ((size_t)b * p.T + t) * 256 + (i0 & 255));
#pragma unroll
          for (int i = 0; i < 4; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        }
      }
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 4) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

cudaError_t launch_grouped_attention(const CUtensorMap& tm_q, const CUtensorMap& tm_k, const CUtensorMap& tm_p,
                                     const CUtensorMap& tm_vt, const GroupedAttnParams& p, cudaStream_t st) {
  if (p.H != 4) return cudaErrorInvalidValue;  // any key length: more than GA_SLOTS key blocks take the recompute path
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(grouped_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GA_SMEM_TOTAL);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  dim3 grid((p.Tg + 127) / 128, p.H, p.B);
  cudaError_t le = launch_pdl(grouped_attention_kernel, grid, dim3(GA_THREADS), (size_t)GA_SMEM_TOTAL, st, tm_q, tm_k, tm_p, tm_vt, p);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------------------------
// pos_g[t, 0:256] = linear_pos(pos_emb)[t] for t < T, zero for the padded frames (pad4group, attention.py:73-77); viewed as
// [ceil(T/3), 768] by the attention kernel.
__global__ void grouped_pos_kernel(const __nv_bfloat16* __restrict__ tab, int ldtab, int col0, int T, int Tpad,
                                   __nv_bfloat16* __restrict__ out) {
  const int t = blockIdx.x;
  const int c = threadIdx.x * 8;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (t < T) v = *reinterpret_cast<const uint4*>(tab + (size_t)t * ldtab + col0 + c);
  if (t < Tpad) *reinterpret_cast<uint4*>(out + (size_t)t * 256 + c) = v;
}

cudaError_t launch_grouped_pos(const __nv_bfloat16* tab, int ldtab, int col0, int T, int Tpad, __nv_bfloat16* out,
                               cudaStream_t st) {
  grouped_pos_kernel<<<Tpad, 32, 0, st>>>(tab, ldtab, col0, T, Tpad, out);
  count_launch();
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------------------------
// Strided depthwise conv of the StrideConformerEncoderLayer's conv module + norm + Swish (reference:
// efficient_conformer/convolution.py:57-63,120-129): out[b, to, c] = swish(norm(bias[c] + sum_k w[c,k] g[b, s*to + k - lpad, c]))
// rows before 0 read `pad_left` (causal: GLU(bias), the value of a zero frame after pointwise_conv1 + GLU) or zero,
// rows >= T read zero. One CTA per output frame, thread = channel (C = 256).
__global__ void __launch_bounds__(256)
dwconv_stride_kernel(const __nv_bfloat16* __restrict__ g, const float* __restrict__ w, const float* __restrict__ bias,
                     const float* __restrict__ pad_left, const float* __restrict__ ng, const float* __restrict__ nb,
                     int layer_norm, __nv_bfloat16* __restrict__ z, int T, int Tout, int K, int lpad, int stride, float eps,
                     const int* __restrict__ zero_lens) {
  __shared__ float red[2][8];
  pdl_wait();
  pdl_launch_dependents();
  const int b = blockIdx.y, to = blockIdx.x, c = threadIdx.x;
  const int warp = c >> 5, lane = c & 31;
  float acc = bias[c];
  for (int k = 0; k < K; ++k) {
    const int t = stride * to + k - lpad;
    float v = 0.f;
    if (t < 0) v = pad_left ? pad_left[c] : 0.f;
    else if (t < T) v = __bfloat162float(g[((size_t)b * T + t) * 256 + c]);
    acc = fmaf(w[c * K + k], v, acc);
  }
  float y;
  if (layer_norm) {
    float s = warp_sum(acc);
    if (lane == 0) red[0][warp] = s;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += red[0][i];
    const float mean = tot * (1.0f / 256.0f);
    float q = warp_sum((acc - mean) * (acc - mean));
    if (lane == 0) red[1][warp] = q;
    __syncthreads();
    float qt = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) qt += red[1][i];
    y = (acc - mean) * rsqrtf(qt * (1.0f / 256.0f) + eps) * ng[c] + nb[c];
  } else {
    y = acc * ng[c] + nb[c];  // folded eval-mode BatchNorm
  }
  y = swish_precise(y);
  if (zero_lens && to >= zero_lens[b]) y = 0.f;
  z[((size_t)b * Tout + to) * 256 + c] = __float2bfloat16_rn(y);
}

cudaError_t launch_dwconv_stride(const __nv_bfloat16* g, const float* w, const float* bias, const float* pad_left,
                                 const float* ng, const float* nb, int layer_norm, __nv_bfloat16* z, int B, int T, int Tout,
                                 int C, int K, int lpad, int stride, float eps, const int* zero_lens, cudaStream_t st) {
  if (C != 256) return cudaErrorInvalidValue;
  cudaError_t le = launch_pdl(dwconv_stride_kernel, dim3(Tout, B), dim3(256), (size_t)0, st, g, w, bias, pad_left, ng, nb,
                              layer_norm, z, T, Tout, K, lpad, stride, eps, zero_lens);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

// AvgPool1D(kernel 2, stride 2, ceil_mode, exclusive) over time on the fp32 residual stream (efficient_conformer/
// encoder.py:171-172,523-526): out[b, to] = mean(x[b, 2 to], x[b, 2 to + 1]) or x[b, 2 to] when the second frame is missing.
__global__ void avgpool2_kernel(const float* __restrict__ x, float* __restrict__ out, int T, int Tout, int C) {
  pdl_wait();
  pdl_launch_dependents();
  const int b = blockIdx.y, to = blockIdx.x;
  for (int c = threadIdx.x * 4; c < C; c += blockDim.x * 4) {
    float4 a = *reinterpret_cast<const float4*>(x + ((size_t)b * T + 2 * to) * C + c);
    if (2 * to + 1 < T) {
      const float4 d = *reinterpret_cast<const float4*>(x + ((size_t)b * T + 2 * to + 1) * C + c);
      a.x = (a.x + d.x) * 0.5f, a.y = (a.y + d.y) * 0.5f, a.z = (a.z + d.z) * 0.5f, a.w = (a.w + d.w) * 0.5f;
    }
    *reinterpret_cast<float4*>(out + ((size_t)b * Tout + to) * C + c) = a;
  }
}

cudaError_t launch_avgpool2(const float* x, float* out, int B, int T, int Tout, int C, cudaStream_t st) {
  cudaError_t le = launch_pdl(avgpool2_kernel, dim3(Tout, B), dim3(64), (size_t)0, st, x, out, T, Tout, C);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

}  // namespace ppasr
