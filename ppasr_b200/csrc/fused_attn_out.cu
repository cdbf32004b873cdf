// Fused tail of the attention block + head of the convolution module for sm_100a, one CTA per 128 rows:
//
//   x <- x + Wo . att + bo                                        (linear_out + residual, encoder.py:389-402)
//   y  = LN(x; g, b)  with pad rows zeroed                        (norm_conv + masked_fill, encoder.py:407-410,
//                                                                  convolution.py:104-106)
//   g_out = GLU(Wpw1 . y + bpw1)                                  (pointwise_conv1 + glu, convolution.py:119-123)
//
// Same row-tile skeleton as fused_ffn.cu. The out-projection starts from zero in the TMEM accumulator (O, columns
// [256,512)) as soon as the att tile has landed; the row owners add the old residual (prefetched into registers with
// coalesced loads while the TMA / MMA run) and bo in the same slab pass that writes x back: v = O + x_old + bo ->
// statistics, x_new -> TMEM O and -> global. They then normalise straight from TMEM and write the bf16 LayerNorm output
// into the (reused) A tiles in shared memory -- y never goes to HBM -- then the 512-wide pointwise_conv1 runs as two
// 128x256x16 MMA groups (gate/value rows are interleaved so GLU is thread-local) and g is written with coalesced stores
// through an smem staging tile.
#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"
#include "row_tile.cuh"

#include <mutex>

namespace ppasr {

void count_launch();

constexpr int AO_THREADS = 384;
constexpr int AO_TILE = 128 * 64 * 2;       // 16 KB
constexpr int AO_SMEM_A = 0;                // 4 tiles: att, later y
constexpr int AO_SMEM_H = 4 * AO_TILE;      // 64 KB scratch: residual slabs, x write-out slabs, exchange
constexpr int AO_SMEM_W = 8 * AO_TILE;      // ring 3 x 32 KB
constexpr int AO_RING = 3;
constexpr int AO_SMEM_BAR = 14 * AO_TILE;
constexpr int AO_SMEM_TOTAL = AO_SMEM_BAR + 512 + 1024;
constexpr int AO_SLAB_PITCH = 68;           // fp32 slab [128][68]
constexpr int AO_G_PITCH = 264;             // bf16 staging [128][264] for g

struct AttnOutParams {
  int M;
  float* x;             // fp32 residual stream, updated in place
  __nv_bfloat16* g;     // bf16 GLU output [M, 256]
  const float* bo;      // [256]
  const float *ln_g, *ln_b;
  const float* bpw1;    // [512] interleaved (value, gate) like the weight rows
  const int* lens;      // valid frames per utterance (nullable): pad rows get y = 0
  int T;
  float eps;
};

__global__ void __launch_bounds__(AO_THREADS, 1)
fused_attn_out_kernel(const __grid_constant__ CUtensorMap tm_att, const __grid_constant__ CUtensorMap tm_wo,
                      const __grid_constant__ CUtensorMap tm_wpw1, const AttnOutParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_a = smem + AO_SMEM_A;
  uint8_t* s_h = smem + AO_SMEM_H;
  uint8_t* s_w = smem + AO_SMEM_W;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + AO_SMEM_BAR);
  uint64_t* a_full = bars;        // TMA att tile
  uint64_t* w_full = bars + 1;    // [3]
  uint64_t* w_empty = bars + 4;   // [3]
  uint64_t* pre_full = bars + 7;  // out-projection accumulated
  uint64_t* a_ready = bars + 8;   // 256: y in A tiles, O drained
  uint64_t* g_full = bars + 9;    // [2] halves of pointwise_conv1
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 11);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * 128;

  if (warp_idx == 0 && elect_one()) {
    tma_prefetch_desc(&tm_att);
    tma_prefetch_desc(&tm_wo);
    tma_prefetch_desc(&tm_wpw1);
  }
  if (warp_idx == 1 && elect_one()) {
    mbar_init(a_full, 1);
    for (int i = 0; i < AO_RING; ++i) {
      mbar_init(&w_full[i], 1);
      mbar_init(&w_empty[i], 1);
    }
    mbar_init(pre_full, 1);
    mbar_init(a_ready, 256);
    mbar_init(&g_full[0], 1);
    mbar_init(&g_full[1], 1);
    fence_barrier_init();
    fence_proxy_async_smem();
  }
  if (warp_idx == 2) tmem_alloc<512>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t tmem_o = tmem_base + 256;
  pdl_wait();
  pdl_launch_dependents();

  if (warp_idx == 0) {
    // ============================ TMA producer ============================
    if (elect_one()) {
      mbar_arrive_expect_tx(a_full, 4 * AO_TILE);
      for (int kb = 0; kb < 4; ++kb) tma_load_2d(s_a + kb * AO_TILE, &tm_att, a_full, kb * 64, m0);
      int slot = 0;
      uint32_t phase = 0;
      auto load_rows256 = [&](const CUtensorMap* tm, int k0, int row0) {
        mbar_wait(&w_empty[slot], phase ^ 1);
        mbar_arrive_expect_tx(&w_full[slot], 2 * AO_TILE);
        tma_load_2d(s_w + slot * 2 * AO_TILE, tm, &w_full[slot], k0, row0);
        if (++slot == AO_RING) slot = 0, phase ^= 1;
      };
      for (int kb = 0; kb < 4; ++kb) load_rows256(&tm_wo, kb * 64, 0);
      for (int nh = 0; nh < 2; ++nh)
        for (int kb = 0; kb < 4; ++kb) load_rows256(&tm_wpw1, kb * 64, nh * 256);
    }
  } else if (warp_idx == 1) {
    // ============================ MMA issuer ============================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, 256);
      int slot = 0;
      uint32_t phase = 0;
      const uint32_t a_addr = smem_u32(s_a);
      auto gemm256 = [&](uint32_t tmem_d) {
        for (int kb = 0; kb < 4; ++kb) {
          mbar_wait(&w_full[slot], phase);
          tc_fence_after();
          const uint32_t w_addr = smem_u32(s_w + slot * 2 * AO_TILE);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_d, umma_desc_k_sw128(a_addr + kb * AO_TILE + k * 32), umma_desc_k_sw128(w_addr + k * 32), idesc,
                      (kb | k) != 0 ? 1u : 0u);
          umma_commit(&w_empty[slot]);
          if (++slot == AO_RING) slot = 0, phase ^= 1;
        }
      };
      mbar_wait(a_full, 0);
      tc_fence_after();
      gemm256(tmem_o);  // O = att . Wo^T (the row owners add the residual)
      umma_commit(pre_full);
      mbar_wait(a_ready, 0);  // y replaced att in the A tiles; O has been drained
      tc_fence_after();
      gemm256(tmem_base);  // G[:, 0:256]
      umma_commit(&g_full[0]);
      gemm256(tmem_o);     // G[:, 256:512]
      umma_commit(&g_full[1]);
    }
  } else if (warp_idx >= 4) {
    // ============================ compute warps ============================
    const int ew = warp_idx - 4;
    const int quad = ew & 3;
    const int half = ew >> 2;
    const int r = quad * 32 + lane;
    const int ct = threadIdx.x - 128;
    const uint32_t lane_base = ((uint32_t)(quad * 32)) << 16;
    const int row_g = m0 + r;
    bool pad = false;
    if (p.lens != nullptr && row_g < p.M) {
      const int b = row_g / p.T;
      pad = (row_g - b * p.T) >= __ldg(p.lens + b);
    }
    float* slab = reinterpret_cast<float*>(s_h);
    const int cq = ct & 15;
    float4 pre[8];  // this thread's share of the next residual slab (16 rows apart, 16 B per row segment)
    auto prefetch = [&](int s) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = (ct >> 4) + 16 * i;
        pre[i] = ((m0 + rr) < p.M) ? __ldcg(reinterpret_cast<const float4*>(p.x + (size_t)(m0 + rr) * 256 + s * 64) + cq)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    prefetch(0);
    mbar_wait(pre_full, 0);
    tc_fence_after();
    FfnStat st{0.f, 0.f, 0.f};
    for (int s = 0; s < 4; ++s) {
#pragma unroll
      for (int i = 0; i < 8; ++i) *reinterpret_cast<float4*>(slab + ((ct >> 4) + 16 * i) * AO_SLAB_PITCH + cq * 4) = pre[i];
      if (s + 1 < 4) prefetch(s + 1);
      named_bar_sync(1, 256);
      if (half == (s >> 1)) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int cc = s * 64 + c * 32;
          uint32_t ro[32];
          tmem_ld_32x32b_x32(tmem_o + lane_base + cc, ro);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 xo = *reinterpret_cast<const float4*>(slab + r * AO_SLAB_PITCH + c * 32 + 4 * j);
            const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bo + cc) + j);
            v[4 * j + 0] = __uint_as_float(ro[4 * j + 0]) + xo.x + bb.x;
            v[4 * j + 1] = __uint_as_float(ro[4 * j + 1]) + xo.y + bb.y;
            v[4 * j + 2] = __uint_as_float(ro[4 * j + 2]) + xo.z + bb.z;
            v[4 * j + 3] = __uint_as_float(ro[4 * j + 3]) + xo.w + bb.w;
            *reinterpret_cast<float4*>(slab + r * AO_SLAB_PITCH + c * 32 + 4 * j) =
                make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            ro[4 * j + 0] = __float_as_uint(v[4 * j + 0]), ro[4 * j + 1] = __float_as_uint(v[4 * j + 1]);
            ro[4 * j + 2] = __float_as_uint(v[4 * j + 2]), ro[4 * j + 3] = __float_as_uint(v[4 * j + 3]);
          }
          tmem_st_32x32b_x32(tmem_o + lane_base + cc, ro);  // x_new stays in O for the LayerNorm pass
          ffn_add_chunk(st, v);
        }
      }
      named_bar_sync(1, 256);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = (ct >> 4) + 16 * i;
        if ((m0 + rr) < p.M)
          *(reinterpret_cast<float4*>(p.x + (size_t)(m0 + rr) * 256 + s * 64) + cq) =
              *reinterpret_cast<const float4*>(slab + rr * AO_SLAB_PITCH + cq * 4);
      }
      named_bar_sync(1, 256);
    }
    tmem_st_wait();
    float4* sc = reinterpret_cast<float4*>(s_h + 128 * AO_SLAB_PITCH * 4);
    ffn_exchange(st, sc, r, half, 2);
    const float mean = st.mean;
    const float rstd = rsqrtf(st.m2 * (1.0f / 256.0f) + p.eps);
    // y = LN(x_new) -> A tiles (this thread's 128 columns, read back from O)
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      const int cc = half * 128 + c * 32;
      uint32_t ro[32];
      tmem_ld_32x32b_x32(tmem_o + lane_base + cc, ro);
      tmem_ld_wait();
      uint32_t pk[16];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 gg = __ldg(reinterpret_cast<const float4*>(p.ln_g + cc) + j);
        const float4 bb = __ldg(reinterpret_cast<const float4*>(p.ln_b + cc) + j);
        const float y0 = (__uint_as_float(ro[4 * j + 0]) - mean) * rstd * gg.x + bb.x;
        const float y1 = (__uint_as_float(ro[4 * j + 1]) - mean) * rstd * gg.y + bb.y;
        const float y2 = (__uint_as_float(ro[4 * j + 2]) - mean) * rstd * gg.z + bb.z;
        const float y3 = (__uint_as_float(ro[4 * j + 3]) - mean) * rstd * gg.w + bb.w;
        pk[2 * j] = pad ? 0u : pack_bf16x2(y0, y1);
        pk[2 * j + 1] = pad ? 0u : pack_bf16x2(y2, y3);
      }
      uint8_t* atile = s_a + (cc >> 6) * AO_TILE + r * 128;
      const int ch0 = (cc & 63) >> 3;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4)
        *reinterpret_cast<uint4*>(atile + (((ch0 + q4) ^ (r & 7)) << 4)) =
            make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
    }
    tc_fence_before();
    fence_proxy_async_smem();
    mbar_arrive(a_ready);
    // ---- GLU epilogue: G columns (2c, 2c+1) = (value, gate) of channel c; staged for coalesced stores ----
    __nv_bfloat16* gs = reinterpret_cast<__nv_bfloat16*>(smem);  // [128][AO_G_PITCH] over the A + H regions
    mbar_wait(&g_full[half], 0);
    tc_fence_after();
    if (half == 0) {
      // both halves must be complete before the staging tile may overwrite the A tiles (MMA operands)
      mbar_wait(&g_full[1], 0);
      tc_fence_after();
    }
    named_bar_sync(1, 256);
#pragma unroll 1
    for (int c = 0; c < 8; c += 2) {
      uint32_t ro[2][32];
      tmem_ld_32x32b_x32(tmem_base + lane_base + half * 256 + c * 32, ro[0]);
      tmem_ld_32x32b_x32(tmem_base + lane_base + half * 256 + c * 32 + 32, ro[1]);
      tmem_ld_wait();
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int gc = half * 256 + (c + u) * 32;  // first G column of this chunk
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bpw1 + gc) + j);
          const float a0 = __uint_as_float(ro[u][4 * j + 0]) + bb.x;
          const float g0 = __uint_as_float(ro[u][4 * j + 1]) + bb.y;
          const float a1 = __uint_as_float(ro[u][4 * j + 2]) + bb.z;
          const float g1 = __uint_as_float(ro[u][4 * j + 3]) + bb.w;
          pk[j] = pack_bf16x2(a0 * sigmoid_f(g0), a1 * sigmoid_f(g1));
        }
        uint4* dst = reinterpret_cast<uint4*>(gs + (size_t)r * AO_G_PITCH + (gc >> 1));
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
    }
    named_bar_sync(1, 256);
    for (int row = ew; row < 128; row += 8) {
      if (m0 + row >= p.M) break;
      const uint4 v = *reinterpret_cast<const uint4*>(gs + (size_t)row * AO_G_PITCH + lane * 8);
      *reinterpret_cast<uint4*>(p.g + (size_t)(m0 + row) * 256 + lane * 8) = v;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

cudaError_t launch_fused_attn_out(const CUtensorMap& tm_att, const CUtensorMap& tm_wo, const CUtensorMap& tm_wpw1, int M,
                                  float* x, __nv_bfloat16* g, const float* bo, const float* ln_g, const float* ln_b,
                                  const float* bpw1, const int* lens, int T, float eps, cudaStream_t st) {
  if (M <= 0) return cudaErrorInvalidValue;
  static std::once_flag once;
  static cudaError_t cfg_err = cudaSuccess;
  std::call_once(once, [] {
    cfg_err = cudaFuncSetAttribute(fused_attn_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AO_SMEM_TOTAL);
  });
  if (cfg_err != cudaSuccess) return cfg_err;
  AttnOutParams p;
  p.M = M, p.x = x, p.g = g, p.bo = bo, p.ln_g = ln_g, p.ln_b = ln_b, p.bpw1 = bpw1, p.lens = lens, p.T = T, p.eps = eps;
  cudaError_t le = launch_pdl(fused_attn_out_kernel, dim3((M + 127) / 128), dim3(AO_THREADS), (size_t)AO_SMEM_TOTAL, st, tm_att,
                              tm_wo, tm_wpw1, p);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

}  // namespace ppasr
