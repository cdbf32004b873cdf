// GlobalCMVN + Conv2d(1 -> 256, 3x3, stride 2) + ReLU on the tensor cores (sm_100a), writing the four stride-phase
// images the conv2 GEMM reads (DESIGN.md §3 `phase`).
//
// Reference: ppasr/model_utils/utils/cmvn.py:29-32, ppasr/model_utils/conformer/subsampling.py:84-85,110.
//
// Why a GEMM for a K = 9 convolution: the CUDA-core kernel (kernels.cu::conv1_subsample_kernel) spends ~12 issue slots
// per output element (91 M warp instructions per C2 step, 141 us, 55 % issue utilisation -- ncu r2_conv) while the
// output it has to write (326 MB of bf16) needs ~50 us of HBM time. Here one output row (a conv1 position) is a GEMM
// row, the 256 channels are N, and the 3x3 window is K; the CUDA cores only build the 128-byte im2col row per position
// and convert the accumulators, ~1.2 issue slots per element.
//
// fp32 accuracy from tf32 tensor cores: x = x_hi + x_lo and w = w_hi + w_lo with x_hi, w_hi rounded to tf32
// (10 mantissa bits; x_lo = x - x_hi is exact in fp32 and keeps 10 more bits after its own rounding). The K dimension
// carries  [x_hi | x_lo | x_hi | 1 | 1 | 0 0 0] . [w_hi | w_hi | w_lo | b_hi | b_lo | 0 0 0]  (9 + 9 + 9 + 2 + 3 = 32),
// i.e. every product except x_lo * w_lo (2^-22 relative) and the bias, accumulated in fp32 by the tensor core. The
// result agrees with the fp32 FMA chain of the CUDA-core kernel to ~1e-6 relative, far inside one bf16 ulp.
//
// Tile = 128 consecutive raster rows r = (b*Th + th)*FH + f2 of ONE phase image (ph = 2*(t1&1) + (f1&1),
// t1 = 2 th + pt, f1 = 2 f2 + pf) x 256 channels = 64 KB contiguous in global memory.
//   warps 0-3 : A producers (thread = row): 9 inputs -> normalise -> hi/lo split -> one swizzled 128-byte K-major row
//   warps 4-7 : epilogue: TMEM -> ReLU + bf16 (cvt.rn.relu.bf16x2.f32) -> 128B-swizzled staging -> TMA tensor store
//   warp  8   : MMA issuer (4 x tcgen05.mma kind::tf32 128x256x8 per tile), TMEM alloc (2 x 256 columns)
// Everything is double-buffered (A tile, accumulator, output staging) so the kernel runs at the rate the 64 KB tile
// stores drain to HBM. Rows outside the image (t1 >= T1, f1 >= F1, r >= Mr) are zero K-rows -> relu(0) = 0, as before.
#include <mutex>
#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"

namespace ppasr {

void count_launch();

constexpr int C1_BLOCK_M = 128;
constexpr int C1_N = 256;
constexpr int C1_THREADS = 288;
constexpr int C1_B_BYTES = C1_N * 128;          // 32 KB: [256 channels][32 tf32]
constexpr int C1_A_BYTES = C1_BLOCK_M * 128;    // 16 KB: [128 rows][32 tf32]
constexpr int C1_OUT_BYTES = C1_BLOCK_M * C1_N * 2;  // 64 KB: 4 boxes of [128 rows][64 bf16]
constexpr int C1_SMEM_A = C1_B_BYTES;
constexpr int C1_SMEM_OUT = C1_SMEM_A + 2 * C1_A_BYTES;
constexpr int C1_SMEM_BAR = C1_SMEM_OUT + 2 * C1_OUT_BYTES;
constexpr int C1_SMEM_CMVN = C1_SMEM_BAR + 128;   // mean[256], istd[256]
constexpr int C1_SMEM_TOTAL = C1_SMEM_CMVN + 2048 + 1024;

struct Conv1TcParams {
  const float* feats;  // [B, T, F]
  const float* mean;   // [F]
  const float* istd;   // [F]
  const float* w;      // [256, 9]
  const float* bias;   // [256]
  int B, T, F, T1, F1, Th, FH;
  int Mr;              // B * Th * FH raster rows per phase image
  int mtiles;          // ceil(Mr / 128)
  int num_tiles;       // 4 * mtiles
};

DEVINL uint32_t tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// {lo half: a, hi half: b}, each max(x, 0) rounded to nearest-even bf16
DEVINL uint32_t relu_pack_bf16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
DEVINL void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::tf32, A and B K-major tf32, fp32 accumulate (cute/arch/mma_sm100_desc.hpp: F16F32Format::TF32 = 2)
__host__ __device__ constexpr uint32_t umma_idesc_tf32(uint32_t M, uint32_t N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
DEVINL void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
DEVINL void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
DEVINL void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
DEVINL void bulk_wait_group_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__global__ void __launch_bounds__(C1_THREADS, 1)
conv1_tc_kernel(const __grid_constant__ CUtensorMap tmap_phase, const Conv1TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_b = smem;
  uint8_t* smem_a = smem + C1_SMEM_A;
  uint8_t* smem_out = smem + C1_SMEM_OUT;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + C1_SMEM_BAR);
  uint64_t* a_empty = a_full + 2;
  uint64_t* acc_full = a_empty + 2;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* s_mean = reinterpret_cast<float*>(smem + C1_SMEM_CMVN);
  float* s_istd = s_mean + 256;

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp_idx == 0 && elect_one()) {
    tma_prefetch_desc(&tmap_phase);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], 4);     // one arrival per producer warp
      mbar_init(&a_empty[i], 1);    // tcgen05.commit
      mbar_init(&acc_full[i], 1);   // tcgen05.commit
      mbar_init(&acc_empty[i], 4);  // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp_idx == 8) tmem_alloc<512>(tmem_ptr_smem);
  // B operand (constants, may be read before the grid dependency resolves): [w_hi | w_hi | w_lo | b_hi b_lo 0 0 0]
  for (int idx = threadIdx.x; idx < C1_N * 8; idx += C1_THREADS) {
    const int c = idx >> 3, j = idx & 7;
    uint32_t v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = 4 * j + e;
      uint32_t o = 0;
      if (k < 27) {
        const float w = __ldg(p.w + c * 9 + (k % 9));
        const uint32_t hi = tf32_rna(w);
        o = k < 18 ? hi : tf32_rna(w - __uint_as_float(hi));
      } else if (k < 29) {
        const float b = __ldg(p.bias + c);
        const uint32_t hi = tf32_rna(b);
        o = k == 27 ? hi : tf32_rna(b - __uint_as_float(hi));
      }
      v[e] = o;
    }
    *reinterpret_cast<uint4*>(smem_b + c * 128 + ((j ^ (c & 7)) << 4)) = make_uint4(v[0], v[1], v[2], v[3]);
  }
  for (int i = threadIdx.x; i < p.F; i += C1_THREADS) s_mean[i] = __ldg(p.mean + i), s_istd[i] = __ldg(p.istd + i);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();
  pdl_launch_dependents();

  if (warp_idx < 4) {
    // ===================== A producers: one im2col row per thread =====================
    // The raw inputs of the next two tiles are already in flight (registers) while the current row is converted: the loads
    // miss to L2 / HBM underneath 3+ TB/s of phase-image writes, and one tile period (~1.5 us) does not cover that latency.
    const int row = threadIdx.x;  // 0..127
    const int sw = row & 7;
    float x0[9], x1[9], x2[9];
    int c0 = -1, c1 = -1, c2 = -1;  // first input column of the window (2 * f1), -1 = row outside the image
    auto fetch = [&](int tile, float (&x)[9], int& col) {
      col = -1;
#pragma unroll
      for (int i = 0; i < 9; ++i) x[i] = 0.f;
      if (tile >= p.num_tiles) return;
      const int ph = tile & 3, mt = tile >> 2;
      const int r = mt * C1_BLOCK_M + row;
      const int bl = r / p.FH;
      const int f2 = r - bl * p.FH;
      const int b = bl / p.Th;
      const int th = bl - b * p.Th;
      const int t1 = 2 * th + (ph >> 1), f1 = 2 * f2 + (ph & 1);
      if (r < p.Mr && t1 < p.T1 && f1 < p.F1) {
        col = 2 * f1;
        const float* src = p.feats + ((size_t)b * p.T + 2 * t1) * p.F + col;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) x[kh * 3 + kw] = __ldg(src + kh * p.F + kw);
      }
    };
    fetch(blockIdx.x, x0, c0);
    fetch(blockIdx.x + gridDim.x, x1, c1);
    int s = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      fetch(tile + 2 * gridDim.x, x2, c2);
      const bool valid = c0 >= 0;
      uint32_t hi[9], lo[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) hi[i] = 0u, lo[i] = 0u;
      if (valid) {
        float m[3], sd[3];
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) m[kw] = s_mean[c0 + kw], sd[kw] = s_istd[c0 + kw];
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          const float x = (x0[i] - m[i % 3]) * sd[i % 3];
          const uint32_t h = tf32_rna(x);
          hi[i] = h;
          lo[i] = tf32_rna(x - __uint_as_float(h));
        }
      }
      const uint32_t one = valid ? 0x3F800000u : 0u;
      mbar_wait(&a_empty[s], phase ^ 1);
      uint8_t* arow = smem_a + s * C1_A_BYTES + row * 128;
      // k: 0-8 x_hi, 9-17 x_lo, 18-26 x_hi, 27-28 one, 29-31 zero
      *reinterpret_cast<uint4*>(arow + ((0 ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<uint4*>(arow + ((1 ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
      *reinterpret_cast<uint4*>(arow + ((2 ^ sw) << 4)) = make_uint4(hi[8], lo[0], lo[1], lo[2]);
      *reinterpret_cast<uint4*>(arow + ((3 ^ sw) << 4)) = make_uint4(lo[3], lo[4], lo[5], lo[6]);
      *reinterpret_cast<uint4*>(arow + ((4 ^ sw) << 4)) = make_uint4(lo[7], lo[8], hi[0], hi[1]);
      *reinterpret_cast<uint4*>(arow + ((5 ^ sw) << 4)) = make_uint4(hi[2], hi[3], hi[4], hi[5]);
      *reinterpret_cast<uint4*>(arow + ((6 ^ sw) << 4)) = make_uint4(hi[6], hi[7], hi[8], one);
      *reinterpret_cast<uint4*>(arow + ((7 ^ sw) << 4)) = make_uint4(one, 0u, 0u, 0u);
      fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_full[s]);
      if (++s == 2) s = 0, phase ^= 1;
#pragma unroll
      for (int i = 0; i < 9; ++i) x0[i] = x1[i], x1[i] = x2[i];
      c0 = c1, c1 = c2;
    }
  } else if (warp_idx < 8) {
    // ===================== epilogue: ReLU + bf16 -> swizzled staging -> TMA store =====================
    const int quad = warp_idx - 4;
    const int row = quad * 32 + lane;
    const int sw = row & 7;
    const bool issuer = threadIdx.x == 128;
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int ph = tile & 3, mt = tile >> 2;
      uint8_t* obuf = smem_out + as * C1_OUT_BYTES;
      if (issuer) bulk_wait_group_read<1>();  // the store issued two tiles ago has finished reading this buffer
      named_bar_sync(1, 128);
      mbar_wait(&acc_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + as * C1_N;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + c * 32, v);
        tmem_ld_wait();
        uint8_t* orow = obuf + (c >> 1) * (C1_BLOCK_M * 128) + row * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 o;
          o.x = relu_pack_bf16x2(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]));
          o.y = relu_pack_bf16x2(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
          o.z = relu_pack_bf16x2(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
          o.w = relu_pack_bf16x2(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
          *reinterpret_cast<uint4*>(orow + ((((c & 1) * 4 + j) ^ sw) << 4)) = o;
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();  // staging writes -> visible to the TMA store (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[as]);
      named_bar_sync(1, 128);
      if (issuer) {
#pragma unroll
        for (int g = 0; g < 4; ++g) tma_store_3d(&tmap_phase, obuf + g * (C1_BLOCK_M * 128), g * 64, mt * C1_BLOCK_M, ph);
        bulk_commit_group();
      }
      if (++as == 2) as = 0, aphase ^= 1;
    }
    if (issuer) bulk_wait_group_all();
  } else {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_tf32(C1_BLOCK_M, C1_N);
      const uint32_t b_addr = smem_u32(smem_b);
      int s = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        mbar_wait(&acc_empty[s], phase ^ 1);
        mbar_wait(&a_full[s], phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem_a + s * C1_A_BYTES);
        const uint32_t tmem_d = tmem_base + s * C1_N;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_tf32(tmem_d, umma_desc_k_sw128(a_addr + k * 32), umma_desc_k_sw128(b_addr + k * 32), idesc, k != 0 ? 1u : 0u);
        umma_commit(&a_empty[s]);
        umma_commit(&acc_full[s]);
        if (++s == 2) s = 0, phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 8) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------
// Fused front end: the conv1 GEMM above becomes the A-operand producer of the conv2 GEMM (gemm.cuh CONV mode) -- the phase
// images (326 MB written by conv1, read 2.25x by conv2's nine taps) never exist.
//
// Reference: ppasr/model_utils/conformer/subsampling.py:84-87,110-111 (conv -> ReLU -> conv -> ReLU).
//
// conv2 tile = 128 raster rows R = (b*Th + t')*FH + f' x 256 output channels, K = 9 taps x 256 conv1 channels (36 k-blocks of
// 64, same order as the stand-alone GEMM). For tap (kh, kw) row R needs conv1 at (2t'+kh, 2f'+kw), all 256 channels: ONE
// split-tf32 conv1 GEMM per tap (A1 = [128 rows x 32] im2col of the normalised features, exactly the rows conv1_tc_kernel
// builds), issued as two N = 128 halves ("half-taps") so that the conv1 accumulators double-buffer in 2 x 128 TMEM columns
// next to the 256 columns of the conv2 accumulator.
//   warp 0      : TMA producer of the conv2 weight k-blocks (3 x 32 KB ring)
//   warp 1      : issuer of the conv2 MMAs (bf16 128x256x16, 4 per k-block)
//   warp 3      : issuer of the conv1 MMAs (tf32 128x128x8, 4 per half-tap); runs ahead of warp 1 by the two conv1 accumulators,
//                 so epilogue-1 of half-tap u+1 runs underneath the conv2 k-blocks of u
//   warp 2      : TMEM alloc (512 columns)
//   warps 4-11  : epilogue-2: conv2 accumulator + bias -> ReLU -> bf16 -> compact c2 rows (as EpiConv2)
//   warps 12-15 : A1 producers (thread = row), inputs of the next two taps in flight
//   warps 16-23 : epilogue-1: conv1 accumulator -> ReLU -> bf16 -> the 128B-swizzled K-major A2 tile the conv2 MMA reads
// Arithmetic is identical to conv1_tc_kernel + the CONV GEMM (same MMAs in the same order, same roundings): the two paths
// agree bit for bit (tests/test_gpu_parity.py::test_conv_front_tc_bit_identical).
// ------------------------------------------------------------------------------------------------
constexpr int CF2_THREADS = 768;
constexpr int CF2_A1_BYTES = 128 * 128;   // [128 rows][32 tf32]
constexpr int CF2_A2_BYTES = 128 * 128;   // [128 rows][64 bf16]
constexpr int CF2_B_BYTES = 256 * 128;    // [256 out channels][64 bf16]
constexpr int CF2_B_STAGES = 3;
constexpr int CF2_SMEM_A1 = C1_B_BYTES;                        // W1 first (32 KB)
constexpr int CF2_SMEM_A2 = CF2_SMEM_A1 + 2 * CF2_A1_BYTES;
constexpr int CF2_SMEM_B = CF2_SMEM_A2 + 4 * CF2_A2_BYTES;
constexpr int CF2_SMEM_CMVN = CF2_SMEM_B + CF2_B_STAGES * CF2_B_BYTES;  // mean[96], istd[96]
constexpr int CF2_SMEM_BAR = CF2_SMEM_CMVN + 768;
constexpr int CF2_SMEM_TOTAL = CF2_SMEM_BAR + 256 + 1024;
static_assert(CF2_SMEM_TOTAL <= 232448, "227 KB of dynamic shared memory per CTA");

struct ConvFrontTcParams {
  const float* feats;  // [B, T, F]
  const float* mean;   // [F]
  const float* istd;   // [F]
  const float* w1;     // [256, 9]
  const float* b1;     // [256]
  const float* b2;     // [256]
  __nv_bfloat16* out;  // [B*Tout*Fout, 256]
  int B, T, F, T1, F1;
  int Th, FH;          // raster: Th time rows per utterance, FH = pitch
  int Tout, Fout;      // valid outputs per utterance (T', 19)
  int M;               // B * Th * FH raster rows
  int num_tiles;
};

__global__ void __launch_bounds__(CF2_THREADS, 1)
conv_front_tc_kernel(const __grid_constant__ CUtensorMap tmap_w2, const ConvFrontTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_w1 = smem;
  uint8_t* smem_a1 = smem + CF2_SMEM_A1;
  uint8_t* smem_a2 = smem + CF2_SMEM_A2;
  uint8_t* smem_b = smem + CF2_SMEM_B;
  float* s_mean = reinterpret_cast<float*>(smem + CF2_SMEM_CMVN);
  float* s_istd = s_mean + 96;
  uint64_t* a1_full = reinterpret_cast<uint64_t*>(smem + CF2_SMEM_BAR);
  uint64_t* a1_empty = a1_full + 2;
  uint64_t* acc1_full = a1_empty + 2;
  uint64_t* acc1_empty = acc1_full + 2;
  uint64_t* a2_full = acc1_empty + 2;
  uint64_t* a2_empty = a2_full + 4;
  uint64_t* b_full = a2_empty + 4;
  uint64_t* b_empty = b_full + CF2_B_STAGES;
  uint64_t* acc2_full = b_empty + CF2_B_STAGES;
  uint64_t* acc2_empty = acc2_full + 1;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(acc2_empty + 1);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp_idx == 0 && elect_one()) tma_prefetch_desc(&tmap_w2);
  if (warp_idx == 1 && elect_one()) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a1_full[i], 4);     // one arrival per A1 producer warp
      mbar_init(&a1_empty[i], 1);    // tcgen05.commit after the tap's second half
      mbar_init(&acc1_full[i], 1);   // tcgen05.commit
      mbar_init(&acc1_empty[i], 8);  // one arrival per epilogue-1 warp
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&a2_full[i], 4);     // the four epilogue-1 warps that share a column half
      mbar_init(&a2_empty[i], 1);    // tcgen05.commit
    }
    for (int i = 0; i < CF2_B_STAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    mbar_init(acc2_full, 1);
    mbar_init(acc2_empty, 8);        // one arrival per epilogue-2 warp
    fence_barrier_init();
  }
  if (warp_idx == 2) tmem_alloc<512>(tmem_ptr_smem);
  // conv1 B operand (constants): [w_hi | w_hi | w_lo | b_hi b_lo 0 0 0] per channel, as in conv1_tc_kernel
  for (int idx = threadIdx.x; idx < C1_N * 8; idx += CF2_THREADS) {
    const int c = idx >> 3, j = idx & 7;
    uint32_t v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = 4 * j + e;
      uint32_t o = 0;
      if (k < 27) {
        const float w = __ldg(p.w1 + c * 9 + (k % 9));
        const uint32_t hi = tf32_rna(w);
        o = k < 18 ? hi : tf32_rna(w - __uint_as_float(hi));
      } else if (k < 29) {
        const float b = __ldg(p.b1 + c);
        const uint32_t hi = tf32_rna(b);
        o = k == 27 ? hi : tf32_rna(b - __uint_as_float(hi));
      }
      v[e] = o;
    }
    *reinterpret_cast<uint4*>(smem_w1 + c * 128 + ((j ^ (c & 7)) << 4)) = make_uint4(v[0], v[1], v[2], v[3]);
  }
  for (int i = threadIdx.x; i < p.F; i += CF2_THREADS) s_mean[i] = __ldg(p.mean + i), s_istd[i] = __ldg(p.istd + i);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t tmem_acc1 = tmem_base + 256;
  pdl_wait();
  pdl_launch_dependents();

  const int my_tiles = blockIdx.x < p.num_tiles ? (p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp_idx == 0) {
    // ===================== TMA producer of the conv2 weights =====================
    if (elect_one()) {
      const int total = my_tiles * 36;
      for (int J = 0; J < total; ++J) {
        const int st = J % CF2_B_STAGES;
        mbar_wait(&b_empty[st], ((J / CF2_B_STAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&b_full[st], CF2_B_BYTES);
        tma_load_2d(smem_b + st * CF2_B_BYTES, &tmap_w2, &b_full[st], (J % 36) * 64, 0);
      }
    }
  } else if (warp_idx == 3) {
    // ===================== MMA1 issuer: the split-tf32 conv1 GEMM of every half-tap =====================
    // A thread of its own: it runs ahead of the conv2 issuer as far as the two conv1 accumulators allow, and neither thread's
    // mbarrier round trips delay the other's MMAs (tcgen05.commit tracks the issuing thread's MMAs only).
    if (elect_one()) {
      constexpr uint32_t idesc1 = umma_idesc_tf32(128, 128);
      const uint32_t w1_addr = smem_u32(smem_w1);
      const int total = my_tiles * 18;  // half-taps
      for (int U = 0; U < total; ++U) {
        const int Tn = U >> 1, hh = U & 1, s1 = Tn & 1, sa = U & 1;
        if (hh == 0) mbar_wait(&a1_full[s1], (Tn >> 1) & 1);
        mbar_wait(&acc1_empty[sa], ((U >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem_a1 + s1 * CF2_A1_BYTES);
        const uint32_t b_addr = w1_addr + hh * (128 * 128);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_tf32(tmem_acc1 + sa * 128, umma_desc_k_sw128(a_addr + k * 32), umma_desc_k_sw128(b_addr + k * 32), idesc1,
                    k != 0 ? 1u : 0u);
        umma_commit(&acc1_full[sa]);
        if (hh == 1) umma_commit(&a1_empty[s1]);
      }
    }
  } else if (warp_idx == 1) {
    // ===================== MMA2 issuer: the conv2 k-blocks =====================
    if (elect_one()) {
      constexpr uint32_t idesc2 = umma_idesc_bf16(128, 256);
      const int total = my_tiles * 36;  // k-blocks
      for (int J = 0; J < total; ++J) {
        const int kb = J % 36;
        if (kb == 0) {
          mbar_wait(acc2_empty, ((J / 36) & 1) ^ 1);
          tc_fence_after();
        }
        const int sa2 = J & 3, sb = J % CF2_B_STAGES;
        mbar_wait(&a2_full[sa2], (J >> 2) & 1);
        mbar_wait(&b_full[sb], (J / CF2_B_STAGES) & 1);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem_a2 + sa2 * CF2_A2_BYTES);
        const uint32_t b_addr = smem_u32(smem_b + sb * CF2_B_BYTES);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_base, umma_desc_k_sw128(a_addr + k * 32), umma_desc_k_sw128(b_addr + k * 32), idesc2,
                    (kb | k) != 0 ? 1u : 0u);
        umma_commit(&a2_empty[sa2]);
        umma_commit(&b_empty[sb]);
        if (kb == 35) umma_commit(acc2_full);
      }
    }
  } else if (warp_idx >= 4 && warp_idx < 12) {
    // ===================== epilogue-2: +bias2, ReLU, bf16, compact raster =====================
    const int ew = warp_idx - 4;
    const int quad = ew & 3, half = ew >> 2;
    for (int ti = 0; ti < my_tiles; ++ti) {
      const int tile = blockIdx.x + ti * gridDim.x;
      const int row = tile * C1_BLOCK_M + quad * 32 + lane;
      bool valid = false;
      size_t orow = 0;
      if (row < p.M) {
        const int b = row / (p.Th * p.FH);
        const int rem = row - b * (p.Th * p.FH);
        const int t = rem / p.FH;
        const int f = rem - t * p.FH;
        valid = (t < p.Tout) && (f < p.Fout);
        orow = ((size_t)b * p.Tout + t) * p.Fout + f;
      }
      mbar_wait(acc2_full, ti & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + half * 128;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + c * 32, r);
        tmem_ld_wait();
        if (valid) {
          const int col = half * 128 + c * 32;
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 bv = __ldg(reinterpret_cast<const float4*>(p.b2 + col) + j);
            pk[2 * j] = pack_bf16x2(fmaxf(__uint_as_float(r[4 * j]) + bv.x, 0.f), fmaxf(__uint_as_float(r[4 * j + 1]) + bv.y, 0.f));
            pk[2 * j + 1] =
                pack_bf16x2(fmaxf(__uint_as_float(r[4 * j + 2]) + bv.z, 0.f), fmaxf(__uint_as_float(r[4 * j + 3]) + bv.w, 0.f));
          }
          uint4* dst = reinterpret_cast<uint4*>(p.out + orow * 256 + col);
#pragma unroll
          for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc2_empty);
    }
  } else if (warp_idx >= 12 && warp_idx < 16) {
    // ===================== A1 producers: one im2col row per thread and tap =====================
    const int row = threadIdx.x - 12 * 32;  // 0..127
    const int sw = row & 7;
    const int total = my_tiles * 9;         // taps
    float x0[9], x1[9], x2[9];
    int c0 = -1, c1 = -1, c2 = -1;          // first input column of the window, -1 = zero row
    auto fetch = [&](int Tn, float (&x)[9], int& col) {
      col = -1;
#pragma unroll
      for (int i = 0; i < 9; ++i) x[i] = 0.f;
      if (Tn >= total) return;
      const int ti = Tn / 9, tap = Tn - ti * 9;
      const int kh = tap / 3, kw = tap - kh * 3;
      const int r = (blockIdx.x + ti * gridDim.x) * C1_BLOCK_M + row;
      const int bl = r / p.FH;
      const int f2 = r - bl * p.FH;
      const int b = bl / p.Th;
      const int th = bl - b * p.Th;
      const int t1 = 2 * th + kh, f1 = 2 * f2 + kw;   // conv1 position read by this tap
      if (r < p.M && t1 < p.T1 && f1 < p.F1) {
        col = 2 * f1;
        const float* src = p.feats + ((size_t)b * p.T + 2 * t1) * p.F + col;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) x[i * 3 + j] = __ldg(src + i * p.F + j);
      }
    };
    fetch(0, x0, c0);
    fetch(1, x1, c1);
    for (int Tn = 0; Tn < total; ++Tn) {
      fetch(Tn + 2, x2, c2);
      const bool valid = c0 >= 0;
      uint32_t hi[9], lo[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) hi[i] = 0u, lo[i] = 0u;
      if (valid) {
        float m[3], sd[3];
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) m[kw] = s_mean[c0 + kw], sd[kw] = s_istd[c0 + kw];
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          const float x = (x0[i] - m[i % 3]) * sd[i % 3];
          const uint32_t h = tf32_rna(x);
          hi[i] = h;
          lo[i] = tf32_rna(x - __uint_as_float(h));
        }
      }
      const uint32_t one = valid ? 0x3F800000u : 0u;
      const int s = Tn & 1;
      mbar_wait(&a1_empty[s], ((Tn >> 1) & 1) ^ 1);
      uint8_t* arow = smem_a1 + s * CF2_A1_BYTES + row * 128;
      *reinterpret_cast<uint4*>(arow + ((0 ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<uint4*>(arow + ((1 ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
      *reinterpret_cast<uint4*>(arow + ((2 ^ sw) << 4)) = make_uint4(hi[8], lo[0], lo[1], lo[2]);
      *reinterpret_cast<uint4*>(arow + ((3 ^ sw) << 4)) = make_uint4(lo[3], lo[4], lo[5], lo[6]);
      *reinterpret_cast<uint4*>(arow + ((4 ^ sw) << 4)) = make_uint4(lo[7], lo[8], hi[0], hi[1]);
      *reinterpret_cast<uint4*>(arow + ((5 ^ sw) << 4)) = make_uint4(hi[2], hi[3], hi[4], hi[5]);
      *reinterpret_cast<uint4*>(arow + ((6 ^ sw) << 4)) = make_uint4(hi[6], hi[7], hi[8], one);
      *reinterpret_cast<uint4*>(arow + ((7 ^ sw) << 4)) = make_uint4(one, 0u, 0u, 0u);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&a1_full[s]);
#pragma unroll
      for (int i = 0; i < 9; ++i) x0[i] = x1[i], x1[i] = x2[i];
      c0 = c1, c1 = c2;
    }
  } else if (warp_idx >= 16) {
    // ===================== epilogue-1: conv1 accumulator -> ReLU -> bf16 -> swizzled A2 tile =====================
    const int ew = warp_idx - 16;
    const int quad = ew & 3, ch = ew >> 2;   // TMEM lane quadrant (== warp_idx % 4), 64-channel half of the half-tap
    const int row = quad * 32 + lane;
    const int sw = row & 7;
    const int total = my_tiles * 18;
    for (int U = 0; U < total; ++U) {
      const int sa = U & 1;
      const int J = 2 * U + ch;              // A2 tile = conv2 k-block index
      const int sa2 = J & 3;
      mbar_wait(&acc1_full[sa], (U >> 1) & 1);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      const uint32_t taddr = tmem_acc1 + ((uint32_t)(quad * 32) << 16) + sa * 128 + ch * 64;
      tmem_ld_32x32b_x32(taddr, v0);
      tmem_ld_32x32b_x32(taddr + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc1_empty[sa]);   // the accumulator half is in registers
      mbar_wait(&a2_empty[sa2], ((J >> 2) & 1) ^ 1);
      uint8_t* orow = smem_a2 + sa2 * CF2_A2_BYTES + row * 128;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 o;
        o.x = relu_pack_bf16x2(__uint_as_float(v0[8 * j + 0]), __uint_as_float(v0[8 * j + 1]));
        o.y = relu_pack_bf16x2(__uint_as_float(v0[8 * j + 2]), __uint_as_float(v0[8 * j + 3]));
        o.z = relu_pack_bf16x2(__uint_as_float(v0[8 * j + 4]), __uint_as_float(v0[8 * j + 5]));
        o.w = relu_pack_bf16x2(__uint_as_float(v0[8 * j + 6]), __uint_as_float(v0[8 * j + 7]));
        *reinterpret_cast<uint4*>(orow + ((j ^ sw) << 4)) = o;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 o;
        o.x = relu_pack_bf16x2(__uint_as_float(v1[8 * j + 0]), __uint_as_float(v1[8 * j + 1]));
        o.y = relu_pack_bf16x2(__uint_as_float(v1[8 * j + 2]), __uint_as_float(v1[8 * j + 3]));
        o.z = relu_pack_bf16x2(__uint_as_float(v1[8 * j + 4]), __uint_as_float(v1[8 * j + 5]));
        o.w = relu_pack_bf16x2(__uint_as_float(v1[8 * j + 6]), __uint_as_float(v1[8 * j + 7]));
        *reinterpret_cast<uint4*>(orow + (((4 + j) ^ sw) << 4)) = o;
      }
      fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&a2_full[sa2]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

cudaError_t launch_conv_front_tc(const CUtensorMap& tmap_w2, const float* feats, const float* mean, const float* istd,
                                 const float* w1, const float* b1, const float* b2, __nv_bfloat16* out, int B, int T, int F,
                                 int T1, int F1, int Th, int FH, int Tout, int Fout, int num_sms, cudaStream_t st) {
  static std::once_flag once;
  static cudaError_t cfg_err = cudaSuccess;
  std::call_once(once, [] {
    cfg_err = cudaFuncSetAttribute(conv_front_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CF2_SMEM_TOTAL);
  });
  if (cfg_err != cudaSuccess) return cfg_err;
  if (F > 96) return cudaErrorInvalidValue;  // s_mean / s_istd staging
  ConvFrontTcParams p;
  p.feats = feats, p.mean = mean, p.istd = istd, p.w1 = w1, p.b1 = b1, p.b2 = b2, p.out = out;
  p.B = B, p.T = T, p.F = F, p.T1 = T1, p.F1 = F1, p.Th = Th, p.FH = FH, p.Tout = Tout, p.Fout = Fout;
  p.M = B * Th * FH;
  p.num_tiles = (p.M + C1_BLOCK_M - 1) / C1_BLOCK_M;
  const int grid = p.num_tiles < num_sms ? p.num_tiles : num_sms;
  cudaError_t le = launch_pdl(conv_front_tc_kernel, dim3(grid), dim3(CF2_THREADS), (size_t)CF2_SMEM_TOTAL, st, tmap_w2, p);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t launch_conv1_tc(const CUtensorMap& tmap_phase, const float* feats, const float* mean, const float* istd,
                            const float* w, const float* bias, int B, int T, int F, int T1, int F1, int Th, int FH,
                            int num_sms, cudaStream_t st) {
  static std::once_flag once;
  static cudaError_t cfg_err = cudaSuccess;
  std::call_once(once, [] {
    cfg_err = cudaFuncSetAttribute(conv1_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, C1_SMEM_TOTAL);
  });
  if (cfg_err != cudaSuccess) return cfg_err;
  if (F > 256) return cudaErrorInvalidValue;  // s_mean / s_istd staging
  Conv1TcParams p;
  p.feats = feats, p.mean = mean, p.istd = istd, p.w = w, p.bias = bias;
  p.B = B, p.T = T, p.F = F, p.T1 = T1, p.F1 = F1, p.Th = Th, p.FH = FH;
  p.Mr = B * Th * FH;
  p.mtiles = (p.Mr + C1_BLOCK_M - 1) / C1_BLOCK_M;
  p.num_tiles = 4 * p.mtiles;
  const int grid = p.num_tiles < num_sms ? p.num_tiles : num_sms;
  cudaError_t le = launch_pdl(conv1_tc_kernel, dim3(grid), dim3(C1_THREADS), (size_t)C1_SMEM_TOTAL, st, tmap_phase, p);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

}  // namespace ppasr
