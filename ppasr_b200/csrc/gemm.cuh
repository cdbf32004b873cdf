// Persistent warp-specialised bf16 GEMM for sm_100a:  C[M,N] = epilogue(A[M,K] * W[N,K]^T)
//
//   warp 0       : TMA producer   (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx-count)
//   warp 1       : MMA issuer     (one elected thread, tcgen05.mma cta_group::1 kind::f16, 128 x BLOCK_N x 16)
//   warp 2       : TMEM allocator (tcgen05.alloc / dealloc)
//   warps 4..11  : epilogue       (tcgen05.ld 32x32b -> registers -> fused epilogue -> global).
//                  Warp w reads TMEM lane quadrant w%4; warps 4..7 take the low half of the tile's
//                  columns, warps 8..11 the high half. The tile's bias slice is staged in smem.
//
// Accumulators live in TMEM (fp32), double buffered so the epilogue of tile i overlaps the MMAs of
// tile i+1. A and W are both K-major bf16 (PyTorch "Linear.weight [out,in]" layout for W).
//
// The CONV template flag turns the k-loop into the 9-tap "shifted GEMM" used for the second
// subsampling convolution (reference: ppasr/model_utils/conformer/subsampling.py:84-87,110-111):
// A is a 3-D tensor [phase(4)][row][256] and k-block kb reads tap kb/kc at row offset
// (kh>>1)*pitch + (kw>>1) of phase (kh&1)*2 + (kw&1).
#pragma once
#include "launch.h"
#include "ptx.cuh"

namespace ppasr {

void count_launch();

constexpr int GEMM_BLOCK_M = 128;
constexpr int GEMM_BLOCK_K = 64;  // 64 bf16 = 128 bytes = one swizzle-128B row
constexpr int GEMM_UMMA_K = 16;
constexpr int GEMM_EPI_WARPS = 8;
constexpr int GEMM_THREADS = 128 + GEMM_EPI_WARPS * 32;  // 384

struct GemmShape {
  int M;             // rows of A / C actually valid
  int N;             // valid output columns
  int num_k_blocks;  // K / 64 (for CONV: 9 taps * Cin/64)
  int num_m_tiles;
  int num_n_tiles;
  int conv_pitch;    // CONV only: row pitch of the (t, f) raster (20)
  int conv_kc;       // CONV only: k-blocks per tap (Cin / 64)
};

template <int BLOCK_N, int STAGES>
struct GemmSmem {
  static constexpr int A_BYTES = GEMM_BLOCK_M * GEMM_BLOCK_K * 2;
  static constexpr int B_BYTES = BLOCK_N * GEMM_BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BIAS_OFFSET = STAGES * STAGE_BYTES;       // 2 x BLOCK_N floats
  static constexpr int SCRATCH_OFFSET = BIAS_OFFSET + 2 * BLOCK_N * 4;  // epilogue exchange area (LayerNorm stats)
  static constexpr int SCRATCH_BYTES = 2 * 128 * 2 * 16;
  static constexpr int BAR_OFFSET = SCRATCH_OFFSET + SCRATCH_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + 256 + 1024;           // + barriers + alignment slack
};

template <int BLOCK_N>
struct GemmAcc {
  static constexpr int ACC_STAGES = (BLOCK_N * 2 <= 512) ? 2 : 1;
  static constexpr int TMEM_COLS = (BLOCK_N * ACC_STAGES <= 32)    ? 32
                                   : (BLOCK_N * ACC_STAGES <= 64)  ? 64
                                   : (BLOCK_N * ACC_STAGES <= 128) ? 128
                                   : (BLOCK_N * ACC_STAGES <= 256) ? 256
                                                                   : 512;
};

// ------------------------------------------------------------------------------------------------
// Epilogue helpers. Every epilogue functor implements
//   __device__ void tile(uint32_t taddr, int row, int n0, int n_tile, int half, const float* sbias, float4* scratch) const
// where taddr addresses (this thread's TMEM lane, first column of the accumulator stage), `row` is
// the global output row owned by this thread, n0 the first output column of the tile, `half`
// selects which BLOCK_N/2 columns this warp handles and sbias[j] is the bias of column n0 + j.
// ------------------------------------------------------------------------------------------------
enum : int { ACT_NONE = 0, ACT_RELU = 1, ACT_SWISH = 2 };

template <int ACT>
DEVINL float apply_act(float v) {
  if (ACT == ACT_RELU) return fmaxf(v, 0.0f);
  if (ACT == ACT_SWISH) return swish_f(v);
  return v;
}

// Software-pipelined walk over this warp's NCH 32-column chunks: the TMEM load of chunk c+1 is in
// flight while chunk c is processed. f(cc, r) gets the chunk's column offset inside the tile.
template <int BLOCK_N, int PARTS = 2, class F>
DEVINL void epi_for_chunks(uint32_t taddr, int half, F&& f) {
  constexpr int NCH = BLOCK_N / (32 * PARTS);
  static_assert(NCH >= 1, "a column part is at least one 32-column chunk");
  const int c0 = half * NCH;
  uint32_t r[2][32];
  tmem_ld_32x32b_x32(taddr + c0 * 32, r[0]);
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    tmem_ld_wait();
    if (c + 1 < NCH) tmem_ld_32x32b_x32(taddr + (c0 + c + 1) * 32, r[(c + 1) & 1]);
    f((c0 + c) * 32, r[c & 1]);
  }
}

// out_bf16[row, n] = act(acc + bias[n])
template <int BLOCK_N, int ACT>
struct EpiStoreBF16 {
  __nv_bfloat16* out;
  const float* bias;
  int ldo;  // elements
  int M, N;
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (row < M && col < N) {
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bv = *reinterpret_cast<const float4*>(sbias + cc + 4 * j);
          pk[2 * j] = pack_bf16x2(apply_act<ACT>(__uint_as_float(r[4 * j]) + bv.x),
                                  apply_act<ACT>(__uint_as_float(r[4 * j + 1]) + bv.y));
          pk[2 * j + 1] = pack_bf16x2(apply_act<ACT>(__uint_as_float(r[4 * j + 2]) + bv.z),
                                      apply_act<ACT>(__uint_as_float(r[4 * j + 3]) + bv.w));
        }
        uint4* dst = reinterpret_cast<uint4*>(out + (size_t)row * ldo + col);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      }
    });
  }
};

// Residual-stream update in fp32:  x[row, n] = (residual ? x[row, n] : 0) + alpha * (acc + bias[n])
// Rows with t >= valid_len[b] contribute 0 when `lens` is given (conv-module pad masking,
// reference: ppasr/model_utils/conformer/convolution.py:138-140).
template <int BLOCK_N>
struct EpiResidF32 {
  float* x;
  const float* bias;
  int ldx;
  int M, N;
  float alpha;
  int residual;
  const int* lens;  // per-utterance valid frame count (nullable)
  int T;            // frames per utterance (row = b*T + t)
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    bool masked = false;
    if (lens != nullptr && row < M) {
      int b = row / T;
      masked = (row - b * T) >= __ldg(lens + b);
    }
    const float a = masked ? 0.f : alpha;
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (row < M && col < N) {
        float4* dst = reinterpret_cast<float4*>(x + (size_t)row * ldx + col);
        float4 o[8];
        if (residual) {
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = dst[j];  // all 8 loads in flight before first use
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bv = *reinterpret_cast<const float4*>(sbias + cc + 4 * j);
          o[j].x = fmaf(a, __uint_as_float(r[4 * j + 0]) + bv.x, o[j].x);
          o[j].y = fmaf(a, __uint_as_float(r[4 * j + 1]) + bv.y, o[j].y);
          o[j].z = fmaf(a, __uint_as_float(r[4 * j + 2]) + bv.z, o[j].z);
          o[j].w = fmaf(a, __uint_as_float(r[4 * j + 3]) + bv.w, o[j].w);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[j] = o[j];
      }
    });
  }
};

// Residual update fused with the LayerNorm(s) that follow it. Requires BLOCK_N == N == 256: the CTA owns
// complete rows (two epilogue threads per row, 128 columns each; statistics are combined through shared
// memory with Chan's parallel mean/M2 update, so the variance is as robust as a two-pass LayerNorm).
//   x_new = (residual ? x : 0) + alpha * (acc + bias)         (rows t >= lens[b] keep x when mask_resid)
//   single (g2 == null): y = LN(x_new; g1, b1)                (rows t >= lens[b] -> 0 when zero_y_pad)
//   double            : x <- LN(x_new; g1, b1),  y = LN(x; g2, b2)
// TMEM plan (kXbuf): one accumulator stage in columns [0,256) and a 256-column "X buffer" in [256,512).
// While the mainloop runs, the epilogue threads prefetch the fp32 residual tile into the X buffer; pass 1
// writes x_new back over the accumulator columns, so the later passes read TMEM instead of re-reading HBM.
// Reference: the LayerNorms of ConformerEncoderLayer (conformer/encoder.py:327-336, 380-429) following
// feed_forward_macaron / self_attn / conv_module / feed_forward, and `after_norm` (encoder.py:201-202).
template <int BLOCK_N>
struct EpiResidLN {
  static constexpr int kXbuf = 1;
  float* x;
  const float* bias;
  int ldx;
  int M, N;
  float alpha;
  int residual;
  const int* lens;
  int T;
  int mask_resid;
  int zero_y_pad;
  const float *g1, *b1, *g2, *b2;
  __nv_bfloat16* y;
  float eps;
  // post-norm models (Squeezeformer, squeezeformer/encoder.py:468-504): with g2 != null and y_affine the bf16 output is the
  // element-wise affine y = g2 * x + b2 of the stored fp32 row (the next module's adaptive scale/bias, attention.py:120-123)
  // instead of a second LayerNorm; no_norm additionally skips LN1 (x = x_new; time-reduction output, encoder.py:213).
  int y_affine = 0;
  int no_norm = 0;

  struct Stat {
    float n, mean, m2;
  };
  static DEVINL void chan(Stat& a, float nb, float mb, float m2b) {
    const float n = a.n + nb;
    const float d = mb - a.mean;
    a.mean += d * (nb / n);
    a.m2 += m2b + d * d * (a.n * nb / n);
    a.n = n;
  }
  static DEVINL void add_chunk(Stat& a, const float (&v)[32]) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) s += v[j];
    const float m = s * (1.0f / 32.0f);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) q += (v[j] - m) * (v[j] - m);
    if (a.n == 0.f) {
      a.n = 32.f, a.mean = m, a.m2 = q;
    } else {
      chan(a, 32.f, m, q);
    }
  }
  // combine with the partner thread that owns the other 128 columns of this row
  static DEVINL void exchange(Stat& a, float4* scratch, int r, int half) {
    scratch[r * 2 + half] = make_float4(a.n, a.mean, a.m2, 0.f);
    named_bar_sync(2, GEMM_EPI_WARPS * 32);
    const float4 o = scratch[r * 2 + (half ^ 1)];
    // fixed combination order (half 0 then half 1) so both partner threads get bit-identical statistics
    const float4 lo = half ? o : make_float4(a.n, a.mean, a.m2, 0.f);
    const float4 hi = half ? make_float4(a.n, a.mean, a.m2, 0.f) : o;
    Stat t{lo.x, lo.y, lo.z};
    chan(t, hi.x, hi.y, hi.z);
    a = t;
  }

  // residual tile -> TMEM X buffer (runs while the MMAs of this tile are in flight)
  DEVINL void prefetch(uint32_t taddr_x, int row, int half) const {
    if (!residual) return;
    constexpr int NCH = BLOCK_N / 64;
    const bool in = row < M;
    const float* xr = x + (size_t)(in ? row : 0) * ldx;
#pragma unroll
    for (int c = 0; c < NCH; c += 2) {
      uint32_t v[2][32];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int cc = (half * NCH + c + u) * 32;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 t = in ? __ldcg(reinterpret_cast<const float4*>(xr + cc) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
          v[u][4 * j] = __float_as_uint(t.x), v[u][4 * j + 1] = __float_as_uint(t.y);
          v[u][4 * j + 2] = __float_as_uint(t.z), v[u][4 * j + 3] = __float_as_uint(t.w);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) tmem_st_32x32b_x32(taddr_x + (half * NCH + c + u) * 32, v[u]);
    }
    tmem_st_wait();
  }

  // taddr: accumulator columns of this thread's lane; taddr + BLOCK_N: the X buffer
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4* scratch) const {
    static_assert(BLOCK_N == 256, "EpiResidLN needs the whole 256-wide row in one CTA");
    constexpr int NCH = BLOCK_N / 64;
    const int r = row & (GEMM_BLOCK_M - 1);
    const bool in = row < M;
    bool pad = false;
    if (lens != nullptr && in) {
      const int b = row / T;
      pad = (row - b * T) >= __ldg(lens + b);
    }
    const float a = (pad && mask_resid) ? 0.f : alpha;
    float* xr = x + (size_t)row * ldx;
    Stat st{0.f, 0.f, 0.f};
    // pass 1: x_new = x_old + a * (acc + bias) -> TMEM (over the accumulator) [+ global when it is final]
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
      const int cc = (half * NCH + c) * 32;
      uint32_t ra[32], rx[32];
      tmem_ld_32x32b_x32(taddr + cc, ra);
      if (residual) tmem_ld_32x32b_x32(taddr + BLOCK_N + cc, rx);
      tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float xo = residual ? __uint_as_float(rx[j]) : 0.f;
        v[j] = fmaf(a, __uint_as_float(ra[j]) + sbias[cc + j], xo);
        ra[j] = __float_as_uint(v[j]);
      }
      tmem_st_32x32b_x32(taddr + cc, ra);
      if (in && (g2 == nullptr || no_norm)) {
        float4* dst = reinterpret_cast<float4*>(xr + cc);
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
      add_chunk(st, v);
    }
    tmem_st_wait();
    exchange(st, scratch, r, half);
    float mean = st.mean;
    float rstd = rsqrtf(st.m2 * (1.0f / 256.0f) + eps);
    if (g2 != nullptr && !no_norm) {
      // pass 2: x <- LN1(x_new) (final residual stream value) -> global + TMEM, statistics of the result
      Stat s2{0.f, 0.f, 0.f};
#pragma unroll 1
      for (int c = 0; c < NCH; ++c) {
        const int cc = (half * NCH + c) * 32;
        uint32_t ra[32];
        tmem_ld_32x32b_x32(taddr + cc, ra);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 gv = __ldg(reinterpret_cast<const float4*>(g1 + cc) + j);
          const float4 bv = __ldg(reinterpret_cast<const float4*>(b1 + cc) + j);
          v[4 * j + 0] = (__uint_as_float(ra[4 * j + 0]) - mean) * rstd * gv.x + bv.x;
          v[4 * j + 1] = (__uint_as_float(ra[4 * j + 1]) - mean) * rstd * gv.y + bv.y;
          v[4 * j + 2] = (__uint_as_float(ra[4 * j + 2]) - mean) * rstd * gv.z + bv.z;
          v[4 * j + 3] = (__uint_as_float(ra[4 * j + 3]) - mean) * rstd * gv.w + bv.w;
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) ra[j] = __float_as_uint(v[j]);
        tmem_st_32x32b_x32(taddr + cc, ra);
        if (in) {
          float4* dst = reinterpret_cast<float4*>(xr + cc);
#pragma unroll
          for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        add_chunk(s2, v);
      }
      tmem_st_wait();
      if (!y_affine) {
        exchange(s2, scratch + 2 * GEMM_BLOCK_M, r, half);
        mean = s2.mean;
        rstd = rsqrtf(s2.m2 * (1.0f / 256.0f) + eps);
      }
    }
    if (g2 != nullptr && y_affine) mean = 0.f, rstd = 1.f;
    // final pass: y = LN(x; gl, bl) as bf16
    const float* gl = g2 ? g2 : g1;
    const float* bl = g2 ? b2 : b1;
    const bool zero = pad && zero_y_pad;
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
      const int cc = (half * NCH + c) * 32;
      uint32_t ra[32];
      tmem_ld_32x32b_x32(taddr + cc, ra);
      tmem_ld_wait();
      if (in) {
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 gv = __ldg(reinterpret_cast<const float4*>(gl + cc) + j);
          const float4 bv = __ldg(reinterpret_cast<const float4*>(bl + cc) + j);
          const float y0 = (__uint_as_float(ra[4 * j + 0]) - mean) * rstd * gv.x + bv.x;
          const float y1 = (__uint_as_float(ra[4 * j + 1]) - mean) * rstd * gv.y + bv.y;
          const float y2 = (__uint_as_float(ra[4 * j + 2]) - mean) * rstd * gv.z + bv.z;
          const float y3 = (__uint_as_float(ra[4 * j + 3]) - mean) * rstd * gv.w + bv.w;
          pk[2 * j] = zero ? 0u : pack_bf16x2(y0, y1);
          pk[2 * j + 1] = zero ? 0u : pack_bf16x2(y2, y3);
        }
        uint4* dst = reinterpret_cast<uint4*>(y + (size_t)row * BLOCK_N + cc);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      }
    }
  }
};

// Squeezeformer recover step (squeezeformer/encoder.py:216-230): the GEMM rows are the time-reduced frames (b, tr);
//   v = acc + bias  = time_recover_layer(x_reduced[b, tr])
//   for t in {2 tr, 2 tr + 1} (t < T):  x[b, t] <- x[b, t] + v  (x holds the activations saved before the reduction)
//                                       y[b, t]  = ada_scale * x[b, t] + ada_bias   (bf16, next module's input)
// i.e. repeat_interleave(xs, 2) -> Linear -> [:T] -> + recover_tensor without materialising the repeated tensor.
template <int BLOCK_N>
struct EpiRecover {
  float* x;           // [B*T, N] fp32 (in/out)
  __nv_bfloat16* y;   // [B*T, N]
  const float* bias;
  const float *ys, *yb;  // affine of the bf16 output
  int M;              // B * Tr reduced rows
  int N;
  int Tr, T;
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    const bool in = row < M;
    const int b = in ? row / Tr : 0;
    const int tr = row - b * Tr;
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (!in || col >= N) return;
#pragma unroll 1
      for (int u = 0; u < 2; ++u) {
        const int t = 2 * tr + u;
        if (t >= T) break;
        float* xr = x + ((size_t)b * T + t) * N + col;
        __nv_bfloat16* yr = y + ((size_t)b * T + t) * N + col;
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 xo = *reinterpret_cast<const float4*>(xr + 4 * j);
          const float4 bv = *reinterpret_cast<const float4*>(sbias + cc + 4 * j);
          const float4 sv = __ldg(reinterpret_cast<const float4*>(ys + col) + j);
          const float4 ov = __ldg(reinterpret_cast<const float4*>(yb + col) + j);
          xo.x += __uint_as_float(r[4 * j + 0]) + bv.x;
          xo.y += __uint_as_float(r[4 * j + 1]) + bv.y;
          xo.z += __uint_as_float(r[4 * j + 2]) + bv.z;
          xo.w += __uint_as_float(r[4 * j + 3]) + bv.w;
          *reinterpret_cast<float4*>(xr + 4 * j) = xo;
          pk[2 * j] = pack_bf16x2(fmaf(sv.x, xo.x, ov.x), fmaf(sv.y, xo.y, ov.y));
          pk[2 * j + 1] = pack_bf16x2(fmaf(sv.z, xo.z, ov.z), fmaf(sv.w, xo.w, ov.w));
        }
        uint4* dst = reinterpret_cast<uint4*>(yr);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      }
    });
  }
};

// GLU over interleaved columns: packed column 2c = "a" channel c, 2c+1 = gate channel c.
// out_bf16[row, c] = (acc_a + bias_a) * sigmoid(acc_b + bias_b)
// (reference: ppasr/model_utils/conformer/convolution.py:121-123, paddle glu = a * sigmoid(b))
template <int BLOCK_N>
struct EpiGLU {
  __nv_bfloat16* out;
  const float* bias;  // interleaved like the weight rows
  int ldo;
  int M, N;  // N = 2 * channels
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (row < M && col < N) {
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bv = *reinterpret_cast<const float4*>(sbias + cc + 4 * j);
          float a0 = __uint_as_float(r[4 * j + 0]) + bv.x;
          float g0 = __uint_as_float(r[4 * j + 1]) + bv.y;
          float a1 = __uint_as_float(r[4 * j + 2]) + bv.z;
          float g1 = __uint_as_float(r[4 * j + 3]) + bv.w;
          pk[j] = pack_bf16x2(a0 * sigmoid_f(g0), a1 * sigmoid_f(g1));
        }
        uint4* dst = reinterpret_cast<uint4*>(out + (size_t)row * ldo + (col >> 1));
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
    });
  }
};

// Fused QKV projection epilogue (reference: ppasr/model_utils/conformer/attention.py:76-84,235-245).
// Packed output columns: [0,D) = q, [D,2D) = k, [2D,3D) = v  with column = h*64 + d.
//   q2[b,h,t, 0:64 ] = q + pos_bias_u[h]      (bf16)
//   q2[b,h,t,64:128] = q + pos_bias_v[h]
//   kk[b,h,tk,0:64 ] = k                      (tk = kofs + t : KV-cache append position)
//   vt[b,h,d,tk]     = v  (transposed so P.V^T is a K-major UMMA B operand)
template <int BLOCK_N>
struct EpiQKV {
  static constexpr int kEpiWarps = 16;  // four column parts, one 32-column chunk per warp and 128-wide tile
  __nv_bfloat16* q2;
  __nv_bfloat16* kk;
  __nv_bfloat16* vt;
  const float* bias;    // [3D]
  const float* bias_u;  // [H*64]
  const float* bias_v;  // [H*64]
  int M;                // B*T
  int T;                // new frames per utterance
  int H;                // heads
  int Tk;               // rows per (b,h) in kk
  int Tkp;              // padded key pitch of vt
  int kofs;             // first key position written
  // ragged streaming sessions (ppasr_b200_sessions_step): utterance b of the batch lives in cache slot slots[b] and appends
  // its keys at position kofs_b[b]; null = lock-step streams (slot b, position kofs)
  const int* kofs_b = nullptr;
  const int* slots = nullptr;
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    const int D = H * 64;
    int b = 0, t = 0;
    if (row < M) {
      b = row / T;
      t = row - b * T;
    }
    const int kb = slots ? __ldg(slots + b) : b;               // cache slot of the K / V rows
    const int kofs = kofs_b ? __ldg(kofs_b + b) : this->kofs;  // shadows the member on purpose
    epi_for_chunks<BLOCK_N, kEpiWarps / 4>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (row >= M || col >= 3 * D) return;
      const int which = col / D;
      const int hd = col - which * D;
      const int h = hd >> 6;
      const int d0 = hd & 63;
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + sbias[cc + j];
      if (which == 0) {
        __nv_bfloat16* dst = q2 + ((size_t)(b * H + h) * T + t) * 128 + d0;
        uint32_t pu[16], pv[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 u = __ldg(reinterpret_cast<const float2*>(bias_u + hd) + j);
          const float2 w = __ldg(reinterpret_cast<const float2*>(bias_v + hd) + j);
          pu[j] = pack_bf16x2(v[2 * j] + u.x, v[2 * j + 1] + u.y);
          pv[j] = pack_bf16x2(v[2 * j] + w.x, v[2 * j + 1] + w.y);
        }
        uint4* du = reinterpret_cast<uint4*>(dst);
        uint4* dv = reinterpret_cast<uint4*>(dst + 64);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          du[j] = make_uint4(pu[4 * j], pu[4 * j + 1], pu[4 * j + 2], pu[4 * j + 3]);
          dv[j] = make_uint4(pv[4 * j], pv[4 * j + 1], pv[4 * j + 2], pv[4 * j + 3]);
        }
      } else if (which == 1) {
        __nv_bfloat16* dst = kk + ((size_t)(kb * H + h) * Tk + kofs + t) * 64 + d0;
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
        uint4* dk = reinterpret_cast<uint4*>(dst);
#pragma unroll
        for (int j = 0; j < 4; ++j) dk[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      } else {
        __nv_bfloat16* dst = vt + ((size_t)(kb * H + h) * 64 + d0) * Tkp + kofs + t;
#pragma unroll
        for (int j = 0; j < 32; ++j) dst[(size_t)j * Tkp] = __float2bfloat16_rn(v[j]);
      }
    });
  }
};

// Fused QKV projection epilogue for GroupedRelPositionMultiHeadedAttention (reference:
// ppasr/model_utils/efficient_conformer/attention.py:40-79,128-193; group size 3, H heads of 64).
// pad4group views the zero-padded (B, Tpad, H*64) q / k / v tensors as (B, Tpad/3, H, 192): with
//   i = (t % 3) * 256 + column,  g = t / 3,  h' = i / 192,  d' = i % 192
//   q2g[b,h',g, d'] = q + pos_bias_u[h'][d'],  q2g[b,h',g,192+d'] = q + pos_bias_v[h'][d']     (bf16)
//   kkg[b,h',g, d'] = k ;  vtg[b,h',d',g] = v (transposed: K-major B operand of P.V)
// The thread that owns the last frame of an utterance also writes the zero-padded frames t = T .. 3*Tg-1
// (q = 0 -> bias only, k = v = 0).
template <int BLOCK_N>
struct EpiQKVGrouped {
  __nv_bfloat16* q2g;   // [B*H*Tg, 384]
  __nv_bfloat16* kkg;   // [B*H*Tg, 192]
  __nv_bfloat16* vtg;   // [B*H*192, Tgp]
  const float* bias;    // [3D]
  const float* bias_u;  // [H*192]
  const float* bias_v;  // [H*192]
  int M, T, H, Tg, Tgp;
  // chunk streaming: K / V go to the append-only grouped cache at ABSOLUTE frame kofs + t (group = frame / 3, the cache
  // starts zeroed so a partially filled last group reads zeros), queries stay grouped from the chunk start.
  // Tgk = group pitch of the K cache per (b, h) (0 = offline: Tg); the V^T pitch is Tgp in both modes.
  int kofs = 0, Tgk = 0;
  DEVINL void put(int b, int t, int which, int c0, const float (&v)[32]) const {
    const int tf = which == 0 ? t : t + kofs;
    const int i0 = (tf % 3) * 256 + c0;
    const int g = tf / 3;
    const int hp = i0 / 192;
    const int dp = i0 - hp * 192;
    const size_t bh = (size_t)b * H + hp;
    if (which == 0) {
      __nv_bfloat16* dst = q2g + (bh * Tg + g) * 384 + dp;
      uint32_t pu[16], pv[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float2 u = __ldg(reinterpret_cast<const float2*>(bias_u + hp * 192 + dp) + j);
        const float2 w = __ldg(reinterpret_cast<const float2*>(bias_v + hp * 192 + dp) + j);
        pu[j] = pack_bf16x2(v[2 * j] + u.x, v[2 * j + 1] + u.y);
        pv[j] = pack_bf16x2(v[2 * j] + w.x, v[2 * j + 1] + w.y);
      }
      uint4* du = reinterpret_cast<uint4*>(dst);
      uint4* dv = reinterpret_cast<uint4*>(dst + 192);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        du[j] = make_uint4(pu[4 * j], pu[4 * j + 1], pu[4 * j + 2], pu[4 * j + 3]);
        dv[j] = make_uint4(pv[4 * j], pv[4 * j + 1], pv[4 * j + 2], pv[4 * j + 3]);
      }
    } else if (which == 1) {
      __nv_bfloat16* dst = kkg + (bh * (Tgk > 0 ? Tgk : Tg) + g) * 192 + dp;
      uint32_t pk[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
      uint4* dk = reinterpret_cast<uint4*>(dst);
#pragma unroll
      for (int j = 0; j < 4; ++j) dk[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
    } else {
      __nv_bfloat16* dst = vtg + (bh * 192 + dp) * Tgp + g;
#pragma unroll
      for (int j = 0; j < 32; ++j) dst[(size_t)j * Tgp] = __float2bfloat16_rn(v[j]);
    }
  }
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    const int D = H * 64;
    int b = 0, t = 0;
    if (row < M) {
      b = row / T;
      t = row - b * T;
    }
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (row >= M || col >= 3 * D) return;
      const int which = col / D;
      const int c0 = col - which * D;
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + sbias[cc + j];
      put(b, t, which, c0, v);
      if (t == T - 1 && (Tgk == 0 || which == 0)) {  // streaming: only the query padding; the cache is append-only
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
        for (int tp = T; tp < 3 * Tg; ++tp) put(b, tp, which, c0, v);
      }
    });
  }
};

// Second subsampling conv: rows are the padded raster R = (b*Th + t')*pitch + f'; valid rows are
// written compactly as out[((b*Tout + t')*Fout + f'), n] = relu(acc + bias[n]) in bf16.
template <int BLOCK_N>
struct EpiConv2 {
  __nv_bfloat16* out;
  const float* bias;
  int M;      // padded raster rows = B*Th*pitch
  int N;      // 256
  int Th;     // raster rows per utterance (time)
  int pitch;  // 20
  int Tout;   // valid output frames per utterance
  int Fout;   // valid output freq bins (19)
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    bool valid = false;
    size_t orow = 0;
    if (row < M) {
      int b = row / (Th * pitch);
      int rem = row - b * (Th * pitch);
      int t = rem / pitch;
      int f = rem - t * pitch;
      valid = (t < Tout) && (f < Fout);
      orow = ((size_t)b * Tout + t) * Fout + f;
    }
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (valid && col < N) {
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bv = *reinterpret_cast<const float4*>(sbias + cc + 4 * j);
          pk[2 * j] = pack_bf16x2(fmaxf(__uint_as_float(r[4 * j]) + bv.x, 0.f),
                                  fmaxf(__uint_as_float(r[4 * j + 1]) + bv.y, 0.f));
          pk[2 * j + 1] = pack_bf16x2(fmaxf(__uint_as_float(r[4 * j + 2]) + bv.z, 0.f),
                                      fmaxf(__uint_as_float(r[4 * j + 3]) + bv.w, 0.f));
        }
        uint4* dst = reinterpret_cast<uint4*>(out + orow * N + col);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      }
    });
  }
};

// CTC head, materialising path: logits_f32[row, n] = acc + bias[n]   (ld multiple of 4)
template <int BLOCK_N>
struct EpiLogitsF32 {
  float* out;
  const float* bias;  // padded to num_n_tiles*BLOCK_N
  int ldo;
  int M, N;
  DEVINL void tile(uint32_t taddr, int row, int n0, int, int half, const float* sbias, float4*) const {
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (row < M && col < ldo) {
        float4* dst = reinterpret_cast<float4*>(out + (size_t)row * ldo + col);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (col + 4 * j < ldo) {
            const float4 bv = *reinterpret_cast<const float4*>(sbias + cc + 4 * j);
            dst[j] = make_float4(__uint_as_float(r[4 * j + 0]) + bv.x, __uint_as_float(r[4 * j + 1]) + bv.y,
                                 __uint_as_float(r[4 * j + 2]) + bv.z, __uint_as_float(r[4 * j + 3]) + bv.w);
          }
        }
      }
    });
  }
};

// CTC head, fused path: per (row, n_tile, half) partial soft-max statistics, never writing the logits:
//   pmax[row, p], parg[row, p] (first index of the max), psum[row, p] = sum exp(l - pmax),  p = 2*n_tile + half
// (reference: ppasr/model_utils/loss/ctc.py:62-70 followed by ppasr/decoders/ctc_greedy_decoder.py:21)
template <int BLOCK_N>
struct EpiCtcStats {
  float* pmax;
  int* parg;
  float* psum;
  const float* bias;  // padded
  int M, N;           // N = vocab size (valid columns)
  int num_parts;      // 2 * num_n_tiles
  DEVINL void tile(uint32_t taddr, int row, int n0, int n_tile, int half, const float* sbias, float4*) const {
    float m = -INFINITY, s = 0.f;
    int am = 0;
    epi_for_chunks<BLOCK_N>(taddr, half, [&](int cc, const uint32_t(&r)[32]) {
      const int col = n0 + cc;
      if (col >= N) return;
      float v[32];
      float cm = -INFINITY;
      int ca = 0;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        v[j] = (col + j < N) ? __uint_as_float(r[j]) + sbias[cc + j] : -INFINITY;
        if (v[j] > cm) {
          cm = v[j];
          ca = col + j;
        }
      }
      if (cm > m) {
        s *= __expf(m - cm);  // m = -inf on the first chunk -> s stays 0
        m = cm;
        am = ca;
      }
      float cs = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) cs += __expf(v[j] - m);
      s += cs;
    });
    if (row < M) {
      const size_t o = (size_t)row * num_parts + 2 * n_tile + half;
      pmax[o] = m;
      parg[o] = am;
      psum[o] = s;
    }
  }
};

// epilogues that keep a second TMEM buffer (kXbuf) run with one accumulator stage
template <class Epi, class = void>
struct EpiUsesXbuf {
  static constexpr bool value = false;
};
template <class Epi>
struct EpiUsesXbuf<Epi, decltype((void)Epi::kXbuf)> {
  static constexpr bool value = Epi::kXbuf != 0;
};

// epilogue warps per CTA: 8 (two column halves per TMEM lane quadrant) unless the epilogue asks for more. The epilogues of
// the K = 256 GEMMs are per-warp latency chains (ncu r2_qkv: 12 cycles per instruction, 600 instructions per warp and tile,
// 13 % tensor-pipe activity), so an epilogue with that much work per element declares kEpiWarps = 16 (four column parts).
template <class Epi, class = void>
struct EpiWarps {
  static constexpr int value = GEMM_EPI_WARPS;
};
template <class Epi>
struct EpiWarps<Epi, decltype((void)Epi::kEpiWarps)> {
  static constexpr int value = Epi::kEpiWarps;
};

// ------------------------------------------------------------------------------------------------
// The kernel
// ------------------------------------------------------------------------------------------------
template <int BLOCK_N, int STAGES, bool CONV, class Epi>
__global__ void __launch_bounds__(128 + EpiWarps<Epi>::value * 32, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const GemmShape shape, const Epi epi) {
  using SM = GemmSmem<BLOCK_N, STAGES>;
  using ACC = GemmAcc<BLOCK_N>;
  constexpr bool XBUF = EpiUsesXbuf<Epi>::value;
  constexpr int EPI_WARPS = EpiWarps<Epi>::value;
  static_assert(EPI_WARPS % 4 == 0 && BLOCK_N % (8 * EPI_WARPS) == 0, "column parts of whole 32-column chunks");
  constexpr int ACC_STAGES = XBUF ? 1 : ACC::ACC_STAGES;
  static_assert(!XBUF || BLOCK_N == 256, "X buffer layout assumes 2 x 256 TMEM columns");
  static_assert(BLOCK_N % 64 == 0 && BLOCK_N >= 64 && BLOCK_N <= 256, "BLOCK_N");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * SM::A_BYTES;
  float* smem_bias = reinterpret_cast<float*>(smem + SM::BIAS_OFFSET);
  float4* smem_scratch = reinterpret_cast<float4*>(smem + SM::SCRATCH_OFFSET);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + SM::BAR_OFFSET);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + ACC_STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + ACC_STAGES);

  const int warp_idx = threadIdx.x / 32;
  const int num_tiles = shape.num_m_tiles * shape.num_n_tiles;

  if (warp_idx == 0 && elect_one()) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp_idx == 1 && elect_one()) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < ACC_STAGES; ++i) {
      mbar_init(&tmem_full_bar[i], 1);
      mbar_init(&tmem_empty_bar[i], EPI_WARPS * 32);
    }
    fence_barrier_init();
    fence_proxy_async_smem();
  }
  if (warp_idx == 2) {
    tmem_alloc<ACC::TMEM_COLS>(tmem_ptr_smem);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();               // everything above overlapped the previous kernel's tail
  pdl_launch_dependents();  // let the next kernel start its own set-up

  if (warp_idx == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_tile = tile / shape.num_n_tiles;
        const int n_tile = tile - m_tile * shape.num_n_tiles;
        const int m0 = m_tile * GEMM_BLOCK_M;
        const int n0 = n_tile * BLOCK_N;
        for (int kb = 0; kb < shape.num_k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], SM::STAGE_BYTES);
          if (CONV) {
            const int tap = kb / shape.conv_kc;
            const int kc = kb - tap * shape.conv_kc;
            const int kh = tap / 3, kw = tap - kh * 3;
            const int ph = (kh & 1) * 2 + (kw & 1);
            const int shift = (kh >> 1) * shape.conv_pitch + (kw >> 1);
            tma_load_3d(smem_a + stage * SM::A_BYTES, &tmap_a, &full_bar[stage], kc * GEMM_BLOCK_K, m0 + shift, ph);
          } else {
            tma_load_2d(smem_a + stage * SM::A_BYTES, &tmap_a, &full_bar[stage], kb * GEMM_BLOCK_K, m0);
          }
          tma_load_2d(smem_b + stage * SM::B_BYTES, &tmap_b, &full_bar[stage], kb * GEMM_BLOCK_K, n0);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(GEMM_BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tmem_empty_bar[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BLOCK_N;
        for (int kb = 0; kb < shape.num_k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + stage * SM::A_BYTES);
          const uint32_t b_addr = smem_u32(smem_b + stage * SM::B_BYTES);
#pragma unroll
          for (int k = 0; k < GEMM_BLOCK_K / GEMM_UMMA_K; ++k) {
            umma_bf16(tmem_d, umma_desc_k_sw128(a_addr + k * GEMM_UMMA_K * 2),
                      umma_desc_k_sw128(b_addr + k * GEMM_UMMA_K * 2), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot when the MMAs have read it
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tmem_full_bar[as]);  // accumulator complete -> epilogue
        if (++as == ACC_STAGES) {
          as = 0;
          aphase ^= 1;
        }
      }
    }
  } else if (warp_idx >= 4) {
    // ===================== epilogue =====================
    const int ew = warp_idx - 4;
    const int quad = ew & 3;  // == warp_idx % 4 : TMEM lane quadrant
    const int half = ew >> 2;
    const int lane = threadIdx.x & 31;
    const int etid = threadIdx.x - 128;  // 0 .. EPI_WARPS * 32
    int as = 0;
    uint32_t aphase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int m_tile = tile / shape.num_n_tiles;
      const int n_tile = tile - m_tile * shape.num_n_tiles;
      // stage this tile's bias slice (double buffered by tile parity; one named barrier per tile)
      float* sbias = smem_bias + (it & 1) * BLOCK_N;
      if (etid < BLOCK_N) sbias[etid] = __ldg(epi.bias + n_tile * BLOCK_N + etid);
      named_bar_sync(1, EPI_WARPS * 32);
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + as * BLOCK_N;
      if constexpr (XBUF) epi.prefetch(taddr + BLOCK_N, m_tile * GEMM_BLOCK_M + quad * 32 + lane, half);
      mbar_wait(&tmem_full_bar[as], aphase);
      tc_fence_after();
      epi.tile(taddr, m_tile * GEMM_BLOCK_M + quad * 32 + lane, n_tile * BLOCK_N, n_tile, half, sbias, smem_scratch);
      tc_fence_before();
      mbar_arrive(&tmem_empty_bar[as]);
      if (++as == ACC_STAGES) {
        as = 0;
        aphase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc<ACC::TMEM_COLS>(tmem_base);
  }
}

// Host-side launcher. `num_sms` bounds the persistent grid. The bias pointer of every epilogue must
// be readable for num_n_tiles * BLOCK_N floats.
template <int BLOCK_N, int STAGES, bool CONV, class Epi>
inline cudaError_t launch_gemm(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const GemmShape& shape,
                               const Epi& epi, int num_sms, cudaStream_t stream) {
  using SM = GemmSmem<BLOCK_N, STAGES>;
  auto kern = gemm_bf16_tcgen05_kernel<BLOCK_N, STAGES, CONV, Epi>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  const int num_tiles = shape.num_m_tiles * shape.num_n_tiles;
  if (num_tiles <= 0) return cudaSuccess;
  const int grid = num_tiles < num_sms ? num_tiles : num_sms;
  cudaError_t le = launch_pdl(kern, dim3(grid), dim3(128 + EpiWarps<Epi>::value * 32), (size_t)SM::TOTAL, stream, tmap_a, tmap_b, shape, epi);
  count_launch();
  return le != cudaSuccess ? le : cudaGetLastError();
}

}  // namespace ppasr
