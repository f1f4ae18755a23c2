// Aggregation fused with the decoder's skip convolution (SURVEY.md section 8f, rank 1), forward and backward:
//   y[b,o,p] = relu( scale[o] * sum_c W[o,c] * skip[b,c,p] + shift[o] ),   skip = TemporalAggregator(att_group)
// which is UpConvBlock.skip_conv = Conv2d(d,d,1) -> BatchNorm2d (eval) -> ReLU (conv.py:378-382) applied to the
// aggregator's output (utae.py:225-229) without the skip map ever visiting HBM.  One CTA = one sample x ALL 64
// channels x 128 pixels: the producer issues ONE 3-D tensor-map copy per valid frame (box = 128 pixels x 64 channels
// x 1 frame, 16 KB per stage; 64 separate 256-byte bulk copies per frame were issue-bound at a third of the HBM
// rate), the consumers accumulate 4 channels x 8 pixels each exactly like agg_pipe_kernel, then the
// [64 x 128] skip tile goes to shared memory as bf16 (the value the unfused bf16 path would have stored) and the
// 1x1 convolution runs as mma.sync m16n8k16 with W split into bf16 hi + lo (two products, fp32 accumulation).
//
// The backward recomputes the skip map with the same prologue, producer, bilinear geometry, tap interpolation, weights
// and accumulation as the forward, in the forward's frame order, so its bf16 s is the forward's bit for bit: the
// BatchNorm-weight and conv-weight gradients rely on that.
//
// With the BatchNorm in training mode (batch statistics) the statistics must be complete before any output can be
// normalised, and the x sweep is too expensive to repeat, so the pre-BatchNorm z = W s + b crosses HBM once in bf16 (the
// value the unfused bf16 convolution stores): the sweep (BSTATS instantiation) writes z and per-CTA mean / M2 partials,
// skipconv_bstats_finish_kernel merges them, skipconv_bstats_apply_kernel writes relu(scale z + shift).
#include <initializer_list>

#include "c2s_sm100.cuh"

namespace c2s {
namespace {

constexpr int kScC = 64;            // channels of the skip map (= in and out channels of the 1x1 convolution)
constexpr int kScPB = 128;          // pixels per CTA
constexpr int kScVec = 8;           // pixels per consumer thread (one 16-byte bf16 vector)
constexpr int kScConsumers = 256;   // thread = (attention head, 8-pixel vector)
constexpr int kScStageBytes = kScC * kScPB * 2;
constexpr int kScTileStride = kScPB * 2 + 16;  // bytes per channel row of a bf16 tile (padded: ldmatrix conflict-free)
constexpr int kScFrags = 4 * 4 * 32;           // uint4 A fragments of one 64 x 64 bf16 matrix (m-tile, k-step, lane)
// stages the mbarriers are sized for, and the backward's ring (one CTA per SM: the grad_s and s registers rule out two)
constexpr int kScMaxStages = 6;
constexpr int kScGsStride = kScPB + 4;              // backward: floats per channel row of the fp32 grad_s tile
constexpr int kScPartial = kScC * kScC + 2 * kScC;  // backward: floats per CTA: g_y s^T, sum g_y, sum g_y (z - mean)

struct SkipConvShape {  // filled by skipconv_plan, read by both kernels
  int B, T, H, W, hw, ha, wa;
  float sy, sx;    // ATen's area_pixel_compute_scale: float(in) / out
  int tap_floats;  // per head and stage: staged attention rows of the pixel block (0: taps from global memory)
  int n_stages;
};

struct SkipConvArgs {
  SkipConvShape g;
  const float* attn;   // [16 heads, B, T, ha, wa]
  const uint8_t* pad;  // [B, T] or nullptr
  __nv_bfloat16* out;  // BSTATS: z
  const uint4* wfrag;  // [hi|lo][m-tile 4][k-step 4][lane 32] A fragments of W (bf16 pairs)
  const float* scale;  // [64]  gamma / sqrt(var + eps)
  const float* shift;  // [64]  (conv_bias - mean) * scale + beta; BSTATS: conv_bias or nullptr
  float* partial;      // BSTATS: [mean | M2][64][CTAs] of the tile's z
};

struct SkipConvBwdArgs {
  SkipConvShape g;
  const float* attn;
  const uint8_t* pad;
  const __nv_bfloat16* out;
  const __nv_bfloat16* gout;
  __nv_bfloat16* gx;
  float* gattn;
  const uint4* wfrag;   // [hi|lo] A fragments of W            (z = W s)
  const uint4* afrag;   // [hi|lo] A fragments of (alpha W)^T  (grad_s = (alpha W)^T g_y)
  const float* zshift;  // [64] conv_bias - running_mean; BSTATS: -batch mean of z
  float* partial;       // [CTAs][kScPartial] or nullptr (no parameter gradient wanted)
};

// the backward's inputs with batch statistics: a separate parameter, empty for the eval instantiation (whose code and
// registers stay those of a kernel without it)
template <bool BSTATS>
struct SkipConvBstatsIn {
  const __nv_bfloat16* z;  // the forward's pre-BatchNorm z [B,64,H,W]
  const float* inv_std;    // [64] 1 / sqrt(batch var + eps)
  const float* gmean;      // [2][64] mean_N(g_y), mean_N(g_y zhat)
};
template <>
struct SkipConvBstatsIn<false> {};

// ---------------------------------------------------------------------------------------------------------------------
// weight preparation
// ---------------------------------------------------------------------------------------------------------------------
// BatchNorm (eval) scale gamma / sqrt(var + eps): the forward's output scale and the backward's alpha
__device__ __forceinline__ float bn_scale(const float* bn_w, const float* bn_var, float eps, int o) {
  return (bn_w ? bn_w[o] : 1.f) / sqrtf(bn_var[o] + eps);
}

// A fragments (row-major 16 x 16 tiles, mma.sync m16n8k16) of the 64 x 64 matrix m(r, c) as bf16 hi and the bf16 of the
// residual: frag[idx] and frag[kScFrags + idx], idx = (m-tile, k-step, lane) in the order skipconv_tile_mma reads them
template <class Mat>
__device__ __forceinline__ void write_frags(const Mat& m, int idx, uint4* __restrict__ frag) {
  const int lane = idx & 31, ks = (idx >> 5) & 3, mt = idx >> 7;
  const int r0 = mt * 16 + (lane >> 2), c0 = ks * 16 + (lane & 3) * 2;
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {  // a0:(r, c) a1:(r+8, c) a2:(r, c+8) a3:(r+8, c+8)
    const int r = r0 + (q & 1) * 8, c = c0 + (q >> 1) * 8;
    const float v0 = m(r, c), v1 = m(r, c + 1);
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
    hi[q] = Elem<__nv_bfloat16>::pack2(__bfloat162float(h0), __bfloat162float(h1));
    lo[q] = Elem<__nv_bfloat16>::pack2(v0 - __bfloat162float(h0), v1 - __bfloat162float(h1));
  }
  frag[idx] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  frag[kScFrags + idx] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// W[o][c] fp32 -> A fragments; block 2: the scale / shift of conv bias + eval BatchNorm
__global__ void skipconv_prep_kernel(const float* __restrict__ w, uint4* __restrict__ frag, const float* conv_bias,
                                     const float* bn_w, const float* bn_b, const float* bn_mean, const float* bn_var,
                                     float eps, float* scale, float* shift) {
  if (blockIdx.x == 2) {
    const int o = threadIdx.x;
    if (o < kScC) {
      const float sc = bn_scale(bn_w, bn_var, eps, o);
      scale[o] = sc;
      shift[o] = ((conv_bias ? conv_bias[o] : 0.f) - bn_mean[o]) * sc + (bn_b ? bn_b[o] : 0.f);
    }
    return;
  }
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kScFrags) return;
  write_frags([&](int r, int c) { return w[r * kScC + c]; }, idx, frag);
}

// A fragments of W and of (alpha W)^T; block 2: the per-channel constants
__global__ void skipconv_bwd_prep_kernel(const float* __restrict__ w, const float* conv_bias, const float* bn_w,
                                         const float* bn_mean, const float* bn_var, float eps, uint4* __restrict__ wfrag,
                                         uint4* __restrict__ afrag, float* alpha, float* inv_std, float* zshift) {
  if (blockIdx.x == 2) {
    const int o = threadIdx.x;
    if (o < kScC) {
      inv_std[o] = 1.f / sqrtf(bn_var[o] + eps);
      alpha[o] = bn_scale(bn_w, bn_var, eps, o);
      zshift[o] = (conv_bias ? conv_bias[o] : 0.f) - bn_mean[o];
    }
    return;
  }
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kScFrags) return;
  write_frags([&](int r, int c) { return w[r * kScC + c]; }, idx, wfrag);
  // (alpha W)^T [c_in = r][c_out = c]
  write_frags([&](int r, int c) { return bn_scale(bn_w, bn_var, eps, c) * w[c * kScC + r]; }, idx, afrag);
}

// ---------------------------------------------------------------------------------------------------------------------
// pieces of both kernels
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sts_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Warp 0 lists the valid frames of sample b in order (and, given s_pad, flags every padded frame there); thread 0
// initialises the ring's mbarriers: full = bars[s] (the producer's arrival + transaction bytes) and empty =
// bars[n_stages + s] (one arrival per consumer warp).  Returns the number of valid frames to every thread of the block.
__device__ __forceinline__ int skipconv_frames(const SkipConvShape& g, const uint8_t* pad, int b, short* frames,
                                               int* n_frames_s, unsigned long long* bars, uint8_t* s_pad = nullptr) {
  if (threadIdx.x < 32) {
    int count = 0;
    for (int base = 0; base < g.T; base += 32) {
      const int t = base + threadIdx.x;
      const bool valid = t < g.T && (pad == nullptr || pad[b * g.T + t] == 0);
      if (s_pad != nullptr && t < g.T) s_pad[t] = !valid;
      const unsigned m = __ballot_sync(0xffffffffu, valid);
      if (valid) frames[count + __popc(m & ((1u << threadIdx.x) - 1u))] = static_cast<short>(t);
      count += __popc(m);
    }
    if (threadIdx.x == 0) {
      *n_frames_s = count;
      for (int s = 0; s < g.n_stages; ++s) {
        mbar_init(s32(&bars[s]), 1);
        mbar_init(s32(&bars[g.n_stages + s]), kScConsumers / 32);
      }
      fence_mbarrier_init();
    }
  }
  __syncthreads();
  return *n_frames_s;
}

// first attention row of the staged slice: the upper tap row of the pixel block's first pixel
__device__ __forceinline__ int staged_row0(const SkipConvShape& g, int pblk) {
  int r_lo, i1;
  float l1;
  source_index(g.sy, (pblk * kScPB) / g.W, g.ha, r_lo, i1, l1);
  return r_lo;
}

// The producer thread: per valid frame one box {128 pixels, 64 channels, 1 frame} of x and, with staged taps, one box
// {tap_floats of the map from row r_lo, 1 frame, 16 heads} of the attention (16 separate bulk copies of 128-256 bytes
// per frame were measured: issue-bound, slower than the global-memory taps)
template <bool TAPS>
__device__ __forceinline__ void skipconv_produce(const CUtensorMap* map_x, const CUtensorMap* map_att, const SkipConvShape& g,
                                                 int b, int pblk, int r_lo, const short* frames, int n_frames,
                                                 uint32_t stage0, uint32_t stage_stride, unsigned long long* bars) {
  const uint32_t tap_bytes = TAPS ? 16u * g.tap_floats * 4u : 0u;
  for (int i = 0; i < n_frames; ++i) {
    const int s = i % g.n_stages, round = i / g.n_stages;
    if (round > 0) mbar_wait(s32(&bars[g.n_stages + s]), (round - 1) & 1);
    const uint32_t full = s32(&bars[s]);
    mbar_expect_tx(full, kScStageBytes + tap_bytes);
    tma_load_3d(stage0 + s * stage_stride, map_x, pblk * kScPB, 0, b * g.T + frames[i], full);
    if (TAPS) tma_load_3d(stage0 + s * stage_stride + kScStageBytes, map_att, r_lo * g.wa, b * g.T + frames[i], 0, full);
  }
}

// Bilinear geometry of a consumer's 8-pixel vector at xS up-sampling (the vector covers whole attention cells): its two
// attention rows, in the map and in the staged slice, their weights, the window of NCOL low-resolution columns it
// touches and the horizontal weight of each pixel
template <int S>
struct SkipGeom {
  static constexpr int NCOL = kScVec / S + 2;
  int row0, row1;    // rows of the map, times wa
  int trow0, trow1;  // rows inside the staged slice, times wa
  float ly0, ly1;
  int cmin;          // first window column before clamping
  int col[NCOL];
  float lx1[kScVec];

  __device__ __forceinline__ SkipGeom(const SkipConvShape& g, int p0, int r_lo) {
    const int y = p0 / g.W;
    const int x0 = p0 - y * g.W;
    int iy0, iy1;
    source_index(g.sy, y, g.ha, iy0, iy1, ly1);
    ly0 = 1.f - ly1;
    row0 = iy0 * g.wa, row1 = iy1 * g.wa;
    trow0 = (iy0 - r_lo) * g.wa, trow1 = (iy1 - r_lo) * g.wa;
#pragma unroll
    for (int j = 0; j < kScVec; ++j) {
      int i0, i1;
      source_index(g.sx, x0 + j, g.wa, i0, i1, lx1[j]);
    }
    cmin = x0 / S - 1;
#pragma unroll
    for (int j = 0; j < NCOL; ++j) {
      const int cj = cmin + j;
      col[j] = cj < 0 ? 0 : (cj > g.wa - 1 ? g.wa - 1 : cj);
    }
  }
  // window column of pixel j's left tap (its right tap is the next column)
  static __device__ __forceinline__ constexpr int cell(int j) { return j / S + ((j % S) < S / 2 ? 0 : 1); }

  // one frame's attention at the two rows and the window columns: the frame's map in global memory (read-only path) or
  // the staged slice of the head in shared memory
  __device__ __forceinline__ void rows(const float* m, bool staged, float (&top)[NCOL], float (&bot)[NCOL]) const {
#pragma unroll
    for (int j = 0; j < NCOL; ++j) {
      top[j] = staged ? m[trow0 + col[j]] : __ldg(m + row0 + col[j]);
      bot[j] = staged ? m[trow1 + col[j]] : __ldg(m + row1 + col[j]);
    }
  }
  // one frame's vertical interpolation at the window columns
  __device__ __forceinline__ void vertical(const float (&top)[NCOL], const float (&bot)[NCOL], float (&r)[NCOL]) const {
#pragma unroll
    for (int j = 0; j < NCOL; ++j) r[j] = fmaf(ly1, bot[j], ly0 * top[j]);
  }
  // the up-sampled attention of the 8 pixels from one frame's vertical interpolation
  __device__ __forceinline__ void weights(const float (&r)[NCOL], float (&w)[kScVec]) const {
#pragma unroll
    for (int j = 0; j < kScVec; ++j) w[j] = fmaf(lx1[j], r[cell(j) + 1], (1.f - lx1[j]) * r[cell(j)]);
  }
};

// one frame's term of the skip value of one channel at the 8 pixels
__device__ __forceinline__ void skip_accumulate(float (&acc)[kScVec], const float (&w)[kScVec], const float (&f)[kScVec]) {
#pragma unroll
  for (int j = 0; j < kScVec; ++j) acc[j] = fmaf(w[j], f[j], acc[j]);
}

// [64 rows][128 pixels] = A[64 x 64] (hi + lo fragments) x tile[64 channels][128 pixels] (bf16, row stride kScTileStride);
// warp w: pixels [16 w, 16 w + 16).  D fragment: rows mt*16 + lane/4 (+8), pixels 16 w + 8 nt + 2 (lane % 4) (+1).
__device__ __forceinline__ void skipconv_tile_mma(float (&d)[4][2][4], const uint4* frag, uint32_t tile, int warp, int lane) {
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) d[mt][nt][e] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    // B fragments: ldmatrix.x4.trans of the four 8x8 blocks (k 0-7 | 8-15) x (n 0-7 | 8-15) of this k-step
    const int mrow = ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;  // channel row this lane addresses
    const int ncol = warp * 16 + (lane >> 4) * 8;                   // first pixel of the 8x8 block
    uint32_t bf[4];
    ldsm_x4_trans(bf, tile + mrow * kScTileStride + ncol * 2);
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
      const uint4 h4 = __ldg(frag + (mt * 4 + ks) * 32 + lane);
      const uint4 l4 = __ldg(frag + kScFrags + (mt * 4 + ks) * 32 + lane);
      const uint32_t ah[4] = {h4.x, h4.y, h4.z, h4.w}, al[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        mma_bf16(d[mt][nt], ah, bf[2 * nt], bf[2 * nt + 1]);
        mma_bf16(d[mt][nt], al, bf[2 * nt], bf[2 * nt + 1]);
      }
    }
  }
}

// g_y = grad_out masked by the forward's ReLU decision, 8 bf16 pixels (exact): a positive bf16 has a clear sign bit and a
// non-zero magnitude
__device__ __forceinline__ uint4 relu_masked(const uint4& gv, const uint4& o) {
  const uint32_t gw[4] = {gv.x, gv.y, gv.z, gv.w}, ow[4] = {o.x, o.y, o.z, o.w};
  uint32_t m[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t lo_pos = ((ow[q] & 0x8000u) == 0 && (ow[q] & 0x7fffu) != 0) ? 0x0000ffffu : 0u;
    const uint32_t hi_pos = ((ow[q] & 0x80000000u) == 0 && (ow[q] & 0x7fff0000u) != 0) ? 0xffff0000u : 0u;
    m[q] = gw[q] & (lo_pos | hi_pos);
  }
  return make_uint4(m[0], m[1], m[2], m[3]);
}

// Reduction of one value per thread over a 256-thread block in a fixed order (deterministic); thread 0 gets the result
template <class V, class Merge>
__device__ __forceinline__ V block_reduce_fixed(V v, Merge merge) {
  __shared__ V vals[256];
  vals[threadIdx.x] = v;
  __syncthreads();
  for (int stride = 128; stride > 0; stride >>= 1) {
    if (threadIdx.x < stride) vals[threadIdx.x] = merge(vals[threadIdx.x], vals[threadIdx.x + stride]);
    __syncthreads();
  }
  return vals[0];
}

// ---------------------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------------------
// Batch-statistics epilogue of the sweep: z = W s + bias -> bf16 (no BatchNorm, no ReLU), and per output channel the mean
// and M2 of the bf16-rounded z over the tile's 128 pixels: two passes over the registers (the mean first, then the
// squared deviations from it), not sums of z and z^2, whose difference cancels in fp32.  `red` holds 2 x 8 x 64 floats.
__device__ __forceinline__ void skipconv_z_epilogue(float (&d)[4][2][4], const float* bias, __nv_bfloat16* op, int hw,
                                                    int warp, int lane, float* red, float* partial, int cta, int n_ctas) {
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      const int o = mt * 16 + (lane >> 2) + hrow * 8;
      const float bz = bias != nullptr ? __ldg(bias + o) : 0.f;
      float sum = 0.f;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        float* v = &d[mt][nt][hrow * 2];
        v[0] = __bfloat162float(__float2bfloat16_rn(v[0] + bz));
        v[1] = __bfloat162float(__float2bfloat16_rn(v[1] + bz));
        *reinterpret_cast<uint32_t*>(op + static_cast<size_t>(o) * hw + nt * 8) = Elem<__nv_bfloat16>::pack2(v[0], v[1]);
        sum += v[0] + v[1];
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      if ((lane & 3) == 0) red[warp * kScC + o] = sum;
    }
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");
  auto tile_mean = [&](int o) {
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += red[w8 * kScC + o];
    return s * (1.f / kScPB);
  };
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      const int o = mt * 16 + (lane >> 2) + hrow * 8;
      const float mean = tile_mean(o);
      float q = 0.f;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float dv = d[mt][nt][hrow * 2 + e] - mean;
          q = fmaf(dv, dv, q);
        }
      q += __shfl_xor_sync(0xffffffffu, q, 1);
      q += __shfl_xor_sync(0xffffffffu, q, 2);
      if ((lane & 3) == 0) red[8 * kScC + warp * kScC + o] = q;
    }
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");
  if (threadIdx.x < kScC) {
    const int o = threadIdx.x;
    float m2 = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) m2 += red[8 * kScC + w8 * kScC + o];
    partial[static_cast<size_t>(o) * n_ctas + cta] = tile_mean(o);
    partial[static_cast<size_t>(kScC + o) * n_ctas + cta] = m2;
  }
}

template <int S, bool TAPS, bool BSTATS>
__global__ void __launch_bounds__(kScConsumers + 32, 2) agg_skipconv_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                             const __grid_constant__ CUtensorMap map_att,
                                                                             const SkipConvArgs k) {
  using T = __nv_bfloat16;
  using Geom = SkipGeom<S>;
  constexpr int NCOL = Geom::NCOL;
  const SkipConvShape& g = k.g;
  extern __shared__ __align__(128) unsigned char pipe_smem[];  // stages, then the epilogue tile
  __shared__ short frames[kAggMaxT];
  __shared__ int n_frames_s;
  __shared__ __align__(8) unsigned long long bars[2 * kScMaxStages];

  const int b = blockIdx.y, pblk = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t stage_stride = kScStageBytes + 16u * g.tap_floats * 4u;
  const int r_lo = TAPS ? staged_row0(g, pblk) : 0;
  const int n_frames = skipconv_frames(g, k.pad, b, frames, &n_frames_s, bars);
  const uint32_t stage0 = s32(pipe_smem);

  if (warp == kScConsumers / 32) {
    if (lane == 0) skipconv_produce<TAPS>(&map_x, &map_att, g, b, pblk, r_lo, frames, n_frames, stage0, stage_stride, bars);
    return;
  }

  // ---- consumers: thread = (attention head, 8-pixel vector) -----------------------------------------------------------
  const int head = threadIdx.x >> 4, pv = threadIdx.x & 15;
  const Geom geo(g, pblk * kScPB + pv * kScVec, r_lo);
  const int amap = g.ha * g.wa;
  const float* ab = k.attn + (static_cast<size_t>(head) * g.B + b) * g.T * amap;

  float acc[4][kScVec];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int j = 0; j < kScVec; ++j) acc[c][j] = 0.f;

  float top[NCOL], bot[NCOL];  // global-memory taps: the next frame's rows travel while this one is consumed
  if (!TAPS && n_frames > 0) geo.rows(ab + static_cast<size_t>(frames[0]) * amap, false, top, bot);
  const uint32_t my_off = (head * 4) * (kScPB * 2) + pv * 16;
  for (int i = 0; i < n_frames; ++i) {
    float r[NCOL];
    if (!TAPS) {
      geo.vertical(top, bot, r);
      if (i + 1 < n_frames) geo.rows(ab + static_cast<size_t>(frames[i + 1]) * amap, false, top, bot);
    }
    const int s = i % g.n_stages;
    mbar_wait(s32(&bars[s]), (i / g.n_stages) & 1);
    uint4 xv[4];
    const uint32_t base = stage0 + s * stage_stride + my_off;
#pragma unroll
    for (int c = 0; c < 4; ++c) xv[c] = lds_v4(base + c * (kScPB * 2));
    if (TAPS) {
      geo.rows(reinterpret_cast<const float*>(pipe_smem + s * stage_stride + kScStageBytes) + head * g.tap_floats, true, top, bot);
      geo.vertical(top, bot, r);
    }
    fence_proxy_async();  // the stage's shared loads before the producer's next bulk copy into it
    __syncwarp();
    if (lane == 0) mbar_arrive(s32(&bars[g.n_stages + s]));

    float w[kScVec];
    geo.weights(r, w);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float f[kScVec];
      Elem<T>::unpack(xv[c], f);
      skip_accumulate(acc[c], w, f);
    }
  }

  // ---- epilogue: skip tile [64 channels][128 pixels] bf16 -> shared memory, 1x1 convolution on the tensor cores -------
  const uint32_t tile = stage0 + g.n_stages * stage_stride;
#pragma unroll
  for (int c = 0; c < 4; ++c) sts_v4(tile + (head * 4 + c) * kScTileStride + pv * 16, Elem<T>::pack(acc[c]));
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");  // the producer warp has left; consumers only

  float d[4][2][4];
  skipconv_tile_mma(d, k.wfrag, tile, warp, lane);
  T* op = k.out + static_cast<size_t>(b) * kScC * g.hw + static_cast<size_t>(pblk) * kScPB + warp * 16 + (lane & 3) * 2;
  if constexpr (BSTATS) {  // the stages are drained: every consumer has passed the barrier above
    skipconv_z_epilogue(d, k.shift, op, g.hw, warp, lane, reinterpret_cast<float*>(pipe_smem), k.partial,
                        b * gridDim.x + pblk, gridDim.x * gridDim.y);
  } else {
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int o = mt * 16 + (lane >> 2) + hrow * 8;
        const float sc = __ldg(k.scale + o), sh = __ldg(k.shift + o);
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          const float v0 = fmaxf(fmaf(sc, d[mt][nt][hrow * 2], sh), 0.f), v1 = fmaxf(fmaf(sc, d[mt][nt][hrow * 2 + 1], sh), 0.f);
          *reinterpret_cast<uint32_t*>(op + static_cast<size_t>(o) * g.hw + nt * 8) = Elem<T>::pack2(v0, v1);
        }
      }
  }
}

// Chan's parallel merge of (count, mean, M2) summaries
struct MeanM2 {
  float n, mean, m2;
};
__device__ __forceinline__ MeanM2 chan_merge(const MeanM2& a, const MeanM2& b) {
  const float n = a.n + b.n;
  if (b.n == 0.f) return a;
  const float delta = b.mean - a.mean, fb = b.n / n;
  return MeanM2{n, fmaf(delta, fb, a.mean), a.m2 + b.m2 + delta * delta * a.n * fb};
}

// One block per channel: the CTA partials merged in a fixed order (thread i takes CTAs i, i + 256, ...; then a fixed
// tree), so the statistics are bit-identical from run to run.  Writes the batch mean, the biased variance and the scale /
// shift of BatchNorm-affine + ReLU.
__global__ void __launch_bounds__(256) skipconv_bstats_finish_kernel(const float* __restrict__ partial, int n_ctas,
                                                                     const float* bn_w, const float* bn_b, float eps,
                                                                     float* mean, float* var, float* scale, float* shift) {
  const int o = blockIdx.x;
  MeanM2 acc{0.f, 0.f, 0.f};
  for (int i = threadIdx.x; i < n_ctas; i += 256)
    acc = chan_merge(acc, MeanM2{static_cast<float>(kScPB), partial[static_cast<size_t>(o) * n_ctas + i],
                                 partial[static_cast<size_t>(kScC + o) * n_ctas + i]});
  acc = block_reduce_fixed(acc, chan_merge);
  if (threadIdx.x != 0) return;
  const float v = acc.m2 / acc.n;
  const float sc = (bn_w ? bn_w[o] : 1.f) / sqrtf(v + eps);
  mean[o] = acc.mean, var[o] = v;
  scale[o] = sc, shift[o] = (bn_b ? bn_b[o] : 0.f) - acc.mean * sc;
}

// out = relu(scale z + shift), 8 bf16 pixels per thread; blockIdx.x = (sample, channel) plane, 32-bit offsets inside it.
// out may be z (plain loads: no read-only path on data this kernel writes).
__global__ void __launch_bounds__(256) skipconv_bstats_apply_kernel(const __nv_bfloat16* z, __nv_bfloat16* out,
                                                                    const float* __restrict__ scale,
                                                                    const float* __restrict__ shift, int hw_vec) {
  const int v = blockIdx.y * 256 + threadIdx.x;
  if (v >= hw_vec) return;
  const int o = blockIdx.x % kScC;
  const size_t off = static_cast<size_t>(blockIdx.x) * hw_vec * kScVec + static_cast<uint32_t>(v) * kScVec;
  const float sc = __ldg(scale + o), sh = __ldg(shift + o);
  float f[kScVec];
  Elem<__nv_bfloat16>::unpack(*reinterpret_cast<const uint4*>(z + off), f);
#pragma unroll
  for (int j = 0; j < kScVec; ++j) f[j] = fmaxf(fmaf(sc, f[j], sh), 0.f);
  st_stream_v4(out + off, Elem<__nv_bfloat16>::pack(f));
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward with the BatchNorm in eval mode, for one sample and pixel p (s = the bf16 skip map, z = W s + b,
// alpha = gamma / sqrt(var + eps)):
//   g_y = grad_out * [out > 0]                      grad_s = W^T (alpha * g_y)
//   grad_bn_bias = sum g_y   grad_bn_weight = sum g_y (z - mean) / sqrt(var + eps)
//   grad_conv_bias = alpha * sum g_y                grad_conv_weight = alpha * sum_p g_y s^T
// then the aggregator's backward with grad_out = grad_s.  One CTA = one sample x 64 channels x 128 pixels, as in the
// forward.  Before any frame arrives grad_s is formed on the tensor cores from grad_out and out alone (the A operand is
// (alpha W)^T as bf16 hi + lo; g_y is exact in bf16).  The valid frames then stream once through the TMA ring: the
// consumers write grad_x, scatter the bilinear adjoint into grad_attn (as agg_backward_pipe_kernel) and re-accumulate s
// with the forward's code in the forward's frame order.  After the sweep, z = W s (hi + lo, the forward's products) gives
// the BatchNorm sums and g_y s^T the weight gradient; each CTA writes its partials to the workspace and
// skipconv_bwd_finish_kernel reduces them in a fixed order (deterministic).
//
// BSTATS (BatchNorm with batch statistics mean mu and variance var; zhat = (z - mu) / sqrt(var + eps), alpha as above
// with var):
//   g_z = alpha * g_z',  g_z' = g_y - mean_N(g_y) - zhat * mean_N(g_y zhat)
//   grad_s = (alpha W)^T g_z'   grad_conv_weight = alpha * sum_p g_z' s^T   grad_conv_bias = 0
//   grad_bn_bias = sum g_y      grad_bn_weight = sum g_y zhat
// The two means are global, so skipconv_bstats_bwd_sums_kernel and its finish run first.  The prologue forms g_z' per
// pixel in fp32 from grad_out, out and the forward's z; it is not exact in bf16, so it goes to shared memory as bf16 hi +
// lo tiles and both products (grad_s and g_z' s^T) take the two.  (The expanded form (alpha W)^T g_y - (.. W)^T z + const
// would lose g_z' to cancellation when grad_out is nearly constant per channel.)  The sweep is unchanged.
// ---------------------------------------------------------------------------------------------------------------------
template <int S, bool TAPS, bool BSTATS>
__global__ void __launch_bounds__(kScConsumers + 32, 1) agg_skipconv_backward_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                                      const __grid_constant__ CUtensorMap map_att,
                                                                                      const SkipConvBwdArgs a,
                                                                                      const SkipConvBstatsIn<BSTATS> bs) {
  using T = __nv_bfloat16;
  using Geom = SkipGeom<S>;
  constexpr int VEC = kScVec;
  constexpr int M = VEC / S;  // attention cells per thread
  constexpr int NCOL = Geom::NCOL;
  const SkipConvShape& g = a.g;
  // stages | g_y tile (bf16; BSTATS: g_z' hi) | grad_s (fp32), later the s tile | BSTATS: g_z' lo tile
  extern __shared__ __align__(128) unsigned char sb_smem[];
  __shared__ short frames[kAggMaxT];
  __shared__ uint8_t s_pad[kAggMaxT];
  __shared__ int n_frames_s;
  __shared__ __align__(8) unsigned long long bars[2 * kScMaxStages];

  const int b = blockIdx.y, pblk = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_stages = g.n_stages;
  const uint32_t stage_stride = kScStageBytes + 16u * g.tap_floats * 4u;
  const int r_lo = TAPS ? staged_row0(g, pblk) : 0;
  const int n_frames = skipconv_frames(g, a.pad, b, frames, &n_frames_s, bars, s_pad);
  const uint32_t stage0 = s32(sb_smem);

  if (warp == kScConsumers / 32) {
    if (lane == 0) skipconv_produce<TAPS>(&map_x, &map_att, g, b, pblk, r_lo, frames, n_frames, stage0, stage_stride, bars);
    return;
  }

  // ---- consumers: thread = (attention head, 8-pixel vector) ------------------------------------------------------------
  const int head = threadIdx.x >> 4, pv = threadIdx.x & 15;
  const int p0 = pblk * kScPB + pv * VEC;
  const uint32_t gy_tile = stage0 + n_stages * stage_stride;
  const uint32_t gs_tile = gy_tile + kScC * kScTileStride;  // grad_s fp32 [64][kScGsStride]; after the sweep the s tile
  float* gs_smem = reinterpret_cast<float*>(sb_smem + n_stages * stage_stride + kScC * kScTileStride);
  const size_t plane = static_cast<size_t>(b) * kScC * g.hw + p0;
  const uint32_t glo_tile = gs_tile + kScC * kScGsStride * 4;  // BSTATS

  // g_y = grad_out masked by the forward's ReLU decision (bf16, exact) -> shared tile; BSTATS: g_z' as hi + lo tiles
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int ch = head * 4 + c;
    const size_t off = plane + static_cast<size_t>(ch) * g.hw;
    if constexpr (BSTATS) {
      float gf[VEC], zf[VEC], hi[VEC], lo[VEC];
      Elem<T>::unpack(relu_masked(ld_stream_v4(a.gout + off), ld_stream_v4(a.out + off)), gf);
      Elem<T>::unpack(ld_stream_v4(bs.z + off), zf);
      const float is = __ldg(bs.inv_std + ch), zs = __ldg(a.zshift + ch);
      const float m1 = __ldg(bs.gmean + ch), m2 = __ldg(bs.gmean + kScC + ch);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float gz = gf[j] - m1 - (zf[j] + zs) * is * m2;
        hi[j] = __bfloat162float(__float2bfloat16_rn(gz));
        lo[j] = gz - hi[j];
      }
      sts_v4(gy_tile + ch * kScTileStride + pv * 16, Elem<T>::pack(hi));
      sts_v4(glo_tile + ch * kScTileStride + pv * 16, Elem<T>::pack(lo));
    } else {
      sts_v4(gy_tile + ch * kScTileStride + pv * 16, relu_masked(ld_stream_v4(a.gout + off), ld_stream_v4(a.out + off)));
    }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");  // consumers only (the producer warp has its own loop)
  {  // grad_s = (alpha W)^T g_y (BSTATS: g_z' hi + lo) -> shared memory (fp32)
    float d[4][2][4];
    skipconv_tile_mma(d, a.afrag, gy_tile, warp, lane);
    if constexpr (BSTATS) {
      float dl[4][2][4];
      skipconv_tile_mma(dl, a.afrag, glo_tile, warp, lane);
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int e = 0; e < 4; ++e) d[mt][nt][e] += dl[mt][nt][e];
    }
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          const int c = mt * 16 + (lane >> 2) + hrow * 8, p = warp * 16 + nt * 8 + (lane & 3) * 2;
          *reinterpret_cast<float2*>(gs_smem + c * kScGsStride + p) = make_float2(d[mt][nt][hrow * 2], d[mt][nt][hrow * 2 + 1]);
        }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");
  float gs[4][VEC];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 v0 = *reinterpret_cast<const float4*>(gs_smem + (head * 4 + c) * kScGsStride + pv * VEC);
    const float4 v1 = *reinterpret_cast<const float4*>(gs_smem + (head * 4 + c) * kScGsStride + pv * VEC + 4);
    gs[c][0] = v0.x, gs[c][1] = v0.y, gs[c][2] = v0.z, gs[c][3] = v0.w;
    gs[c][4] = v1.x, gs[c][5] = v1.y, gs[c][6] = v1.z, gs[c][7] = v1.w;
  }

  const Geom geo(g, p0, r_lo);
  const int amap = g.ha * g.wa;
  const size_t abase = (static_cast<size_t>(head) * g.B + b) * g.T * amap;
  // 16 lanes of a head cover the 128 pixels in order: a lane's left / right neighbour in the image row sits next to it
  const int lanes_per_row = g.W / VEC;
  const int lane_in_row = (p0 / VEC) % lanes_per_row;
  const bool has_left = pv > 0 && lane_in_row > 0;
  const bool has_right = pv < 15 && lane_in_row < lanes_per_row - 1;
  const size_t frame_stride = static_cast<size_t>(kScC) * g.hw;
  T* gxb = a.gx != nullptr ? a.gx + static_cast<size_t>(b) * g.T * frame_stride + static_cast<size_t>(head * 4) * g.hw + p0 : nullptr;

  float acc[4][VEC];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[c][j] = 0.f;

  const uint32_t my_off = (head * 4) * (kScPB * 2) + pv * 16;
  for (int i = 0; i < n_frames; ++i) {
    const int t = frames[i];
    float top[NCOL], bot[NCOL], r[NCOL];
    if (!TAPS) {
      geo.rows(a.attn + abase + static_cast<size_t>(t) * amap, false, top, bot);
      geo.vertical(top, bot, r);
    }
    const int s = i % n_stages;
    mbar_wait(s32(&bars[s]), (i / n_stages) & 1);
    uint4 xv[4];
    const uint32_t base = stage0 + s * stage_stride + my_off;
#pragma unroll
    for (int c = 0; c < 4; ++c) xv[c] = lds_v4(base + c * (kScPB * 2));
    if (TAPS) {
      geo.rows(reinterpret_cast<const float*>(sb_smem + s * stage_stride + kScStageBytes) + head * g.tap_floats, true, top, bot);
      geo.vertical(top, bot, r);
    }
    fence_proxy_async();  // the stage's shared loads before the producer's next bulk copy into it
    __syncwarp();
    if (lane == 0) mbar_arrive(s32(&bars[g.n_stages + s]));

    float w[VEC];
    geo.weights(r, w);
    float gsum[VEC];  // sum_c x * grad_s of this thread's pixels
#pragma unroll
    for (int j = 0; j < VEC; ++j) gsum[j] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float f[VEC], dx[VEC];
      Elem<T>::unpack(xv[c], f);
      skip_accumulate(acc[c], w, f);  // the forward's accumulation
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        gsum[j] = fmaf(f[j], gs[c][j], gsum[j]);
        dx[j] = w[j] * gs[c][j];
      }
      if (gxb != nullptr) st_stream_v4(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(c) * g.hw, Elem<T>::pack(dx));
    }
    if (a.gattn == nullptr) continue;
    // horizontal adjoint into the NCOL-column window, then edge columns travel to the neighbouring lanes
    float* gp = a.gattn + abase + static_cast<size_t>(t) * amap;
    float win[NCOL];
#pragma unroll
    for (int jj = 0; jj < NCOL; ++jj) win[jj] = 0.f;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      win[Geom::cell(j)] = fmaf(gsum[j], 1.f - geo.lx1[j], win[Geom::cell(j)]);
      win[Geom::cell(j) + 1] = fmaf(gsum[j], geo.lx1[j], win[Geom::cell(j) + 1]);
    }
    const float from_left = __shfl_up_sync(0xffffffffu, win[NCOL - 1], 1);
    const float from_right = __shfl_down_sync(0xffffffffu, win[0], 1);
    float own[M];
#pragma unroll
    for (int q = 0; q < M; ++q) own[q] = win[q + 1];
    if (has_left) own[0] += from_left;
    if (has_right) own[M - 1] += from_right;
#pragma unroll
    for (int q = 0; q < M; ++q) {
      const int cj = geo.cmin + 1 + q;  // own columns are always inside [0, wa)
      atomicAdd(gp + geo.row0 + cj, geo.ly0 * own[q]);
      if (geo.ly1 != 0.f) atomicAdd(gp + geo.row1 + cj, geo.ly1 * own[q]);
    }
    if (!has_left) {  // edge columns nobody picked up (image border: clamped; head or row boundary)
      atomicAdd(gp + geo.row0 + geo.col[0], geo.ly0 * win[0]);
      if (geo.ly1 != 0.f) atomicAdd(gp + geo.row1 + geo.col[0], geo.ly1 * win[0]);
    }
    if (!has_right) {
      atomicAdd(gp + geo.row0 + geo.col[NCOL - 1], geo.ly0 * win[NCOL - 1]);
      if (geo.ly1 != 0.f) atomicAdd(gp + geo.row1 + geo.col[NCOL - 1], geo.ly1 * win[NCOL - 1]);
    }
  }
  if (gxb != nullptr && n_frames < g.T) {  // padded frames receive exactly zero
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (int t = 0; t < g.T; ++t)
      if (s_pad[t])
#pragma unroll
        for (int c = 0; c < 4; ++c) st_stream_v4(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(c) * g.hw, z);
  }
  if (a.partial == nullptr) return;

  // ---- parameter gradients of the tile: the s tile (bf16, the forward's value) replaces grad_s in shared memory -------
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");  // every consumer has its grad_s in registers
  const uint32_t s_tile = gs_tile;
#pragma unroll
  for (int c = 0; c < 4; ++c) sts_v4(s_tile + (head * 4 + c) * kScTileStride + pv * 16, Elem<T>::pack(acc[c]));
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");
  float* part = a.partial + (static_cast<size_t>(b) * gridDim.x + pblk) * kScPartial;
  float(*red)[8][kScC] = reinterpret_cast<float(*)[8][kScC]>(sb_smem);  // per-warp sums; the stages are drained by now
  if constexpr (!BSTATS) {  // z - mean = W s + (bias - mean): sums of g_y and g_y (z - mean) per output channel
    float d[4][2][4];
    skipconv_tile_mma(d, a.wfrag, s_tile, warp, lane);
    const unsigned char* gyb = sb_smem + n_stages * stage_stride;
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int o = mt * 16 + (lane >> 2) + hrow * 8;
        const float zs = __ldg(a.zshift + o);
        float sg = 0.f, sgz = 0.f;
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          const int p = warp * 16 + nt * 8 + (lane & 3) * 2;
          const __nv_bfloat162 gy2 = *reinterpret_cast<const __nv_bfloat162*>(gyb + o * kScTileStride + p * 2);
          const float g0 = __low2float(gy2), g1 = __high2float(gy2);
          sg += g0 + g1;
          sgz = fmaf(g0, d[mt][nt][hrow * 2] + zs, sgz);
          sgz = fmaf(g1, d[mt][nt][hrow * 2 + 1] + zs, sgz);
        }
        sg += __shfl_xor_sync(0xffffffffu, sg, 1);
        sg += __shfl_xor_sync(0xffffffffu, sg, 2);
        sgz += __shfl_xor_sync(0xffffffffu, sgz, 1);
        sgz += __shfl_xor_sync(0xffffffffu, sgz, 2);
        if ((lane & 3) == 0) red[0][warp][o] = sg, red[1][warp][o] = sgz;
      }
  }
  {  // g_y s^T [64 out][64 in] over the 128 pixels: warp w takes m-tile w / 2 and n-tiles 4 (w % 2) .. + 3, K = pixels
    const int mt = warp >> 1, nt0 = (warp & 1) * 4;
    float d[4][4];
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) d[n][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < kScPB / 16; ++ks) {
      uint32_t af[4], al[4];
      ldsm_x4(af, gy_tile + (mt * 16 + (lane & 15)) * kScTileStride + (ks * 16 + (lane >> 4) * 8) * 2);
      if constexpr (BSTATS) ldsm_x4(al, glo_tile + (mt * 16 + (lane & 15)) * kScTileStride + (ks * 16 + (lane >> 4) * 8) * 2);
#pragma unroll
      for (int np = 0; np < 2; ++np) {  // two n-tiles per ldmatrix.x4: (n 0-7 | 8-15) x (k 0-7 | 8-15)
        uint32_t bf[4];
        const int crow = (nt0 + 2 * np) * 8 + (lane & 7) + ((lane >> 4) & 1) * 8;
        ldsm_x4(bf, s_tile + crow * kScTileStride + (ks * 16 + ((lane >> 3) & 1) * 8) * 2);
        mma_bf16(d[2 * np], af, bf[0], bf[1]);
        mma_bf16(d[2 * np + 1], af, bf[2], bf[3]);
        if constexpr (BSTATS) {
          mma_bf16(d[2 * np], al, bf[0], bf[1]);
          mma_bf16(d[2 * np + 1], al, bf[2], bf[3]);
        }
      }
    }
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int o = mt * 16 + (lane >> 2) + hrow * 8, c = (nt0 + n) * 8 + (lane & 3) * 2;
        *reinterpret_cast<float2*>(part + o * kScC + c) = make_float2(d[n][hrow * 2], d[n][hrow * 2 + 1]);
      }
  }
  if constexpr (BSTATS) return;  // the BatchNorm sums came from skipconv_bstats_bwd_sums_kernel
  asm volatile("bar.sync 1, %0;" ::"n"(kScConsumers) : "memory");
  if (threadIdx.x < 2 * kScC) {  // fixed order over the warps
    const int q = threadIdx.x / kScC, o = threadIdx.x % kScC;
    float v = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) v += red[q][w8][o];
    part[kScC * kScC + q * kScC + o] = v;
  }
}

// Sum of the CTA partials in a fixed order (warp w takes CTAs w, w + 8, ...; the 8 warp sums are added in order), then
// the chain to the parameters: grad_conv_weight = alpha g_y s^T, grad_conv_bias = alpha sum g_y, grad_bn_bias = sum g_y,
// grad_bn_weight = sum g_y (z - mean) / sqrt(var + eps).
__global__ void __launch_bounds__(256) skipconv_bwd_finish_kernel(const float* __restrict__ partial, int n_ctas,
                                                                  const float* __restrict__ alpha, const float* __restrict__ inv_std,
                                                                  float* gw, float* gb, float* gbn_w, float* gbn_b) {
  __shared__ float sums[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = blockIdx.x * 32 + lane;
  float v = 0.f;
  if (e < kScPartial)
    for (int i = warp; i < n_ctas; i += 8) v += partial[static_cast<size_t>(i) * kScPartial + e];
  sums[warp][lane] = v;
  __syncthreads();
  if (warp != 0 || e >= kScPartial) return;
  float total = 0.f;
#pragma unroll
  for (int w8 = 0; w8 < 8; ++w8) total += sums[w8][lane];
  if (e < kScC * kScC) {
    if (gw != nullptr) gw[e] = alpha[e / kScC] * total;
  } else if (e < kScC * kScC + kScC) {
    const int o = e - kScC * kScC;
    if (gb != nullptr) gb[o] = alpha[o] * total;
    if (gbn_b != nullptr) gbn_b[o] = total;
  } else {
    const int o = e - kScC * kScC - kScC;
    if (gbn_w != nullptr) gbn_w[o] = inv_std[o] * total;
  }
}

// BSTATS pre-pass with the main kernel's tiling (one sample x 128 pixels; thread = 4 channels x 8 pixels): per CTA and
// channel, sum g_y and sum g_y zhat -> partial [2][64][CTAs]
__global__ void __launch_bounds__(kScConsumers) skipconv_bstats_bwd_sums_kernel(
    const __nv_bfloat16* __restrict__ gout, const __nv_bfloat16* __restrict__ out, const __nv_bfloat16* __restrict__ z,
    const float* __restrict__ inv_std, const float* __restrict__ zshift, int hw, float* __restrict__ partial) {
  const int head = threadIdx.x >> 4, pv = threadIdx.x & 15;
  const int n_ctas = gridDim.x * gridDim.y, cta = blockIdx.y * gridDim.x + blockIdx.x;
  const size_t plane = static_cast<size_t>(blockIdx.y) * kScC * hw + blockIdx.x * kScPB + pv * kScVec;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int ch = head * 4 + c;
    const size_t off = plane + static_cast<size_t>(ch) * hw;
    float gf[kScVec], zf[kScVec];
    Elem<__nv_bfloat16>::unpack(relu_masked(ld_stream_v4(gout + off), ld_stream_v4(out + off)), gf);
    Elem<__nv_bfloat16>::unpack(ld_stream_v4(z + off), zf);
    const float is = __ldg(inv_std + ch), zs = __ldg(zshift + ch);
    float sg = 0.f, sgz = 0.f;
#pragma unroll
    for (int j = 0; j < kScVec; ++j) {
      sg += gf[j];
      sgz = fmaf(gf[j], (zf[j] + zs) * is, sgz);
    }
#pragma unroll
    for (int m = 1; m < 16; m <<= 1) {  // the 16 lanes of this channel group, fixed order
      sg += __shfl_xor_sync(0xffffffffu, sg, m);
      sgz += __shfl_xor_sync(0xffffffffu, sgz, m);
    }
    if (pv == 0) {
      partial[static_cast<size_t>(ch) * n_ctas + cta] = sg;
      partial[static_cast<size_t>(kScC + ch) * n_ctas + cta] = sgz;
    }
  }
}

// One block per channel, fixed order: grad_bn_bias = sum g_y, grad_bn_weight = sum g_y zhat, and their means over the
// N = B H W pixels for the main kernel's g_z'
__global__ void __launch_bounds__(256) skipconv_bstats_bwd_means_kernel(const float* __restrict__ partial, int n_ctas,
                                                                        float* gmean, float* gbn_w, float* gbn_b) {
  const int o = blockIdx.x;
  float2 acc = make_float2(0.f, 0.f);
  for (int i = threadIdx.x; i < n_ctas; i += 256) {
    acc.x += partial[static_cast<size_t>(o) * n_ctas + i];
    acc.y += partial[static_cast<size_t>(kScC + o) * n_ctas + i];
  }
  acc = block_reduce_fixed(acc, [](float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); });
  if (threadIdx.x != 0) return;
  const float inv_n = 1.f / (static_cast<float>(n_ctas) * kScPB);
  gmean[o] = acc.x * inv_n, gmean[kScC + o] = acc.y * inv_n;
  if (gbn_b != nullptr) gbn_b[o] = acc.x;
  if (gbn_w != nullptr) gbn_w[o] = acc.y;
}

// ---------------------------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------------------------
struct SkipConvPlan {
  SkipConvShape g;  // n_stages is the caller's
  int scale_class;  // 2 / 4 / 8
  CUtensorMap map_x, map_att;
};

constexpr int kScNotServed = -1;

// Host side of both directions.  Returns kScNotServed, before any device call, when the fused kernels do not serve the
// call (att_group, bf16, C = 64, 16 heads, x2 / x4 / x8 up-sampling, H*W % 128 == 0, T <= kAggMaxT, 16-byte aligned
// `tensors`); each entry point reports that with its own status and message.  Otherwise checks the device, chooses the
// staged attention rows (none at x2 unless staged_taps_at_x2, none under C2S_OPT_AGG_TAPS) and encodes the tensor maps:
// C2S_OK or the error.
int skipconv_plan(const c2s_agg_desc* d, const void* x, const float* attn, std::initializer_list<const void*> tensors,
                  bool staged_taps_at_x2, SkipConvPlan* p) {
  p->scale_class = 0;
  for (int s : {2, 4, 8})
    if (d->H == s * d->ha && d->W == s * d->wa) p->scale_class = s;
  const int hw = d->H * d->W;
  bool aligned = true;
  for (const void* t : tensors) aligned = aligned && reinterpret_cast<uintptr_t>(t) % 16 == 0;  // nullptr: not passed
  if (d->mode != C2S_AGG_ATT_GROUP || d->dtype != C2S_BF16 || d->C != kScC || d->n_heads != 16 || p->scale_class == 0 ||
      hw % kScPB != 0 || d->W % 8 != 0 || d->T > kAggMaxT || d->B > 65535 || !aligned)
    return kScNotServed;
  int status = check_device();
  if (status != C2S_OK) return status;

  SkipConvShape& g = p->g;
  g = SkipConvShape{};
  g.B = d->B, g.T = d->T, g.H = d->H, g.W = d->W, g.hw = hw, g.ha = d->ha, g.wa = d->wa;
  g.sy = static_cast<float>(d->ha) / static_cast<float>(d->H);
  g.sx = static_cast<float>(d->wa) / static_cast<float>(d->W);
  {  // staged attention rows: the rows a 128-pixel block can touch, per head (16-byte aligned slices of the map)
    const int rows_out = (kScPB + d->W - 1) / d->W + 1;
    int rows_att = rows_out / p->scale_class + 3;
    rows_att = rows_att > d->ha ? d->ha : rows_att;
    const int tap_floats = ((rows_att * d->wa + 3) / 4) * 4;
    const bool taps = option(C2S_OPT_AGG_TAPS) == 0 && d->wa % 4 == 0 && reinterpret_cast<uintptr_t>(attn) % 16 == 0 &&
                      tap_floats <= 256 && (staged_taps_at_x2 || p->scale_class >= 4);
    g.tap_floats = taps ? tap_floats : 0;
  }
  // x as [B*T][C][H*W] bf16; box = 128 pixels x 64 channels x 1 frame, dense in shared memory
  const cuuint64_t dims[3] = {static_cast<cuuint64_t>(hw), static_cast<cuuint64_t>(kScC), static_cast<cuuint64_t>(d->B) * d->T};
  const cuuint64_t strides[2] = {static_cast<cuuint64_t>(hw) * 2, static_cast<cuuint64_t>(kScC) * hw * 2};
  const cuuint32_t box[3] = {kScPB, kScC, 1};
  status = encode_tensor_map(&p->map_x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_NONE, "skip features");
  if (status != C2S_OK) return status;
  p->map_att = p->map_x;  // attention as [16 heads][B*T][ha*wa] fp32; box = tap_floats of one map x 1 frame x 16 heads
  if (g.tap_floats == 0) return C2S_OK;
  const cuuint64_t amap = static_cast<cuuint64_t>(d->ha) * d->wa;
  const cuuint64_t adims[3] = {amap, static_cast<cuuint64_t>(d->B) * d->T, 16};
  const cuuint64_t astrides[2] = {amap * 4, static_cast<cuuint64_t>(d->B) * d->T * amap * 4};
  const cuuint32_t abox[3] = {static_cast<cuuint32_t>(g.tap_floats), 1, 16};
  return encode_tensor_map(&p->map_att, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, attn, adims, astrides, abox,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, "attention");
}

template <int S, bool TAPS, bool BSTATS>
int launch_skipconv_t(const SkipConvPlan& p, const SkipConvArgs& k, cudaStream_t stream, const char* name) {
  const size_t smem = static_cast<size_t>(k.g.n_stages) * (kScStageBytes + 16 * k.g.tap_floats * 4) + kScC * kScTileStride;
  C2S_SMEM_ATTR((agg_skipconv_kernel<S, TAPS, BSTATS>), 227 * 1024);  // once per instantiation and device (smem varies per call)
  dim3 grid(k.g.hw / kScPB, k.g.B);
  agg_skipconv_kernel<S, TAPS, BSTATS><<<grid, kScConsumers + 32, smem, stream>>>(p.map_x, p.map_att, k);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <int S, bool BSTATS>
int launch_skipconv(const SkipConvPlan& p, const SkipConvArgs& k, cudaStream_t stream, const char* name) {
  return k.g.tap_floats > 0 ? launch_skipconv_t<S, true, BSTATS>(p, k, stream, name)
                            : launch_skipconv_t<S, false, BSTATS>(p, k, stream, name);
}

// stages | g_y tile | grad_s (then s) tile | BSTATS: g_z' lo tile
size_t skipconv_bwd_smem(int n_stages, int tap_floats, bool bstats) {
  return static_cast<size_t>(n_stages) * (kScStageBytes + 16 * tap_floats * 4) + kScC * kScTileStride + kScC * kScGsStride * 4 +
         (bstats ? kScC * kScTileStride : 0);
}

template <int S, bool TAPS, bool BSTATS>
int launch_skipconv_bwd_t(const SkipConvPlan& p, const SkipConvBwdArgs& k, const SkipConvBstatsIn<BSTATS>& bs,
                          cudaStream_t stream, const char* name) {
  const size_t smem = skipconv_bwd_smem(k.g.n_stages, k.g.tap_floats, BSTATS);
  C2S_SMEM_ATTR((agg_skipconv_backward_kernel<S, TAPS, BSTATS>), 227 * 1024);  // once per instantiation and device
  dim3 grid(k.g.hw / kScPB, k.g.B);
  agg_skipconv_backward_kernel<S, TAPS, BSTATS><<<grid, kScConsumers + 32, smem, stream>>>(p.map_x, p.map_att, k, bs);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <int S, bool BSTATS>
int launch_skipconv_bwd(const SkipConvPlan& p, const SkipConvBwdArgs& k, const SkipConvBstatsIn<BSTATS>& bs,
                        cudaStream_t stream, const char* name) {
  return k.g.tap_floats > 0 ? launch_skipconv_bwd_t<S, true, BSTATS>(p, k, bs, stream, name)
                            : launch_skipconv_bwd_t<S, false, BSTATS>(p, k, bs, stream, name);
}

// stages for the backward's ring: fewer if the staged rows make them too large for one CTA (227 KB with the static part)
int skipconv_bwd_stages(int tap_floats, bool bstats) {
  int n = kScMaxStages;
  while (n > 2 && skipconv_bwd_smem(n, tap_floats, bstats) > 220 * 1024) --n;
  return n;
}

// backward workspace: W and (alpha W)^T fragments, alpha / inv_std / zshift, then the CTA partials (16-byte aligned throughout)
constexpr size_t kScBwdFixedBytes = 2 * 2 * kScFrags * sizeof(uint4) + 3 * kScC * sizeof(float);
size_t skipconv_bwd_ctas(const c2s_agg_desc* d) {
  return d->B > 0 && d->H > 0 && d->W > 0 ? static_cast<size_t>(d->B) * ((static_cast<size_t>(d->H) * d->W) / kScPB) : 0;
}
// batch-statistics forward workspace: W fragments, scale, shift, then the [mean | M2][64][CTAs] partials
constexpr size_t kScBstatsFixedBytes = 2 * kScFrags * sizeof(uint4) + 2 * kScC * sizeof(float);
// batch-statistics backward workspace: the backward's fixed part, the two g_y means [2][64], the main kernel's CTA partials
// (kScPartial floats each, of which the 64 x 64 weight term is used), then the pre-pass partials [2][64][CTAs]
constexpr size_t kScBstatsBwdFixedBytes = kScBwdFixedBytes + 2 * kScC * sizeof(float);

}  // namespace
}  // namespace c2s

extern "C" {

size_t c2s_agg_skipconv_workspace_bytes(const c2s_agg_desc* d) {
  (void)d;
  return 2 * c2s::kScFrags * sizeof(uint4) + 2 * c2s::kScC * sizeof(float);  // W fragments (hi, lo), scale, shift
}

int c2s_agg_skipconv_forward(const c2s_agg_desc* d, const void* x, const float* attn, const uint8_t* pad_mask,
                             const c2s_skipconv_params* p, void* out, void* workspace, size_t workspace_bytes,
                             void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(d != nullptr && p != nullptr, "c2s_agg_skipconv_forward: desc/params is NULL");
  C2S_CHECK_ARG(x != nullptr && out != nullptr && attn != nullptr, "c2s_agg_skipconv_forward: x/attn/out is NULL");
  C2S_CHECK_ARG(p->conv_weight != nullptr && p->bn_running_mean != nullptr && p->bn_running_var != nullptr,
                "c2s_agg_skipconv_forward: conv weight and BatchNorm running statistics are required");
  C2S_CHECK_ARG(d->B > 0 && d->T > 0 && d->H > 0 && d->W > 0, "c2s_agg_skipconv_forward: non-positive dimension");
  C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= c2s_agg_skipconv_workspace_bytes(d),
                "c2s_agg_skipconv_forward: needs %zu workspace bytes", c2s_agg_skipconv_workspace_bytes(d));
  C2S_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 16 == 0, "c2s_agg_skipconv_forward: workspace must be 16-byte aligned");
  SkipConvPlan plan;
  // x2: measured slower with staged taps here (0.151 vs 0.109 ms at 32 x 32), so that level keeps the global-memory taps
  int status = skipconv_plan(d, x, attn, {x, out}, /*staged_taps_at_x2=*/false, &plan);
  if (status == kScNotServed)
    C2S_UNSUPPORTED("c2s_agg_skipconv_forward: the fused path serves att_group, bf16, C=64, 16 heads, x2/x4/x8 up-sampling, "
                    "H*W %% 128 == 0 (got mode %d dtype %d C %d heads %d %dx%d from %dx%d); run c2s_agg_forward and the "
                    "convolution separately", d->mode, d->dtype, d->C, d->n_heads, d->H, d->W, d->ha, d->wa);
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);

  uint4* wfrag = static_cast<uint4*>(workspace);
  float* scale = reinterpret_cast<float*>(wfrag + 2 * kScFrags);
  float* shift = scale + kScC;
  skipconv_prep_kernel<<<3, 256, 0, stream>>>(p->conv_weight, wfrag, p->conv_bias, p->bn_weight, p->bn_bias,
                                              p->bn_running_mean, p->bn_running_var, p->bn_eps, scale, shift);
  C2S_LAUNCH_CHECK("skipconv_prep");
  SkipConvArgs k{};
  k.g = plan.g;
  k.g.n_stages = 4;
  k.attn = attn, k.pad = pad_mask, k.out = static_cast<__nv_bfloat16*>(out);
  k.wfrag = wfrag, k.scale = scale, k.shift = shift;
  switch (plan.scale_class) {
    case 2: return launch_skipconv<2, false>(plan, k, stream, "agg_skipconv<x2>");
    case 4: return launch_skipconv<4, false>(plan, k, stream, "agg_skipconv<x4>");
    default: return launch_skipconv<8, false>(plan, k, stream, "agg_skipconv<x8>");
  }
}

size_t c2s_agg_skipconv_backward_workspace_bytes(const c2s_agg_desc* d) {
  if (d == nullptr) return 0;
  return c2s::kScBwdFixedBytes + c2s::skipconv_bwd_ctas(d) * c2s::kScPartial * sizeof(float);
}

int c2s_agg_skipconv_backward(const c2s_agg_desc* d, const void* x, const float* attn, const uint8_t* pad_mask,
                              const c2s_skipconv_params* p, const void* out, const void* grad_out,
                              const c2s_skipconv_bwd_io* io, void* workspace, size_t workspace_bytes, void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(d != nullptr && p != nullptr && io != nullptr, "c2s_agg_skipconv_backward: desc/params/io is NULL");
  C2S_CHECK_ARG(x != nullptr && attn != nullptr && out != nullptr && grad_out != nullptr,
                "c2s_agg_skipconv_backward: x/attn/out/grad_out is NULL");
  C2S_CHECK_ARG(p->conv_weight != nullptr && p->bn_running_mean != nullptr && p->bn_running_var != nullptr,
                "c2s_agg_skipconv_backward: conv weight and BatchNorm running statistics are required");
  C2S_CHECK_ARG(d->B > 0 && d->T > 0 && d->H > 0 && d->W > 0, "c2s_agg_skipconv_backward: non-positive dimension");
  SkipConvPlan plan;
  int status = skipconv_plan(d, x, attn, {x, out, grad_out, io->grad_x}, /*staged_taps_at_x2=*/true, &plan);
  C2S_CHECK_ARG(status != kScNotServed,
                "c2s_agg_skipconv_backward: the fused backward serves what the fused forward serves: att_group, bf16, C=64, "
                "16 heads, x2/x4/x8 up-sampling, H*W %% 128 == 0, 16-byte aligned tensors (got mode %d dtype %d C %d heads "
                "%d %dx%d from %dx%d)", d->mode, d->dtype, d->C, d->n_heads, d->H, d->W, d->ha, d->wa);
  if (status != C2S_OK) return status;
  const bool want_params = io->grad_conv_weight != nullptr || io->grad_conv_bias != nullptr || io->grad_bn_weight != nullptr ||
                           io->grad_bn_bias != nullptr;
  if (!want_params && io->grad_x == nullptr && io->grad_attn == nullptr) return C2S_OK;  // nothing asked for
  const size_t need = c2s_agg_skipconv_backward_workspace_bytes(d);
  C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= need && reinterpret_cast<uintptr_t>(workspace) % 16 == 0,
                "c2s_agg_skipconv_backward: needs %zu workspace bytes, 16-byte aligned", need);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);

  uint4* wfrag = static_cast<uint4*>(workspace);
  uint4* afrag = wfrag + 2 * kScFrags;
  float* alpha = reinterpret_cast<float*>(afrag + 2 * kScFrags);
  float* inv_std = alpha + kScC;
  float* zshift = inv_std + kScC;
  float* partial = reinterpret_cast<float*>(static_cast<char*>(workspace) + kScBwdFixedBytes);
  skipconv_bwd_prep_kernel<<<3, 256, 0, stream>>>(p->conv_weight, p->conv_bias, p->bn_weight, p->bn_running_mean,
                                                  p->bn_running_var, p->bn_eps, wfrag, afrag, alpha, inv_std, zshift);
  C2S_LAUNCH_CHECK("agg_skipconv_backward<prep>");

  SkipConvBwdArgs k{};
  k.g = plan.g;
  k.g.n_stages = skipconv_bwd_stages(k.g.tap_floats, false);
  k.attn = attn, k.pad = pad_mask;
  k.out = static_cast<const __nv_bfloat16*>(out), k.gout = static_cast<const __nv_bfloat16*>(grad_out);
  k.gx = static_cast<__nv_bfloat16*>(io->grad_x), k.gattn = io->grad_attn;
  k.wfrag = wfrag, k.afrag = afrag, k.zshift = zshift, k.partial = want_params ? partial : nullptr;
  switch (plan.scale_class) {
    case 2: status = launch_skipconv_bwd<2, false>(plan, k, {}, stream, "agg_skipconv_backward<x2>"); break;
    case 4: status = launch_skipconv_bwd<4, false>(plan, k, {}, stream, "agg_skipconv_backward<x4>"); break;
    default: status = launch_skipconv_bwd<8, false>(plan, k, {}, stream, "agg_skipconv_backward<x8>"); break;
  }
  if (status != C2S_OK || !want_params) return status;
  skipconv_bwd_finish_kernel<<<ceil_div(kScPartial, 32), 256, 0, stream>>>(
      partial, static_cast<int>(skipconv_bwd_ctas(d)), alpha, inv_std, io->grad_conv_weight, io->grad_conv_bias,
      io->grad_bn_weight, io->grad_bn_bias);
  C2S_LAUNCH_CHECK("agg_skipconv_backward<reduce>");
  return C2S_OK;
}

size_t c2s_agg_skipconv_bstats_workspace_bytes(const c2s_agg_desc* d) {
  if (d == nullptr) return 0;
  return c2s::kScBstatsFixedBytes + c2s::skipconv_bwd_ctas(d) * 2 * c2s::kScC * sizeof(float);
}

int c2s_agg_skipconv_bstats_forward(const c2s_agg_desc* d, const void* x, const float* attn, const uint8_t* pad_mask,
                                    const c2s_skipconv_params* p, void* z, void* out, float* bn_batch_mean,
                                    float* bn_batch_var, void* workspace, size_t workspace_bytes, void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(d != nullptr && p != nullptr, "c2s_agg_skipconv_bstats_forward: desc/params is NULL");
  C2S_CHECK_ARG(x != nullptr && attn != nullptr && z != nullptr && out != nullptr && bn_batch_mean != nullptr &&
                    bn_batch_var != nullptr && p->conv_weight != nullptr,
                "c2s_agg_skipconv_bstats_forward: x/attn/z/out/bn_batch_mean/bn_batch_var/conv_weight is NULL");
  C2S_CHECK_ARG(d->B > 0 && d->T > 0 && d->H > 0 && d->W > 0, "c2s_agg_skipconv_bstats_forward: non-positive dimension");
  SkipConvPlan plan;
  int status = skipconv_plan(d, x, attn, {x, z, out}, /*staged_taps_at_x2=*/false, &plan);
  if (status == kScNotServed)
    C2S_UNSUPPORTED("c2s_agg_skipconv_bstats_forward: the fused path serves att_group, bf16, C=64, 16 heads, x2/x4/x8 "
                    "up-sampling, H*W %% 128 == 0 (got mode %d dtype %d C %d heads %d %dx%d from %dx%d); run c2s_agg_forward "
                    "and the convolution separately", d->mode, d->dtype, d->C, d->n_heads, d->H, d->W, d->ha, d->wa);
  if (status != C2S_OK) return status;
  const size_t need = c2s_agg_skipconv_bstats_workspace_bytes(d);
  C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= need && reinterpret_cast<uintptr_t>(workspace) % 16 == 0,
                "c2s_agg_skipconv_bstats_forward: needs %zu workspace bytes, 16-byte aligned", need);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  const int n_ctas = static_cast<int>(skipconv_bwd_ctas(d));

  uint4* wfrag = static_cast<uint4*>(workspace);
  float* scale = reinterpret_cast<float*>(wfrag + 2 * kScFrags);
  float* shift = scale + kScC;
  float* partial = reinterpret_cast<float*>(static_cast<char*>(workspace) + kScBstatsFixedBytes);
  // blocks 0-1 only: the W fragments (block 2 would read the running statistics)
  skipconv_prep_kernel<<<2, 256, 0, stream>>>(p->conv_weight, wfrag, nullptr, nullptr, nullptr, nullptr, nullptr, 0.f,
                                              nullptr, nullptr);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats<prep>");
  SkipConvArgs k{};
  k.g = plan.g;
  k.g.n_stages = 4;
  k.attn = attn, k.pad = pad_mask, k.out = static_cast<__nv_bfloat16*>(z);
  k.wfrag = wfrag, k.shift = p->conv_bias, k.partial = partial;
  switch (plan.scale_class) {
    case 2: status = launch_skipconv<2, true>(plan, k, stream, "agg_skipconv_bstats<x2>"); break;
    case 4: status = launch_skipconv<4, true>(plan, k, stream, "agg_skipconv_bstats<x4>"); break;
    default: status = launch_skipconv<8, true>(plan, k, stream, "agg_skipconv_bstats<x8>"); break;
  }
  if (status != C2S_OK) return status;
  skipconv_bstats_finish_kernel<<<kScC, 256, 0, stream>>>(partial, n_ctas, p->bn_weight, p->bn_bias, p->bn_eps,
                                                          bn_batch_mean, bn_batch_var, scale, shift);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats<stats>");
  const int hw_vec = plan.g.hw / kScVec;
  skipconv_bstats_apply_kernel<<<dim3(d->B * kScC, ceil_div(hw_vec, 256)), 256, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(z), static_cast<__nv_bfloat16*>(out), scale, shift, hw_vec);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats<apply>");
  return C2S_OK;
}

size_t c2s_agg_skipconv_bstats_backward_workspace_bytes(const c2s_agg_desc* d) {
  if (d == nullptr) return 0;
  return c2s::kScBstatsBwdFixedBytes + c2s::skipconv_bwd_ctas(d) * (c2s::kScPartial + 2 * c2s::kScC) * sizeof(float);
}

int c2s_agg_skipconv_bstats_backward(const c2s_agg_desc* d, const void* x, const float* attn, const uint8_t* pad_mask,
                                     const c2s_skipconv_params* p, const void* z, const float* bn_batch_mean,
                                     const float* bn_batch_var, const void* out, const void* grad_out,
                                     const c2s_skipconv_bwd_io* io, void* workspace, size_t workspace_bytes,
                                     void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(d != nullptr && p != nullptr && io != nullptr, "c2s_agg_skipconv_bstats_backward: desc/params/io is NULL");
  C2S_CHECK_ARG(x != nullptr && attn != nullptr && z != nullptr && bn_batch_mean != nullptr && bn_batch_var != nullptr &&
                    out != nullptr && grad_out != nullptr && p->conv_weight != nullptr,
                "c2s_agg_skipconv_bstats_backward: x/attn/z/bn_batch_mean/bn_batch_var/out/grad_out/conv_weight is NULL");
  C2S_CHECK_ARG(d->B > 0 && d->T > 0 && d->H > 0 && d->W > 0, "c2s_agg_skipconv_bstats_backward: non-positive dimension");
  SkipConvPlan plan;
  int status = skipconv_plan(d, x, attn, {x, z, out, grad_out, io->grad_x}, /*staged_taps_at_x2=*/true, &plan);
  C2S_CHECK_ARG(status != kScNotServed,
                "c2s_agg_skipconv_bstats_backward: the fused backward serves what the fused forward serves: att_group, "
                "bf16, C=64, 16 heads, x2/x4/x8 up-sampling, H*W %% 128 == 0, 16-byte aligned tensors (got mode %d dtype "
                "%d C %d heads %d %dx%d from %dx%d)", d->mode, d->dtype, d->C, d->n_heads, d->H, d->W, d->ha, d->wa);
  if (status != C2S_OK) return status;
  const bool want_main = io->grad_x != nullptr || io->grad_attn != nullptr || io->grad_conv_weight != nullptr;
  const bool want_bn = io->grad_bn_weight != nullptr || io->grad_bn_bias != nullptr;
  if (!want_main && !want_bn && io->grad_conv_bias == nullptr) return C2S_OK;  // nothing asked for
  const size_t need = c2s_agg_skipconv_bstats_backward_workspace_bytes(d);
  C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= need && reinterpret_cast<uintptr_t>(workspace) % 16 == 0,
                "c2s_agg_skipconv_bstats_backward: needs %zu workspace bytes, 16-byte aligned", need);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  // batch statistics remove any per-channel constant of z, so the convolution bias has no effect on the output
  if (io->grad_conv_bias != nullptr) C2S_CUDA(cudaMemsetAsync(io->grad_conv_bias, 0, kScC * sizeof(float), stream));
  if (!want_main && !want_bn) return C2S_OK;
  const int n_ctas = static_cast<int>(skipconv_bwd_ctas(d));

  uint4* wfrag = static_cast<uint4*>(workspace);
  uint4* afrag = wfrag + 2 * kScFrags;
  float* alpha = reinterpret_cast<float*>(afrag + 2 * kScFrags);
  float* inv_std = alpha + kScC;
  float* zshift = inv_std + kScC;
  float* gmean = zshift + kScC;
  float* partial = reinterpret_cast<float*>(static_cast<char*>(workspace) + kScBstatsBwdFixedBytes);
  float* sums = partial + static_cast<size_t>(n_ctas) * kScPartial;
  // the eval backward's preparation on the batch statistics, without the conv bias: zshift = -mean, alpha = gamma inv_std
  skipconv_bwd_prep_kernel<<<3, 256, 0, stream>>>(p->conv_weight, nullptr, p->bn_weight, bn_batch_mean, bn_batch_var,
                                                  p->bn_eps, wfrag, afrag, alpha, inv_std, zshift);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats_backward<prep>");
  const dim3 grid(plan.g.hw / kScPB, d->B);
  skipconv_bstats_bwd_sums_kernel<<<grid, kScConsumers, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(grad_out), static_cast<const __nv_bfloat16*>(out),
      static_cast<const __nv_bfloat16*>(z), inv_std, zshift, plan.g.hw, sums);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats_backward<sums>");
  skipconv_bstats_bwd_means_kernel<<<kScC, 256, 0, stream>>>(sums, n_ctas, gmean, io->grad_bn_weight, io->grad_bn_bias);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats_backward<means>");
  if (!want_main) return C2S_OK;

  SkipConvBwdArgs k{};
  k.g = plan.g;
  k.g.n_stages = skipconv_bwd_stages(k.g.tap_floats, true);
  k.attn = attn, k.pad = pad_mask;
  k.out = static_cast<const __nv_bfloat16*>(out), k.gout = static_cast<const __nv_bfloat16*>(grad_out);
  k.gx = static_cast<__nv_bfloat16*>(io->grad_x), k.gattn = io->grad_attn;
  k.wfrag = wfrag, k.afrag = afrag, k.zshift = zshift, k.partial = io->grad_conv_weight != nullptr ? partial : nullptr;
  const SkipConvBstatsIn<true> bs{static_cast<const __nv_bfloat16*>(z), inv_std, gmean};
  switch (plan.scale_class) {
    case 2: status = launch_skipconv_bwd<2, true>(plan, k, bs, stream, "agg_skipconv_bstats_backward<x2>"); break;
    case 4: status = launch_skipconv_bwd<4, true>(plan, k, bs, stream, "agg_skipconv_bstats_backward<x4>"); break;
    default: status = launch_skipconv_bwd<8, true>(plan, k, bs, stream, "agg_skipconv_bstats_backward<x8>"); break;
  }
  if (status != C2S_OK || io->grad_conv_weight == nullptr) return status;
  // the 64 x 64 weight entries only: grad_conv_weight = alpha sum g_z' s^T
  skipconv_bwd_finish_kernel<<<kScC * kScC / 32, 256, 0, stream>>>(partial, n_ctas, alpha, inv_std, io->grad_conv_weight,
                                                                   nullptr, nullptr, nullptr);
  C2S_LAUNCH_CHECK("agg_skipconv_bstats_backward<reduce>");
  return C2S_OK;
}

}  // extern "C"
