// TemporalAggregator forward for sm_100a.
//
// Replaces TemporalAggregator.forward (reference src/backbones/temporal_aggregator.py:14-77):
//   out[b,c,y,x] = sum_t  resize(attn)[c / (C/h), b, t, y, x] * (pad[b,t] ? 0 : 1) * x[b,t,c,y,x]
// The reference materialises the up-sampled attention (nn.Upsample, :17-19,27), a head-major copy
// of x (torch.stack(x.chunk), :35) and the full-size product (:37) in HBM.  Here every byte of x is
// read exactly once with 128-bit streaming loads, the bilinear weights are rebuilt in registers
// from the low-resolution attention map (which stays L1/L2 resident: h*T*ha*wa*4 B = 1 MB per
// sample at the shipped shapes), padded frames are never read, and only out[B,C,H,W] is written.
//
// Work decomposition: one thread owns VEC consecutive pixels (one 16-byte vector) of CPT
// consecutive channels that share one attention head, loops over the valid frames of its sample
// and keeps VEC*CPT fp32 accumulators in registers.  A warp therefore reads 512 contiguous bytes
// per (frame, channel); CPT*U independent 16-byte loads are in flight per thread.
//
// HBM roofline: algorithmic bytes = e*T_valid*C*H*W (x) + e*C*H*W (out) per sample, see DESIGN.md.
#include <cstdlib>
#include <type_traits>

#include "c2s_sm100.cuh"

namespace c2s {
namespace {

constexpr int kAggThreads = 256;

struct AggArgs {
  const void* x;
  const float* attn;  // [n_heads, B, T, ha, wa] or nullptr (uniform weights)
  const uint8_t* pad;  // [B, T] or nullptr
  const int* order;    // [B] samples by decreasing number of valid frames (pipelined kernel) or nullptr
  void* out;
  int B, T, C, H, W;
  int n_heads, ha, wa;
  int cpg;           // channels per attention head = C / n_heads
  int uniform_div;   // 'mean' mode: weights are 1 and the sum is divided by the number of frames read
  float sy, sx;      // ATen's area_pixel_compute_scale: float(in) / out
  int hw;            // H * W
  int pv_per_plane;  // hw / VEC
  int items_per_b;   // (C / CPT) * pv_per_plane
};

template <typename T, int VEC>
struct PixelVec;  // VEC pixels of one channel

template <>
struct PixelVec<float, 4> {
  uint4 v;
  __device__ __forceinline__ void load(const float* p) { v = ld_stream_v4(p); }
  __device__ __forceinline__ void get(float (&f)[4]) const { Elem<float>::unpack(v, f); }
  __device__ static __forceinline__ void store(float* p, const float (&f)[4]) { st_stream_v4(p, Elem<float>::pack(f)); }
};
template <>
struct PixelVec<__nv_bfloat16, 8> {
  uint4 v;
  __device__ __forceinline__ void load(const __nv_bfloat16* p) { v = ld_stream_v4(p); }
  __device__ __forceinline__ void get(float (&f)[8]) const { Elem<__nv_bfloat16>::unpack(v, f); }
  __device__ static __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    st_stream_v4(p, Elem<__nv_bfloat16>::pack(f));
  }
};
template <typename T>
struct PixelVec<T, 1> {  // scalar fallback: any W, any alignment
  T v;
  __device__ __forceinline__ void load(const T* p) { v = *p; }
  __device__ __forceinline__ void get(float (&f)[1]) const { f[0] = Elem<T>::load(&v); }
  __device__ static __forceinline__ void store(T* p, const float (&f)[1]) { Elem<T>::store(p, f[0]); }
};

// S > 0 : H == S*ha and W == S*wa with S a power of two; the VEC pixels of a thread touch a
//         compile-time window of NCOL low-resolution columns (2 rows x NCOL loads per frame).
// S == 0: any size ratio; 4 attention loads per pixel and frame.
// S == -1: no attention map (mode 'mean').
template <int VEC, int S>
struct Window {
  static constexpr int kCols = (S > 0) ? ((VEC >= S) ? VEC / S + 2 : 2) : 1;
};

template <typename T, int VEC, int CPT, int S>
__global__ void __launch_bounds__(kAggThreads) agg_forward_kernel(const AggArgs a) {
  __shared__ short frames[kAggMaxT];
  __shared__ int n_frames_s;

  const int b = blockIdx.y;
  if (threadIdx.x < 32) {  // ordered list of the frames that are not padded
    int count = 0;
    for (int base = 0; base < a.T; base += 32) {
      const int t = base + threadIdx.x;
      const bool valid = t < a.T && (a.pad == nullptr || a.pad[b * a.T + t] == 0);
      const unsigned m = __ballot_sync(0xffffffffu, valid);
      if (valid) frames[count + __popc(m & ((1u << threadIdx.x) - 1u))] = static_cast<short>(t);
      count += __popc(m);
    }
    if (threadIdx.x == 0) n_frames_s = count;
  }
  __syncthreads();
  const int n_frames = n_frames_s;

  const int item = blockIdx.x * kAggThreads + threadIdx.x;
  if (item >= a.items_per_b) return;
  const int cchunk = item / a.pv_per_plane;
  const int pv = item - cchunk * a.pv_per_plane;
  const int c0 = cchunk * CPT;
  const int p0 = pv * VEC;
  const int y = p0 / a.W;
  const int x0 = p0 - y * a.W;

  constexpr int NCOL = Window<VEC, S>::kCols;
  // vertical taps (shared by the VEC pixels) and horizontal taps
  int row0 = 0, row1 = 0;
  float ly1 = 0.f;
  int col[(S > 0) ? NCOL : 1];
  int gcol0[(S == 0) ? VEC : 1], gcol1[(S == 0) ? VEC : 1];
  float lx1[VEC];
  if constexpr (S >= 0) {
    int iy0, iy1;
    source_index(a.sy, y, a.ha, iy0, iy1, ly1);
    row0 = iy0 * a.wa;
    row1 = iy1 * a.wa;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      int i0, i1;
      source_index(a.sx, x0 + j, a.wa, i0, i1, lx1[j]);
      if constexpr (S == 0) {
        gcol0[j] = i0;
        gcol1[j] = i1;
      }
    }
    if constexpr (S > 0) {
      int cmin = x0 / S - 1;
      if constexpr (VEC < S) cmin += ((x0 % S) >= S / 2) ? 1 : 0;
#pragma unroll
      for (int j = 0; j < NCOL; ++j) {
        int cj = cmin + j;
        cj = cj < 0 ? 0 : cj;
        col[j] = cj > a.wa - 1 ? a.wa - 1 : cj;
      }
    }
  }
  const float ly0 = 1.f - ly1;

  const size_t frame_stride = static_cast<size_t>(a.C) * a.hw;
  const T* xb = static_cast<const T*>(a.x) + static_cast<size_t>(b) * a.T * frame_stride +
                static_cast<size_t>(c0) * a.hw + p0;
  const int amap = a.ha * a.wa;
  const float* ab = nullptr;
  if constexpr (S >= 0) {
    const int g = c0 / a.cpg;
    ab = a.attn + (static_cast<size_t>(g) * a.B + b) * a.T * amap;
  }

  float acc[CPT][VEC];
#pragma unroll
  for (int k = 0; k < CPT; ++k)
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[k][j] = 0.f;

  // one group of U frames: all global loads are issued before the first use
  auto step = [&](auto u_tag, int i) {
    constexpr int U = decltype(u_tag)::value;
    PixelVec<T, VEC> xv[U][CPT];
    float top[U][(S > 0) ? NCOL : ((S == 0) ? 2 * VEC : 1)];
    float bot[U][(S > 0) ? NCOL : ((S == 0) ? 2 * VEC : 1)];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = frames[i + u];
      const T* xp = xb + static_cast<size_t>(t) * frame_stride;
#pragma unroll
      for (int k = 0; k < CPT; ++k) xv[u][k].load(xp + static_cast<size_t>(k) * a.hw);
      if constexpr (S > 0) {
        const float* ap = ab + static_cast<size_t>(t) * amap;
#pragma unroll
        for (int j = 0; j < NCOL; ++j) {
          top[u][j] = __ldg(ap + row0 + col[j]);
          bot[u][j] = __ldg(ap + row1 + col[j]);
        }
      } else if constexpr (S == 0) {
        const float* ap = ab + static_cast<size_t>(t) * amap;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          top[u][2 * j] = __ldg(ap + row0 + gcol0[j]);
          top[u][2 * j + 1] = __ldg(ap + row0 + gcol1[j]);
          bot[u][2 * j] = __ldg(ap + row1 + gcol0[j]);
          bot[u][2 * j + 1] = __ldg(ap + row1 + gcol1[j]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float w[VEC];
      if constexpr (S > 0) {
        float r[NCOL];
#pragma unroll
        for (int j = 0; j < NCOL; ++j) r[j] = fmaf(ly1, bot[u][j], ly0 * top[u][j]);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const int i0w = (VEC >= S) ? (j / S + ((j % S) < S / 2 ? 0 : 1)) : 0;
          w[j] = fmaf(lx1[j], r[i0w + 1], (1.f - lx1[j]) * r[i0w]);
        }
      } else if constexpr (S == 0) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float l0 = 1.f - lx1[j];
          const float tp = fmaf(lx1[j], top[u][2 * j + 1], l0 * top[u][2 * j]);
          const float bt = fmaf(lx1[j], bot[u][2 * j + 1], l0 * bot[u][2 * j]);
          w[j] = fmaf(ly1, bt, ly0 * tp);
        }
      }
#pragma unroll
      for (int k = 0; k < CPT; ++k) {
        float f[VEC];
        xv[u][k].get(f);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          if constexpr (S >= 0)
            acc[k][j] = fmaf(w[j], f[j], acc[k][j]);
          else
            acc[k][j] += f[j];
        }
      }
    }
  };

  constexpr int U = (sizeof(T) * VEC * CPT >= 64) ? 2 : 4;  // >= 128 B of x in flight per thread
  int i = 0;
  for (; i + U <= n_frames; i += U) step(std::integral_constant<int, U>{}, i);
  for (; i < n_frames; ++i) step(std::integral_constant<int, 1>{}, i);

  T* op = static_cast<T*>(a.out) + (static_cast<size_t>(b) * a.C + c0) * a.hw + p0;
#pragma unroll
  for (int k = 0; k < CPT; ++k) {
    if (a.uniform_div) {  // no valid frame: 0 / 0 = nan, as in the reference
#pragma unroll
      for (int j = 0; j < VEC; ++j) acc[k][j] = acc[k][j] / static_cast<float>(n_frames);
    }
    PixelVec<T, VEC>::store(op + static_cast<size_t>(k) * a.hw, acc[k]);
  }
}

// attn_mean[b,t,y,x] = mean_h attn[h,b,t,y,x]          (temporal_aggregator.py:48 / :72)
__global__ void head_mean_kernel(const float* __restrict__ attn, float* __restrict__ out, int n_heads, size_t n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int h = 0; h < n_heads; ++h) s += attn[static_cast<size_t>(h) * n + i];
  out[i] = s / static_cast<float>(n_heads);
}

// nn.AvgPool2d(kernel_size=k) on the last two axes (temporal_aggregator.py:29): stride k, floor.
__global__ void avg_pool_kernel(const float* __restrict__ in, float* __restrict__ out, int hi, int wi, int ho,
                                int wo, int k, size_t n_out) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const int x = static_cast<int>(i % wo);
  const int y = static_cast<int>((i / wo) % ho);
  const size_t map = i / (static_cast<size_t>(wo) * ho);
  const float* p = in + map * hi * wi + static_cast<size_t>(y) * k * wi + static_cast<size_t>(x) * k;
  float s = 0.f;
  for (int dy = 0; dy < k; ++dy)
    for (int dx = 0; dx < k; ++dx) s += p[dy * wi + dx];
  out[i] = s / static_cast<float>(k * k);
}


// ---------------------------------------------------------------------------------------------------
// Pipelined variant: the feature stream goes HBM -> shared memory through the bulk-copy engine
// (cp.async.bulk + mbarrier transaction counts), so the number of bytes in flight per SM is set by the
// ring of stages (2 CTAs x 6 stages x 16 KB = 192 KB) instead of by registers.  One producer thread
// issues four 4 KB row copies (the 4 channels of one attention head x PB pixels) per frame; the
// consumer warps read their 16-byte vectors back with conflict-free LDS.128 and release the stage.
// ---------------------------------------------------------------------------------------------------
constexpr int kPipeCPT = 4;
constexpr int kPipeMaxConsumers = 256;

// The CTAs of a sample do work proportional to its number of valid frames (27 .. 61 in the benchmark) and the hardware
// hands CTAs out in grid order, so the kernel's tail is whatever the last samples happen to be.  One small CTA sorts the
// samples by decreasing length (rank by counting, stable) and the pipelined kernel walks the grid's y dimension through
// that permutation: longest-processing-time-first, the tail is made of the shortest series.
__global__ void __launch_bounds__(1024) agg_order_kernel(const uint8_t* __restrict__ pad, int* __restrict__ order, int B, int T) {
  __shared__ short len[1024];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int s = warp; s < B; s += 32) {  // one warp per sample: T / 32 coalesced byte loads and a ballot instead of T loads per thread
    int n = 0;
    for (int t0 = 0; t0 < T; t0 += 32) {
      const int t = t0 + lane;
      n += __popc(__ballot_sync(0xffffffffu, t < T && pad[s * T + t] == 0));
    }
    if (lane == 0) len[s] = static_cast<short>(n);
  }
  __syncthreads();
  const int i = threadIdx.x;
  if (i >= B) return;
  const int n = len[i];
  int rank = 0;
  for (int q = 0; q < B; ++q) rank += (len[q] > n) || (len[q] == n && q < i);
  order[rank] = i;
}

// TAPS: the attention rows a pixel block needs (a contiguous slice of the low-resolution map, at most a few hundred
// floats) ride along with every frame as one more bulk copy into the stage, and the consumers read their bilinear taps
// from shared memory.  Without it every consumer thread issues 2 * NCOL global loads per frame for them -- measured as
// the largest cost after the feature bytes themselves (x2 / x4 / x8: 0.103 / 0.304 / 0.928 ms with, 0.078 / 0.228 /
// 0.857 ms without any tap loads).  TAPS needs 16-byte aligned attention rows (wa % 4 == 0).
template <typename T, int S, bool TAPS>
__global__ void __launch_bounds__(kPipeMaxConsumers + 32, (S >= 4 && sizeof(T) == 2 && TAPS) || (S == 8 && sizeof(T) == 2) ? 3 : 2) agg_pipe_kernel(const AggArgs a, int n_stages,
                                                                            int n_consumers, int pblocks, int tap_floats) {
  constexpr int VEC = Elem<T>::kVec;
  constexpr int NCOL = Window<VEC, S>::kCols;
  extern __shared__ __align__(128) unsigned char pipe_smem[];
  __shared__ short frames[kAggMaxT];
  __shared__ int n_frames_s;
  __shared__ __align__(8) unsigned long long bars[2 * 16];  // full[0..15], empty[0..15]

  const int b = a.order != nullptr ? a.order[blockIdx.y] : blockIdx.y;  // longest series first: the last wave is the short ones
  const int cchunk = blockIdx.x / pblocks;
  const int pblk = blockIdx.x - cchunk * pblocks;
  const int c0 = cchunk * kPipeCPT;
  const int pb = n_consumers * VEC;                 // pixels per block
  const uint32_t row_bytes = pb * sizeof(T);        // one channel row of the block
  const uint32_t stage_bytes = kPipeCPT * row_bytes;
  const uint32_t stage_stride = stage_bytes + (TAPS ? tap_floats * 4 : 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_cwarps = n_consumers >> 5;
  // attention rows [r_lo, r_hi] feed this pixel block (the rows of its first and last pixel, clamped like source_index)
  int r_lo = 0, n_rows_att = 0;
  if (TAPS) {
    int i0, i1;
    float l1;
    source_index(a.sy, (pblk * pb) / a.W, a.ha, i0, i1, l1);
    r_lo = i0;
    source_index(a.sy, (pblk * pb + pb - 1) / a.W, a.ha, i0, i1, l1);
    n_rows_att = i1 - r_lo + 1;
  }

  if (threadIdx.x < 32) {
    int count = 0;
    for (int base = 0; base < a.T; base += 32) {
      const int t = base + threadIdx.x;
      const bool valid = t < a.T && (a.pad == nullptr || a.pad[b * a.T + t] == 0);
      const unsigned m = __ballot_sync(0xffffffffu, valid);
      if (valid) frames[count + __popc(m & ((1u << threadIdx.x) - 1u))] = static_cast<short>(t);
      count += __popc(m);
    }
    if (threadIdx.x == 0) {
      n_frames_s = count;
      for (int s = 0; s < n_stages; ++s) {
        mbar_init(s32(&bars[s]), 1);
        mbar_init(s32(&bars[16 + s]), n_cwarps);
      }
      fence_mbarrier_init();
    }
  }
  __syncthreads();
  const int n_frames = n_frames_s;
  const size_t frame_stride = static_cast<size_t>(a.C) * a.hw;
  const uint32_t stage0 = s32(pipe_smem);

  if (warp == n_cwarps) {  // ---- producer -------------------------------------------------------------
    if (lane == 0) {
      const T* src = static_cast<const T*>(a.x) + static_cast<size_t>(b) * a.T * frame_stride +
                     static_cast<size_t>(c0) * a.hw + static_cast<size_t>(pblk) * pb;
      const int amap_p = a.ha * a.wa;
      const float* att_src = TAPS ? a.attn + (static_cast<size_t>(c0 / a.cpg) * a.B + b) * a.T * amap_p + r_lo * a.wa : nullptr;
      const uint32_t tap_bytes = TAPS ? static_cast<uint32_t>(n_rows_att * a.wa) * 4u : 0u;
      for (int i = 0; i < n_frames; ++i) {
        const int s = i % n_stages, round = i / n_stages;
        if (round > 0) mbar_wait(s32(&bars[16 + s]), (round - 1) & 1);
        const uint32_t full = s32(&bars[s]);
        mbar_expect_tx(full, stage_bytes + tap_bytes);
        const T* fp = src + static_cast<size_t>(frames[i]) * frame_stride;
#pragma unroll
        for (int k = 0; k < kPipeCPT; ++k)
          bulk_g2s(stage0 + s * stage_stride + k * row_bytes, fp + static_cast<size_t>(k) * a.hw, row_bytes, full);
        if (TAPS) bulk_g2s(stage0 + s * stage_stride + stage_bytes, att_src + static_cast<size_t>(frames[i]) * amap_p, tap_bytes, full);
      }
    }
    return;
  }

  // ---- consumers -------------------------------------------------------------------------------------
  const int p0 = pblk * pb + threadIdx.x * VEC;
  const int y = p0 / a.W;
  const int x0 = p0 - y * a.W;
  int iy0, iy1;
  float ly1;
  source_index(a.sy, y, a.ha, iy0, iy1, ly1);
  const float ly0 = 1.f - ly1;
  const int row0 = iy0 * a.wa, row1 = iy1 * a.wa;
  float lx1[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    int i0, i1;
    source_index(a.sx, x0 + j, a.wa, i0, i1, lx1[j]);
  }
  int col[NCOL];
  {
    int cmin = x0 / S - 1;
    if constexpr (VEC < S) cmin += ((x0 % S) >= S / 2) ? 1 : 0;
#pragma unroll
    for (int j = 0; j < NCOL; ++j) {
      int cj = cmin + j;
      cj = cj < 0 ? 0 : cj;
      col[j] = cj > a.wa - 1 ? a.wa - 1 : cj;
    }
  }
  const int amap = a.ha * a.wa;
  const float* ab = a.attn + (static_cast<size_t>(c0 / a.cpg) * a.B + b) * a.T * amap;

  float acc[kPipeCPT][VEC];
#pragma unroll
  for (int k = 0; k < kPipeCPT; ++k)
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[k][j] = 0.f;

  float top_n[NCOL], bot_n[NCOL];
  if (!TAPS && n_frames > 0) {
    const float* ap = ab + static_cast<size_t>(frames[0]) * amap;
#pragma unroll
    for (int j = 0; j < NCOL; ++j) top_n[j] = __ldg(ap + row0 + col[j]), bot_n[j] = __ldg(ap + row1 + col[j]);
  }
  const int trow0 = (iy0 - r_lo) * a.wa, trow1 = (iy1 - r_lo) * a.wa;  // TAPS: rows inside the staged slice
  const uint32_t my_off = threadIdx.x * 16;
  for (int i = 0; i < n_frames; ++i) {
    float r[NCOL];
    if (!TAPS) {
#pragma unroll
      for (int j = 0; j < NCOL; ++j) r[j] = fmaf(ly1, bot_n[j], ly0 * top_n[j]);
      if (i + 1 < n_frames) {  // attention taps of the next frame travel while this one is consumed
        const float* ap = ab + static_cast<size_t>(frames[i + 1]) * amap;
#pragma unroll
        for (int j = 0; j < NCOL; ++j) top_n[j] = __ldg(ap + row0 + col[j]), bot_n[j] = __ldg(ap + row1 + col[j]);
      }
    }
    const int s = i % n_stages;
    mbar_wait(s32(&bars[s]), (i / n_stages) & 1);
    uint4 xv[kPipeCPT];
    const uint32_t base = stage0 + s * stage_stride + my_off;
#pragma unroll
    for (int k = 0; k < kPipeCPT; ++k) xv[k] = lds_v4(base + k * row_bytes);
    if (TAPS) {
      const float* tp = reinterpret_cast<const float*>(pipe_smem + s * stage_stride + stage_bytes);
#pragma unroll
      for (int j = 0; j < NCOL; ++j) r[j] = fmaf(ly1, tp[trow1 + col[j]], ly0 * tp[trow0 + col[j]]);
    }
    fence_proxy_async();  // the stage's shared loads before the producer's next bulk copy into it (see agg_backward_pipe)
    __syncwarp();
    if (lane == 0) mbar_arrive(s32(&bars[16 + s]));  // the stage's data now lives in registers

    float w[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int i0w = (VEC >= S) ? (j / S + ((j % S) < S / 2 ? 0 : 1)) : 0;
      w[j] = fmaf(lx1[j], r[i0w + 1], (1.f - lx1[j]) * r[i0w]);
    }
#pragma unroll
    for (int k = 0; k < kPipeCPT; ++k) {
      float f[VEC];
      Elem<T>::unpack(xv[k], f);
#pragma unroll
      for (int j = 0; j < VEC; ++j) acc[k][j] = fmaf(w[j], f[j], acc[k][j]);
    }
  }
  T* op = static_cast<T*>(a.out) + (static_cast<size_t>(b) * a.C + c0) * a.hw + p0;
#pragma unroll
  for (int k = 0; k < kPipeCPT; ++k) PixelVec<T, VEC>::store(op + static_cast<size_t>(k) * a.hw, acc[k]);
}

template <typename T, int S, bool TAPS>
int launch_pipe_st(const AggArgs& a, int n_consumers, int n_stages, int tap_floats, cudaStream_t stream, const char* name) {
  constexpr int VEC = Elem<T>::kVec;
  const int pblocks = a.hw / (n_consumers * VEC);
  const size_t smem = static_cast<size_t>(n_stages) * (static_cast<size_t>(kPipeCPT) * n_consumers * 16 + (TAPS ? tap_floats * 4 : 0));
  C2S_SMEM_ATTR((agg_pipe_kernel<T, S, TAPS>), 13 * 16384);  // once per instantiation and device
  dim3 grid((a.C / kPipeCPT) * pblocks, a.B);
  agg_pipe_kernel<T, S, TAPS><<<grid, n_consumers + 32, smem, stream>>>(a, n_stages, n_consumers, pblocks, tap_floats);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <typename T, int S>
int launch_pipe_s(const AggArgs& a, int n_consumers, int n_stages, cudaStream_t stream, const char* name) {
  constexpr int VEC = Elem<T>::kVec;
  // staged attention rows: 16-byte aligned slices of the map, small enough to ride in the stage
  const int rows_out = (n_consumers * VEC + a.W - 1) / a.W + 1;  // output rows a pixel block can touch
  int rows_att = rows_out / S + 3;
  rows_att = rows_att > a.ha ? a.ha : rows_att;
  const int tap_floats = ((rows_att * a.wa + 3) / 4) * 4;
  const bool taps = option(C2S_OPT_AGG_TAPS) == 0 && a.wa % 4 == 0 && reinterpret_cast<uintptr_t>(a.attn) % 16 == 0 &&
                    tap_floats <= 1024;
  if (taps)  // fewer stages if they do not fit once the rows ride along
    while (n_stages > 2 && static_cast<size_t>(n_stages) * (static_cast<size_t>(kPipeCPT) * n_consumers * 16 + tap_floats * 4) > 13 * 16384)
      --n_stages;
  return taps ? launch_pipe_st<T, S, true>(a, n_consumers, n_stages, tap_floats, stream, name)
              : launch_pipe_st<T, S, false>(a, n_consumers, n_stages, 0, stream, name);
}

template <typename T>
int launch_pipe(const AggArgs& a, int s, int n_consumers, int n_stages, cudaStream_t stream) {
  switch (s) {
    case 2: return launch_pipe_s<T, 2>(a, n_consumers, n_stages, stream, "agg_forward_pipe<x2>");
    case 4: return launch_pipe_s<T, 4>(a, n_consumers, n_stages, stream, "agg_forward_pipe<x4>");
    default: return launch_pipe_s<T, 8>(a, n_consumers, n_stages, stream, "agg_forward_pipe<x8>");
  }
}

template <typename T, int VEC, int CPT, int S>
int launch_variant(const AggArgs& a, cudaStream_t stream, const char* name) {
  dim3 grid(ceil_div(a.items_per_b, kAggThreads), a.B);
  agg_forward_kernel<T, VEC, CPT, S><<<grid, kAggThreads, 0, stream>>>(a);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <typename T, int VEC, int CPT>
int launch_scale(const AggArgs& a, int s, cudaStream_t stream) {
  if constexpr (VEC > 1) {
    switch (s) {
      case 2: return launch_variant<T, VEC, CPT, 2>(a, stream, "agg_forward<x2>");
      case 4: return launch_variant<T, VEC, CPT, 4>(a, stream, "agg_forward<x4>");
      case 8: return launch_variant<T, VEC, CPT, 8>(a, stream, "agg_forward<x8>");
      default: break;
    }
  }
  if (s == -1) return launch_variant<T, VEC, CPT, -1>(a, stream, "agg_forward<mean>");
  return launch_variant<T, VEC, CPT, 0>(a, stream, "agg_forward<generic>");
}

template <typename T, int VEC>
int launch_cpt(const AggArgs& a, int cpt, int s, cudaStream_t stream) {
  switch (cpt) {
    case 4: return launch_scale<T, VEC, 4>(a, s, stream);
    case 2: return launch_scale<T, VEC, 2>(a, s, stream);
    default: return launch_scale<T, VEC, 1>(a, s, stream);
  }
}

// the sample order of the pipelined kernel sits behind the pooled / averaged attention maps in the workspace
inline size_t order_offset(size_t map_bytes) { return (map_bytes + 15) & ~static_cast<size_t>(15); }

size_t attn_elems(const c2s_agg_desc* d, int heads, int h, int w) {
  return static_cast<size_t>(heads) * d->B * d->T * h * w;
}

// The AvgPool2d branch is taken when x is not taller than the attention map is wide
// (temporal_aggregator.py:26-29 compares x.shape[-2] with the attention width).
bool uses_pool(const c2s_agg_desc* d) { return d->mode == C2S_AGG_ATT_GROUP && !(d->H > d->wa); }

}  // namespace
}  // namespace c2s

extern "C" {

size_t c2s_agg_workspace_bytes(const c2s_agg_desc* d) {
  if (d == nullptr) return 0;
  size_t n = 0;
  if (d->mode == C2S_AGG_ATT_MEAN) n = c2s::attn_elems(d, 1, d->ha, d->wa);
  if (c2s::uses_pool(d)) {
    const int k = d->wa / (d->H > 0 ? d->H : 1);
    if (k >= 1) n = c2s::attn_elems(d, d->n_heads, d->ha / k, d->wa / k);
  }
  return c2s::order_offset(n * sizeof(float)) + static_cast<size_t>(d->B > 0 ? d->B : 0) * sizeof(int);
}

int c2s_agg_forward(const c2s_agg_desc* d, const void* x, const float* attn, const uint8_t* pad_mask, void* out,
                    void* workspace, size_t workspace_bytes, void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(d != nullptr, "c2s_agg_forward: desc is NULL");
  C2S_CHECK_ARG(x != nullptr && out != nullptr, "c2s_agg_forward: x/out is NULL");
  C2S_CHECK_ARG(d->B > 0 && d->T > 0 && d->C > 0 && d->H > 0 && d->W > 0,
                "c2s_agg_forward: non-positive dimension in x[%d,%d,%d,%d,%d]", d->B, d->T, d->C, d->H, d->W);
  C2S_CHECK_ARG(d->dtype == C2S_F32 || d->dtype == C2S_BF16, "c2s_agg_forward: unknown dtype %d", d->dtype);
  C2S_CHECK_ARG(d->mode >= C2S_AGG_ATT_GROUP && d->mode <= C2S_AGG_MEAN, "c2s_agg_forward: unknown mode %d", d->mode);
  if (d->T > kAggMaxT) C2S_UNSUPPORTED("c2s_agg_forward: T=%d exceeds the supported %d frames", d->T, kAggMaxT);
  if (d->B > 65535) C2S_UNSUPPORTED("c2s_agg_forward: B=%d exceeds 65535 samples per call", d->B);
  if (static_cast<long long>(d->H) * d->W > (1ll << 30)) C2S_UNSUPPORTED("c2s_agg_forward: H*W too large");
  int status = check_device();
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);

  AggArgs a{};
  a.x = x;
  a.pad = pad_mask;
  a.out = out;
  a.B = d->B, a.T = d->T, a.C = d->C, a.H = d->H, a.W = d->W;
  a.hw = d->H * d->W;
  int scale_class = 0;
  size_t map_bytes = 0;  // workspace bytes taken by the averaged / pooled attention maps

  if (d->mode == C2S_AGG_MEAN) {
    a.attn = nullptr;
    a.n_heads = 1, a.ha = 1, a.wa = 1, a.cpg = d->C;
    // masked: sum / count (temporal_aggregator.py:54-55); unmasked: x.mean(dim=1) (:77)
    a.uniform_div = 1;
    scale_class = -1;
  } else {
    C2S_CHECK_ARG(attn != nullptr, "c2s_agg_forward: attn is NULL for an attention mode");
    C2S_CHECK_ARG(d->n_heads > 0 && d->ha > 0 && d->wa > 0, "c2s_agg_forward: bad attention shape [%d,.,.,%d,%d]",
                  d->n_heads, d->ha, d->wa);
    const float* amap = attn;
    int heads = d->n_heads, ha = d->ha, wa = d->wa;
    if (d->mode == C2S_AGG_ATT_MEAN) {
      const size_t n = attn_elems(d, 1, ha, wa);
      C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= n * sizeof(float),
                    "c2s_agg_forward: att_mean needs %zu workspace bytes", n * sizeof(float));
      head_mean_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(attn, static_cast<float*>(workspace), heads, n);
      C2S_LAUNCH_CHECK("head_mean");
      amap = static_cast<const float*>(workspace);
      map_bytes = n * sizeof(float);
      heads = 1;
    } else if (uses_pool(d)) {
      const int k = d->wa / d->H;
      C2S_CHECK_ARG(k >= 1, "c2s_agg_forward: AvgPool2d kernel size would be 0");
      const int ho = ha / k, wo = wa / k;
      C2S_CHECK_ARG(ho == d->H && wo == d->W,
                    "c2s_agg_forward: pooled attention %dx%d does not match x %dx%d (the reference fails to broadcast)",
                    ho, wo, d->H, d->W);
      if (k > 1) {
        const size_t n = attn_elems(d, heads, ho, wo);
        C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= n * sizeof(float),
                      "c2s_agg_forward: pooled attention needs %zu workspace bytes", n * sizeof(float));
        avg_pool_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(attn, static_cast<float*>(workspace), ha, wa, ho, wo,
                                                              k, n);
        C2S_LAUNCH_CHECK("avg_pool");
        amap = static_cast<const float*>(workspace);
        map_bytes = n * sizeof(float);
      }
      ha = ho, wa = wo;
    }
    C2S_CHECK_ARG(d->C % heads == 0, "c2s_agg_forward: C=%d is not divisible by n_heads=%d", d->C, heads);
    a.attn = amap;
    a.n_heads = heads, a.ha = ha, a.wa = wa, a.cpg = d->C / heads;
    a.sy = static_cast<float>(ha) / static_cast<float>(d->H);
    a.sx = static_cast<float>(wa) / static_cast<float>(d->W);
    for (int s : {2, 4, 8})
      if (d->H == s * ha && d->W == s * wa) scale_class = s;
  }

  const int cpt = (a.cpg % 4 == 0) ? 4 : (a.cpg % 2 == 0 ? 2 : 1);
  const bool bf16 = d->dtype == C2S_BF16;
  const int vec_full = bf16 ? 8 : 4;
  const bool aligned = (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
  const int vec = (d->W % vec_full == 0 && aligned) ? vec_full : 1;
  a.pv_per_plane = a.hw / vec;
  a.items_per_b = (d->C / cpt) * a.pv_per_plane;
  if (vec == 1 && scale_class > 0) scale_class = 0;

  // pipelined (bulk-copy) variant: power-of-two up-sampling, 4-channel head groups, whole 16-byte vectors
  const bool no_pipe = option(C2S_OPT_AGG_KERNEL) == 1;  // parity tests: A/B against the register kernel
  if (!no_pipe && scale_class > 0 && vec == vec_full && a.cpg % kPipeCPT == 0) {
    const int vecs = a.hw / vec;
    int n_consumers = vecs < kPipeMaxConsumers ? vecs : kPipeMaxConsumers;
    if (n_consumers >= 64 && n_consumers % 32 == 0 && vecs % n_consumers == 0) {
      int n_stages = bf16 ? 3 : 4;  // 16 KB stages; bf16: 3 (x8: three CTAs per SM = 144 KB, the rest stays L1 for the attention taps: 0.927 vs 0.967 ms with 4)
      while (static_cast<size_t>(n_stages) * kPipeCPT * n_consumers * 16 > 12 * 16384) --n_stages;
      // ragged series: walk the samples longest first (one 1-CTA launch; skipped when the caller gave no room for it)
      const size_t off = order_offset(map_bytes);
      if (pad_mask != nullptr && d->B > 1 && d->B <= 1024 && workspace != nullptr &&
          workspace_bytes >= off + static_cast<size_t>(d->B) * sizeof(int)) {
        int* order = reinterpret_cast<int*>(static_cast<char*>(workspace) + off);
        agg_order_kernel<<<1, 1024, 0, stream>>>(pad_mask, order, d->B, d->T);
        C2S_LAUNCH_CHECK("agg_order");
        a.order = order;
      }
      return bf16 ? launch_pipe<__nv_bfloat16>(a, scale_class, n_consumers, n_stages, stream)
                  : launch_pipe<float>(a, scale_class, n_consumers, n_stages, stream);
    }
  }

  if (bf16) {
    return vec == 8 ? launch_cpt<__nv_bfloat16, 8>(a, cpt, scale_class, stream)
                    : launch_cpt<__nv_bfloat16, 1>(a, cpt, scale_class, stream);
  }
  return vec == 4 ? launch_cpt<float, 4>(a, cpt, scale_class, stream) : launch_cpt<float, 1>(a, cpt, scale_class, stream);
}

}  // extern "C"
