// TemporalAggregator backward for sm_100a (autograd of reference src/backbones/temporal_aggregator.py:14-77).
//
//   grad_x[b,t,c,y,x]     = w[g(c),b,t,y,x] * grad_out[b,c,y,x]          w = bilinear(attn) on valid frames, else 0
//   grad_attn[g,b,t,:,:]  = bilinear^T( sum_{c in g} x[b,t,c,:,:] * grad_out[b,c,:,:] )
//
// Same work decomposition as the forward register kernel: one thread owns VEC pixels x CPT channels of one
// attention head, keeps grad_out for them in registers and streams over the frames once: it reads x (only when
// grad_attn is wanted), writes grad_x with 128-bit streaming stores and scatters the bilinear adjoint.  For the
// power-of-two up-sampling of the shipped models the adjoint is first reduced across the lanes of an image row
// with two warp shuffles per attention row, so a lane issues 2 * VEC/S float atomics per frame instead of 4 * VEC.
// HBM traffic: e*T_valid*C*H*W read (x) + e*T*C*H*W written (grad_x) + e*C*H*W (grad_out) per sample.
#include <type_traits>

#include <cstdlib>

#include "c2s_sm100.cuh"

namespace c2s {
namespace {

constexpr int kBwdThreads = 256;

struct AggBwdArgs {
  const void* x;
  const float* attn;
  const uint8_t* pad;
  const void* gout;
  void* gx;
  float* gattn;
  int B, T, C, H, W;
  int n_heads, ha, wa, cpg;
  int uniform;       // 'mean' mode
  float sy, sx;
  int hw, vecs_per_plane;
  int t_chunks, t_per_chunk;  // the frame loop is split over blockIdx.z (set by launch_bwd)
};

template <typename T, int VEC>
struct BVec {
  static_assert(VEC == 1, "scalar fallback");
  static __device__ __forceinline__ void load(const T* p, float (&f)[1]) { f[0] = Elem<T>::load(p); }
  static __device__ __forceinline__ void store(T* p, const float (&f)[1]) { Elem<T>::store(p, f[0]); }
};
template <>
struct BVec<float, 4> {
  static __device__ __forceinline__ void load(const float* p, float (&f)[4]) { Elem<float>::unpack(ld_stream_v4(p), f); }
  static __device__ __forceinline__ void store(float* p, const float (&f)[4]) { st_stream_v4(p, Elem<float>::pack(f)); }
};
template <>
struct BVec<__nv_bfloat16, 8> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
    Elem<__nv_bfloat16>::unpack(ld_stream_v4(p), f);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    st_stream_v4(p, Elem<__nv_bfloat16>::pack(f));
  }
};

// S > 0: H == S*ha, W == S*wa, VEC >= S (whole attention cells per thread): shuffle-reduced adjoint.
// S == 0: any ratio: one atomic per tap and pixel.    S == -1: 'mean' mode (no attention).
template <typename T, int VEC, int CPT, int S>
__global__ void __launch_bounds__(kBwdThreads) agg_backward_kernel(const AggBwdArgs a) {
  __shared__ uint8_t s_pad[1024];
  __shared__ int s_nvalid;
  // blockIdx.z = sample * t_chunks + chunk: the frames are independent (grad_x per frame, grad_attn per frame), so small
  // planes, which have few pixel blocks, are also split over T to fill the SMs
  const int b = blockIdx.z / a.t_chunks;
  const int t_begin = (blockIdx.z - b * a.t_chunks) * a.t_per_chunk;
  const int t_end = min(a.T, t_begin + a.t_per_chunk);
  if (threadIdx.x < 32) {
    int count = 0;
    for (int base = 0; base < a.T; base += 32) {
      const int t = base + threadIdx.x;
      const bool pd = t < a.T && a.pad != nullptr && a.pad[b * a.T + t] != 0;
      if (t < a.T) s_pad[t] = pd;
      count += __popc(__ballot_sync(0xffffffffu, t < a.T && !pd));
    }
    if (threadIdx.x == 0) s_nvalid = count;
  }
  __syncthreads();
  const int pv = blockIdx.x * kBwdThreads + threadIdx.x;
  const bool active = pv < a.vecs_per_plane;  // inactive lanes still take part in the shuffles
  const int c0 = blockIdx.y * CPT;
  const int p0 = (active ? pv : 0) * VEC;
  const int y = p0 / a.W, x0 = p0 - y * a.W;

  constexpr int M = (S > 0) ? VEC / S : 1;  // attention cells per thread
  constexpr int NCOL = (S > 0) ? M + 2 : 1;
  int row0 = 0, row1 = 0, cmin = 0;
  float ly1 = 0.f;
  float lx1[VEC];
  int gcol0[(S == 0) ? VEC : 1], gcol1[(S == 0) ? VEC : 1];
  if constexpr (S >= 0) {
    int iy0, iy1;
    source_index(a.sy, y, a.ha, iy0, iy1, ly1);
    row0 = iy0 * a.wa, row1 = iy1 * a.wa;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      int i0, i1;
      source_index(a.sx, x0 + j, a.wa, i0, i1, lx1[j]);
      if constexpr (S == 0) gcol0[j] = i0, gcol1[j] = i1;
    }
    if constexpr (S > 0) cmin = x0 / S - 1;
  }
  const float ly0 = 1.f - ly1;
  auto clampc = [&](int c) { return c < 0 ? 0 : (c > a.wa - 1 ? a.wa - 1 : c); };

  const size_t frame_stride = static_cast<size_t>(a.C) * a.hw;
  const size_t plane0 = static_cast<size_t>(c0) * a.hw + p0;
  const T* xb = static_cast<const T*>(a.x) + static_cast<size_t>(b) * a.T * frame_stride + plane0;
  T* gxb = static_cast<T*>(a.gx) + static_cast<size_t>(b) * a.T * frame_stride + plane0;
  const int amap = a.ha * a.wa;
  const size_t abase = (S >= 0) ? (static_cast<size_t>(c0 / a.cpg) * a.B + b) * a.T * amap : 0;

  float go[CPT][VEC];
#pragma unroll
  for (int k = 0; k < CPT; ++k) {
    if (active) {
      BVec<T, VEC>::load(static_cast<const T*>(a.gout) + (static_cast<size_t>(b) * a.C + c0 + k) * a.hw + p0, go[k]);
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) go[k][j] = 0.f;
    }
  }
  const float inv_n = 1.f / static_cast<float>(s_nvalid);

  // lanes of the same image row that sit next to each other in the warp exchange their edge columns
  const int lane = threadIdx.x & 31;
  const int lanes_per_row = a.W / VEC;
  const int lane_in_row = (active ? pv : 0) % lanes_per_row;
  const bool has_left = active && lane > 0 && lane_in_row > 0;
  const bool has_right = active && lane < 31 && lane_in_row < lanes_per_row - 1 && (pv + 1) < a.vecs_per_plane;

  for (int t = t_begin; t < t_end; ++t) {
    const bool padded = s_pad[t] != 0;  // block-uniform
    float w[VEC];
    if (padded) {
      if (a.gx != nullptr && active) {
        float z[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) z[j] = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) BVec<T, VEC>::store(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(k) * a.hw, z);
      }
      continue;
    }
    // forward weights (identical arithmetic to agg_forward_kernel)
    if constexpr (S > 0) {
      const float* ap = a.attn + abase + static_cast<size_t>(t) * amap;
      float r[NCOL];
#pragma unroll
      for (int jj = 0; jj < NCOL; ++jj) {
        const int cj = clampc(cmin + jj);
        r[jj] = fmaf(ly1, __ldg(ap + row1 + cj), ly0 * __ldg(ap + row0 + cj));
      }
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int i0w = j / S + ((j % S) < S / 2 ? 0 : 1);
        w[j] = fmaf(lx1[j], r[i0w + 1], (1.f - lx1[j]) * r[i0w]);
      }
    } else if constexpr (S == 0) {
      const float* ap = a.attn + abase + static_cast<size_t>(t) * amap;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float l0 = 1.f - lx1[j];
        const float tp = fmaf(lx1[j], __ldg(ap + row0 + gcol1[j]), l0 * __ldg(ap + row0 + gcol0[j]));
        const float bt = fmaf(lx1[j], __ldg(ap + row1 + gcol1[j]), l0 * __ldg(ap + row1 + gcol0[j]));
        w[j] = fmaf(ly1, bt, ly0 * tp);
      }
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) w[j] = inv_n;
    }
    float g[VEC];  // sum_c x * grad_out of this thread's pixels
#pragma unroll
    for (int j = 0; j < VEC; ++j) g[j] = 0.f;
    const bool want_attn = (S >= 0) && a.gattn != nullptr;
    if (active) {
#pragma unroll
      for (int k = 0; k < CPT; ++k) {
        const size_t off = static_cast<size_t>(t) * frame_stride + static_cast<size_t>(k) * a.hw;
        if (want_attn) {
          float xv[VEC];
          BVec<T, VEC>::load(xb + off, xv);
#pragma unroll
          for (int j = 0; j < VEC; ++j) g[j] = fmaf(xv[j], go[k][j], g[j]);
        }
        if (a.gx != nullptr) {
          float d[VEC];
#pragma unroll
          for (int j = 0; j < VEC; ++j) d[j] = w[j] * go[k][j];
          BVec<T, VEC>::store(gxb + off, d);
        }
      }
    }
    if (!want_attn) continue;
    float* gp = a.gattn + abase + static_cast<size_t>(t) * amap;
    if constexpr (S > 0) {
      // horizontal adjoint into the NCOL-column window, then edge columns travel to the neighbouring lanes
      float win[NCOL];
#pragma unroll
      for (int jj = 0; jj < NCOL; ++jj) win[jj] = 0.f;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int i0w = j / S + ((j % S) < S / 2 ? 0 : 1);
        win[i0w] = fmaf(g[j], 1.f - lx1[j], win[i0w]);
        win[i0w + 1] = fmaf(g[j], lx1[j], win[i0w + 1]);
      }
      const float from_left = __shfl_up_sync(0xffffffffu, win[NCOL - 1], 1);   // left lane's column cmin + M + 1 == my first own
      const float from_right = __shfl_down_sync(0xffffffffu, win[0], 1);       // right lane's column cmin' == my last own
      float own[M];
#pragma unroll
      for (int i = 0; i < M; ++i) own[i] = win[i + 1];
      if (has_left) own[0] += from_left;
      if (has_right) own[M - 1] += from_right;
      if (active) {
#pragma unroll
        for (int i = 0; i < M; ++i) {
          const int cj = cmin + 1 + i;  // own columns are always inside [0, wa)
          atomicAdd(gp + row0 + cj, ly0 * own[i]);
          if (ly1 != 0.f) atomicAdd(gp + row1 + cj, ly1 * own[i]);
        }
        // edge columns nobody picked up (image border: clamped; warp or row boundary: the neighbour is elsewhere)
        const bool left_taken = lane > 0 && lane_in_row > 0;                                   // right neighbour of lane-1 is me
        const bool right_taken = lane < 31 && lane_in_row < lanes_per_row - 1 && (pv + 1) < a.vecs_per_plane;
        if (!left_taken) {
          const int cj = clampc(cmin);
          atomicAdd(gp + row0 + cj, ly0 * win[0]);
          if (ly1 != 0.f) atomicAdd(gp + row1 + cj, ly1 * win[0]);
        }
        if (!right_taken) {
          const int cj = clampc(cmin + NCOL - 1);
          atomicAdd(gp + row0 + cj, ly0 * win[NCOL - 1]);
          if (ly1 != 0.f) atomicAdd(gp + row1 + cj, ly1 * win[NCOL - 1]);
        }
      }
    } else if constexpr (S == 0) {
      if (active) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float l0 = 1.f - lx1[j];
          atomicAdd(gp + row0 + gcol0[j], ly0 * l0 * g[j]);
          atomicAdd(gp + row0 + gcol1[j], ly0 * lx1[j] * g[j]);
          atomicAdd(gp + row1 + gcol0[j], ly1 * l0 * g[j]);
          atomicAdd(gp + row1 + gcol1[j], ly1 * lx1[j] * g[j]);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Pipelined variant for the shipped shapes (power-of-two up-sampling S with VEC >= S, 4-channel head groups, whole
// 16-byte vectors, grad_x AND grad_attn wanted): same arithmetic as agg_backward_kernel, but x travels HBM -> shared
// memory through the bulk-copy engine (cp.async.bulk + mbarrier transaction counts, as in agg_pipe_kernel of the
// forward), so the bytes in flight per SM are set by the ring of stages, not by the registers of the consumers, which
// are busy with the stores of grad_x and the adjoint.  One CTA = one sample x one head (4 channels) x n_consumers
// pixel vectors x one chunk of frames; one producer thread issues four row copies per valid frame.
// ---------------------------------------------------------------------------------------------------
constexpr int kBwdPipeCPT = 4;
constexpr int kBwdPipeMaxConsumers = 256;

// TAPS: as in the forward (c2s_aggregator.cu), the attention rows of the pixel block ride in the stage as one more bulk
// copy and the consumers read their taps from shared memory instead of 2 * NCOL global loads per thread and frame.
template <typename T, int S, bool TAPS>
__global__ void __launch_bounds__(kBwdPipeMaxConsumers + 32, 2)
agg_backward_pipe_kernel(const AggBwdArgs a, int n_stages, int n_consumers, int pblocks, int tap_floats) {
  constexpr int VEC = Elem<T>::kVec;
  constexpr int CPT = kBwdPipeCPT;
  constexpr int M = VEC / S;   // attention cells per thread
  constexpr int NCOL = M + 2;
  extern __shared__ __align__(128) unsigned char bpipe_smem[];
  __shared__ uint8_t s_pad[1024];
  __shared__ __align__(8) unsigned long long bars[2 * 16];  // full[0..15], empty[0..15]

  const int b = blockIdx.y / a.t_chunks;
  const int t_begin = (blockIdx.y - b * a.t_chunks) * a.t_per_chunk;
  const int t_end = min(a.T, t_begin + a.t_per_chunk);
  const int cchunk = blockIdx.x / pblocks;
  const int pblk = blockIdx.x - cchunk * pblocks;
  const int c0 = cchunk * CPT;
  const uint32_t row_bytes = n_consumers * 16;
  const uint32_t stage_bytes = CPT * row_bytes;
  const uint32_t stage_stride = stage_bytes + (TAPS ? tap_floats * 4 : 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_cwarps = n_consumers >> 5;
  int r_lo = 0, n_rows_att = 0;  // attention rows [r_lo, r_lo + n_rows_att) feed this pixel block
  if (TAPS) {
    const int pb = n_consumers * VEC;
    int i0, i1;
    float l1;
    source_index(a.sy, (pblk * pb) / a.W, a.ha, i0, i1, l1);
    r_lo = i0;
    source_index(a.sy, (pblk * pb + pb - 1) / a.W, a.ha, i0, i1, l1);
    n_rows_att = i1 - r_lo + 1;
  }

  for (int t = threadIdx.x; t < a.T; t += blockDim.x) s_pad[t] = a.pad != nullptr && a.pad[b * a.T + t] != 0;
  if (threadIdx.x == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(s32(&bars[s]), 1);
      mbar_init(s32(&bars[16 + s]), n_cwarps);
    }
    fence_mbarrier_init();
  }
  __syncthreads();
  const size_t frame_stride = static_cast<size_t>(a.C) * a.hw;
  const uint32_t stage0 = s32(bpipe_smem);
  const size_t plane0 = static_cast<size_t>(c0) * a.hw + static_cast<size_t>(pblk) * n_consumers * VEC;

  if (warp == n_cwarps) {  // ---- producer: the valid frames of the chunk, in order ------------------------
    if (lane == 0) {
      const T* src = static_cast<const T*>(a.x) + static_cast<size_t>(b) * a.T * frame_stride + plane0;
      const int amap_p = a.ha * a.wa;
      const float* att_src = TAPS ? a.attn + (static_cast<size_t>(c0 / a.cpg) * a.B + b) * a.T * amap_p + r_lo * a.wa : nullptr;
      const uint32_t tap_bytes = TAPS ? static_cast<uint32_t>(n_rows_att * a.wa) * 4u : 0u;
      int i = 0;
      for (int t = t_begin; t < t_end; ++t) {
        if (s_pad[t]) continue;
        const int s = i % n_stages, round = i / n_stages;
        if (round > 0) mbar_wait(s32(&bars[16 + s]), (round - 1) & 1);
        const uint32_t full = s32(&bars[s]);
        mbar_expect_tx(full, stage_bytes + tap_bytes);
        const T* fp = src + static_cast<size_t>(t) * frame_stride;
#pragma unroll
        for (int k = 0; k < CPT; ++k)
          bulk_g2s(stage0 + s * stage_stride + k * row_bytes, fp + static_cast<size_t>(k) * a.hw, row_bytes, full);
        if (TAPS) bulk_g2s(stage0 + s * stage_stride + stage_bytes, att_src + static_cast<size_t>(t) * amap_p, tap_bytes, full);
        ++i;
      }
    }
    return;
  }

  // ---- consumers ------------------------------------------------------------------------------------------
  const int pv = pblk * n_consumers + threadIdx.x;  // pixel vector of the plane
  const int p0 = pv * VEC;
  const int y = p0 / a.W, x0 = p0 - y * a.W;
  int iy0, iy1;
  float ly1;
  source_index(a.sy, y, a.ha, iy0, iy1, ly1);
  const int row0 = iy0 * a.wa, row1 = iy1 * a.wa;
  const float ly0 = 1.f - ly1;
  float lx1[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    int i0, i1;
    source_index(a.sx, x0 + j, a.wa, i0, i1, lx1[j]);
  }
  const int cmin = x0 / S - 1;
  auto clampc = [&](int c) { return c < 0 ? 0 : (c > a.wa - 1 ? a.wa - 1 : c); };
  T* gxb = static_cast<T*>(a.gx) + static_cast<size_t>(b) * a.T * frame_stride + plane0 + static_cast<size_t>(threadIdx.x) * VEC;
  const int amap = a.ha * a.wa;
  const size_t abase = (static_cast<size_t>(c0 / a.cpg) * a.B + b) * a.T * amap;

  float go[CPT][VEC];
#pragma unroll
  for (int k = 0; k < CPT; ++k)
    BVec<T, VEC>::load(static_cast<const T*>(a.gout) + (static_cast<size_t>(b) * a.C + c0 + k) * a.hw + p0, go[k]);

  // lanes of the same image row that sit next to each other in the warp exchange their edge columns
  const int lanes_per_row = a.W / VEC;
  const int lane_in_row = pv % lanes_per_row;
  const bool has_left = lane > 0 && lane_in_row > 0;
  const bool has_right = lane < 31 && lane_in_row < lanes_per_row - 1;
  const uint32_t my_off = threadIdx.x * 16;

  int i = 0;
  for (int t = t_begin; t < t_end; ++t) {
    if (s_pad[t]) {  // block-uniform
      float z[VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) z[j] = 0.f;
#pragma unroll
      for (int k = 0; k < CPT; ++k) BVec<T, VEC>::store(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(k) * a.hw, z);
      continue;
    }
    // forward weights (identical arithmetic to agg_forward_kernel); the taps travel while the stage is awaited
    float r[NCOL];
    if (!TAPS) {
      const float* ap = a.attn + abase + static_cast<size_t>(t) * amap;
#pragma unroll
      for (int jj = 0; jj < NCOL; ++jj) {
        const int cj = clampc(cmin + jj);
        r[jj] = fmaf(ly1, __ldg(ap + row1 + cj), ly0 * __ldg(ap + row0 + cj));
      }
    }
    const int s = i % n_stages;
    mbar_wait(s32(&bars[s]), (i / n_stages) & 1);
    uint4 xv[CPT];
    const uint32_t base = stage0 + s * stage_stride + my_off;
#pragma unroll
    for (int k = 0; k < CPT; ++k) xv[k] = lds_v4(base + k * row_bytes);
    if (TAPS) {
      const float* tp = reinterpret_cast<const float*>(bpipe_smem + s * stage_stride + stage_bytes);
      const int trow0 = row0 - r_lo * a.wa, trow1 = row1 - r_lo * a.wa;
#pragma unroll
      for (int jj = 0; jj < NCOL; ++jj) {
        const int cj = clampc(cmin + jj);
        r[jj] = fmaf(ly1, tp[trow1 + cj], ly0 * tp[trow0 + cj]);
      }
    }
    // the stage's reads (generic proxy) must be performed before the producer's next bulk copy (async proxy) into it:
    // without the fence the arrive can overtake the shared loads and the first frames of a time chunk read their
    // successors' rows
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(s32(&bars[16 + s]));  // the stage's data now lives in registers
    ++i;

    float g[VEC];  // sum_c x * grad_out of this thread's pixels
#pragma unroll
    for (int j = 0; j < VEC; ++j) g[j] = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
      float f[VEC], d[VEC];
      Elem<T>::unpack(xv[k], f);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int i0w = j / S + ((j % S) < S / 2 ? 0 : 1);
        const float w = fmaf(lx1[j], r[i0w + 1], (1.f - lx1[j]) * r[i0w]);
        g[j] = fmaf(f[j], go[k][j], g[j]);
        d[j] = w * go[k][j];
      }
      BVec<T, VEC>::store(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(k) * a.hw, d);
    }
    // horizontal adjoint into the NCOL-column window, then edge columns travel to the neighbouring lanes
    float* gp = a.gattn + abase + static_cast<size_t>(t) * amap;
    float win[NCOL];
#pragma unroll
    for (int jj = 0; jj < NCOL; ++jj) win[jj] = 0.f;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int i0w = j / S + ((j % S) < S / 2 ? 0 : 1);
      win[i0w] = fmaf(g[j], 1.f - lx1[j], win[i0w]);
      win[i0w + 1] = fmaf(g[j], lx1[j], win[i0w + 1]);
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
      const int cj = cmin + 1 + q;  // own columns are always inside [0, wa)
      atomicAdd(gp + row0 + cj, ly0 * own[q]);
      if (ly1 != 0.f) atomicAdd(gp + row1 + cj, ly1 * own[q]);
    }
    if (!has_left) {  // edge columns nobody picked up (image border: clamped; warp or row boundary)
      const int cj = clampc(cmin);
      atomicAdd(gp + row0 + cj, ly0 * win[0]);
      if (ly1 != 0.f) atomicAdd(gp + row1 + cj, ly1 * win[0]);
    }
    if (!has_right) {
      const int cj = clampc(cmin + NCOL - 1);
      atomicAdd(gp + row0 + cj, ly0 * win[NCOL - 1]);
      if (ly1 != 0.f) atomicAdd(gp + row1 + cj, ly1 * win[NCOL - 1]);
    }
  }
}

template <typename T, int S, bool TAPS>
int launch_bwd_pipe_st(const AggBwdArgs& b, int n_consumers, int n_stages, int pblocks, int tap_floats, cudaStream_t stream,
                       const char* name) {
  const size_t smem = static_cast<size_t>(n_stages) * (static_cast<size_t>(kBwdPipeCPT) * n_consumers * 16 + (TAPS ? tap_floats * 4 : 0));
  C2S_SMEM_ATTR((agg_backward_pipe_kernel<T, S, TAPS>), 13 * 16384);  // once per instantiation and device
  dim3 grid((b.C / kBwdPipeCPT) * pblocks, b.B * b.t_chunks);
  agg_backward_pipe_kernel<T, S, TAPS><<<grid, n_consumers + 32, smem, stream>>>(b, n_stages, n_consumers, pblocks, tap_floats);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <typename T, int S>
int launch_bwd_pipe_s(const AggBwdArgs& a, int n_consumers, int n_stages, cudaStream_t stream, const char* name) {
  constexpr int VEC = Elem<T>::kVec;
  AggBwdArgs b = a;
  const int pblocks = a.vecs_per_plane / n_consumers;
  const long long ctas = static_cast<long long>(a.C / kBwdPipeCPT) * pblocks * a.B;
  int chunks = 1;
  while (ctas * chunks < 8 * 148 && ceil_div(a.T, chunks * 2) >= 8 && static_cast<long long>(a.B) * chunks * 2 <= 65535) chunks *= 2;
  b.t_per_chunk = ceil_div(a.T, chunks);
  b.t_chunks = ceil_div(a.T, b.t_per_chunk);
  // staged attention rows (see agg_pipe_kernel): 16-byte aligned slices of the map
  const int rows_out = (n_consumers * VEC + a.W - 1) / a.W + 1;
  int rows_att = rows_out / S + 3;
  rows_att = rows_att > a.ha ? a.ha : rows_att;
  const int tap_floats = ((rows_att * a.wa + 3) / 4) * 4;
  const bool taps = option(C2S_OPT_AGG_TAPS) == 0 && a.wa % 4 == 0 && reinterpret_cast<uintptr_t>(a.attn) % 16 == 0 &&
                    tap_floats <= 1024;
  if (taps)  // fewer stages if they do not fit once the rows ride along
    while (n_stages > 2 && static_cast<size_t>(n_stages) * (static_cast<size_t>(kBwdPipeCPT) * n_consumers * 16 + tap_floats * 4) > 13 * 16384)
      --n_stages;
  return taps ? launch_bwd_pipe_st<T, S, true>(b, n_consumers, n_stages, pblocks, tap_floats, stream, name)
              : launch_bwd_pipe_st<T, S, false>(b, n_consumers, n_stages, pblocks, 0, stream, name);
}

// att_mean: every head receives grad(mean) / n_heads                       (temporal_aggregator.py:48)
__global__ void spread_head_mean_kernel(const float* __restrict__ gmean, float* __restrict__ gattn, int n_heads, size_t n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = gmean[i] / static_cast<float>(n_heads);
  for (int h = 0; h < n_heads; ++h) gattn[static_cast<size_t>(h) * n + i] += v;
}
__global__ void head_mean_bwd_fwd_kernel(const float* __restrict__ attn, float* __restrict__ out, int n_heads, size_t n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int h = 0; h < n_heads; ++h) s += attn[static_cast<size_t>(h) * n + i];
  out[i] = s / static_cast<float>(n_heads);
}

template <typename T, int VEC, int CPT, int S>
int launch_bwd(const AggBwdArgs& a, cudaStream_t stream, const char* name) {
  AggBwdArgs b = a;
  const long long ctas = static_cast<long long>(ceil_div(a.vecs_per_plane, kBwdThreads)) * (a.C / CPT) * a.B;
  int chunks = 1;  // enough CTAs for ~8 per SM, at least 8 frames per CTA (the prologue loads grad_out once per CTA)
  while (ctas * chunks < 8 * 148 && ceil_div(a.T, chunks * 2) >= 8 && static_cast<long long>(a.B) * chunks * 2 <= 65535) chunks *= 2;
  b.t_per_chunk = ceil_div(a.T, chunks);
  b.t_chunks = ceil_div(a.T, b.t_per_chunk);
  dim3 grid(ceil_div(a.vecs_per_plane, kBwdThreads), a.C / CPT, a.B * b.t_chunks);
  agg_backward_kernel<T, VEC, CPT, S><<<grid, kBwdThreads, 0, stream>>>(b);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <typename T, int VEC, int CPT>
int launch_bwd_scale(const AggBwdArgs& a, int s, cudaStream_t stream) {
  if constexpr (VEC > 1) {
    if (s == 2 && VEC >= 2) return launch_bwd<T, VEC, CPT, 2>(a, stream, "agg_backward<x2>");
    if (s == 4 && VEC >= 4) return launch_bwd<T, VEC, CPT, 4>(a, stream, "agg_backward<x4>");
    if constexpr (VEC >= 8)
      if (s == 8) return launch_bwd<T, VEC, CPT, 8>(a, stream, "agg_backward<x8>");
  }
  if (s == -1) return launch_bwd<T, VEC, CPT, -1>(a, stream, "agg_backward<mean>");
  return launch_bwd<T, VEC, CPT, 0>(a, stream, "agg_backward<generic>");
}

template <typename T, int VEC>
int launch_bwd_cpt(const AggBwdArgs& a, int cpt, int s, cudaStream_t stream) {
  switch (cpt) {
    case 4: return launch_bwd_scale<T, VEC, 4>(a, s, stream);
    case 2: return launch_bwd_scale<T, VEC, 2>(a, s, stream);
    default: return launch_bwd_scale<T, VEC, 1>(a, s, stream);
  }
}

// nn.AvgPool2d(kernel_size=k) of the attention maps (temporal_aggregator.py:28-29: the branch taken when the attention
// is not coarser than x) and its adjoint: every cell of a k x k window receives grad / k^2, the rows and columns that
// the floor of the pooling drops receive nothing
__global__ void pool_attn_kernel(const float* __restrict__ in, float* __restrict__ out, int hi, int wi, int ho, int wo, int k,
                                 size_t n_out) {
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
__global__ void unpool_grad_kernel(const float* __restrict__ gpooled, float* __restrict__ gattn, int hi, int wi, int ho,
                                   int wo, int k, size_t n_in) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_in) return;
  const int x = static_cast<int>(i % wi);
  const int y = static_cast<int>((i / wi) % hi);
  const size_t map = i / (static_cast<size_t>(wi) * hi);
  const int py = y / k, px = x / k;
  if (py >= ho || px >= wo) return;
  gattn[i] += gpooled[(map * ho + py) * wo + px] / static_cast<float>(k * k);
}

bool bwd_uses_pool(const c2s_agg_desc* d) { return d->mode == C2S_AGG_ATT_GROUP && !(d->H > d->wa); }

}  // namespace
}  // namespace c2s

extern "C" {

size_t c2s_agg_backward_workspace_bytes(const c2s_agg_desc* d) {
  if (d == nullptr) return 0;
  if (c2s::bwd_uses_pool(d)) {  // pooled attention + its gradient (nothing for the same-resolution case k = 1)
    const int k = d->H > 0 ? d->wa / d->H : 0;
    return k > 1 ? 2 * static_cast<size_t>(d->n_heads) * d->B * d->T * d->H * d->W * sizeof(float) : 0;
  }
  if (d->mode != C2S_AGG_ATT_MEAN) return 0;
  // mean attention map + its gradient
  return 2 * static_cast<size_t>(d->B) * d->T * d->ha * d->wa * sizeof(float);
}

int c2s_agg_backward(const c2s_agg_desc* d, const void* x, const float* attn, const uint8_t* pad_mask,
                     const void* grad_out, void* grad_x, float* grad_attn, void* workspace, size_t workspace_bytes,
                     void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(d != nullptr, "c2s_agg_backward: desc is NULL");
  C2S_CHECK_ARG(grad_out != nullptr, "c2s_agg_backward: grad_out is NULL");
  C2S_CHECK_ARG(grad_x != nullptr || grad_attn != nullptr, "c2s_agg_backward: nothing to compute");
  C2S_CHECK_ARG(d->B > 0 && d->T > 0 && d->C > 0 && d->H > 0 && d->W > 0,
                "c2s_agg_backward: non-positive dimension in x[%d,%d,%d,%d,%d]", d->B, d->T, d->C, d->H, d->W);
  C2S_CHECK_ARG(d->dtype == C2S_F32 || d->dtype == C2S_BF16, "c2s_agg_backward: unknown dtype %d", d->dtype);
  C2S_CHECK_ARG(d->mode >= C2S_AGG_ATT_GROUP && d->mode <= C2S_AGG_MEAN, "c2s_agg_backward: unknown mode %d", d->mode);
  if (d->T > 1024) C2S_UNSUPPORTED("c2s_agg_backward: T=%d exceeds the supported 1024 frames", d->T);
  if (d->B > 65535 || d->C > 65535) C2S_UNSUPPORTED("c2s_agg_backward: B or C exceeds 65535");
  int status = check_device();
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);

  AggBwdArgs a{};
  a.x = x, a.pad = pad_mask, a.gout = grad_out, a.gx = grad_x;
  a.B = d->B, a.T = d->T, a.C = d->C, a.H = d->H, a.W = d->W, a.hw = d->H * d->W;
  int scale_class = 0;
  float* gmean = nullptr;
  size_t n_mean = 0;
  float* gpool = nullptr;  // AvgPool2d branch: gradient of the pooled maps, spread over the windows at the end
  size_t n_pool = 0;
  int pool_k = 0;
  if (d->mode == C2S_AGG_MEAN) {
    a.attn = nullptr, a.gattn = nullptr;
    a.n_heads = 1, a.ha = 1, a.wa = 1, a.cpg = d->C, a.uniform = 1;
    scale_class = -1;
    C2S_CHECK_ARG(grad_x != nullptr, "c2s_agg_backward: mode 'mean' has no attention gradient");
  } else {
    C2S_CHECK_ARG(attn != nullptr, "c2s_agg_backward: attn is NULL for an attention mode");
    C2S_CHECK_ARG(grad_attn == nullptr || x != nullptr, "c2s_agg_backward: x is needed for grad_attn");
    C2S_CHECK_ARG(d->n_heads > 0 && d->ha > 0 && d->wa > 0, "c2s_agg_backward: bad attention shape");
    int heads = d->n_heads;
    const float* amap = attn;
    float* gmap = grad_attn;
    int ha = d->ha, wa = d->wa;
    if (bwd_uses_pool(d)) {  // temporal_aggregator.py:28-29
      pool_k = d->wa / d->H;
      C2S_CHECK_ARG(pool_k >= 1, "c2s_agg_backward: AvgPool2d kernel size would be 0");
      const int ho = d->ha / pool_k, wo = d->wa / pool_k;
      C2S_CHECK_ARG(ho == d->H && wo == d->W,
                    "c2s_agg_backward: pooled attention %dx%d does not match x %dx%d (the reference fails to broadcast)",
                    ho, wo, d->H, d->W);
      if (pool_k > 1) {
        n_pool = static_cast<size_t>(heads) * d->B * d->T * ho * wo;
        C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= 2 * n_pool * sizeof(float),
                      "c2s_agg_backward: the AvgPool2d branch needs %zu workspace bytes", 2 * n_pool * sizeof(float));
        float* pooled = static_cast<float*>(workspace);
        pool_attn_kernel<<<ceil_div(n_pool, 256), 256, 0, stream>>>(attn, pooled, d->ha, d->wa, ho, wo, pool_k, n_pool);
        C2S_LAUNCH_CHECK("avg_pool");
        amap = pooled;
        if (grad_attn != nullptr) {
          gpool = pooled + n_pool;
          C2S_CUDA(cudaMemsetAsync(gpool, 0, n_pool * sizeof(float), stream));
          gmap = gpool;
        }
      }
      ha = ho, wa = wo;
    }
    if (d->mode == C2S_AGG_ATT_MEAN) {
      n_mean = static_cast<size_t>(d->B) * d->T * d->ha * d->wa;
      C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= 2 * n_mean * sizeof(float),
                    "c2s_agg_backward: att_mean needs %zu workspace bytes", 2 * n_mean * sizeof(float));
      float* mean = static_cast<float*>(workspace);
      head_mean_bwd_fwd_kernel<<<ceil_div(n_mean, 256), 256, 0, stream>>>(attn, mean, heads, n_mean);
      C2S_LAUNCH_CHECK("head_mean");
      amap = mean;
      if (grad_attn != nullptr) {
        gmean = mean + n_mean;
        C2S_CUDA(cudaMemsetAsync(gmean, 0, n_mean * sizeof(float), stream));
        gmap = gmean;
      }
      heads = 1;
    }
    C2S_CHECK_ARG(d->C % heads == 0, "c2s_agg_backward: C=%d is not divisible by n_heads=%d", d->C, heads);
    a.attn = amap, a.gattn = gmap;
    a.n_heads = heads, a.ha = ha, a.wa = wa, a.cpg = d->C / heads;
    a.sy = static_cast<float>(ha) / static_cast<float>(d->H);
    a.sx = static_cast<float>(wa) / static_cast<float>(d->W);
    for (int s : {2, 4, 8})
      if (d->H == s * ha && d->W == s * wa) scale_class = s;
  }
  const int cpt = (a.cpg % 4 == 0) ? 4 : (a.cpg % 2 == 0 ? 2 : 1);
  const bool bf16 = d->dtype == C2S_BF16;
  const int vec_full = bf16 ? 8 : 4;
  auto al16 = [](const void* p) { return p == nullptr || reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  const int vec = (d->W % vec_full == 0 && al16(x) && al16(grad_out) && al16(grad_x)) ? vec_full : 1;
  a.vecs_per_plane = a.hw / vec;
  if (scale_class > 0 && (vec == 1 || vec < scale_class)) scale_class = 0;  // whole attention cells per thread only

  // pipelined variant: both gradients wanted, power-of-two up-sampling with whole attention cells per thread
  const bool no_pipe = option(C2S_OPT_AGG_KERNEL) == 1;  // parity tests: A/B against the register kernel
  if (!no_pipe && scale_class > 0 && vec == vec_full && vec >= scale_class && a.cpg % kBwdPipeCPT == 0 && a.gx != nullptr &&
      a.gattn != nullptr && x != nullptr && a.W % vec == 0) {
    const int vecs = a.vecs_per_plane;
    int n_consumers = vecs < kBwdPipeMaxConsumers ? vecs : kBwdPipeMaxConsumers;
    if (n_consumers >= 64 && n_consumers % 32 == 0 && vecs % n_consumers == 0) {
      int n_stages = 4;
      while (static_cast<size_t>(n_stages) * kBwdPipeCPT * n_consumers * 16 > 12 * 16384) --n_stages;
      auto go = [&](auto tag) {
        using TT = decltype(tag);
        switch (scale_class) {
          case 2: return launch_bwd_pipe_s<TT, 2>(a, n_consumers, n_stages, stream, "agg_backward_pipe<x2>");
          case 4: return launch_bwd_pipe_s<TT, 4>(a, n_consumers, n_stages, stream, "agg_backward_pipe<x4>");
          default:
            if constexpr (Elem<TT>::kVec >= 8)
              return launch_bwd_pipe_s<TT, 8>(a, n_consumers, n_stages, stream, "agg_backward_pipe<x8>");
            else
              return -1;  // fp32 vectors hold 4 pixels: no whole x8 cell per thread, the register kernel takes it
        }
      };
      status = bf16 ? go(__nv_bfloat16{}) : go(float{});
      if (status != -1) {
        if (status != C2S_OK) return status;
        if (gmean != nullptr) {
          spread_head_mean_kernel<<<ceil_div(n_mean, 256), 256, 0, stream>>>(gmean, grad_attn, d->n_heads, n_mean);
          C2S_LAUNCH_CHECK("spread_head_mean");
        }
        return C2S_OK;
      }
    }
  }
  if (bf16)
    status = vec == 8 ? launch_bwd_cpt<__nv_bfloat16, 8>(a, cpt, scale_class, stream)
                      : launch_bwd_cpt<__nv_bfloat16, 1>(a, cpt, scale_class, stream);
  else
    status = vec == 4 ? launch_bwd_cpt<float, 4>(a, cpt, scale_class, stream)
                      : launch_bwd_cpt<float, 1>(a, cpt, scale_class, stream);
  if (status != C2S_OK) return status;
  if (gmean != nullptr) {
    spread_head_mean_kernel<<<ceil_div(n_mean, 256), 256, 0, stream>>>(gmean, grad_attn, d->n_heads, n_mean);
    C2S_LAUNCH_CHECK("spread_head_mean");
  }
  if (gpool != nullptr) {
    const size_t n_in = static_cast<size_t>(d->n_heads) * d->B * d->T * d->ha * d->wa;
    unpool_grad_kernel<<<ceil_div(n_in, 256), 256, 0, stream>>>(gpool, grad_attn, d->ha, d->wa, d->H, d->W, pool_k, n_in);
    C2S_LAUNCH_CHECK("avg_unpool");
  }
  return C2S_OK;
}

}  // extern "C"
