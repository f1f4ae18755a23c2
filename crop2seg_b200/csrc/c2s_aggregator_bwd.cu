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

// ---------------------------------------------------------------------------------------------------
// Backward of the aggregation fused with the skip convolution (agg_skipconv_kernel of c2s_aggregator.cu) with the
// BatchNorm in eval mode, for one sample and pixel p (s = the bf16 skip map, z = W s + b, alpha = gamma / sqrt(var + eps)):
//   g_y = grad_out * [out > 0]                      grad_s = W^T (alpha * g_y)
//   grad_bn_bias = sum g_y   grad_bn_weight = sum g_y (z - mean) / sqrt(var + eps)
//   grad_conv_bias = alpha * sum g_y                grad_conv_weight = alpha * sum_p g_y s^T
// then the aggregator's backward with grad_out = grad_s.  One CTA = one sample x 64 channels x 128 pixels, as in the
// forward.  Before any frame arrives grad_s is formed on the tensor cores from grad_out and out alone (the A operand is
// (alpha W)^T as bf16 hi + lo; g_y is exact in bf16).  The valid frames then stream once through the TMA ring: the
// consumers write grad_x, scatter the bilinear adjoint into grad_attn (as agg_backward_pipe_kernel) and re-accumulate s
// with the forward's arithmetic in the forward's frame order, so the bf16 s is the forward's bit for bit.  After the
// sweep, z = W s (hi + lo, the forward's products) gives the BatchNorm sums and g_y s^T the weight gradient; each CTA
// writes its partials to the workspace and skipconv_bwd_finish_kernel reduces them in a fixed order (deterministic).
// ---------------------------------------------------------------------------------------------------
constexpr int kSbC = 64;                       // channels of the skip map (in and out channels of the 1x1 convolution)
constexpr int kSbPB = 128;                     // pixels per CTA
constexpr int kSbConsumers = 256;              // thread = (attention head, 8-pixel vector)
constexpr int kSbStageBytes = kSbC * kSbPB * 2;
constexpr int kSbTileStride = kSbPB * 2 + 16;  // bytes per channel row of a bf16 tile (padded: ldmatrix conflict-free)
constexpr int kSbGsStride = kSbPB + 4;         // floats per channel row of the fp32 grad_s tile
constexpr int kSbFrags = 4 * 4 * 32;           // uint4 A fragments of one 64 x 64 bf16 matrix (m-tile, k-step, lane)
constexpr int kSbPartial = kSbC * kSbC + 2 * kSbC;  // floats per CTA: g_y s^T, sum g_y, sum g_y (z - mean)
constexpr int kSbMaxStages = 6;  // one CTA per SM (the grad_s and s registers rule out two): 96 KB of x in flight

struct SkipConvBwdArgs {
  const float* attn;
  const uint8_t* pad;
  const __nv_bfloat16* out;
  const __nv_bfloat16* gout;
  __nv_bfloat16* gx;
  float* gattn;
  const uint4* wfrag;   // [hi|lo] A fragments of W            (z = W s)
  const uint4* afrag;   // [hi|lo] A fragments of (alpha W)^T  (grad_s = (alpha W)^T g_y)
  const float* zshift;  // [64] conv_bias - running_mean
  float* partial;       // [CTAs][kSbPartial] or nullptr (no parameter gradient wanted)
  int B, T, H, W, hw, ha, wa;
  float sy, sx;
  int tap_floats;       // per head and stage: staged attention rows of the pixel block (0: taps from global memory)
  int n_stages;
};

// A fragments (row-major 16 x 16 tiles, mma.sync m16n8k16) of W and of (alpha W)^T, each as bf16 hi + bf16 residual,
// in the order of skipconv_prep_kernel (c2s_aggregator.cu); block 2: the per-channel constants
__global__ void skipconv_bwd_prep_kernel(const float* __restrict__ w, const float* conv_bias, const float* bn_w,
                                         const float* bn_mean, const float* bn_var, float eps, uint4* __restrict__ wfrag,
                                         uint4* __restrict__ afrag, float* alpha, float* inv_std, float* zshift) {
  if (blockIdx.x == 2) {
    const int o = threadIdx.x;
    if (o < kSbC) {
      const float is = 1.f / sqrtf(bn_var[o] + eps);
      inv_std[o] = is;
      alpha[o] = (bn_w ? bn_w[o] : 1.f) / sqrtf(bn_var[o] + eps);  // the forward's scale, same arithmetic
      zshift[o] = (conv_bias ? conv_bias[o] : 0.f) - bn_mean[o];
    }
    return;
  }
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // (mt, ks, lane)
  if (idx >= kSbFrags) return;
  const int lane = idx & 31, ks = (idx >> 5) & 3, mt = idx >> 7;
  const int r0 = mt * 16 + (lane >> 2), c0 = ks * 16 + (lane & 3) * 2;
  for (int which = 0; which < 2; ++which) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {  // a0:(r, c) a1:(r+8, c) a2:(r, c+8) a3:(r+8, c+8)
      const int r = r0 + (q & 1) * 8, c = c0 + (q >> 1) * 8;
      float v0, v1;
      if (which == 0) {
        v0 = w[r * kSbC + c], v1 = w[r * kSbC + c + 1];
      } else {  // (alpha W)^T [c_in = r][c_out = c]
        const float a0 = (bn_w ? bn_w[c] : 1.f) / sqrtf(bn_var[c] + eps), a1 = (bn_w ? bn_w[c + 1] : 1.f) / sqrtf(bn_var[c + 1] + eps);
        v0 = a0 * w[c * kSbC + r], v1 = a1 * w[(c + 1) * kSbC + r];
      }
      const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
      hi[q] = Elem<__nv_bfloat16>::pack2(__bfloat162float(h0), __bfloat162float(h1));
      lo[q] = Elem<__nv_bfloat16>::pack2(v0 - __bfloat162float(h0), v1 - __bfloat162float(h1));
    }
    uint4* f = which == 0 ? wfrag : afrag;
    f[idx] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    f[kSbFrags + idx] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// [64 rows][128 pixels] = A[64 x 64] (hi + lo fragments) x tile[64 channels][128 pixels] (bf16, row stride kSbTileStride);
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
    const int mrow = ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
    const int ncol = warp * 16 + (lane >> 4) * 8;
    uint32_t bf[4];
    ldsm_x4_trans(bf, tile + mrow * kSbTileStride + ncol * 2);
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
      const uint4 h4 = __ldg(frag + (mt * 4 + ks) * 32 + lane);
      const uint4 l4 = __ldg(frag + kSbFrags + (mt * 4 + ks) * 32 + lane);
      const uint32_t ah[4] = {h4.x, h4.y, h4.z, h4.w}, al[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        mma_bf16(d[mt][nt], ah, bf[2 * nt], bf[2 * nt + 1]);
        mma_bf16(d[mt][nt], al, bf[2 * nt], bf[2 * nt + 1]);
      }
    }
  }
}

__device__ __forceinline__ void sts_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int S, bool TAPS>
__global__ void __launch_bounds__(kSbConsumers + 32, 1) agg_skipconv_backward_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                                      const __grid_constant__ CUtensorMap map_att,
                                                                                      const SkipConvBwdArgs a) {
  using T = __nv_bfloat16;
  constexpr int VEC = 8;
  constexpr int M = VEC / S;  // attention cells per thread
  constexpr int NCOL = M + 2;
  extern __shared__ __align__(128) unsigned char sb_smem[];  // stages | g_y tile (bf16) | grad_s (fp32), later the s tile
  __shared__ short frames[1024];
  __shared__ uint8_t s_pad[1024];
  __shared__ int n_frames_s;
  __shared__ __align__(8) unsigned long long bars[2 * kSbMaxStages];

  const int b = blockIdx.y, pblk = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int n_cwarps = kSbConsumers / 32;
  const int n_stages = a.n_stages;
  const uint32_t stage_stride = kSbStageBytes + 16u * a.tap_floats * 4u;
  int r_lo = 0;  // first attention row of the staged slice (the rows of the block's first pixel)
  if (TAPS) {
    int i1;
    float l1;
    source_index(a.sy, (pblk * kSbPB) / a.W, a.ha, r_lo, i1, l1);
  }

  if (threadIdx.x < 32) {  // ordered list of the frames that are not padded
    int count = 0;
    for (int base = 0; base < a.T; base += 32) {
      const int t = base + threadIdx.x;
      const bool valid = t < a.T && (a.pad == nullptr || a.pad[b * a.T + t] == 0);
      if (t < a.T) s_pad[t] = !valid;
      const unsigned m = __ballot_sync(0xffffffffu, valid);
      if (valid) frames[count + __popc(m & ((1u << threadIdx.x) - 1u))] = static_cast<short>(t);
      count += __popc(m);
    }
    if (threadIdx.x == 0) {
      n_frames_s = count;
      for (int s = 0; s < n_stages; ++s) {
        mbar_init(s32(&bars[s]), 1);
        mbar_init(s32(&bars[n_stages + s]), n_cwarps);
      }
      fence_mbarrier_init();
    }
  }
  __syncthreads();
  const int n_frames = n_frames_s;
  const uint32_t stage0 = s32(sb_smem);

  if (warp == n_cwarps) {  // ---- producer: one box {128 pixels, 64 channels, 1 frame} (+ the attention rows) per frame
    if (lane == 0) {
      const uint32_t tap_bytes = TAPS ? 16u * a.tap_floats * 4u : 0u;
      for (int i = 0; i < n_frames; ++i) {
        const int s = i % n_stages, round = i / n_stages;
        if (round > 0) mbar_wait(s32(&bars[n_stages + s]), (round - 1) & 1);
        const uint32_t full = s32(&bars[s]);
        mbar_expect_tx(full, kSbStageBytes + tap_bytes);
        tma_load_3d(stage0 + s * stage_stride, &map_x, pblk * kSbPB, 0, b * a.T + frames[i], full);
        if (TAPS) tma_load_3d(stage0 + s * stage_stride + kSbStageBytes, &map_att, r_lo * a.wa, b * a.T + frames[i], 0, full);
      }
    }
    return;
  }

  // ---- consumers: thread = (attention head, 8-pixel vector) ------------------------------------------------------------
  const int head = threadIdx.x >> 4, pv = threadIdx.x & 15;
  const int p0 = pblk * kSbPB + pv * VEC;
  const uint32_t gy_tile = stage0 + n_stages * stage_stride;
  const uint32_t gs_tile = gy_tile + kSbC * kSbTileStride;  // grad_s fp32 [64][kSbGsStride]; after the sweep the s tile
  float* gs_smem = reinterpret_cast<float*>(sb_smem + n_stages * stage_stride + kSbC * kSbTileStride);
  const size_t plane = static_cast<size_t>(b) * kSbC * a.hw + p0;

  // g_y = grad_out masked by the forward's ReLU decision (bf16, exact) -> shared tile
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const size_t off = plane + static_cast<size_t>(head * 4 + c) * a.hw;
    const uint4 g = ld_stream_v4(a.gout + off), o = ld_stream_v4(a.out + off);
    const uint32_t gw[4] = {g.x, g.y, g.z, g.w}, ow[4] = {o.x, o.y, o.z, o.w};
    uint32_t m[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {  // bf16 pairs: a positive bf16 has a clear sign bit and a non-zero magnitude
      const uint32_t lo_pos = ((ow[q] & 0x8000u) == 0 && (ow[q] & 0x7fffu) != 0) ? 0x0000ffffu : 0u;
      const uint32_t hi_pos = ((ow[q] & 0x80000000u) == 0 && (ow[q] & 0x7fff0000u) != 0) ? 0xffff0000u : 0u;
      m[q] = gw[q] & (lo_pos | hi_pos);
    }
    sts_v4(gy_tile + (head * 4 + c) * kSbTileStride + pv * 16, make_uint4(m[0], m[1], m[2], m[3]));
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kSbConsumers) : "memory");  // consumers only (the producer warp has its own loop)
  {  // grad_s = (alpha W)^T g_y -> shared memory (fp32)
    float d[4][2][4];
    skipconv_tile_mma(d, a.afrag, gy_tile, warp, lane);
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          const int c = mt * 16 + (lane >> 2) + hrow * 8, p = warp * 16 + nt * 8 + (lane & 3) * 2;
          *reinterpret_cast<float2*>(gs_smem + c * kSbGsStride + p) = make_float2(d[mt][nt][hrow * 2], d[mt][nt][hrow * 2 + 1]);
        }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kSbConsumers) : "memory");
  float gs[4][VEC];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 v0 = *reinterpret_cast<const float4*>(gs_smem + (head * 4 + c) * kSbGsStride + pv * VEC);
    const float4 v1 = *reinterpret_cast<const float4*>(gs_smem + (head * 4 + c) * kSbGsStride + pv * VEC + 4);
    gs[c][0] = v0.x, gs[c][1] = v0.y, gs[c][2] = v0.z, gs[c][3] = v0.w;
    gs[c][4] = v1.x, gs[c][5] = v1.y, gs[c][6] = v1.z, gs[c][7] = v1.w;
  }

  // bilinear geometry (identical to agg_skipconv_kernel)
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
  const int cmin = x0 / S - 1;
  int col[NCOL];
#pragma unroll
  for (int j = 0; j < NCOL; ++j) {
    const int cj = cmin + j;
    col[j] = cj < 0 ? 0 : (cj > a.wa - 1 ? a.wa - 1 : cj);
  }
  const int amap = a.ha * a.wa;
  const size_t abase = (static_cast<size_t>(head) * a.B + b) * a.T * amap;
  const int trow0 = (iy0 - r_lo) * a.wa, trow1 = (iy1 - r_lo) * a.wa;
  // 16 lanes of a head cover the 128 pixels in order: a lane's left / right neighbour in the image row sits next to it
  const int lanes_per_row = a.W / VEC;
  const int lane_in_row = (p0 / VEC) % lanes_per_row;
  const bool has_left = pv > 0 && lane_in_row > 0;
  const bool has_right = pv < 15 && lane_in_row < lanes_per_row - 1;
  const size_t frame_stride = static_cast<size_t>(kSbC) * a.hw;
  T* gxb = a.gx != nullptr ? a.gx + static_cast<size_t>(b) * a.T * frame_stride + static_cast<size_t>(head * 4) * a.hw + p0 : nullptr;

  float acc[4][VEC];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[c][j] = 0.f;

  const uint32_t my_off = (head * 4) * (kSbPB * 2) + pv * 16;
  for (int i = 0; i < n_frames; ++i) {
    const int t = frames[i];
    float r[NCOL];
    if (!TAPS) {
      const float* ap = a.attn + abase + static_cast<size_t>(t) * amap;
#pragma unroll
      for (int j = 0; j < NCOL; ++j) r[j] = fmaf(ly1, __ldg(ap + row1 + col[j]), ly0 * __ldg(ap + row0 + col[j]));
    }
    const int s = i % n_stages;
    mbar_wait(s32(&bars[s]), (i / n_stages) & 1);
    uint4 xv[4];
    const uint32_t base = stage0 + s * stage_stride + my_off;
#pragma unroll
    for (int c = 0; c < 4; ++c) xv[c] = lds_v4(base + c * (kSbPB * 2));
    if (TAPS) {
      const float* tp = reinterpret_cast<const float*>(sb_smem + s * stage_stride + kSbStageBytes) + head * a.tap_floats;
#pragma unroll
      for (int j = 0; j < NCOL; ++j) r[j] = fmaf(ly1, tp[trow1 + col[j]], ly0 * tp[trow0 + col[j]]);
    }
    fence_proxy_async();  // the stage's shared loads before the producer's next bulk copy into it
    __syncwarp();
    if (lane == 0) mbar_arrive(s32(&bars[n_stages + s]));

    float w[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int i0w = j / S + ((j % S) < S / 2 ? 0 : 1);
      w[j] = fmaf(lx1[j], r[i0w + 1], (1.f - lx1[j]) * r[i0w]);
    }
    float g[VEC];  // sum_c x * grad_s of this thread's pixels
#pragma unroll
    for (int j = 0; j < VEC; ++j) g[j] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float f[VEC], dx[VEC];
      Elem<T>::unpack(xv[c], f);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        acc[c][j] = fmaf(w[j], f[j], acc[c][j]);  // the forward's accumulation
        g[j] = fmaf(f[j], gs[c][j], g[j]);
        dx[j] = w[j] * gs[c][j];
      }
      if (gxb != nullptr) st_stream_v4(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(c) * a.hw, Elem<T>::pack(dx));
    }
    if (a.gattn == nullptr) continue;
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
    if (!has_left) {  // edge columns nobody picked up (image border: clamped; head or row boundary)
      atomicAdd(gp + row0 + col[0], ly0 * win[0]);
      if (ly1 != 0.f) atomicAdd(gp + row1 + col[0], ly1 * win[0]);
    }
    if (!has_right) {
      atomicAdd(gp + row0 + col[NCOL - 1], ly0 * win[NCOL - 1]);
      if (ly1 != 0.f) atomicAdd(gp + row1 + col[NCOL - 1], ly1 * win[NCOL - 1]);
    }
  }
  if (gxb != nullptr && n_frames < a.T) {  // padded frames receive exactly zero
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (int t = 0; t < a.T; ++t)
      if (s_pad[t])
#pragma unroll
        for (int c = 0; c < 4; ++c) st_stream_v4(gxb + static_cast<size_t>(t) * frame_stride + static_cast<size_t>(c) * a.hw, z);
  }
  if (a.partial == nullptr) return;

  // ---- parameter gradients of the tile: the s tile (bf16, the forward's value) replaces grad_s in shared memory -------
  asm volatile("bar.sync 1, %0;" ::"n"(kSbConsumers) : "memory");  // every consumer has its grad_s in registers
  const uint32_t s_tile = gs_tile;
#pragma unroll
  for (int c = 0; c < 4; ++c) sts_v4(s_tile + (head * 4 + c) * kSbTileStride + pv * 16, Elem<T>::pack(acc[c]));
  asm volatile("bar.sync 1, %0;" ::"n"(kSbConsumers) : "memory");
  float* part = a.partial + (static_cast<size_t>(b) * gridDim.x + pblk) * kSbPartial;
  float(*red)[8][kSbC] = reinterpret_cast<float(*)[8][kSbC]>(sb_smem);  // per-warp sums; the stages are drained by now
  {  // z - mean = W s + (bias - mean): sums of g_y and g_y (z - mean) per output channel
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
          const __nv_bfloat162 gy2 = *reinterpret_cast<const __nv_bfloat162*>(gyb + o * kSbTileStride + p * 2);
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
    for (int ks = 0; ks < kSbPB / 16; ++ks) {
      uint32_t af[4];
      ldsm_x4(af, gy_tile + (mt * 16 + (lane & 15)) * kSbTileStride + (ks * 16 + (lane >> 4) * 8) * 2);
#pragma unroll
      for (int np = 0; np < 2; ++np) {  // two n-tiles per ldmatrix.x4: (n 0-7 | 8-15) x (k 0-7 | 8-15)
        uint32_t bf[4];
        const int crow = (nt0 + 2 * np) * 8 + (lane & 7) + ((lane >> 4) & 1) * 8;
        ldsm_x4(bf, s_tile + crow * kSbTileStride + (ks * 16 + ((lane >> 3) & 1) * 8) * 2);
        mma_bf16(d[2 * np], af, bf[0], bf[1]);
        mma_bf16(d[2 * np + 1], af, bf[2], bf[3]);
      }
    }
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int o = mt * 16 + (lane >> 2) + hrow * 8, c = (nt0 + n) * 8 + (lane & 3) * 2;
        *reinterpret_cast<float2*>(part + o * kSbC + c) = make_float2(d[n][hrow * 2], d[n][hrow * 2 + 1]);
      }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kSbConsumers) : "memory");
  if (threadIdx.x < 2 * kSbC) {  // fixed order over the warps
    const int q = threadIdx.x / kSbC, o = threadIdx.x % kSbC;
    float v = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) v += red[q][w8][o];
    part[kSbC * kSbC + q * kSbC + o] = v;
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
  if (e < kSbPartial)
    for (int i = warp; i < n_ctas; i += 8) v += partial[static_cast<size_t>(i) * kSbPartial + e];
  sums[warp][lane] = v;
  __syncthreads();
  if (warp != 0 || e >= kSbPartial) return;
  float total = 0.f;
#pragma unroll
  for (int w8 = 0; w8 < 8; ++w8) total += sums[w8][lane];
  if (e < kSbC * kSbC) {
    if (gw != nullptr) gw[e] = alpha[e / kSbC] * total;
  } else if (e < kSbC * kSbC + kSbC) {
    const int o = e - kSbC * kSbC;
    if (gb != nullptr) gb[o] = alpha[o] * total;
    if (gbn_b != nullptr) gbn_b[o] = total;
  } else {
    const int o = e - kSbC * kSbC - kSbC;
    if (gbn_w != nullptr) gbn_w[o] = inv_std[o] * total;
  }
}

size_t skipconv_bwd_smem(int n_stages, int tap_floats) {  // stages | g_y tile | grad_s (then s) tile
  return static_cast<size_t>(n_stages) * (kSbStageBytes + 16 * tap_floats * 4) + kSbC * kSbTileStride + kSbC * kSbGsStride * 4;
}

template <int S, bool TAPS>
int launch_skipconv_bwd_t(const CUtensorMap& map_x, const CUtensorMap& map_att, const SkipConvBwdArgs& k, cudaStream_t stream,
                          const char* name) {
  const size_t smem = skipconv_bwd_smem(k.n_stages, k.tap_floats);
  C2S_SMEM_ATTR((agg_skipconv_backward_kernel<S, TAPS>), 227 * 1024);  // once per instantiation and device
  dim3 grid(k.hw / kSbPB, k.B);
  agg_skipconv_backward_kernel<S, TAPS><<<grid, kSbConsumers + 32, smem, stream>>>(map_x, map_att, k);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

template <int S>
int launch_skipconv_bwd(const CUtensorMap& map_x, const CUtensorMap& map_att, const SkipConvBwdArgs& k, cudaStream_t stream,
                        const char* name) {
  return k.tap_floats > 0 ? launch_skipconv_bwd_t<S, true>(map_x, map_att, k, stream, name)
                          : launch_skipconv_bwd_t<S, false>(map_x, map_att, k, stream, name);
}

// workspace: W and (alpha W)^T fragments, alpha / inv_std / zshift, then the CTA partials (16-byte aligned throughout)
constexpr size_t kSbFixedBytes = 2 * 2 * kSbFrags * sizeof(uint4) + 3 * kSbC * sizeof(float);
size_t skipconv_bwd_ctas(const c2s_agg_desc* d) {
  return d->B > 0 && d->H > 0 && d->W > 0 ? static_cast<size_t>(d->B) * ((static_cast<size_t>(d->H) * d->W) / kSbPB) : 0;
}

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

size_t c2s_agg_skipconv_backward_workspace_bytes(const c2s_agg_desc* d) {
  if (d == nullptr) return 0;
  return c2s::kSbFixedBytes + c2s::skipconv_bwd_ctas(d) * c2s::kSbPartial * sizeof(float);
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
  int scale_class = 0;
  for (int s : {2, 4, 8})
    if (d->H == s * d->ha && d->W == s * d->wa) scale_class = s;
  const int hw = d->H * d->W;
  auto al16 = [](const void* q) { return q == nullptr || reinterpret_cast<uintptr_t>(q) % 16 == 0; };
  C2S_CHECK_ARG(d->mode == C2S_AGG_ATT_GROUP && d->dtype == C2S_BF16 && d->C == kSbC && d->n_heads == 16 && scale_class != 0 &&
                    hw % kSbPB == 0 && d->W % 8 == 0 && d->T <= 1024 && d->B <= 65535 && al16(x) && al16(out) &&
                    al16(grad_out) && al16(io->grad_x),
                "c2s_agg_skipconv_backward: the fused backward serves what the fused forward serves: att_group, bf16, C=64, "
                "16 heads, x2/x4/x8 up-sampling, H*W %% 128 == 0, 16-byte aligned tensors (got mode %d dtype %d C %d heads "
                "%d %dx%d from %dx%d)", d->mode, d->dtype, d->C, d->n_heads, d->H, d->W, d->ha, d->wa);
  const bool want_params = io->grad_conv_weight != nullptr || io->grad_conv_bias != nullptr || io->grad_bn_weight != nullptr ||
                           io->grad_bn_bias != nullptr;
  if (!want_params && io->grad_x == nullptr && io->grad_attn == nullptr) return C2S_OK;  // nothing asked for
  const size_t need = c2s_agg_skipconv_backward_workspace_bytes(d);
  C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= need && reinterpret_cast<uintptr_t>(workspace) % 16 == 0,
                "c2s_agg_skipconv_backward: needs %zu workspace bytes, 16-byte aligned", need);
  int status = check_device();
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);

  uint4* wfrag = static_cast<uint4*>(workspace);
  uint4* afrag = wfrag + 2 * kSbFrags;
  float* alpha = reinterpret_cast<float*>(afrag + 2 * kSbFrags);
  float* inv_std = alpha + kSbC;
  float* zshift = inv_std + kSbC;
  float* partial = reinterpret_cast<float*>(static_cast<char*>(workspace) + kSbFixedBytes);
  skipconv_bwd_prep_kernel<<<3, 256, 0, stream>>>(p->conv_weight, p->conv_bias, p->bn_weight, p->bn_running_mean,
                                                  p->bn_running_var, p->bn_eps, wfrag, afrag, alpha, inv_std, zshift);
  C2S_LAUNCH_CHECK("agg_skipconv_backward<prep>");

  SkipConvBwdArgs k{};
  k.attn = attn, k.pad = pad_mask;
  k.out = static_cast<const __nv_bfloat16*>(out), k.gout = static_cast<const __nv_bfloat16*>(grad_out);
  k.gx = static_cast<__nv_bfloat16*>(io->grad_x), k.gattn = io->grad_attn;
  k.wfrag = wfrag, k.afrag = afrag, k.zshift = zshift, k.partial = want_params ? partial : nullptr;
  k.B = d->B, k.T = d->T, k.H = d->H, k.W = d->W, k.hw = hw, k.ha = d->ha, k.wa = d->wa;
  k.sy = static_cast<float>(d->ha) / static_cast<float>(d->H);
  k.sx = static_cast<float>(d->wa) / static_cast<float>(d->W);
  {  // staged attention rows: the rows a 128-pixel block can touch, per head (as in c2s_agg_skipconv_forward)
    const int rows_out = (kSbPB + d->W - 1) / d->W + 1;
    int rows_att = rows_out / scale_class + 3;
    rows_att = rows_att > d->ha ? d->ha : rows_att;
    const int tap_floats = ((rows_att * d->wa + 3) / 4) * 4;
    const bool taps = option(C2S_OPT_AGG_TAPS) == 0 && d->wa % 4 == 0 && reinterpret_cast<uintptr_t>(attn) % 16 == 0 &&
                      tap_floats <= 256;
    k.tap_floats = taps ? tap_floats : 0;
  }
  k.n_stages = kSbMaxStages;  // fewer if the staged rows make them too large for one CTA (227 KB with the static part)
  while (k.n_stages > 2 && skipconv_bwd_smem(k.n_stages, k.tap_floats) > 220 * 1024) --k.n_stages;
  CUtensorMap map_x;  // x as [B*T][C][H*W] bf16; box = 128 pixels x 64 channels x 1 frame
  const cuuint64_t dims[3] = {static_cast<cuuint64_t>(hw), static_cast<cuuint64_t>(kSbC), static_cast<cuuint64_t>(d->B) * d->T};
  const cuuint64_t strides[2] = {static_cast<cuuint64_t>(hw) * 2, static_cast<cuuint64_t>(kSbC) * hw * 2};
  const cuuint32_t box[3] = {kSbPB, kSbC, 1};
  status = encode_tensor_map(&map_x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_NONE, "skip features");
  if (status != C2S_OK) return status;
  CUtensorMap map_att = map_x;  // attention as [16 heads][B*T][ha*wa] fp32; box = tap_floats of one map x 1 frame x 16 heads
  if (k.tap_floats > 0) {
    const cuuint64_t amap = static_cast<cuuint64_t>(d->ha) * d->wa;
    const cuuint64_t adims[3] = {amap, static_cast<cuuint64_t>(d->B) * d->T, 16};
    const cuuint64_t astrides[2] = {amap * 4, static_cast<cuuint64_t>(d->B) * d->T * amap * 4};
    const cuuint32_t abox[3] = {static_cast<cuuint32_t>(k.tap_floats), 1, 16};
    status = encode_tensor_map(&map_att, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, attn, adims, astrides, abox,
                               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, "attention");
    if (status != C2S_OK) return status;
  }
  switch (scale_class) {
    case 2: status = launch_skipconv_bwd<2>(map_x, map_att, k, stream, "agg_skipconv_backward<x2>"); break;
    case 4: status = launch_skipconv_bwd<4>(map_x, map_att, k, stream, "agg_skipconv_backward<x4>"); break;
    default: status = launch_skipconv_bwd<8>(map_x, map_att, k, stream, "agg_skipconv_backward<x8>"); break;
  }
  if (status != C2S_OK || !want_params) return status;
  skipconv_bwd_finish_kernel<<<ceil_div(kSbPartial, 32), 256, 0, stream>>>(
      partial, static_cast<int>(skipconv_bwd_ctas(d)), alpha, inv_std, io->grad_conv_weight, io->grad_conv_bias,
      io->grad_bn_weight, io->grad_bn_bias);
  C2S_LAUNCH_CHECK("agg_skipconv_backward<reduce>");
  return C2S_OK;
}

}  // extern "C"
