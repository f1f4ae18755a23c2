// MLP of the L-TAE as a row GEMM on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
//   y[row, j] = sum_d o[row, d] * Wm[j, d] + bm[j]          rows = B*H*W pixel rows, d = 256, j < c_out   tae.py:443
//   -> BatchNorm1d (eval: folded scale/shift) -> ReLU -> Dropout mask -> GroupNorm(16 groups) -> out[b, j, y, x]
//                                                                                              tae.py:444-448, 488
// One CTA = 128 rows.  o (bf16 hi + lo, written by ltae_mma_kernel) and mlp.0.weight (bf16 hi + lo) are K-major;
// TMA (cp.async.bulk.tensor, 128-byte swizzle) brings 64-wide K chunks into a 2-stage ring, one elected thread
// issues the tcgen05 products (umma_bf16: M = 128, N = c_out, K = 16 per instruction) for hi*hi + lo*hi + hi*lo into
// one fp32 accumulator in tensor memory, umma_commit signals an mbarrier, and the four warps read their 32 TMEM
// lanes (= 32 pixel rows) back with tmem_ld32 for the epilogue, which needs every channel of a pixel in one thread.
#include "c2s_ltae_prep.cuh"
#include "c2s_sm100.cuh"

namespace c2s {
namespace {

constexpr int kRows = 128;    // UMMA M
constexpr int kK = 256;       // d_model
constexpr int kChunk = 64;    // K elements per TMA box row: 128 bytes = one swizzle atom
constexpr int kNumChunks = kK / kChunk;
constexpr int kTcThreads = 128;

struct MlpArgs {
  const float* bm;
  const float* bnf;      // [2, c_out] or nullptr (training: pre-BatchNorm rows go to ypre)
  const float* on_w;
  const float* on_b;
  const uint8_t* mlp_keep;
  float mlp_keep_scale;
  float gn_eps;
  float* ypre;
  __nv_bfloat16* out;
  int n_rows, hw, c_out, tmem_cols;
};

__global__ void __launch_bounds__(kTcThreads, 1)
ltae_mlp_tc_kernel(const __grid_constant__ CUtensorMap map_o_hi, const __grid_constant__ CUtensorMap map_o_lo,
                   const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                   const MlpArgs a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) unsigned long long bars[5];  // full[2], mma_done[2], acc_ready
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row0 = blockIdx.x * kRows;
  const uint32_t a_tile = kRows * kChunk * 2;               // 16 KB: 128 rows x 128 B
  const uint32_t b_tile = static_cast<uint32_t>(a.c_out) * kChunk * 2;
  const uint32_t stage_bytes = 2 * a_tile + 2 * b_tile;
  const uint32_t smem0 = (s32(smem) + 1023u) & ~1023u;  // swizzle atoms are 1024-byte aligned
  unsigned char* smem_al = smem + (smem0 - s32(smem));

  if (tid == 0) {
    for (int i = 0; i < 5; ++i) mbar_init(s32(&bars[i]), 1);
    fence_mbarrier_init();
  }
  if (warp == 0) {  // one warp allocates the accumulator columns in tensor memory
    tmem_alloc(s32(&tmem_base_s), a.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = tmem_base_s;

  if (tid == 0) {  // ---- TMA producer + MMA issuer (one thread) ----------------------------------------------
    auto load_chunk = [&](int kc) {
      const int s = kc & 1;
      const uint32_t full = s32(&bars[s]);
      const uint32_t base = smem0 + s * stage_bytes;
      mbar_expect_tx(full, stage_bytes);
      tma_load_2d(base, &map_o_hi, kc * kChunk, row0, full);
      tma_load_2d(base + a_tile, &map_o_lo, kc * kChunk, row0, full);
      tma_load_2d(base + 2 * a_tile, &map_w_hi, kc * kChunk, 0, full);
      tma_load_2d(base + 2 * a_tile + b_tile, &map_w_lo, kc * kChunk, 0, full);
    };
    const uint32_t idesc = umma_idesc_bf16(kRows, a.c_out);
    load_chunk(0);
    load_chunk(1);
    for (int kc = 0; kc < kNumChunks; ++kc) {
      const int s = kc & 1;
      mbar_wait(s32(&bars[s]), (kc >> 1) & 1);
      tc_fence_after();
      const uint32_t base = smem0 + s * stage_bytes;
      const uint64_t d_ohi = umma_desc_k_sw128(base), d_olo = umma_desc_k_sw128(base + a_tile);
      const uint64_t d_whi = umma_desc_k_sw128(base + 2 * a_tile), d_wlo = umma_desc_k_sw128(base + 2 * a_tile + b_tile);
#pragma unroll
      for (int k = 0; k < kChunk / 16; ++k) {  // 16 bf16 = 32 bytes inside the 128-byte swizzle atom: +2 in 16-byte units
        const uint64_t adv = static_cast<uint64_t>(k * 2);
        umma_bf16(tmem_acc, d_ohi + adv, d_whi + adv, idesc, (kc | k) != 0);
        umma_bf16(tmem_acc, d_olo + adv, d_whi + adv, idesc, 1);
        umma_bf16(tmem_acc, d_ohi + adv, d_wlo + adv, idesc, 1);
      }
      umma_commit(s32(&bars[2 + s]));  // arrives when every MMA issued so far has finished reading this stage
      if (kc + 2 < kNumChunks) {
        mbar_wait(s32(&bars[2 + s]), (kc >> 1) & 1);
        load_chunk(kc + 2);
      }
    }
    umma_commit(s32(&bars[4]));
  }

  // ---- epilogue: every warp owns 32 accumulator lanes = 32 pixel rows ------------------------------------
  mbar_wait(s32(&bars[4]), 0);
  tc_fence_after();
  float* ys = reinterpret_cast<float*>(smem_al);  // the operand ring is free now: [128 rows][c_out + 1]
  const int pitch = a.c_out + 1;
  const int row = row0 + tid;
  const bool live = row < a.n_rows;
  const int b = live ? row / a.hw : 0, pix = live ? row - b * a.hw : 0;
  float* yrow = ys + tid * pitch;
  for (int c0 = 0; c0 < a.c_out; c0 += 32) {
    uint32_t r[32];
    tmem_ld32(tmem_acc + (static_cast<uint32_t>(warp * 32) << 16) + c0, r);
    tmem_wait_ld();
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
    const int n = min(32, a.c_out - c0);
    for (int i = 0; i < n; ++i) {
      const int j = c0 + i;
      float y = v[i] + __ldg(a.bm + j);
      if (a.bnf != nullptr) {
        y = fmaxf(fmaf(y, __ldg(a.bnf + j), __ldg(a.bnf + a.c_out + j)), 0.f);
        if (a.mlp_keep != nullptr && live)
          y *= a.mlp_keep[(static_cast<size_t>(b) * a.c_out + j) * a.hw + pix] ? a.mlp_keep_scale : 0.f;
      }
      yrow[j] = y;
    }
  }
  if (live) {
    if (a.bnf == nullptr) {  // training: BatchNorm statistics need every row of the batch first
      for (int j = 0; j < a.c_out; ++j) a.ypre[static_cast<size_t>(row) * a.c_out + j] = yrow[j];
    } else {
      const int cog = a.c_out / 16;
      __nv_bfloat16* ob = a.out + static_cast<size_t>(b) * a.c_out * a.hw + pix;
      for (int g = 0; g < 16; ++g) {
        float m = 0.f;
        for (int k = 0; k < cog; ++k) m += yrow[g * cog + k];
        m /= static_cast<float>(cog);
        float var = 0.f;
        for (int k = 0; k < cog; ++k) {
          const float d = yrow[g * cog + k] - m;
          var = fmaf(d, d, var);
        }
        const float rstd = 1.f / sqrtf(var / static_cast<float>(cog) + a.gn_eps);
        for (int k = 0; k < cog; ++k) {
          const int j = g * cog + k;
          ob[static_cast<size_t>(j) * a.hw] =
              __float2bfloat16_rn(fmaf((yrow[j] - m) * rstd, __ldg(a.on_w + j), __ldg(a.on_b + j)));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_acc, a.tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------------------
// Persistent, warp-specialised version for c_out = 64 / 128 (the shipped MLPs): one CTA per SM walks over the 128-row tiles.
//   warp 0 (one thread)  TMA producer: the weights (hi + lo, all four K chunks) once, then the o chunks of tile after tile
//                        into a ring of 4 (c_out = 64) or 2 (c_out = 128) stages (hi + lo, 32 KB each);
//   warp 1 (one thread)  issues the 48 products (umma_bf16) of a tile into one of TWO accumulators in tensor memory, frees
//                        ring stages and hands accumulators over with umma_commit;
//   warps 2-5            epilogue: 32 TMEM lanes (= pixel rows) each, 32 channels at a time entirely in registers (the
//                        GroupNorm groups of 4 / 8 channels never straddle such a chunk): bias, BatchNorm fold, ReLU, dropout
//                        mask, output GroupNorm, bf16 stores -- while the next tile's loads and products are under way.
// The one-tile-per-CTA kernel above (no overlap, weights re-loaded per tile, epilogue through shared memory with run-time
// loop bounds) took 0.74 ms at the Time-Unet placement (1 M rows: 4x its HBM time) and 36 us at the U-TAE placement.
constexpr int kTc2Threads = 192;
__host__ __device__ constexpr int tc2_stages(int co) { return co <= 64 ? 4 : 2; }  // 128 KB of weights leave room for two

template <int CO>
__global__ void __launch_bounds__(kTc2Threads, 1)
ltae_mlp_tc2_kernel(const __grid_constant__ CUtensorMap map_o_hi, const __grid_constant__ CUtensorMap map_o_lo,
                    const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                    const MlpArgs a, int n_tiles) {
  constexpr uint32_t A_TILE = kRows * kChunk * 2;  // 16 KB: 128 rows x 128 B
  constexpr uint32_t B_TILE = CO * kChunk * 2;     // one K chunk of the weights
  constexpr uint32_t W_BYTES = kNumChunks * 2 * B_TILE;
  constexpr int COG = CO / 16;                     // channels per output GroupNorm group
  constexpr int kStages2 = tc2_stages(CO);
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) unsigned long long bars[1 + 2 * kStages2 + 4];  // wfull, full[S], empty[S], tfull[2], tempty[2]
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_par[5 * CO];                  // bm, bn scale, bn shift, on_w, on_b
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t smem0 = (s32(smem) + 1023u) & ~1023u;
  const uint32_t w_base = smem0, ring = smem0 + W_BYTES;
  const uint32_t bar0 = s32(&bars[0]);
  auto full = [&](int s) { return bar0 + 8u * (1 + s); };
  auto empty = [&](int s) { return bar0 + 8u * (1 + kStages2 + s); };
  auto tfull = [&](int b) { return bar0 + 8u * (1 + 2 * kStages2 + b); };
  auto tempty = [&](int b) { return bar0 + 8u * (1 + 2 * kStages2 + 2 + b); };

  if (tid == 0) {
    mbar_init(bar0, 1);
    for (int s = 0; s < kStages2; ++s) mbar_init(full(s), 1), mbar_init(empty(s), 1);
    for (int b = 0; b < 2; ++b) mbar_init(tfull(b), 1), mbar_init(tempty(b), 4);  // one arrival per epilogue warp
    fence_mbarrier_init();
  }
  if (warp == 0) {
    tmem_alloc(s32(&tmem_base_s), 2 * CO);
    tmem_relinquish();
  }
  for (int i = tid; i < CO; i += kTc2Threads) {
    s_par[i] = a.bm[i];
    s_par[CO + i] = a.bnf != nullptr ? a.bnf[i] : 1.f;
    s_par[2 * CO + i] = a.bnf != nullptr ? a.bnf[CO + i] : 0.f;
    s_par[3 * CO + i] = a.on_w != nullptr ? a.on_w[i] : 1.f;
    s_par[4 * CO + i] = a.on_b != nullptr ? a.on_b[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = tmem_base_s;

  if (warp == 0) {
    // ---- TMA producer ---------------------------------------------------------------------------------------------------
    if (lane == 0) {
      mbar_expect_tx(bar0, W_BYTES);
      for (int kc = 0; kc < kNumChunks; ++kc) {
        tma_load_2d(w_base + (2 * kc) * B_TILE, &map_w_hi, kc * kChunk, 0, bar0);
        tma_load_2d(w_base + (2 * kc + 1) * B_TILE, &map_w_lo, kc * kChunk, 0, bar0);
      }
      uint32_t g = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int kc = 0; kc < kNumChunks; ++kc, ++g) {
          const uint32_t s = g % kStages2;
          if (g >= kStages2) mbar_wait(empty(s), ((g / kStages2) - 1u) & 1u);
          const uint32_t base = ring + s * 2 * A_TILE;
          mbar_expect_tx(full(s), 2 * A_TILE);
          tma_load_2d(base, &map_o_hi, kc * kChunk, tile * kRows, full(s));
          tma_load_2d(base + A_TILE, &map_o_lo, kc * kChunk, tile * kRows, full(s));
        }
      }
    }
  } else if (warp == 1) {
    // ---- MMA issuer ---------------------------------------------------------------------------------------------------
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(kRows, CO);
      mbar_wait(bar0, 0);
      tc_fence_after();
      uint32_t g = 0, it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const uint32_t buf = it & 1u;
        if (it >= 2) mbar_wait(tempty(buf), ((it >> 1) - 1u) & 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_acc + buf * CO;
        for (int kc = 0; kc < kNumChunks; ++kc, ++g) {
          const uint32_t s = g % kStages2;
          mbar_wait(full(s), (g / kStages2) & 1u);
          tc_fence_after();
          const uint32_t base = ring + s * 2 * A_TILE;
          const uint64_t d_ohi = umma_desc_k_sw128(base), d_olo = umma_desc_k_sw128(base + A_TILE);
          const uint64_t d_whi = umma_desc_k_sw128(w_base + (2 * kc) * B_TILE), d_wlo = umma_desc_k_sw128(w_base + (2 * kc + 1) * B_TILE);
#pragma unroll
          for (int k = 0; k < kChunk / 16; ++k) {
            const uint64_t adv = static_cast<uint64_t>(k * 2);
            umma_bf16(d_tmem, d_ohi + adv, d_whi + adv, idesc, (kc | k) != 0);
            umma_bf16(d_tmem, d_olo + adv, d_whi + adv, idesc, 1);
            umma_bf16(d_tmem, d_ohi + adv, d_wlo + adv, idesc, 1);
          }
          umma_commit(empty(s));  // the stage is free once the products issued so far have read it
        }
        umma_commit(tfull(buf));
      }
    }
  } else {
    // ---- epilogue: TMEM lanes 32 q .. 32 q + 31 = pixel rows of the tile ------------------------------------------------
    const int q = warp & 3;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const uint32_t buf = it & 1u;
      const int row = tile * kRows + q * 32 + lane;
      const bool live = row < a.n_rows;
      const int b = live ? row / a.hw : 0, pix = live ? row - b * a.hw : 0;
      mbar_wait(tfull(buf), (it >> 1) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < CO; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(tmem_acc + (static_cast<uint32_t>(q * 32) << 16) + buf * CO + c0, r);
        tmem_wait_ld();
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
        if (c0 + 32 >= CO) {  // the accumulator is in registers: the tile after next may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty(buf));
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += s_par[c0 + i];
        if (a.bnf == nullptr) {  // training: BatchNorm statistics need every row of the batch first
          if (live) {
            float4* dst = reinterpret_cast<float4*>(a.ypre + static_cast<size_t>(row) * CO + c0);
#pragma unroll
            for (int i = 0; i < 8; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
          }
          continue;
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = fmaxf(fmaf(v[i], s_par[CO + c0 + i], s_par[2 * CO + c0 + i]), 0.f);
        if (a.mlp_keep != nullptr && live) {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            v[i] *= a.mlp_keep[(static_cast<size_t>(b) * CO + c0 + i) * a.hw + pix] ? a.mlp_keep_scale : 0.f;
        }
        if (!live) continue;
        __nv_bfloat16* ob = a.out + (static_cast<size_t>(b) * CO + c0) * a.hw + pix;
#pragma unroll
        for (int g0 = 0; g0 < 32; g0 += COG) {  // output GroupNorm over COG consecutive channels (tae.py:488), two passes
          float m = 0.f;
#pragma unroll
          for (int k = 0; k < COG; ++k) m += v[g0 + k];
          m /= static_cast<float>(COG);
          float var = 0.f;
#pragma unroll
          for (int k = 0; k < COG; ++k) {
            const float d = v[g0 + k] - m;
            var = fmaf(d, d, var);
          }
          const float rstd = 1.f / sqrtf(var / static_cast<float>(COG) + a.gn_eps);
#pragma unroll
          for (int k = 0; k < COG; ++k)
            ob[static_cast<size_t>(g0 + k) * a.hw] =
                __float2bfloat16_rn(fmaf((v[g0 + k] - m) * rstd, s_par[3 * CO + c0 + g0 + k], s_par[4 * CO + c0 + g0 + k]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_acc, 2 * CO);
}

// W[rows][cols] fp32 -> bf16 hi and lo planes, same row-major layout
__global__ void split_rows_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                  size_t n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = w[i];
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// [rows][256] bf16 row-major -> boxes of box_rows x 64 elements, 128-byte swizzle, out-of-range rows read as zero
int make_map(CUtensorMap* map, const void* base, uint64_t rows, uint32_t box_rows, const char* what) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(kK), rows};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(kK) * 2};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(kChunk), box_rows};
  return encode_tensor_map(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, what);
}

}  // namespace

size_t ltae_mlp_tc_workspace_floats(const c2s_ltae_desc& d) {
  if (d.flags & C2S_LTAE_ATTN_ONLY) return 0;
  const size_t rows = static_cast<size_t>(d.B) * d.H * d.W;
  // o hi + lo [rows][256] bf16, Wm hi + lo [c_out][256] bf16
  return align64(rows * kK) + align64(static_cast<size_t>(d.c_out) * kK);
}

void ltae_mlp_tc_buffers(const c2s_ltae_desc& d, float* ws, __nv_bfloat16** o_hi, __nv_bfloat16** o_lo,
                         __nv_bfloat16** w_hi, __nv_bfloat16** w_lo) {
  const size_t rows = static_cast<size_t>(d.B) * d.H * d.W;
  __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(ws);
  *o_hi = p;
  *o_lo = p + rows * kK;
  __nv_bfloat16* w = reinterpret_cast<__nv_bfloat16*>(ws + align64(rows * kK));
  *w_hi = w;
  *w_lo = w + static_cast<size_t>(d.c_out) * kK;
}

int ltae_mlp_tc_forward(const c2s_ltae_desc& d, const c2s_ltae_params& p, float* tc_ws, const float* bnf, float* ypre,
                        void* out, cudaStream_t stream) {
  __nv_bfloat16 *o_hi, *o_lo, *w_hi, *w_lo;
  ltae_mlp_tc_buffers(d, tc_ws, &o_hi, &o_lo, &w_hi, &w_lo);
  const size_t rows = static_cast<size_t>(d.B) * d.H * d.W;
  const size_t nw = static_cast<size_t>(d.c_out) * kK;
  if (!(d.flags & C2S_LTAE_REUSE_FOLDED)) {
    split_rows_kernel<<<ceil_div(nw, 256), 256, 0, stream>>>(p.mlp_weight, w_hi, w_lo, nw);
    C2S_LAUNCH_CHECK("ltae_split_mlp_weight");
  }
  CUtensorMap m_ohi, m_olo, m_whi, m_wlo;
  int status = make_map(&m_ohi, o_hi, rows, kRows, "MLP rows hi");
  if (status == C2S_OK) status = make_map(&m_olo, o_lo, rows, kRows, "MLP rows lo");
  if (status == C2S_OK) status = make_map(&m_whi, w_hi, d.c_out, d.c_out, "MLP weight hi");
  if (status == C2S_OK) status = make_map(&m_wlo, w_lo, d.c_out, d.c_out, "MLP weight lo");
  if (status != C2S_OK) return status;
  MlpArgs a{};
  a.bm = p.mlp_bias, a.bnf = bnf, a.on_w = p.out_norm_weight, a.on_b = p.out_norm_bias;
  a.mlp_keep = p.mlp_keep, a.mlp_keep_scale = d.mlp_keep_scale, a.gn_eps = d.gn_eps;
  a.ypre = ypre, a.out = static_cast<__nv_bfloat16*>(out);
  a.n_rows = static_cast<int>(rows), a.hw = d.H * d.W, a.c_out = d.c_out;
  a.tmem_cols = d.c_out <= 32 ? 32 : (d.c_out <= 64 ? 64 : (d.c_out <= 128 ? 128 : 256));
  if (d.c_out == 64 || d.c_out == 128) {  // persistent, warp-specialised kernel
    const int n_tiles = ceil_div(rows, kRows);
    const int sms = sm_count();
    const int grid = n_tiles < sms ? n_tiles : sms;
    const size_t smem2 = static_cast<size_t>(kNumChunks) * 2 * d.c_out * kChunk * 2 + static_cast<size_t>(tc2_stages(d.c_out)) * 2 * kRows * kChunk * 2 + 1024;
    if (d.c_out == 64) {
      C2S_SMEM_ATTR(ltae_mlp_tc2_kernel<64>, smem2);
      ltae_mlp_tc2_kernel<64><<<grid, kTc2Threads, smem2, stream>>>(m_ohi, m_olo, m_whi, m_wlo, a, n_tiles);
    } else {
      C2S_SMEM_ATTR(ltae_mlp_tc2_kernel<128>, smem2);
      ltae_mlp_tc2_kernel<128><<<grid, kTc2Threads, smem2, stream>>>(m_ohi, m_olo, m_whi, m_wlo, a, n_tiles);
    }
    C2S_LAUNCH_CHECK("ltae_mlp<tcgen05>");
    return C2S_OK;
  }
  const size_t stage = 2 * static_cast<size_t>(kRows) * kChunk * 2 + 2 * static_cast<size_t>(d.c_out) * kChunk * 2;
  size_t smem = 2 * stage;
  const size_t ys_bytes = static_cast<size_t>(kRows) * (d.c_out + 1) * sizeof(float);
  if (ys_bytes > smem) smem = ys_bytes;
  smem += 1024;  // alignment slack for the 1024-byte swizzle atoms
  C2S_SMEM_ATTR(ltae_mlp_tc_kernel, 227 * 1024);
  ltae_mlp_tc_kernel<<<ceil_div(rows, kRows), kTcThreads, smem, stream>>>(m_ohi, m_olo, m_whi, m_wlo, a);
  C2S_LAUNCH_CHECK("ltae_mlp<tcgen05>");
  return C2S_OK;
}

}  // namespace c2s
