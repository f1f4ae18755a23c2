// L-TAE backward over the features on the tensor cores (stage A of the backward; bf16 features, 16 heads, d_model 256,
// C in {64, 128}, T <= 64, H*W % 8 == 0), sm_100a.  Reference: autograd through src/backbones/tae.py:451-504, 760-847.
//
// Same algebra and the same outputs as ltae_backward_kernel (c2s_ltae_bwd.cu, whose header carries the derivation), with
// the execution structure of the forward slab kernels (c2s_ltae_team.cu):
//   * a persistent CTA of 8 warps walks over tiles of 8 consecutive pixels; the tile's features arrive as four TMA boxes
//     [16 frames][C][8 px] and are transposed in place to [t][8-channel block][pixel ^ (t & 7)][8 channels] with
//     ldmatrix.trans + stmatrix (the GroupNorm sums come from the same registers);
//   * one warp owns one pixel.  Its seven products run on mma.sync.m16n8k16 (bf16, fp32 accumulation) straight from that
//     slab: scores S = (U r) X^T (hi + lo split of the per-pixel weights, as in the forward), the adjoint of the
//     attention g_at = (gamma gzn r) X^T + Go PE16^T, the two contractions over the frames au = gs X and az = at X,
//     and g_xh = gs^T U + at^T (gamma gzn); gs / at change from accumulator to operand layout in registers (packing for
//     the k = t products, movmatrix.trans for the k = h products);
//   * gzn[h, c] = sum_i Wc[16 h + i, c] grad_o[16 h + i] has a weight shared by all pixels: the 8 pixels of the tile are
//     the N dimension of one product per head (two heads per warp), the result lands in shared memory [pixel][h][c];
//   * grad_x replaces x in the slab (same fragment positions), is transposed back and leaves as four TMA stores (the
//     frame dimension of the 4-D tensor map clips t >= T);
//   * the sums over pixels (grad_U, direct gamma / beta terms, grad_cpos) collect in shared memory (fp32); grad_U and the
//     gamma / beta terms are flushed once per CTA, grad_cpos once per tile.
// 64 HBM bytes per (pixel, frame, 16 channels) are read and written once; at the training placement (4 096 pixels) the
// kernel is latency-bound, the point is the instruction count: ~4 k warp instructions per pixel against ~77 k of the
// CUDA-core kernel.  Serves what ltae_bwd_tc_eligible says; everything else stays on ltae_backward_kernel.
#include "c2s_ltae_fa.cuh"

namespace c2s {


namespace {

constexpr float kLn2 = 0.6931471805599453f;

template <int C>
struct BtSmem {
  static constexpr int kFB = C * 16;                  // one frame: [C/8][8 slots][8 channels] bf16
  static constexpr int kSlab = kTP * kFB;
  static constexpr int kGzRow = (C + 8) * 2;          // one head row of gzn (bf16), bytes
  static constexpr int kGzPix = kH * kGzRow + 16;     // pixel blocks 4 banks apart
  static constexpr int kGuP = 20;                     // pitch of the grad_U accumulators (bank spread)
  static constexpr int kPeRowB = 48;                  // positional rows [t][16 + 8] bf16
  static constexpr int oSlab = 0;
  static constexpr int oGz = oSlab + kSlab;
  static constexpr int oUf = oGz + kPix * kGzPix;     // float4 [C/16][2][32]  score weights (A fragments, times log2 e)
  static constexpr int oUb = oUf + C * 64;            // uint2  [C/8][32]      U as B fragments of the k = h product (bf16)
  static constexpr int oCpos = oUb + C / 8 * 256;     // float  [16][kAP]
  static constexpr int oPe = oCpos + kH * kAP * 4;    // bf16   [64][24]
  static constexpr int oPart = oPe + kTP * kPeRowB;   // float2 [8 warps][72]
  static constexpr int oRm = oPart + 8 * 72 * 8;      // float  [8 warps][48]: rstd, mean * rstd, mean per group
  static constexpr int oM12 = oRm + 8 * 48 * 4;       // float  [8 warps][32]: the two GroupNorm-backward means per group
  static constexpr int oGam = oM12 + 8 * 32 * 4;      // float  gamma[C], beta[C]
  static constexpr int oGp = oGam + 2 * C * 4;        // bf16x2 gamma pairs [C/2]
  static constexpr int oWb = oGp + C * 2;             // float  [256]
  static constexpr int oGu = oWb + kD * 4;            // float  [C][kGuP]      grad_U of this CTA
  static constexpr int oGgb = oGu + C * kGuP * 4;     // float  gg[C], gb[C]   direct gamma / beta terms of this CTA
  static constexpr int oGc = oGgb + 2 * C * 4;        // float  [64][kGuP]     grad_cpos of the tile
  static constexpr int oBar = oGc + kTP * kGuP * 4;
  static constexpr int kTotal = oBar + 64;
  static_assert(kTotal <= 232448, "shared memory budget");
};

__device__ __forceinline__ uint32_t mul_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t v) {
  uint32_t r;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}
__device__ __forceinline__ float2 ldg_f2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
// global loads that must be ISSUED where they are written (the compiler sinks plain loads to their first use, which puts a
// full L2 latency on the critical path)
__device__ __forceinline__ float ldg_f32_now(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ldg_u8_now(const uint8_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// FULL = false: the attention-only encoder of W-TAE (LTAE4WTAE, tae.py:507-635): no value path, so no gzn, no zn / sa rows,
// no direct gamma / beta terms; g_at is the gradient of the returned attention alone.
template <int C, bool FULL>
__global__ void __launch_bounds__(256, 1)
ltae_bwd_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_gx, const BwdTcArgs a) {
  using S = BtSmem<C>;
  constexpr int KS = C / 16;       // k-steps over the channels
  constexpr int CPG = C / kH;      // channels per GroupNorm group
  constexpr int FB = S::kFB;
  constexpr int NQ = C / 32;       // 4-block quads per frame (one ldmatrix.x4 each)
  constexpr int TSTEP = 8 / NQ;    // frames between two items of a warp in the transposition passes
  constexpr int FPG = 16 / TSTEP;  // frames of a 16-frame box per warp
  constexpr int SUB = (C == 64) ? 2 : 1;
  constexpr int GP = S::kGuP;
  extern __shared__ __align__(1024) unsigned char smem[];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = warp;                        // pixel of this warp
  const int j = lane & 3, g = lane >> 2;     // fragment coordinates
  const int mat = lane >> 3, mr = lane & 7;  // ldmatrix: this lane supplies row mr of matrix mat

  unsigned char* slab_ptr = smem + S::oSlab;
  const uint32_t slab = s32(slab_ptr);
  unsigned char* gz_ptr = smem + S::oGz + p * S::kGzPix;  // this pixel's gzn [h][c]
  const float4* s_uf = reinterpret_cast<const float4*>(smem + S::oUf);
  const uint2* s_ub = reinterpret_cast<const uint2*>(smem + S::oUb);
  float* s_cpos = reinterpret_cast<float*>(smem + S::oCpos);
  unsigned char* s_pe = smem + S::oPe;
  float2* s_part = reinterpret_cast<float2*>(smem + S::oPart);
  float* s_rm = reinterpret_cast<float*>(smem + S::oRm) + warp * 48;
  float* s_m12 = reinterpret_cast<float*>(smem + S::oM12) + warp * 32;
  const float* s_gam = reinterpret_cast<const float*>(smem + S::oGam);
  const uint32_t* s_gp = reinterpret_cast<const uint32_t*>(smem + S::oGp);
  const float* s_wb = reinterpret_cast<const float*>(smem + S::oWb);
  float* s_gu = reinterpret_cast<float*>(smem + S::oGu);
  float* s_ggb = reinterpret_cast<float*>(smem + S::oGgb);
  float* s_gc = reinterpret_cast<float*>(smem + S::oGc);
  const uint32_t bars = s32(smem + S::oBar);

  // ---- set-up ------------------------------------------------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(bars + 8 * i, 1);
    fence_mbarrier_init();
  }
  for (int i = tid; i < S::kSlab / 16; i += 256) reinterpret_cast<uint4*>(slab_ptr)[i] = make_uint4(0, 0, 0, 0);  // never NaN
  for (int i = tid; i < kTP * S::kPeRowB / 4; i += 256) reinterpret_cast<uint32_t*>(s_pe)[i] = 0u;
  for (int i = tid; i < C * GP; i += 256) s_gu[i] = 0.f;
  for (int i = tid; i < 2 * C; i += 256) s_ggb[i] = 0.f;
  for (int i = tid; i < kTP * GP; i += 256) s_gc[i] = 0.f;
  {
    float4* uf = reinterpret_cast<float4*>(smem + S::oUf);
    for (int i = tid; i < KS * 64; i += 256) {  // [ks][half][lane]: rows g / g + 8, channels 16 ks + 8 half + 2 j, + 1
      const int ks = i >> 6, hf = (i >> 5) & 1, ln = i & 31, jj = ln & 3, gg = ln >> 2;
      const float* up = a.u + (ks * 16 + hf * 8 + 2 * jj) * kMaxHeads;
      uf[i] = make_float4(__ldg(up + gg) * kLog2e, __ldg(up + kMaxHeads + gg) * kLog2e, __ldg(up + gg + 8) * kLog2e,
                          __ldg(up + kMaxHeads + gg + 8) * kLog2e);
    }
    uint2* ub = reinterpret_cast<uint2*>(smem + S::oUb);
    for (int i = tid; i < C / 8 * 32; i += 256) {  // [n-tile][lane]: B[k = h][n = c] = U[h][c], c = 8 nt + g, h = 2 j (+ 8)
      const int nt = i >> 5, ln = i & 31, jj = ln & 3, gg = ln >> 2;
      const float* up = a.u + (nt * 8 + gg) * kMaxHeads + 2 * jj;
      ub[i] = make_uint2(pack_bf16(__ldg(up), __ldg(up + 1)), pack_bf16(__ldg(up + 8), __ldg(up + 9)));
    }
    float* gam = reinterpret_cast<float*>(smem + S::oGam);
    for (int i = tid; i < C; i += 256) gam[i] = __ldg(a.gamma + i), gam[C + i] = __ldg(a.beta + i);
    uint32_t* gp = reinterpret_cast<uint32_t*>(smem + S::oGp);
    for (int i = tid; i < C / 2; i += 256) gp[i] = pack_bf16(__ldg(a.gamma + 2 * i), __ldg(a.gamma + 2 * i + 1));
    float* wb = reinterpret_cast<float*>(smem + S::oWb);
    for (int i = tid; i < kD; i += 256) wb[i] = __ldg(a.wb + i);
  }
  const float inv_n_all = 1.f / (static_cast<float>(a.T) * CPG);
  const unsigned long long beyond = (a.T >= 64) ? 0ull : (~0ull << a.T);  // frames t >= T
  fence_proxy_async();  // generic zero fill above, bulk-copy writes below
  __syncthreads();

  int cur_b = -1;
  unsigned long long padm = 0;
#pragma unroll 1
  for (int k = 0;; ++k) {
    const int tile = blockIdx.x + k * gridDim.x;
    if (tile >= a.n_tiles) break;
    const uint32_t par = static_cast<uint32_t>(k) & 1u;
    const int b = tile / a.tiles_per_b;
    const int pix0 = (tile - b * a.tiles_per_b) * kPix;
    const size_t row0 = static_cast<size_t>(b) * a.hw + pix0;

    // ---- the tile's boxes (the previous tile's stores have finished reading the slab) ----------------------------------
    if (tid == 0) {
      tma_store_wait_read();
#pragma unroll
      for (int grp = 0; grp < 4; ++grp)
        if (16 * grp < a.T) {
          mbar_expect_tx(bars + 8 * grp, 16 * FB);
          tma_load_4d(slab + 16 * grp * FB, &map_x, pix0, 0, 16 * grp, b, bars + 8 * grp);
        }
    }

    // ---- per-sample constants ---------------------------------------------------------------------------------------------
    if (b != cur_b) {  // CTA-uniform; the readers of the previous tile are behind its last barrier
      cur_b = b;
      for (int i = tid; i < kTP * 16; i += 256) {
        const int t = i >> 4, h = i & 15;
        s_cpos[h * kAP + t] = t < a.T ? __ldg(a.cpos + (static_cast<size_t>(b) * a.T + t) * kMaxHeads + h) * kLog2e : 0.f;
        const float pv = (a.pe != nullptr && t < a.T) ? __ldg(a.pe + (static_cast<size_t>(b) * a.T + t) * kD + h) : 0.f;
        *reinterpret_cast<__nv_bfloat16*>(s_pe + t * S::kPeRowB + h * 2) = __float2bfloat16_rn(pv);
      }
      unsigned long long m = 0;
      if (a.pad != nullptr) {
        const unsigned lo = __ballot_sync(0xffffffffu, lane < a.T && a.pad[b * a.T + lane] != 0);
        const unsigned hi = __ballot_sync(0xffffffffu, lane + 32 < a.T && a.pad[b * a.T + 32 + lane] != 0);
        m = static_cast<unsigned long long>(lo) | (static_cast<unsigned long long>(hi) << 32);
      }
      padm = m;
    }

    // pivots of the shifted GroupNorm sums: first channel of the lane's group in frame 0 (any value works as a shift)
    float npv[4];
    {
      const __nv_bfloat16* xf = a.x + static_cast<size_t>(b) * a.T * C * a.hw + pix0 + g;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c0 = (4 * (warp % NQ) + i) * 8 + (CPG == 4 ? 4 * (j >> 1) : 0);
        npv[i] = -__bfloat162float(xf[static_cast<size_t>(c0) * a.hw]);
      }
    }
    // this pixel's grad_o row as the A operand [h][i] of the positional product (rows g / g + 8, i = 2 j .. and + 8)
    float2 go0 = make_float2(0.f, 0.f), go1 = go0, go2 = go0, go3 = go0;
    if constexpr (FULL) {
      const float* gor = a.g_o + (row0 + p) * kD;
      go0 = ldg_f2(gor + 16 * g + 2 * j), go1 = ldg_f2(gor + 16 * (g + 8) + 2 * j);
      go2 = ldg_f2(gor + 16 * g + 2 * j + 8), go3 = ldg_f2(gor + 16 * (g + 8) + 2 * j + 8);
    }

    // the gradient of the returned attention is the initial value of the g_at accumulators, the dropout realisation two
    // bit masks (rows g / g + 8, bit 2 nt + e <-> frame 8 nt + 2 j + e): requested now, they travel during the phases below
    float gacc[8][4];
    uint32_t km0 = 0xffffffffu, km1 = 0xffffffffu;
    {
      const size_t h8 = static_cast<size_t>(8) * a.B * a.T * a.hw;
      const size_t at0 = ((static_cast<size_t>(g) * a.B + b) * a.T) * a.hw + pix0 + p;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int t = nt * 8 + 2 * j + e;
          float v0 = 0.f, v1 = 0.f;
          if (a.g_attn != nullptr && t < a.T) {
            const float* ga = a.g_attn + at0 + static_cast<size_t>(t) * a.hw;
            v0 = ldg_f32_now(ga), v1 = ldg_f32_now(ga + h8);
          }
          gacc[nt][e] = v0, gacc[nt][2 + e] = v1;
        }
      if (a.attn_keep != nullptr) {
        uint32_t m0 = 0u, m1 = 0u;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int t = nt * 8 + 2 * j + e;
            if (t < a.T) {
              const uint8_t* kp = a.attn_keep + at0 + static_cast<size_t>(t) * a.hw;
              m0 |= (ldg_u8_now(kp) != 0u ? 1u : 0u) << (2 * nt + e);
              m1 |= (ldg_u8_now(kp + h8) != 0u ? 1u : 0u) << (2 * nt + e);
            }
          }
        km0 = m0, km1 = m1;
      }
    }
    const float keep_scale = a.attn_keep != nullptr ? a.attn_keep_scale : 1.f;

    // ---- gzn[pixel][h][c] = sum_i Wc[16 h + i][c] grad_o[pixel][16 h + i]: heads 2 warp, 2 warp + 1; M = c, N = pixel -----
#pragma unroll
    for (int hh = 0; hh < (FULL ? 2 : 0); ++hh) {
      const int h = 2 * warp + hh;
      const float* gor = a.g_o + (row0 + g) * kD + 16 * h + 2 * j;
      const float2 b0f = ldg_f2(gor), b1f = ldg_f2(gor + 8);
      const uint32_t b0 = pack_bf16(b0f.x, b0f.y), b1 = pack_bf16(b1f.x, b1f.y);
      float2 w[C / 16][4];
#pragma unroll
      for (int mt = 0; mt < C / 16; ++mt) {
        const float* wr = a.wct + static_cast<size_t>(16 * mt + g) * kD + 16 * h + 2 * j;
        w[mt][0] = ldg_f2(wr), w[mt][1] = ldg_f2(wr + 8 * kD), w[mt][2] = ldg_f2(wr + 8), w[mt][3] = ldg_f2(wr + 8 * kD + 8);
      }
#pragma unroll
      for (int mt = 0; mt < C / 16; ++mt) {
        uint32_t af[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) af[i] = pack_bf16(w[mt][i].x, w[mt][i].y);
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        mma_bf16(d, af, b0, b1);
        // d0 = (c = 16 mt + g, pixel 2 j), d1 = (c, 2 j + 1), d2 = (c + 8, 2 j), d3 = (c + 8, 2 j + 1)
        unsigned char* dst = smem + S::oGz + h * S::kGzRow + (16 * mt + g) * 2;
        *reinterpret_cast<__nv_bfloat16*>(dst + (2 * j) * S::kGzPix) = __float2bfloat16_rn(d[0]);
        *reinterpret_cast<__nv_bfloat16*>(dst + (2 * j + 1) * S::kGzPix) = __float2bfloat16_rn(d[1]);
        *reinterpret_cast<__nv_bfloat16*>(dst + (2 * j) * S::kGzPix + 16) = __float2bfloat16_rn(d[2]);
        *reinterpret_cast<__nv_bfloat16*>(dst + (2 * j + 1) * S::kGzPix + 16) = __float2bfloat16_rn(d[3]);
      }
    }

    // ---- transposition in place + GroupNorm sums (tae.py:461; all T frames count) ---------------------------------------
    {
      const int q4 = warp % NQ, f0 = warp / NQ;
      const uint32_t blk0 = slab + q4 * 512 + mat * 128;
      unsigned long long s1p[4], s2p[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) s1p[i] = 0ull, s2p[i] = 0ull;
#pragma unroll
      for (int grp = 0; grp < 4; ++grp) {
        if (16 * grp >= a.T) continue;
        mbar_wait(bars + 8 * grp, par);
        uint32_t v[FPG][4];
#pragma unroll
        for (int q = 0; q < FPG; ++q) ldsm_x4_trans(v[q], blk0 + (16 * grp + f0 + TSTEP * q) * FB + mr * 16);
#pragma unroll
        for (int q = 0; q < FPG; ++q) {
          const int t = 16 * grp + f0 + TSTEP * q;
          stsm_x4(blk0 + t * FB + ((mr ^ (t & 7)) << 4), v[q]);  // row = pixel, 8 channels; slot pixel ^ (t & 7)
          if (t < a.T) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const unsigned long long d = bf16x2_plus_f32(v[q][i], npv[i]);
              s1p[i] = add_f32x2(s1p[i], d);
              s2p[i] = fma_f32x2(d, d, s2p[i]);
            }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float lo, hi;
        unpack_f32x2(s1p[i], lo, hi);
        float s1 = lo + hi;
        unpack_f32x2(s2p[i], lo, hi);
        float s2 = lo + hi;
        s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
        s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
        if (CPG == 8) {
          s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
          s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
        }
        const bool writer = (CPG == 8) ? (j == 0) : ((j & 1) == 0);
        if (writer) s_part[warp * 72 + (g * 4 + i) * SUB + (CPG == 4 ? (j >> 1) : 0)] = make_float2(s1, s2);
      }
    }
    __syncthreads();  // the slab is transposed, gzn and the partial sums are written

    // ---- statistics of this warp's pixel: lane = group -----------------------------------------------------------------
    if (lane < kH) {
      const int grp = lane;
      const int cb = (CPG == 8) ? grp : (grp >> 1), sub = (CPG == 8) ? 0 : (grp & 1);
      const int qq = cb >> 2, ii = cb & 3;
      float t1 = 0.f, t2 = 0.f;
#pragma unroll
      for (int m = 0; m < TSTEP; ++m) {
        const float2 v = s_part[(qq + NQ * m) * 72 + (p * 4 + ii) * SUB + sub];
        t1 += v.x, t2 += v.y;
      }
      const int c0 = grp * CPG;
      const float pv = __bfloat162float(
          *reinterpret_cast<const __nv_bfloat16*>(slab_ptr + (c0 >> 3) * 128 + (p << 4) + (c0 & 7) * 2));  // frame 0, slot p ^ 0
      const float m = t1 * inv_n_all;
      float var = fmaf(t2, inv_n_all, -m * m);
      var = var < 0.f ? 0.f : var;
      const float rstd = rsqrtf(var + a.gn_eps);
      s_rm[grp] = rstd;
      s_rm[16 + grp] = (m + pv) * rstd;
      s_rm[32 + grp] = m + pv;
    }
    __syncwarp();

    // ---- scores S[h, t] (hi + lo weights) and g_at[h, t] = sum_c (gamma gzn r)[h, c] x[t, c] + ... in one sweep ------------
    float sacc[8][4], cacc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int t = nt * 8 + 2 * j;
      const float2 c0 = *reinterpret_cast<const float2*>(s_cpos + g * kAP + t);
      const float2 c1 = *reinterpret_cast<const float2*>(s_cpos + (g + 8) * kAP + t);
      sacc[nt][0] = c0.x, sacc[nt][1] = c0.y, sacc[nt][2] = c1.x, sacc[nt][3] = c1.y;
    }
    const uint32_t xbase = slab + ((p ^ mr) << 4) + (mat & 1) * 128 + ((mat >> 1) * 8 + mr) * FB;
    const uint32_t gz_frag = s32(gz_ptr) + ((mat & 1) * 8 + mr) * S::kGzRow + (mat >> 1) * 16;
#pragma unroll 2
    for (int ks = 0; ks < KS; ++ks) {
      const float4 u0 = s_uf[ks * 64 + lane], u1 = s_uf[ks * 64 + 32 + lane];
      const int c_lo = ks * 16 + 2 * j;
      const int g0 = c_lo / CPG, g1 = (c_lo + 8) / CPG;
      const float r0 = s_rm[g0], r1 = s_rm[g1];
      uint32_t ahi[4], alo[4], az[4];
      split_bf16(u0.x * r0, u0.y * r0, ahi[0], alo[0]);  // (row g,     k 2j, 2j+1)
      split_bf16(u0.z * r0, u0.w * r0, ahi[1], alo[1]);  // (row g + 8, k 2j, 2j+1)
      split_bf16(u1.x * r1, u1.y * r1, ahi[2], alo[2]);  // (row g,     k 2j+8, 2j+9)
      split_bf16(u1.z * r1, u1.w * r1, ahi[3], alo[3]);  // (row g + 8, k 2j+8, 2j+9)
      if constexpr (FULL) {
        ldsm_x4(az, gz_frag + ks * 32);                  // gzn[h][c] as the same A fragment
        const uint32_t gp0 = s_gp[c_lo >> 1], gp1 = s_gp[(c_lo + 8) >> 1];
        const uint32_t rr0 = pack_bf16(r0, r0), rr1 = pack_bf16(r1, r1);
        az[0] = mul_bf16x2(mul_bf16x2(az[0], gp0), rr0);
        az[1] = mul_bf16x2(mul_bf16x2(az[1], gp0), rr0);
        az[2] = mul_bf16x2(mul_bf16x2(az[2], gp1), rr1);
        az[3] = mul_bf16x2(mul_bf16x2(az[3], gp1), rr1);
      }
      uint32_t bfr[4][4];  // (frames 16 ntp .. + 7, channels 16 ks .. + 7), (.., + 8 .. 15), (frames + 8 .. 15, ..), (..)
#pragma unroll
      for (int ntp = 0; ntp < 4; ++ntp) ldsm_x4(bfr[ntp], xbase + ntp * 16 * FB + ks * 256);
#pragma unroll
      for (int ntp = 0; ntp < 4; ++ntp) {
        mma_bf16(sacc[2 * ntp], ahi, bfr[ntp][0], bfr[ntp][1]);
        mma_bf16(sacc[2 * ntp + 1], ahi, bfr[ntp][2], bfr[ntp][3]);
        if constexpr (FULL) {
          mma_bf16(gacc[2 * ntp], az, bfr[ntp][0], bfr[ntp][1]);
          mma_bf16(gacc[2 * ntp + 1], az, bfr[ntp][2], bfr[ntp][3]);
        }
      }
#pragma unroll
      for (int ntp = 0; ntp < 4; ++ntp) {
        mma_bf16(sacc[2 * ntp], alo, bfr[ntp][0], bfr[ntp][1]);
        mma_bf16(sacc[2 * ntp + 1], alo, bfr[ntp][2], bfr[ntp][3]);
      }
      // one more column: the group means, so that column 0 collects sum_c (gamma gzn r)[h, c] mean_c  (xh = x r - mean r)
      if constexpr (FULL) {
        const float mu0 = s_rm[32 + g0], mu1 = s_rm[32 + g1];
        mma_bf16(cacc, az, g == 0 ? pack_bf16(mu0, mu0) : 0u, g == 0 ? pack_bf16(mu1, mu1) : 0u);
      }
    }
    // positional term and the constant of a head:  sum_i go[16 h + i] (PE16[t][i] + bc[16 h + i] + (Wc beta)[16 h + i])
    float gsa0 = 0.f, gsa1 = 0.f;
    if constexpr (FULL) {
      const float* wb0 = s_wb + 16 * g + 2 * j;
      const float* wb1 = s_wb + 16 * (g + 8) + 2 * j;
      gsa0 = go0.x * wb0[0] + go0.y * wb0[1] + go2.x * wb0[8] + go2.y * wb0[9];
      gsa1 = go1.x * wb1[0] + go1.y * wb1[1] + go3.x * wb1[8] + go3.y * wb1[9];
      gsa0 += __shfl_xor_sync(0xffffffffu, gsa0, 1);
      gsa0 += __shfl_xor_sync(0xffffffffu, gsa0, 2);
      gsa1 += __shfl_xor_sync(0xffffffffu, gsa1, 1);
      gsa1 += __shfl_xor_sync(0xffffffffu, gsa1, 2);
      if (a.pe != nullptr) {
        uint32_t ago[4] = {pack_bf16(go0.x, go0.y), pack_bf16(go1.x, go1.y), pack_bf16(go2.x, go2.y), pack_bf16(go3.x, go3.y)};
#pragma unroll
        for (int ntp = 0; ntp < 4; ++ntp) {
          uint32_t bp[4];
          ldsm_x4(bp, s32(s_pe) + ((2 * ntp + (mat >> 1)) * 8 + mr) * S::kPeRowB + (mat & 1) * 16);
          mma_bf16(gacc[2 * ntp], ago, bp[0], bp[1]);
          mma_bf16(gacc[2 * ntp + 1], ago, bp[2], bp[3]);
        }
      }
      gsa0 -= __shfl_sync(0xffffffffu, cacc[0], lane & ~3);
      gsa1 -= __shfl_sync(0xffffffffu, cacc[2], lane & ~3);
    }

    // ---- softmax over t (tae.py:831-836), dropout, softmax backward -------------------------------------------------------
    float sa0 = 0.f, sa1 = 0.f, sgs0 = 0.f, sgs1 = 0.f;
    uint32_t gsp[8][2], atp[8][2];  // packed bf16: gs / at of rows g (0) and g + 8 (1), frames 8 nt + 2 j, + 1
    {
      const unsigned long long ov = padm | beyond;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const uint32_t byte = static_cast<uint32_t>(ov >> (8 * nt)) & 0xffu;
        if (byte != 0) {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int t = nt * 8 + 2 * j + e;
            if ((byte >> (2 * j + e)) & 1u) {
              const float v = t >= a.T ? -INFINITY : -1e6f * kLog2e;
              sacc[nt][e] = v, sacc[nt][2 + e] = v;
            }
          }
        }
      }
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(sacc[nt][0], sacc[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(sacc[nt][2], sacc[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      float d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          sacc[nt][e] = ex2(sacc[nt][e] - mx0);
          sacc[nt][2 + e] = ex2(sacc[nt][2 + e] - mx1);
          d0 += sacc[nt][e], d1 += sacc[nt][2 + e];
        }
      }
      d0 += __shfl_xor_sync(0xffffffffu, d0, 1);
      d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
      d1 += __shfl_xor_sync(0xffffffffu, d1, 1);
      d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
      const float inv0 = 1.f / d0, inv1 = 1.f / d1;  // T >= 1: the maximum contributes exp2(0) = 1
      // a = e inv; g_a = g_at keep; at = a keep
      float dot0 = 0.f, dot1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float k0 = ((km0 >> (2 * nt + e)) & 1u) ? keep_scale : 0.f, k1 = ((km1 >> (2 * nt + e)) & 1u) ? keep_scale : 0.f;
          const float a0 = sacc[nt][e] * inv0, a1 = sacc[nt][2 + e] * inv1;
          sacc[nt][e] = a0, sacc[nt][2 + e] = a1;
          const float ga0 = (gacc[nt][e] + gsa0) * k0, ga1 = (gacc[nt][2 + e] + gsa1) * k1;
          gacc[nt][e] = ga0, gacc[nt][2 + e] = ga1;
          dot0 = fmaf(a0, ga0, dot0), dot1 = fmaf(a1, ga1, dot1);
        }
      }
      dot0 += __shfl_xor_sync(0xffffffffu, dot0, 1);
      dot0 += __shfl_xor_sync(0xffffffffu, dot0, 2);
      dot1 += __shfl_xor_sync(0xffffffffu, dot1, 1);
      dot1 += __shfl_xor_sync(0xffffffffu, dot1, 2);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        float gs[4], at[4];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          gs[e] = sacc[nt][e] * (gacc[nt][e] - dot0);
          gs[2 + e] = sacc[nt][2 + e] * (gacc[nt][2 + e] - dot1);
          at[e] = ((km0 >> (2 * nt + e)) & 1u) ? sacc[nt][e] * keep_scale : 0.f;
          at[2 + e] = ((km1 >> (2 * nt + e)) & 1u) ? sacc[nt][2 + e] * keep_scale : 0.f;
          sgs0 += gs[e], sgs1 += gs[2 + e], sa0 += at[e], sa1 += at[2 + e];
          const int t = nt * 8 + 2 * j + e;
          atomicAdd(s_gc + t * GP + g, gs[e]);  // grad_cpos[b][t][h] += gs, summed over the pixels of the tile (fp32: the
          atomicAdd(s_gc + t * GP + g + 8, gs[2 + e]);  // sum over t is analytically zero and must stay at rounding level)
        }
        gsp[nt][0] = pack_bf16(gs[0], gs[1]), gsp[nt][1] = pack_bf16(gs[2], gs[3]);
        atp[nt][0] = pack_bf16(at[0], at[1]), atp[nt][1] = pack_bf16(at[2], at[3]);
      }
      sa0 += __shfl_xor_sync(0xffffffffu, sa0, 1);
      sa0 += __shfl_xor_sync(0xffffffffu, sa0, 2);
      sa1 += __shfl_xor_sync(0xffffffffu, sa1, 1);
      sa1 += __shfl_xor_sync(0xffffffffu, sa1, 2);
      sgs0 += __shfl_xor_sync(0xffffffffu, sgs0, 1);
      sgs0 += __shfl_xor_sync(0xffffffffu, sgs0, 2);
      sgs1 += __shfl_xor_sync(0xffffffffu, sgs1, 1);
      sgs1 += __shfl_xor_sync(0xffffffffu, sgs1, 2);
      if (FULL && j == 0) {
        a.sa_rows[(row0 + p) * kMaxHeads + g] = sa0;
        a.sa_rows[(row0 + p) * kMaxHeads + g + 8] = sa1;
      }
    }

    // ---- au[h, c] = sum_t gs[h, t] xh[t, c], az[h, c] = sum_t at[h, t] xh[t, c], 32 channels at a time; zn rows, grad_U,
    //      direct gamma / beta terms and the two GroupNorm-backward means of every group ----------------------------------
    {
      float* zn_row = FULL ? a.zn_rows + (row0 + p) * kH * C : nullptr;
#pragma unroll 1
      for (int ch = 0; ch < C / 32; ++ch) {
        float au[4][4], azv[4][4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int i = 0; i < 4; ++i) au[nt][i] = 0.f, azv[nt][i] = 0.f;
#pragma unroll
        for (int kg = 0; kg < 4; ++kg) {
          const uint32_t ags[4] = {gsp[2 * kg][0], gsp[2 * kg][1], gsp[2 * kg + 1][0], gsp[2 * kg + 1][1]};
          const uint32_t aat[4] = {atp[2 * kg][0], atp[2 * kg][1], atp[2 * kg + 1][0], atp[2 * kg + 1][1]};
          uint32_t v[2][4];  // (frames 0-7, block 2 cbp), (0-7, 2 cbp + 1), (8-15, 2 cbp), (8-15, 2 cbp + 1)
#pragma unroll
          for (int q = 0; q < 2; ++q) ldsm_x4_trans(v[q], xbase + kg * 16 * FB + (2 * ch + q) * 256);
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            mma_bf16(au[2 * q], ags, v[q][0], v[q][2]);
            mma_bf16(au[2 * q + 1], ags, v[q][1], v[q][3]);
            if constexpr (FULL) {
              mma_bf16(azv[2 * q], aat, v[q][0], v[q][2]);
              mma_bf16(azv[2 * q + 1], aat, v[q][1], v[q][3]);
            }
          }
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const int c = 32 * ch + 8 * nt + 2 * j;
          const int grp = c / CPG;
          const float r = s_rm[grp], m = s_rm[16 + grp];
          const float2 gm = *reinterpret_cast<const float2*>(s_gam + c), bt = *reinterpret_cast<const float2*>(s_gam + C + c);
          // rows g (index 0, 1) and g + 8 (2, 3); channels c (even index) and c + 1 (odd)
          float auv[4], azz[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            auv[i] = fmaf(au[nt][i], r, -m * (i < 2 ? sgs0 : sgs1));
            azz[i] = fmaf(azv[nt][i], r, -m * (i < 2 ? sa0 : sa1));
          }
          if constexpr (FULL) {
            *reinterpret_cast<float2*>(zn_row + g * C + c) = make_float2(fmaf(gm.x, azz[0], bt.x * sa0), fmaf(gm.y, azz[1], bt.y * sa0));
            *reinterpret_cast<float2*>(zn_row + (g + 8) * C + c) =
                make_float2(fmaf(gm.x, azz[2], bt.x * sa1), fmaf(gm.y, azz[3], bt.y * sa1));
          }
          atomicAdd(s_gu + c * GP + g, auv[0]);
          atomicAdd(s_gu + (c + 1) * GP + g, auv[1]);
          atomicAdd(s_gu + c * GP + g + 8, auv[2]);
          atomicAdd(s_gu + (c + 1) * GP + g + 8, auv[3]);
          const uint32_t z0 = FULL ? *reinterpret_cast<const uint32_t*>(gz_ptr + g * S::kGzRow + c * 2) : 0u;
          const uint32_t z1 = FULL ? *reinterpret_cast<const uint32_t*>(gz_ptr + (g + 8) * S::kGzRow + c * 2) : 0u;
          const float zg[4] = {bf16_lo(z0), bf16_hi(z0), bf16_lo(z1), bf16_hi(z1)};
          // score weights of (rows g, g + 8; channels c, c + 1): the A fragment words of k-step c / 16, half (c / 8) & 1
          const float4 uq = s_uf[(c >> 4) * 64 + ((c >> 3) & 1) * 32 + lane];
          float gg0 = zg[0] * azz[0] + zg[2] * azz[2], gg1 = zg[1] * azz[1] + zg[3] * azz[3];  // sum_h gzn az, channels c, c + 1
          float gb0 = zg[0] * sa0 + zg[2] * sa1, gb1 = zg[1] * sa0 + zg[3] * sa1;              // sum_h gzn sa
          float q1 = kLn2 * (uq.x * sgs0 + uq.y * sgs0 + uq.z * sgs1 + uq.w * sgs1);
          float q2 = kLn2 * (uq.x * auv[0] + uq.y * auv[1] + uq.z * auv[2] + uq.w * auv[3]);
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) {
            gg0 += __shfl_xor_sync(0xffffffffu, gg0, o);
            gg1 += __shfl_xor_sync(0xffffffffu, gg1, o);
            gb0 += __shfl_xor_sync(0xffffffffu, gb0, o);
            gb1 += __shfl_xor_sync(0xffffffffu, gb1, o);
            q1 += __shfl_xor_sync(0xffffffffu, q1, o);
            q2 += __shfl_xor_sync(0xffffffffu, q2, o);
          }
          if (FULL && g == 0) {
            atomicAdd(s_ggb + c, gg0);
            atomicAdd(s_ggb + c + 1, gg1);
            atomicAdd(s_ggb + C + c, gb0);
            atomicAdd(s_ggb + C + c + 1, gb1);
          }
          q1 += gm.x * gb0 + gm.y * gb1;
          q2 += gm.x * gg0 + gm.y * gg1;
          q1 += __shfl_xor_sync(0xffffffffu, q1, 1);
          q2 += __shfl_xor_sync(0xffffffffu, q2, 1);
          if (CPG == 8) {
            q1 += __shfl_xor_sync(0xffffffffu, q1, 2);
            q2 += __shfl_xor_sync(0xffffffffu, q2, 2);
          }
          if (lane == 0 || (CPG == 4 && lane == 2)) {
            s_m12[grp] = q1 * inv_n_all;
            s_m12[16 + grp] = q2 * inv_n_all;
          }
        }
      }
    }
    __syncwarp();

    // ---- g_xh[t, c] = sum_h gs[h, t] U[h, c] + gamma_c sum_h at[h, t] gzn[h, c]; GroupNorm backward; grad_x replaces x ------
    {
      uint32_t agsT[4][4], aatT[4][4];  // A fragments [t][h]: (t g, h 2j), (t g + 8, h 2j), (t g, h 2j + 8), (t g + 8, h 2j + 8)
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        agsT[mt][0] = movmatrix_trans(gsp[2 * mt][0]);
        agsT[mt][1] = movmatrix_trans(gsp[2 * mt + 1][0]);
        agsT[mt][2] = movmatrix_trans(gsp[2 * mt][1]);
        agsT[mt][3] = movmatrix_trans(gsp[2 * mt + 1][1]);
        aatT[mt][0] = movmatrix_trans(atp[2 * mt][0]);
        aatT[mt][1] = movmatrix_trans(atp[2 * mt + 1][0]);
        aatT[mt][2] = movmatrix_trans(atp[2 * mt][1]);
        aatT[mt][3] = movmatrix_trans(atp[2 * mt + 1][1]);
      }
      unsigned char* xw = slab_ptr + g * FB + ((p ^ g) << 4) + 4 * j;  // (t = g, block 0): + 8 frames = same slot
#pragma unroll 1
      for (int np = 0; np < C / 16; ++np) {
        float accu[4][2][4], accz[4][2][4];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
          for (int n2 = 0; n2 < 2; ++n2)
#pragma unroll
            for (int i = 0; i < 4; ++i) accu[mt][n2][i] = 0.f, accz[mt][n2][i] = 0.f;
        const uint2 ub0 = s_ub[(2 * np) * 32 + lane], ub1 = s_ub[(2 * np + 1) * 32 + lane];
        uint32_t zb[4];  // gzn as B[k = h][n = c]: (h 0-7, block 2 np), (h 8-15, 2 np), (h 0-7, 2 np + 1), (h 8-15, 2 np + 1)
        if constexpr (FULL) ldsm_x4_trans(zb, gz_frag + np * 32);
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          mma_bf16(accu[mt][0], agsT[mt], ub0.x, ub0.y);
          mma_bf16(accu[mt][1], agsT[mt], ub1.x, ub1.y);
          if constexpr (FULL) {
            mma_bf16(accz[mt][0], aatT[mt], zb[0], zb[1]);
            mma_bf16(accz[mt][1], aatT[mt], zb[2], zb[3]);
          }
        }
#pragma unroll
        for (int n2 = 0; n2 < 2; ++n2) {
          const int c = 16 * np + 8 * n2 + 2 * j;
          const int grp = c / CPG;
          const float r = s_rm[grp], m = s_rm[16 + grp], m1 = s_m12[grp], m2 = s_m12[16 + grp];
          const float2 gm = *reinterpret_cast<const float2*>(s_gam + c);
#pragma unroll
          for (int mt = 0; mt < 4; ++mt) {
            if (16 * mt >= a.T) continue;  // boxes that are never loaded stay zero
#pragma unroll
            for (int rh = 0; rh < 2; ++rh) {
              uint32_t* ptr = reinterpret_cast<uint32_t*>(xw + (16 * mt + 8 * rh) * FB + (2 * np + n2) * 128);
              const uint32_t xv = *ptr;
              const float xh0 = fmaf(bf16_lo(xv), r, -m), xh1 = fmaf(bf16_hi(xv), r, -m);
              const float v0 = fmaf(gm.x, accz[mt][n2][2 * rh], accu[mt][n2][2 * rh]);
              const float v1 = fmaf(gm.y, accz[mt][n2][2 * rh + 1], accu[mt][n2][2 * rh + 1]);
              *ptr = pack_bf16(r * (v0 - m1 - xh0 * m2), r * (v1 - m1 - xh1 * m2));
            }
          }
        }
      }
    }
    __syncthreads();  // grad_x of every pixel is in the slab; the tile's grad_cpos sums are complete

    // ---- back to [t][c][8 px], grad_cpos of the tile, stores ---------------------------------------------------------------
    {
      const int q4 = warp % NQ, f0 = warp / NQ;
      const uint32_t blk0 = slab + q4 * 512 + mat * 128;
#pragma unroll
      for (int grp = 0; grp < 4; ++grp) {
        if (16 * grp >= a.T) continue;
        uint32_t v[FPG][4];
#pragma unroll
        for (int q = 0; q < FPG; ++q) {
          const int t = 16 * grp + f0 + TSTEP * q;
          ldsm_x4_trans(v[q], blk0 + t * FB + ((mr ^ (t & 7)) << 4));
        }
#pragma unroll
        for (int q = 0; q < FPG; ++q) stsm_x4(blk0 + (16 * grp + f0 + TSTEP * q) * FB + mr * 16, v[q]);
      }
      for (int i = tid; i < a.T * kMaxHeads; i += 256) {
        const int t = i >> 4, h = i & 15;
        atomicAdd(a.g_cpos + (static_cast<size_t>(b) * a.T + t) * kMaxHeads + h, s_gc[t * GP + h]);
      }
    }
    fence_proxy_async();  // generic stores above, bulk-copy reads below
    __syncthreads();
    for (int i = tid; i < kTP * GP; i += 256) s_gc[i] = 0.f;  // next adds are behind the next tile's first barrier
    if (tid == 0) {
#pragma unroll
      for (int grp = 0; grp < 4; ++grp)
        if (16 * grp < a.T) tma_store_4d(&map_gx, pix0, 0, 16 * grp, b, slab + 16 * grp * FB);
      tma_store_commit();
    }
  }

  // ---- sums over this CTA's pixels ------------------------------------------------------------------------------------
  __syncthreads();
  for (int i = tid; i < C * kMaxHeads; i += 256) {
    const int c = i >> 4, h = i & 15;
    atomicAdd(a.g_u + i, s_gu[c * GP + h]);
  }
  if constexpr (FULL)
    for (int i = tid; i < C; i += 256) {
      atomicAdd(a.g_gamma + i, s_ggb[i]);
      atomicAdd(a.g_beta + i, s_ggb[C + i]);
    }
  if (tid == 0) tma_store_wait();  // the last stores have left shared memory
}

template <int C, bool FULL>
int bt_launch(const CUtensorMap& map_x, const CUtensorMap& map_gx, const BwdTcArgs& a, cudaStream_t stream, const char* name) {
  using S = BtSmem<C>;
  C2S_SMEM_ATTR((ltae_bwd_tc_kernel<C, FULL>), S::kTotal);
  const int sms = sm_count();
  const int grid = a.n_tiles < sms ? a.n_tiles : sms;
  ltae_bwd_tc_kernel<C, FULL><<<static_cast<unsigned>(grid), 256, S::kTotal, stream>>>(map_x, map_gx, a);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

}  // namespace

bool ltae_bwd_tc_eligible(const c2s_ltae_desc& d, const void* x, const c2s_ltae_bwd_io& io) {
  const bool attn_only = (d.flags & C2S_LTAE_ATTN_ONLY) != 0;
  if (attn_only && io.grad_attn == nullptr) return false;
  if (d.dtype != C2S_BF16 || d.n_head != kH || d.d_model != kD || !d.has_inconv) return false;
  if (d.C != 64 && d.C != 128) return false;
  if (d.T > kTP || d.T < 1 || (d.H * d.W) % kPix != 0) return false;
  if (d.pe_mode == C2S_PE_SINUSOID_LINEAR) return false;  // table differs per head chunk
  if (io.grad_pe != nullptr) return false;                // learnable tables: the general kernel forms grad_pe
  if (reinterpret_cast<uintptr_t>(x) % 16 != 0 || reinterpret_cast<uintptr_t>(io.grad_x) % 16 != 0) return false;
  if (!attn_only && (reinterpret_cast<uintptr_t>(io.grad_o) % 8 != 0 || reinterpret_cast<uintptr_t>(io.zn_rows) % 8 != 0)) return false;
  return true;
}

int ltae_bwd_tc_launch(const c2s_ltae_desc& d, const BwdTcArgs& a0, void* grad_x, cudaStream_t stream) {
  const int C = d.C, hw = d.H * d.W;
  // x / grad_x as [B][T][C][hw] bf16; box = 8 pixels x C channels x 16 frames of one sample: frames t >= T are zero-filled
  // by the loads and clipped by the stores
  CUtensorMap maps[2];
  const void* bases[2] = {a0.x, grad_x};
  const char* what[2] = {"backward features", "backward feature gradients"};
  const cuuint64_t dims[4] = {static_cast<cuuint64_t>(hw), static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(d.T),
                              static_cast<cuuint64_t>(d.B)};
  const cuuint64_t strides[3] = {static_cast<cuuint64_t>(hw) * 2, static_cast<cuuint64_t>(C) * hw * 2,
                                 static_cast<cuuint64_t>(d.T) * C * hw * 2};
  const cuuint32_t box[4] = {kPix, static_cast<cuuint32_t>(C), 16, 1};
  for (int i = 0; i < 2; ++i) {
    const int status = encode_tensor_map(&maps[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, bases[i], dims, strides, box,
                                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, what[i]);
    if (status != C2S_OK) return status;
  }
  BwdTcArgs a = a0;
  a.tiles_per_b = hw / kPix;
  if (static_cast<long long>(d.B) * a.tiles_per_b > 0x3fffffffll) C2S_UNSUPPORTED("c2s_ltae_backward: too many pixel tiles");
  a.n_tiles = d.B * a.tiles_per_b;
  if (a.g_o == nullptr) {  // attention-only encoder
    if (C == 128) return bt_launch<128, false>(maps[0], maps[1], a, stream, "ltae_backward<tc,C=128,attention>");
    return bt_launch<64, false>(maps[0], maps[1], a, stream, "ltae_backward<tc,C=64,attention>");
  }
  if (C == 128) return bt_launch<128, true>(maps[0], maps[1], a, stream, "ltae_backward<tc,C=128>");
  return bt_launch<64, true>(maps[0], maps[1], a, stream, "ltae_backward<tc,C=64>");
}

}  // namespace c2s
