// L-TAE forward, team-pipelined slab kernel (bf16 I/O, 16 heads, d_model 256, T <= 64, H*W % 8 == 0), sm_100a.
// Reference: LTAE.forward, src/backbones/tae.py:451-504 (Time-Unet call site: src/backbones/timeunet.py:178-180).
//
// Same arithmetic as c2s_ltae_fa.cu (collapsed in-projection, hi/lo 16-bit operand splits, fp32 accumulation) with
// another execution structure:
//   * one persistent CTA of 16 warps per SM holds TWO teams of 8 warps (C = 64); a team owns a slab (8 pixels x 64
//     frames x C channels), its own epilogue scratch and its own stream of tiles.  Teams never synchronise with each
//     other: while one waits for its slab or sits in an ALU phase the other one feeds the tensor pipe;
//   * inside a team one warp owns one pixel from the scores to the normalised value sums; the only team-wide
//     barriers are the one behind the cooperative transposition and three around the two rounds of the per-head
//     in-projection (which batches the 8 pixels as the N dimension of mma.sync);
//   * the epilogue (GroupNorm affine, in-projection, stores) works in its own shared memory, so the slab is handed back
//     to the copy engine as soon as the LAST warp of the team is done with the value products: the next tile's TMA
//     boxes are issued by that warp and fly during the whole epilogue (c2s_ltae_fa.cu reloads after the epilogue);
//   * frames that are not read are not zero-filled: their scores are overwritten (tae.py:831), whole 16-frame blocks
//     without a live frame are skipped, and a probability that is exactly 0 meets stale but finite data;
//   * the softmax normalisation is deferred: the value sums use exp2(s - max) and are scaled by 1 / sum with the
//     GroupNorm affine.
// C = 128 (U-TAE): the slab is 128 KB, so there is ONE team of 16 warps, two warps per pixel: the scores and the softmax
// are split over the frames (32 each; maximum and sum meet through shared memory), the value products over the
// CHANNELS (64 each) -- the pair exchanges its probabilities (16 registers per lane) instead of 64 registers of partial
// sums -- and the in-projection of a head is split over k between the two warps of a pair.  The attention (always
// consumed by U-TAE's aggregations) is staged in the epilogue scratch and stored as 32-byte segments.
// Serves what c2s_ltae_team_eligible says (no dropout mask, not attention-only; C = 64 only without the attention
// store); everything else goes to c2s_ltae_fa.cu.
#include <type_traits>

#include "c2s_ltae_fa.cuh"

namespace c2s {
namespace {

template <int C>
struct TeamSmem {
  static constexpr int WPP = C / 64;                 // warps per pixel
  static constexpr int TEAMS = 2 / WPP;              // teams per CTA
  static constexpr int TW = kPix * WPP;              // warps per team
  static constexpr int kFB = C * 16;                 // one frame: [C][8 px] bf16
  static constexpr int kSlab = kTP * kFB;
  static constexpr int HR = 8;                       // heads per in-projection round
  static constexpr int kZnRow = (C + 8) * 2;         // one head row of zn (fp16), bytes
  static constexpr int kZnPix = 2 * HR * kZnRow + 16;  // per pixel: HR hi rows, HR lo rows; pixel blocks 4 banks apart
  static_assert((kZnPix / 4) % 32 == 4, "pixel blocks of zn must sit 4 banks apart");
  static constexpr int kSub = (C == 64) ? 2 : 1;     // GroupNorm groups per 8-channel block
  static constexpr int kOstRows = 8 * 80;            // staging of 8 o-row pieces per projecting warp (80-byte pitch)
  static constexpr int kOst = kOstRows + (WPP == 2 ? 512 : 0);  // + the partner's partial in-projection (WPP = 2)
  static constexpr int kPartW = 72;                  // float2 per warp: [8 px][4 blocks][kSub] + 8 (bank spread)
  static constexpr int kPaPix = 2 * kH * 8 + 4;      // floats per pixel of the positional sums (+4: bank spread)
  // epilogue scratch: zn tiles of one round; with two warps per pixel also the probability exchange
  // ([TW][16 registers][32 lanes]), the partial in-projections and the attention staging ([8 px][kAsP] floats)
  static constexpr int kEx = (WPP == 2) ? TW * 16 * 128 : 0;
  static constexpr int kStage = (WPP == 2) ? kPix * kAsP * 4 : 0;
  static constexpr int kZnAll = kPix * kZnPix;
  static constexpr int kScratch = kZnAll > kEx ? (kZnAll > kStage ? kZnAll : kStage) : (kEx > kStage ? kEx : kStage);
  // ---- per team ----
  static constexpr int oSlab = 0;
  static constexpr int oZn = oSlab + kSlab;
  static constexpr int oPart = oZn + kScratch;                      // float2 [TW][8 px][4][kSub] statistics partials
  static constexpr int oPa = oPart + TW * kPartW * 8;               // float [8 px][i / 8][16 h][i % 8]
  static constexpr int oRm = oPa + kPix * kPaPix * 4;               // float [TW][2][16]: rstd, mean * rstd per group
  static constexpr int oOst = oRm + TW * 2 * 16 * 4;
  static constexpr int oRed = oOst + kPix * kOst;                   // float [8 px][2 warps][max | sum][16] (WPP = 2)
  static constexpr int oSa = oRed + (WPP == 2 ? kPix * 2 * 2 * kH * 4 : 0);    // float [8 px][16]: sum_t of the returned attention
  static constexpr int oCpos = oSa + (WPP == 2 ? kPix * kH * 4 : 0);  // float [16][kAP]
  static constexpr int oPeHi = oCpos + kH * kAP * 4;                // bf16 [16][kPeRow]
  static constexpr int oPeLo = oPeHi + 16 * kPeRow * 2;
  static constexpr int oBar = oPeLo + 16 * kPeRow * 2;              // 4 mbarriers + release counter
  static constexpr int kTeam = ((oBar + 64) + 1023) & ~1023;
  // ---- per CTA ----
  static constexpr int oUf = TEAMS * kTeam;                         // float4 [C/16][2][32] score weights
  static constexpr int oGam = oUf + C * 64;                         // float gamma[C], beta[C]
  static constexpr int oBc = oGam + 2 * C * 4;                      // float inconv.bias[256]
  static constexpr int kTotal = oBc + kD * 4;
  static_assert(kTotal <= 232448, "shared memory budget");
};

// Phase timing for development (build with -DC2S_TEAM_TIMING): warp `C2S_TEAM_TIMING` of team 0 of CTA 0 adds the cycles
// since the start of the tile at every checkpoint into a.dbg[k]; a.dbg[0] counts tiles.  tools/experiments/team_timing.py
#ifdef C2S_TEAM_TIMING
#define TEAM_DBG(k)                                                                                          \
  if (a.dbg != nullptr && warp == (C2S_TEAM_TIMING) && lane == 0 && blockIdx.x == 0)                          \
  a.dbg[k] += static_cast<unsigned long long>(clock64() - dbg_t0)
#else
#define TEAM_DBG(k)
#endif

// global loads that must be ISSUED where they are written (the compiler sinks plain loads to their first use, which
// puts a full L2 latency on the critical path)
__device__ __forceinline__ unsigned long long ldg_u64_now(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ldg_u16_now(const void* p) {
  uint16_t v;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
  return v;
}

__device__ __forceinline__ void team_bar(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// DROP: training-mode dropout on the returned attention (a second instantiation: the eval kernel carries none of it)
template <int C, bool DROP>
__global__ void __launch_bounds__(512, 1)
ltae_team_kernel(const __grid_constant__ CUtensorMap map16, const __grid_constant__ CUtensorMap map4,
                 const __grid_constant__ CUtensorMap map1, const FaArgs a) {
  using S = TeamSmem<C>;
  constexpr int WPP = S::WPP;              // warps per pixel
  constexpr int TW = S::TW, TT = 32 * TW;  // warps / threads of a team
  constexpr int CPG = C / kH;              // channels per GroupNorm group
  constexpr int KS = C / 16;               // k-steps over channels
  constexpr int NQ = C / 32;               // 4-block quads per frame (one ldmatrix.x4 each)
  constexpr int TSTEP = TW / NQ;           // frames between two items of a warp in the transposition pass
  constexpr int FPG = 16 / TSTEP;          // frames of a 16-frame barrier group per warp
  constexpr int FB = S::kFB;
  constexpr int SUB = S::kSub;
  constexpr int HR = S::HR;
  constexpr int FPW = kTP / WPP;           // frames per warp in the scores and the softmax
  constexpr int FN = FPW / 8;              // score n-tiles per warp
  constexpr int CW = C / WPP;              // channels per warp in the value products
  extern __shared__ __align__(1024) unsigned char smem[];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int team = warp / TW, tw = warp % TW, ttid = tid - team * TT;
  const int p = tw / WPP, half = tw % WPP;       // pixel of this warp; which frames (scores) / channels (values) it owns
  const int j = lane & 3, g = lane >> 2;         // fragment coordinates
  const int mat = lane >> 3, mr = lane & 7;      // ldmatrix: this lane supplies row mr of matrix mat
  const int bar_id = 1 + team;

  unsigned char* tb = smem + team * S::kTeam;
  unsigned char* slab_ptr = tb + S::oSlab;
  const uint32_t slab = s32(slab_ptr);
  unsigned char* zn_ptr = tb + S::oZn;
  float2* s_part = reinterpret_cast<float2*>(tb + S::oPart);
  float* s_pa = reinterpret_cast<float*>(tb + S::oPa);
  float* s_rm = reinterpret_cast<float*>(tb + S::oRm) + tw * 32;  // this warp's copy of rstd[16], mean * rstd[16]
  unsigned char* ost = tb + S::oOst + p * S::kOst;
  float* s_red = reinterpret_cast<float*>(tb + S::oRed);
  float* s_sa = reinterpret_cast<float*>(tb + S::oSa);
  const uint32_t pair_bar = 3 + p;               // named barrier of the two warps of a pixel (WPP = 2)
  float* s_cpos = reinterpret_cast<float*>(tb + S::oCpos);
  __nv_bfloat16* s_pe_hi = reinterpret_cast<__nv_bfloat16*>(tb + S::oPeHi);
  __nv_bfloat16* s_pe_lo = reinterpret_cast<__nv_bfloat16*>(tb + S::oPeLo);
  const uint32_t bars = s32(tb + S::oBar);
  int* s_cnt = reinterpret_cast<int*>(tb + S::oBar + 32);
  const float4* s_uf = reinterpret_cast<const float4*>(smem + S::oUf);
  const float* s_gam = reinterpret_cast<const float*>(smem + S::oGam);
  const float* s_bc = reinterpret_cast<const float*>(smem + S::oBc);

  // ---- set-up ------------------------------------------------------------------------------------------------------
  if (ttid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(bars + 8 * i, 1);
    *s_cnt = 0;
    fence_mbarrier_init();
  }
  for (int i = ttid; i < S::kSlab / 16; i += TT) reinterpret_cast<uint4*>(slab_ptr)[i] = make_uint4(0, 0, 0, 0);  // never NaN
  for (int i = ttid; i < 2 * 16 * kPeRow / 2; i += TT) reinterpret_cast<uint32_t*>(s_pe_hi)[i] = 0u;  // hi and lo tables
  {
    float4* uf = reinterpret_cast<float4*>(smem + S::oUf);
    for (int i = tid; i < KS * 64; i += 512) {  // source order [ks][lane][2] -> [ks][2][lane]
      const int ks = i >> 6, e = i & 63;
      uf[ks * 64 + (e & 1) * 32 + (e >> 1)] = __ldg(reinterpret_cast<const float4*>(a.ufrag) + i);
    }
    float* gam = reinterpret_cast<float*>(smem + S::oGam);
    for (int i = tid; i < C; i += 512) gam[i] = __ldg(a.gamma + i), gam[C + i] = __ldg(a.beta + i);
    float* bcs = reinterpret_cast<float*>(smem + S::oBc);
    for (int i = tid; i < kD; i += 512) bcs[i] = __ldg(a.bc + i);
  }
  const float inv_sc = __ldg(a.wscale + 1);
  const float inv_n_all = 1.f / (static_cast<float>(a.T) * CPG);
  fence_proxy_async();  // generic zero fill above, bulk-copy writes below
  __syncthreads();

  // one warp issues the boxes of a tile: lanes 0..15 = quads of frames, boxes of 16 / 4 / 1 frames by the live mask
  auto issue_tile = [&](int tile, unsigned long long live) {
    const int b = tile / a.tiles_per_b;
    const int pix0 = (tile - b * a.tiles_per_b) * kPix;
    if (lane < 16) {
      const int grp = lane >> 2, t4 = 4 * lane;
      const uint32_t m16 = static_cast<uint32_t>(live >> (16 * grp)) & 0xffffu;
      const uint32_t m4 = static_cast<uint32_t>(live >> t4) & 0xfu;
      const uint32_t bar = bars + 8 * grp;
      if ((lane & 3) == 0) mbar_expect_tx(bar, static_cast<uint32_t>(__popc(m16)) * FB);
      if (m16 == 0xffffu) {
        if ((lane & 3) == 0) tma_load_3d(slab + t4 * FB, &map16, pix0, 0, b * a.T + t4, bar);
      } else if (m4 == 0xfu) {
        tma_load_3d(slab + t4 * FB, &map4, pix0, 0, b * a.T + t4, bar);
      } else {
        for (int e = 0; e < 4; ++e)
          if ((m4 >> e) & 1u) tma_load_3d(slab + (t4 + e) * FB, &map1, pix0, 0, b * a.T + t4 + e, bar);
      }
    }
  };

#ifdef C2S_TEAM_ONLY0  // experiment: one team per CTA, the other one leaves (how much do the teams slow each other down?)
  if (team != 0) return;
  const int first = blockIdx.x, stride = gridDim.x;
#else
  const int first = blockIdx.x * S::TEAMS + team, stride = gridDim.x * S::TEAMS;
#endif
  unsigned long long live = 0, padm = 0;
  if (first < a.n_tiles) {
    const int b0 = first / a.tiles_per_b;
    live = __ldg(a.masks + 2 * b0), padm = __ldg(a.masks + 2 * b0 + 1);
    if (tw == 0) issue_tile(first, live);
  }
  const unsigned long long beyond = (a.T >= 64) ? 0ull : (~0ull << a.T);  // frames t >= T
  int cur_b = -1;
  // pivots of the shifted GroupNorm sums: first channel of the lane's group in the first live frame of the tile, read
  // from global memory one tile ahead (4 two-byte loads per lane, in flight during the previous epilogue)
  uint32_t pvn[4] = {0u, 0u, 0u, 0u};  // raw bf16 bits
  auto load_pivots = [&](int tile, unsigned long long lv) {
#pragma unroll
    for (int i = 0; i < 4; ++i) pvn[i] = 0u;
    if (lv == 0) return;
    const int bb = tile / a.tiles_per_b, px0 = (tile - bb * a.tiles_per_b) * kPix;
    const int tf = __ffsll(static_cast<long long>(lv)) - 1;
    const __nv_bfloat16* xf = a.x + (static_cast<size_t>(bb) * a.T + tf) * C * a.hw + px0 + g;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c0 = (4 * (tw % NQ) + i) * 8 + (CPG == 4 ? 4 * (j >> 1) : 0);
      pvn[i] = ldg_u16_now(xf + static_cast<size_t>(c0) * a.hw);
    }
  };
  if (first < a.n_tiles) load_pivots(first, live);

#pragma unroll 1
  for (int k = 0;; ++k) {
    const int tile = first + k * stride;
    if (tile >= a.n_tiles) break;
    const uint32_t par = static_cast<uint32_t>(k) & 1u;
#ifdef C2S_TEAM_TIMING
    const long long dbg_t0 = clock64();
    if (a.dbg != nullptr && warp == (C2S_TEAM_TIMING) && lane == 0 && blockIdx.x == 0) a.dbg[0] += 1;
#endif
    const int n_live = __popcll(live);
    const int b = tile / a.tiles_per_b;
    const int pix0 = (tile - b * a.tiles_per_b) * kPix;
    // blocks of 16 frames that hold a live frame (uniform); all four in the common case
    const uint32_t blk = (((live & 0xffffull) != 0) ? 1u : 0u) | (((live >> 16 & 0xffffull) != 0) ? 2u : 0u) |
                         (((live >> 32 & 0xffffull) != 0) ? 4u : 0u) | (((live >> 48 & 0xffffull) != 0) ? 8u : 0u);

    // ---- per-sample constants of a new sample: the loads go out now and land in shared memory before the barrier ----
    const bool new_b = b != cur_b;  // team-uniform
    cur_b = b;
    float cst[kTP * 16 / TT], pst[kTP * 16 / TT];
    if (new_b) {
#pragma unroll
      for (int q = 0; q < kTP * 16 / TT; ++q) {
        const int i = ttid + q * TT, t = i >> 4, h = i & 15;
        cst[q] = t < a.T ? __ldg(a.cpos + (static_cast<size_t>(b) * a.T + t) * kMaxHeads + h) : 0.f;
        pst[q] = (a.pe != nullptr && t < a.T) ? __ldg(a.pe + (static_cast<size_t>(b) * a.T + t) * kD + h) : 0.f;
      }
    }

    // ---- transposition in place + GroupNorm sums (tae.py:461; all T frames count, frames that are not read as zeros)
    // warp tw owns quad tw % NQ of the frames tw / NQ + k TSTEP; shifted sums, pivot = first live frame
    {
      const int t_first = n_live > 0 ? __ffsll(static_cast<long long>(live)) - 1 : 0;
      const int q4 = tw % NQ, f0 = tw / NQ;
      const uint32_t blk0 = slab + q4 * 512 + mat * 128;
      unsigned long long s1p[4], s2p[4];
      float npv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) s1p[i] = 0ull, s2p[i] = 0ull, npv[i] = -__uint_as_float(pvn[i] << 16);
#pragma unroll
      for (int grp = 0; grp < 4; ++grp) {
        const uint32_t gl = static_cast<uint32_t>(live >> (16 * grp)) & 0xffffu;  // team-uniform
        if (gl == 0) continue;
        mbar_wait(bars + 8 * grp, par);
        uint32_t v[FPG][4];
#pragma unroll
        for (int q = 0; q < FPG; ++q)
          if ((gl >> (f0 + TSTEP * q)) & 1u) ldsm_x4_trans(v[q], blk0 + (16 * grp + f0 + TSTEP * q) * FB + mr * 16);
#pragma unroll
        for (int q = 0; q < FPG; ++q) {
          if (!((gl >> (f0 + TSTEP * q)) & 1u)) continue;
          const int t = 16 * grp + f0 + TSTEP * q;
          stsm_x4(blk0 + t * FB + ((mr ^ (t & 7)) << 4), v[q]);  // row = pixel, 8 channels; slot pixel ^ (t & 7)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const unsigned long long d = bf16x2_plus_f32(v[q][i], npv[i]);
            s1p[i] = add_f32x2(s1p[i], d);
            s2p[i] = fma_f32x2(d, d, s2p[i]);
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
        if (writer) s_part[tw * S::kPartW + (g * 4 + i) * SUB + (CPG == 4 ? (j >> 1) : 0)] = make_float2(s1, s2);
      }
      TEAM_DBG(1);  // transposition + partial sums done
      if (new_b) {
#pragma unroll
        for (int q = 0; q < kTP * 16 / TT; ++q) {
          const int i = ttid + q * TT, t = i >> 4, h = i & 15;
          s_cpos[h * kAP + t] = cst[q] * kLog2e;
          const __nv_bfloat16 hi = __float2bfloat16_rn(pst[q]);
          s_pe_hi[h * kPeRow + t] = hi;
          s_pe_lo[h * kPeRow + t] = __float2bfloat16_rn(pst[q] - __bfloat162float(hi));
        }
      }
      team_bar(bar_id, TT);
      TEAM_DBG(2);  // barrier behind the transposition
      // every warp finalises the 16 groups of ITS pixel: lane = group
      if (lane < kH) {
        const int grp = lane;
        const int cb = (CPG == 8) ? grp : (grp >> 1), sub = (CPG == 8) ? 0 : (grp & 1);
        const int qq = cb >> 2, ii = cb & 3;
        float t1 = 0.f, t2 = 0.f;
#pragma unroll
        for (int m = 0; m < TSTEP; ++m) {
          const float2 v = s_part[(qq + NQ * m) * S::kPartW + (p * 4 + ii) * SUB + sub];
          t1 += v.x, t2 += v.y;
        }
        float pv = 0.f;
        if (n_live > 0) {  // the pivot of (group, pixel): first channel of the group in the first live frame, transposed layout
          const int c0 = grp * CPG;
          pv = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(
              slab_ptr + t_first * FB + (c0 >> 3) * 128 + ((p ^ (t_first & 7)) << 4) + (c0 & 7) * 2));
        }
        const float n_skip = static_cast<float>((a.T - n_live) * CPG);  // frames known to be zero
        t1 -= n_skip * pv;
        t2 = fmaf(n_skip * pv, pv, t2);
        const float m = t1 * inv_n_all;
        float var = fmaf(t2, inv_n_all, -m * m);
        var = var < 0.f ? 0.f : var;
        const float rstd = rsqrtf(var + a.gn_eps);
        s_rm[grp] = rstd;
        s_rm[16 + grp] = (m + pv) * rstd;
      }
      __syncwarp();
    }

    // the masks of this team's next tile (consumed after the value products)
    unsigned long long nlive = 0, npad = 0;
    const int nxt = tile + stride;
    if (nxt < a.n_tiles) {
      const int bn = nxt / a.tiles_per_b;
      nlive = ldg_u64_now(a.masks + 2 * bn), npad = ldg_u64_now(a.masks + 2 * bn + 1);
    }

    TEAM_DBG(3);  // statistics
    // ---- scores S^T[h, t] of pixel p, frames FPW half .. FPW half + FPW - 1 ------------------------- tae.py:827-831
    const uint32_t wblk = (blk >> (FN / 2 * half)) & ((1u << (FN / 2)) - 1u);  // this warp's 16-frame blocks
    float sacc[FN][4];
#pragma unroll
    for (int nt = 0; nt < FN; ++nt) {
      const int t = (FN * half + nt) * 8 + 2 * j;
      const float2 c0 = *reinterpret_cast<const float2*>(s_cpos + g * kAP + t);
      const float2 c1 = *reinterpret_cast<const float2*>(s_cpos + (g + 8) * kAP + t);
      sacc[nt][0] = c0.x, sacc[nt][1] = c0.y, sacc[nt][2] = c1.x, sacc[nt][3] = c1.y;
    }
    const uint32_t xbase = slab + ((p ^ mr) << 4) + (mat & 1) * 128 + ((mat >> 1) * 8 + mr) * FB;
    const uint32_t xrow = xbase + FPW * half * FB;  // first frame of this warp's scores
    auto scores = [&](auto all_) {
      constexpr bool ALL = decltype(all_)::value;
#pragma unroll 2
      for (int ks = 0; ks < KS; ++ks) {
        const float4 u0 = s_uf[ks * 64 + lane], u1 = s_uf[ks * 64 + 32 + lane];
        const int c_lo = ks * 16 + 2 * j;
        const float r0 = s_rm[c_lo / CPG], r1 = s_rm[(c_lo + 8) / CPG];
        uint32_t ahi[4], alo[4];
        split_bf16(u0.x * r0, u0.y * r0, ahi[0], alo[0]);  // (row g,     k 2j, 2j+1)
        split_bf16(u0.z * r0, u0.w * r0, ahi[1], alo[1]);  // (row g + 8, k 2j, 2j+1)
        split_bf16(u1.x * r1, u1.y * r1, ahi[2], alo[2]);  // (row g,     k 2j+8, 2j+9)
        split_bf16(u1.z * r1, u1.w * r1, ahi[3], alo[3]);  // (row g + 8, k 2j+8, 2j+9)
        uint32_t bfr[FN / 2][4];  // (block 2 ntp, channels 16 ks..+7), (.., +8..15), (block 2 ntp + 1, ..), (..)
#pragma unroll
        for (int ntp = 0; ntp < FN / 2; ++ntp)
          if (ALL || ((wblk >> ntp) & 1u)) ldsm_x4(bfr[ntp], xrow + ntp * 16 * FB + ks * 256);
#pragma unroll
        for (int ntp = 0; ntp < FN / 2; ++ntp) {
          if (!ALL && !((wblk >> ntp) & 1u)) continue;
          mma_bf16(sacc[2 * ntp], ahi, bfr[ntp][0], bfr[ntp][1]);
          mma_bf16(sacc[2 * ntp + 1], ahi, bfr[ntp][2], bfr[ntp][3]);
        }
#pragma unroll
        for (int ntp = 0; ntp < FN / 2; ++ntp) {
          if (!ALL && !((wblk >> ntp) & 1u)) continue;
          mma_bf16(sacc[2 * ntp], alo, bfr[ntp][0], bfr[ntp][1]);
          mma_bf16(sacc[2 * ntp + 1], alo, bfr[ntp][2], bfr[ntp][3]);
        }
      }
    };
    if (wblk == (1u << (FN / 2)) - 1u) scores(std::true_type{});
    else scores(std::false_type{});

    TEAM_DBG(4);  // scores
    // ---- softmax over t for rows h = g and g + 8 (base 2; normalisation deferred) ------------------- tae.py:831-836
    float inv0, inv1;
    float sa0 = 1.f, sa1 = 1.f;  // sum_t of the returned attention of rows g / g + 8: 1 unless dropout acts on it (tae.py:837)
    {
      // padded frames and frames behind T: their scores are REPLACED (masked_fill, tae.py:831), whatever the slab holds
      const unsigned long long ov = (padm | beyond) >> (FPW * half);
#pragma unroll
      for (int nt = 0; nt < FN; ++nt) {
        const uint32_t byte = static_cast<uint32_t>(ov >> (8 * nt)) & 0xffu;  // uniform
        if (byte != 0) {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int t = FPW * half + nt * 8 + 2 * j + e;
            if ((byte >> (2 * j + e)) & 1u) {
              const float v = t >= a.T ? -INFINITY : -1e6f * kLog2e;
              sacc[nt][e] = v, sacc[nt][2 + e] = v;
            }
          }
        }
      }
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < FN; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(sacc[nt][0], sacc[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(sacc[nt][2], sacc[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      float* red = s_red + (p * 2 + half) * 2 * kH;
      const float* red_other = s_red + (p * 2 + (half ^ 1)) * 2 * kH;
      if constexpr (WPP == 2) {
        if (j == 0) red[g] = mx0, red[g + 8] = mx1;
        team_bar(pair_bar, 64);
        mx0 = fmaxf(mx0, red_other[g]);  // T >= 1: at least one side is finite
        mx1 = fmaxf(mx1, red_other[g + 8]);
      }
      float d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < FN; ++nt) {
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
      if constexpr (WPP == 2) {  // the sum is formed in the same order by both warps
        if (j == 0) red[kH + g] = d0, red[kH + g + 8] = d1;
        team_bar(pair_bar, 64);
        const float lo0 = half ? red_other[kH + g] : d0, hi0 = half ? d0 : red_other[kH + g];
        const float lo1 = half ? red_other[kH + g + 8] : d1, hi1 = half ? d1 : red_other[kH + g + 8];
        d0 = lo0 + hi0, d1 = lo1 + hi1;
      }
      inv0 = 1.f / d0, inv1 = 1.f / d1;  // T >= 1: the maximum contributes exp2(0) = 1
      if constexpr (DROP) {  // training: the returned attention is a * keep / (1 - p)
        float p0 = 0.f, p1 = 0.f;
        const uint8_t* kp0 = a.attn_keep + ((static_cast<size_t>(g) * a.B + b) * a.T) * a.hw + pix0 + p;
        const size_t h8 = static_cast<size_t>(8) * a.B * a.T * a.hw;
#pragma unroll
        for (int nt = 0; nt < FN; ++nt) {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int t = FPW * half + nt * 8 + 2 * j + e;
            bool k0 = false, k1 = false;
            if (t < a.T) {
              const uint8_t* kp = kp0 + static_cast<size_t>(t) * a.hw;
              k0 = kp[0] != 0, k1 = kp[h8] != 0;
            }
            sacc[nt][e] = k0 ? sacc[nt][e] : 0.f;
            sacc[nt][2 + e] = k1 ? sacc[nt][2 + e] : 0.f;
            p0 += sacc[nt][e], p1 += sacc[nt][2 + e];
          }
        }
        p0 += __shfl_xor_sync(0xffffffffu, p0, 1);
        p0 += __shfl_xor_sync(0xffffffffu, p0, 2);
        p1 += __shfl_xor_sync(0xffffffffu, p1, 1);
        p1 += __shfl_xor_sync(0xffffffffu, p1, 2);
        if constexpr (WPP == 2) {  // the pair adds its halves in the same order on both sides
          float* red = s_red + (p * 2 + half) * 2 * kH;
          const float* red_other = s_red + (p * 2 + (half ^ 1)) * 2 * kH;
          team_bar(pair_bar, 64);  // the partner has read the softmax sums
          if (j == 0) red[kH + g] = p0, red[kH + g + 8] = p1;
          team_bar(pair_bar, 64);
          const float lo0 = half ? red_other[kH + g] : p0, hi0 = half ? p0 : red_other[kH + g];
          const float lo1 = half ? red_other[kH + g + 8] : p1, hi1 = half ? p1 : red_other[kH + g + 8];
          p0 = lo0 + hi0, p1 = lo1 + hi1;
        }
        inv0 *= a.attn_keep_scale, inv1 *= a.attn_keep_scale;
        sa0 = p0 * inv0, sa1 = p1 * inv1;
      }
      if constexpr (DROP && WPP == 2)  // (dropout is served by the two-warps-per-pixel team only)
        if (half == 0 && j == 0) s_sa[p * kH + g] = sa0, s_sa[p * kH + g + 8] = sa1;  // read behind the team barriers of the epilogue
    }

    TEAM_DBG(5);  // softmax
    // ---- values: z[h, c] = sum_t e[h, t] x[t, c] (+ positional columns), un-normalised; all frames, CW channels -- tae.py:839
    constexpr int NP = 2 / WPP;  // positional 8-column tiles per warp
    float zacc[CW / 8][4];
    float pacc[NP][4];
#pragma unroll
    for (int nt = 0; nt < CW / 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) zacc[nt][i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < NP; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) pacc[nt][i] = 0.f;
    {
      // two warps per pixel: the probabilities of this warp's frames (hi / lo A fragments, 16 registers per lane) go to
      // the partner through shared memory, the partner's come back: every warp then owns ALL frames of ITS channels
      uint32_t* ex_mine = reinterpret_cast<uint32_t*>(zn_ptr) + tw * 16 * 32 + lane;
      const uint32_t* ex_theirs = reinterpret_cast<const uint32_t*>(zn_ptr) + (tw ^ 1) * 16 * 32 + lane;
      uint32_t own[WPP == 2 ? FN / 2 : 1][8];
      if constexpr (WPP == 2) {
#pragma unroll
        for (int kl = 0; kl < FN / 2; ++kl) {
          split_bf16(sacc[2 * kl][0], sacc[2 * kl][1], own[kl][0], own[kl][4]);
          split_bf16(sacc[2 * kl][2], sacc[2 * kl][3], own[kl][1], own[kl][5]);
          split_bf16(sacc[2 * kl + 1][0], sacc[2 * kl + 1][1], own[kl][2], own[kl][6]);
          split_bf16(sacc[2 * kl + 1][2], sacc[2 * kl + 1][3], own[kl][3], own[kl][7]);
#pragma unroll
          for (int r = 0; r < 8; ++r) ex_mine[(kl * 8 + r) * 32] = own[kl][r];
        }
        team_bar(pair_bar, 64);
      }
      const uint32_t pe_row = s32((mat >> 1) ? s_pe_lo : s_pe_hi) + static_cast<uint32_t>(mr * kPeRow + (mat & 1) * 8) * 2u;
      const bool has_pe = a.pe != nullptr;
      auto values = [&](auto all_) {
        constexpr bool ALL = decltype(all_)::value;
#pragma unroll
        for (int kg = 0; kg < kTP / 16; ++kg) {
          // a block without a live frame: its probabilities meet rows that are zero in the reference (x = 0 on padded
          // frames), so the feature products are skipped; the positional sums are not (an all-padded series attends
          // uniformly, tae.py:831-836)
          const bool on = ALL || ((blk >> kg) & 1u);
          if (!on && !has_pe) continue;
          uint32_t ahi[4], alo[4];
          if constexpr (WPP == 1) {
            split_bf16(sacc[2 * kg][0], sacc[2 * kg][1], ahi[0], alo[0]);
            split_bf16(sacc[2 * kg][2], sacc[2 * kg][3], ahi[1], alo[1]);
            split_bf16(sacc[2 * kg + 1][0], sacc[2 * kg + 1][1], ahi[2], alo[2]);
            split_bf16(sacc[2 * kg + 1][2], sacc[2 * kg + 1][3], ahi[3], alo[3]);
          } else {
            constexpr int KL = (FN / 2 > 0) ? FN / 2 : 1;
            const int owner = kg / KL, kl = kg % KL;  // compile-time after unrolling
            if (owner == half) {
#pragma unroll
              for (int r = 0; r < 4; ++r) ahi[r] = own[kl][r], alo[r] = own[kl][4 + r];
            } else {
#pragma unroll
              for (int r = 0; r < 4; ++r) ahi[r] = ex_theirs[(kl * 8 + r) * 32], alo[r] = ex_theirs[(kl * 8 + 4 + r) * 32];
            }
          }
          if (on) {
            constexpr int CB = 2;  // channel-block pairs whose fragments are requested together (registers)
#pragma unroll
            for (int cb0 = 0; cb0 < CW / 16; cb0 += CB) {
              uint32_t v[CB][4];  // (frames 0-7, block 2 cbp), (0-7, 2 cbp + 1), (8-15, 2 cbp), (8-15, 2 cbp + 1)
#pragma unroll
              for (int q = 0; q < CB; ++q) ldsm_x4_trans(v[q], xbase + kg * 16 * FB + (CW / 16 * half + cb0 + q) * 256);
#pragma unroll
              for (int q = 0; q < CB; ++q) {
                mma_bf16(zacc[2 * (cb0 + q)], ahi, v[q][0], v[q][2]);
                mma_bf16(zacc[2 * (cb0 + q) + 1], ahi, v[q][1], v[q][3]);
              }
#pragma unroll
              for (int q = 0; q < CB; ++q) {
                mma_bf16(zacc[2 * (cb0 + q)], alo, v[q][0], v[q][2]);
                mma_bf16(zacc[2 * (cb0 + q) + 1], alo, v[q][1], v[q][3]);
              }
            }
          }
          if (has_pe) {  // matrices (hi, frames 0-7), (hi, 8-15), (lo, 0-7), (lo, 8-15) of 8 table columns
            uint32_t bp[NP][4];
#pragma unroll
            for (int nt2 = 0; nt2 < NP; ++nt2)
              ldsm_x4(bp[nt2], pe_row + static_cast<uint32_t>((WPP == 2 ? half : nt2) * 8 * kPeRow + kg * 16) * 2u);
#pragma unroll
            for (int nt2 = 0; nt2 < NP; ++nt2) {
              mma_bf16(pacc[nt2], ahi, bp[nt2][0], bp[nt2][1]);
              mma_bf16(pacc[nt2], alo, bp[nt2][0], bp[nt2][1]);
              mma_bf16(pacc[nt2], ahi, bp[nt2][2], bp[nt2][3]);
            }
          }
        }
      };
      if (blk == 0xfu) values(std::true_type{});
      else values(std::false_type{});
    }

    TEAM_DBG(6);  // values
    // ---- the slab is dead for this warp; the LAST warp of the team hands it to the copy engine for the next tile -----
    // (every ldmatrix of this warp has delivered its registers -- the products that consume them are issued -- so the
    // counter below is ordered behind the warp's last read of the slab)
    {
      int old = 0;
      if (lane == 0) old = atomicAdd(s_cnt, 1);
      old = __shfl_sync(0xffffffffu, old, 0);
      if (old == TW - 1) {
        if (lane == 0) *s_cnt = 0;
        fence_proxy_async();
        if (nxt < a.n_tiles) issue_tile(nxt, nlive);
      }
    }
    if (nxt < a.n_tiles) load_pivots(nxt, nlive);  // consumed at the top of the next tile

    TEAM_DBG(7);  // release + pivots
    const size_t row0 = static_cast<size_t>(b) * a.hw + pix0;
    if constexpr (WPP == 2) {
      // the probability exchange shares its space with the attention staging and the zn tiles: everyone is done reading
      team_bar(bar_id, TT);
      if (a.attn != nullptr && !a.skip_attn_store) {  // attn[h, b, t, pix0 .. pix0 + 7] as 32-byte segments   tae.py:490-493
        float* stage = reinterpret_cast<float*>(zn_ptr);
        float* as = stage + p * kAsP;
#pragma unroll
        for (int nt = 0; nt < FN; ++nt) {
          const int t = (FN * half + nt) * 8 + 2 * j;
          *reinterpret_cast<float2*>(as + g * kAP + t) = make_float2(sacc[nt][0] * inv0, sacc[nt][1] * inv0);
          *reinterpret_cast<float2*>(as + (g + 8) * kAP + t) = make_float2(sacc[nt][2] * inv1, sacc[nt][3] * inv1);
        }
        team_bar(bar_id, TT);
        {
          const int pp = lane & 7, tq = lane >> 3, h = tw;  // TW = 16 warps = 16 heads
          float* dst = a.attn + ((static_cast<size_t>(h) * a.B + b) * a.T + tq) * a.hw + pix0 + pp;
          const float* src = stage + pp * kAsP + h * kAP + tq;
          const size_t step = static_cast<size_t>(4) * a.hw;
          float v[kTP / 4];
#pragma unroll
          for (int u = 0; u < kTP / 4; ++u) v[u] = src[4 * u];  // t = tq + 4 u <= 63: inside the staging rows
#pragma unroll
          for (int u = 0; u < kTP / 4; ++u)
            if (tq + 4 * u < a.T) dst[u * step] = v[u];
        }
        team_bar(bar_id, TT);
      }
    }

    // ---- epilogue, two rounds of 8 heads: GroupNorm affine -> fp16 hi/lo zn tiles, per-head in-projection --------
    constexpr int KSW = KS / WPP;  // k-steps of the in-projection per warp (the pair splits k)
#pragma unroll
    for (int rnd = 0; rnd < 2; ++rnd) {
      // in-projection weights of head 8 rnd + p (fp16 hi + lo A fragments, L2 resident): requested first, they fly
      // while the zn tiles are written and across the barrier
      const int h = 8 * rnd + p;
      uint4 wha[KSW], wla[KSW];
      {
        const uint4* wc = a.wc16 + (h * KS + KSW * half) * 32 + lane;
#pragma unroll
        for (int ks = 0; ks < KSW; ++ks) wha[ks] = __ldg(wc + ks * 32), wla[ks] = __ldg(wc + kD * C * 2 / 16 + ks * 32);
      }
      {
        unsigned char* zb = zn_ptr + p * S::kZnPix + g * S::kZnRow;  // head row g of this round, pixel p
        const float inv = rnd ? inv1 : inv0;
#pragma unroll
        for (int nt = 0; nt < CW / 8; ++nt) {
          const int c = CW * half + nt * 8 + 2 * j;
          const int grp = c / CPG;
          const float sa = rnd ? sa1 : sa0;
          const float r = s_rm[grp] * inv, m = DROP ? s_rm[16 + grp] * sa : s_rm[16 + grp];
          const float2 gm = *reinterpret_cast<const float2*>(s_gam + c), bt = *reinterpret_cast<const float2*>(s_gam + C + c);
          // sum_t a (x rstd - mean rstd) gamma + beta sum_t a, with sum_t a = 1 unless dropout acts on the attention
          const float z0 = fmaf(gm.x, fmaf(zacc[nt][2 * rnd], r, -m), DROP ? bt.x * sa : bt.x);
          const float z1 = fmaf(gm.y, fmaf(zacc[nt][2 * rnd + 1], r, -m), DROP ? bt.y * sa : bt.y);
          uint32_t hi, lo;
          split_f16(z0, z1, hi, lo);
          *reinterpret_cast<uint32_t*>(zb + c * 2) = hi;
          *reinterpret_cast<uint32_t*>(zb + HR * S::kZnRow + c * 2) = lo;
        }
        const int hz = g + 8 * rnd;
#pragma unroll
        for (int q = 0; q < NP; ++q) {
          const int qq = (WPP == 2) ? half : q;  // which half of the 16 positional columns
          *reinterpret_cast<float2*>(s_pa + p * S::kPaPix + (qq * kH + hz) * 8 + 2 * j) =
              make_float2(pacc[q][2 * rnd] * inv, pacc[q][2 * rnd + 1] * inv);
        }
      }
      TEAM_DBG(8 + 4 * rnd);  // zn tiles written, weights requested
      team_bar(bar_id, TT);
      TEAM_DBG(9 + 4 * rnd);  // barrier
      // o[16 h + i, px] = Wc[16 h + i, :] . zn[px, h, :] + bc + sum_t a PE                      tae.py:463, 479, 839
      float acc[3][4];
#pragma unroll
      for (int q = 0; q < 3; ++q)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[q][e] = 0.f;
      {
        const unsigned char* zb = zn_ptr + g * S::kZnPix + p * S::kZnRow + 2 * j * 2 + KSW * half * 32;  // B[k = c][n = pixel g]
#pragma unroll
        for (int ks = 0; ks < KSW; ++ks) {
          const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(zb + ks * 32);
          const uint32_t bh1 = *reinterpret_cast<const uint32_t*>(zb + ks * 32 + 16);
          const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(zb + HR * S::kZnRow + ks * 32);
          const uint32_t bl1 = *reinterpret_cast<const uint32_t*>(zb + HR * S::kZnRow + ks * 32 + 16);
          mma_f16(acc[0], wha[ks], bh0, bh1);
          mma_f16(acc[1], wla[ks], bh0, bh1);
          mma_f16(acc[2], wha[ks], bl0, bl1);
        }
      }
      float sum[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) sum[e] = acc[0][e] + (acc[1][e] + acc[2][e]);
      if constexpr (WPP == 2) {  // the two halves of k meet: the second warp of the pair hands its partial sums over
        float* px = reinterpret_cast<float*>(ost + S::kOstRows) + lane;
        if (half == 1) {
#pragma unroll
          for (int e = 0; e < 4; ++e) px[e * 32] = sum[e];
        }
        team_bar(pair_bar, 64);
        if (half == 0) {
#pragma unroll
          for (int e = 0; e < 4; ++e) sum[e] += px[e * 32];
        }
      }
      if (half == 0) {
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {  // accumulator: rows i = g, g + 8; columns pixel 2j, 2j + 1
          const int i = g + (e >> 1) * 8, pp = 2 * j + (e & 1);
          const int d = h * 16 + i;
          const float bcs = (DROP && WPP == 2) ? s_bc[d] * s_sa[pp * kH + h] : s_bc[d];
          v[e] = fmaf(sum[e], inv_sc, bcs + s_pa[pp * S::kPaPix + ((e >> 1) * kH + h) * 8 + g]);
          if (a.save_o != nullptr) a.save_o[(row0 + pp) * kD + d] = v[e];
        }
        // rows of o for the tcgen05 MLP kernel: stmatrix.trans turns (i, pixel pair) fragments into 16-byte pieces
        // [pixel][8 consecutive i]; matrices: hi i 0-7, hi i 8-15, lo i 0-7, lo i 8-15
        uint32_t m4[4];
        split_bf16(v[0], v[1], m4[0], m4[2]);
        split_bf16(v[2], v[3], m4[1], m4[3]);
        const uint32_t st = s32(ost);
        asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1,%2,%3,%4};" ::"r"(st + mr * 80 + mat * 16),
                     "r"(m4[0]), "r"(m4[1]), "r"(m4[2]), "r"(m4[3])
                     : "memory");
        __syncwarp();
        const int px = lane >> 2, chunk = lane & 3;
        const uint4 piece = *reinterpret_cast<const uint4*>(ost + px * 80 + chunk * 16);
        __nv_bfloat16* dst = ((chunk >> 1) ? a.o_lo : a.o_hi) + (row0 + px) * kD + h * 16 + (chunk & 1) * 8;
        *reinterpret_cast<uint4*>(dst) = piece;
        __syncwarp();
      }
      TEAM_DBG(10 + 4 * rnd);  // in-projection + o rows stored
      if (rnd == 0) team_bar(bar_id, TT);  // round 0's zn tiles are read: round 1 may overwrite them
      TEAM_DBG(11 + 4 * rnd);
    }

    live = nlive, padm = npad;
  }
}

template <int C, bool DROP>
int team_launch(const CUtensorMap& map16, const CUtensorMap& map4, const CUtensorMap& map1, const FaArgs& a,
                cudaStream_t stream, const char* name) {
  using S = TeamSmem<C>;
  C2S_SMEM_ATTR((ltae_team_kernel<C, DROP>), S::kTotal);
  const int sms = sm_count();
  const int teams = (a.n_tiles + S::TEAMS - 1) / S::TEAMS;
  const int grid = teams < sms ? teams : sms;
  ltae_team_kernel<C, DROP><<<static_cast<unsigned>(grid), 512, S::kTotal, stream>>>(map16, map4, map1, a);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

}  // namespace

bool ltae_team_eligible(int C, const FaArgs& a) {
  if (C != 64 && C != 128) return false;
  if (a.attn_only) return false;                     // LTAE4WTAE: c2s_ltae_fa.cu
  if (a.attn_keep != nullptr && C != 128) return false;  // training-mode dropout: the two-warps-per-pixel team only
  // C = 64: two slabs leave no room for the attention staging
  if (C == 64 && a.attn != nullptr && !a.skip_attn_store) return false;
  return true;
}

int ltae_team_launch(int C, const CUtensorMap& map16, const CUtensorMap& map4, const CUtensorMap& map1, const FaArgs& a,
                     cudaStream_t stream) {
  if (C == 64) return team_launch<64, false>(map16, map4, map1, a, stream, "ltae_forward<team,C=64>");
  if (C == 128 && a.attn_keep != nullptr) return team_launch<128, true>(map16, map4, map1, a, stream, "ltae_forward<team,C=128>");
  if (C == 128) return team_launch<128, false>(map16, map4, map1, a, stream, "ltae_forward<team,C=128>");
  set_error("ltae_team_launch: C=%d has no team kernel", C);
  return C2S_ERR_UNSUPPORTED;
}

}  // namespace c2s
