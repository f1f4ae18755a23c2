// L-TAE forward, persistent TMA-fed kernel for the shipped shapes (bf16 I/O, n_head = 16, d_model = 256,
// C in {64, 128}, T <= 64, H*W % 8 == 0), sm_100a.  Same contract as the other L-TAE kernels; reference
// LTAE.forward / LTAE4WTAE.forward, src/backbones/tae.py:451-504, 589-635.
//
// One CTA per SM walks over tiles of 8 consecutive pixels (tile = blockIdx.x + k * gridDim.x, so that the tiles in
// flight at any time are neighbours and share their 32-byte sectors in L2).  Per tile:
//   load       one 3-D TMA box {8 pixels, C channels, 1 frame} per live frame lands the slab in shared memory in its
//              natural layout X[t][c][8 px] (16-byte rows), signalled on four mbarriers (16 frames each).  With C = 64
//              two slabs alternate: the next tile is in flight during the whole computation of the current one.
//   transpose  every 8 channel x 8 pixel block is transposed IN PLACE by ldmatrix.trans + stmatrix (no lane ever
//              shuffles data by hand) into X[t][c / 8][pixel ^ (t & 7)][8 channels]; the xor keeps the eight frame
//              rows of a fragment in eight different 16-byte bank groups.  The GroupNorm sums (tae.py:461, over all
//              T frames, padded frames count as zeros) are taken from the registers on the way (shifted sums).
//   scores     S^T[h, t] = U'[h, c] X[t, c]^T per pixel, mma.sync m16n8k16 with M = 16 heads; U' = U rstd(group,
//              pixel) log2(e) is rebuilt per pixel and split into bf16 hi + lo (x is exact in bf16).  tae.py:827-831
//              The accumulators start from cpos[b, h, t] (positional / bias part of the scores).
//   softmax    over T in the accumulator registers, two warps per pixel (32 frames each), pad -> -1e6.   tae.py:836
//   values     z[h, c] = sum_t a[h, t] x[t, c]: each warp multiplies the probabilities of ITS frames (still in its
//              registers, hi + lo) with all channels; the two partial sums meet after the slab is dead.     tae.py:839
//   epilogue   GroupNorm affine on z, per-head in-projection against fp16 hi + lo weights (scaled by a power of two
//              into [1, 2); activations fp16 hi + lo; three products) that stay resident in shared memory for the life
//              of the CTA (C = 128: the hi half; the lo fragments are streamed from L2 into registers while the
//              partial sums are exchanged), then bf16 hi/lo rows of o for the tcgen05 row GEMM in c2s_ltae_mlp_tc.cu
//              (MLP + BatchNorm + ReLU + output GroupNorm).  A single 16-bit weight term is not enough: the output
//              GroupNorm runs over 4-8 channels and amplifies errors where a group is almost constant.
//                                                                                              tae.py:463, 486-488
// Frame blocks without a live frame are skipped in both products.
#include <cstdlib>
#include <type_traits>

#include "c2s_ltae_fa.cuh"

namespace c2s {
namespace {

template <int C, int WPP>
struct FaSmem {
  static constexpr int NW = kPix * WPP;                            // warps per CTA
  static constexpr int NBUF = (C == 64 && WPP == 2) ? 2 : 1;      // WPP = 1: two CTAs per SM overlap instead
  static constexpr int kFB = C * 16;                              // one frame: [C][8 px] bf16
  static constexpr int kSlab = kTP * kFB;
  static constexpr int oSlab = 0;
  static constexpr int oWc = NBUF * kSlab;                        // resident in-projection weights (fp16 fragments):
  static constexpr int kWcHalf = kD * C * 2;                      // hi and, with C = 64, lo
  static constexpr bool kHiResident = (WPP == 2);                 // WPP = 1: both halves are streamed from L2
  static constexpr bool kLoResident = (WPP == 2 && C == 64);
  static constexpr int kWc = kLoResident ? 2 * kWcHalf : (kHiResident ? kWcHalf : 0);
  static constexpr int oUf = oWc + kWc;                           // float4 [C/16][2][32] score weights
  static constexpr int oCpos = oUf + C * 64;                      // float [16][kAP]
  static constexpr int oPeHi = oCpos + kH * kAP * 4;              // bf16 [16][kPeRow]
  static constexpr int oPeLo = oPeHi + 16 * kPeRow * 2;
  static constexpr int oGam = oPeLo + 16 * kPeRow * 2;            // float gamma[C], beta[C]
  static constexpr int oRstd = oGam + 2 * C * 4;                  // float [16][8]
  static constexpr int oMu = oRstd + kH * kPix * 4;               // float [16][8]  mean * rstd
  static constexpr int oSa = oMu + kH * kPix * 4;                 // float [16][8]  sum_t a
  static constexpr int oRed = oSa + kH * kPix * 4;                // float [8 px][2 warps][max | sum][16]
  static constexpr int oSaP = oRed + kPix * 2 * 2 * kH * 4;       // float [8 px][2 warps][16]
  static constexpr int oPart = oSaP + kPix * 2 * kH * 4;          // float2 [16 warps][4][subgroups][8 px] statistics partials
  static constexpr int kSub = (C == 64) ? 2 : 1;                  // GroupNorm groups per 8-channel block
  static constexpr int oRaw = oPart + NW * 4 * kSub * kPix * 8;  // float cpos[64][16], pe[64][16] of the next sample
  static constexpr int oMask = oRaw + 2 * kTP * 16 * 4;           // frame masks of the tile that takes over the slab, [k & 1][2]
  static constexpr int oBar = oMask + 32;
  static constexpr int kTotal = oBar + 64;
  static_assert(kTotal <= 232448, "shared memory budget");
  // ---- epilogue scratch, aliased onto the slab once every warp is done with x ----
  static constexpr int ZH = C / 16;                               // channel n-tiles finalised per warp
  static constexpr int NR = ZH * 4 + 4;                           // exchanged registers per thread (z + positional)
  static constexpr int kZn = kH * (C + 8) * 2;                    // zn_hi [16 h][C + 8] fp16
  static constexpr int PB = (WPP == 2 ? 2 * NR * 128 : 2 * kZn) + 16;  // per-pixel block: exchange (WPP = 2), then zn hi/lo
  static_assert(2 * kZn <= PB && (PB / 4) % 32 == 4, "zn tiles must fit; pixel blocks 4 banks apart");
  static constexpr int oStage = kPix * PB;                        // attention staging float [8][kAsP]
  static constexpr bool kStageApart = oStage + kPix * kAsP * 4 + 8192 + 2 * kPix * kOsRow * 2 <= kSlab;
  static constexpr int oPa = kStageApart ? oStage + kPix * kAsP * 4 : oStage;  // float [16][16][8]
  static constexpr int oOsHi = oPa + kH * 16 * kPix * 4;          // 16-bit [8][kOsRow]
  static constexpr int oOsLo = oOsHi + kPix * kOsRow * 2;
  static_assert(oOsLo + kPix * kOsRow * 2 <= kSlab, "epilogue scratch must fit in the slab");
  static_assert(kStageApart || kPix * kAsP * 4 <= kSlab, "attention staging must fit in the slab");
};


// Phase timing for development (build with -DC2S_FA_TIMING, run with C2S_FA_DBG=1): warp 1 of CTA 0 accumulates the
// cycles since the start of the tile at every checkpoint; the host prints the means at the next launch.
#ifdef C2S_FA_TIMING
#define FA_DBG(k)                                                                                   \
  if (a.dbg != nullptr && tid == 32 && blockIdx.x == 0) a.dbg[k] += static_cast<unsigned long long>(clock64() - dbg_t0)
#else
#define FA_DBG(k)
#endif

template <int C, int WPP>
__global__ void __launch_bounds__(256 * WPP, WPP == 1 ? 2 : 1)
ltae_fa_kernel(const __grid_constant__ CUtensorMap map16, const __grid_constant__ CUtensorMap map4,
               const __grid_constant__ CUtensorMap map1, const FaArgs a) {
  using S = FaSmem<C, WPP>;
  constexpr int NW = S::NW, NT = 32 * NW;  // warps, threads
  constexpr int CPG = C / kH;            // channels per GroupNorm group (8 or 4)
  constexpr int KS = C / 16;             // k-steps over channels
  constexpr int NQ = C / 32;             // 4-block quads per frame (one ldmatrix.x4 each)
  constexpr int TSTEP = NW / NQ;   // frames between two items of a warp in the transposition pass
  constexpr int NBUF = S::NBUF;
  constexpr int FB = S::kFB;
  constexpr int ZH = S::ZH;
  constexpr int NR = S::NR;
  extern __shared__ __align__(1024) unsigned char smem[];
  float4* s_uf = reinterpret_cast<float4*>(smem + S::oUf);
  float* s_cpos = reinterpret_cast<float*>(smem + S::oCpos);
  __nv_bfloat16* s_pe_hi = reinterpret_cast<__nv_bfloat16*>(smem + S::oPeHi);
  __nv_bfloat16* s_pe_lo = reinterpret_cast<__nv_bfloat16*>(smem + S::oPeLo);
  float* s_gam = reinterpret_cast<float*>(smem + S::oGam);
  float* s_rstd = reinterpret_cast<float*>(smem + S::oRstd);
  float* s_mu = reinterpret_cast<float*>(smem + S::oMu);
  float* s_sa = reinterpret_cast<float*>(smem + S::oSa);
  float* s_red = reinterpret_cast<float*>(smem + S::oRed);
  float* s_sap = reinterpret_cast<float*>(smem + S::oSaP);
  float2* s_part = reinterpret_cast<float2*>(smem + S::oPart);
  float* s_raw = reinterpret_cast<float*>(smem + S::oRaw);
  unsigned long long* s_mask = reinterpret_cast<unsigned long long*>(smem + S::oMask);
  const uint32_t bars = s32(smem + S::oBar);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = warp / WPP, half = warp % WPP;  // pixel of this warp, which part of the frames it owns (WPP = 2)
  constexpr int FPW = kTP / WPP;               // frames per warp
  constexpr int FN = FPW / 8;                  // score n-tiles per warp
  const int j = lane & 3, g = lane >> 2;       // fragment coordinates: row g (and g + 8), column pair 2j
  const int mat = lane >> 3, mr = lane & 7;    // ldmatrix: this lane supplies row mr of matrix mat
  const uint32_t pair_bar = 1 + p;

  // ---- set-up: barriers, resident weights ----------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < NBUF * 4; ++i) mbar_init(bars + 8 * i, 1);
    fence_mbarrier_init();
  }
  {
    uint4* wc = reinterpret_cast<uint4*>(smem + S::oWc);
    if (!a.attn_only && S::kWc > 0)
      for (int i = tid; i < S::kWc / 16; i += NT) wc[i] = __ldg(a.wc16 + i);
    for (int i = tid; i < KS * 64; i += NT) {  // source order [ks][lane][2] -> [ks][2][lane]
      const int ks = i >> 6, e = i & 63;
      s_uf[ks * 64 + (e & 1) * 32 + (e >> 1)] = __ldg(reinterpret_cast<const float4*>(a.ufrag) + i);
    }
    for (int i = tid; i < C; i += NT) s_gam[i] = __ldg(a.gamma + i), s_gam[C + i] = __ldg(a.beta + i);
    for (int i = tid; i < 2 * kTP * 16; i += NT) s_raw[i] = 0.f;  // rows t >= T and a missing table stay zero
  }
  const float inv_sc = a.attn_only ? 1.f : __ldg(a.wscale + 1);
  __syncthreads();

  // cpos[b, t, :] and the first 16 columns of pe[b, t, :] of sample bn -> raw staging (thread i and i + 512 own their
  // elements from the copy to the conversion at the top of the tile that needs them: no barrier in between)
  auto fetch_consts = [&](int bn) {
#pragma unroll
    for (int q = 0; q < kTP * 16 / NT; ++q) {
      const int i = tid + q * NT, t = i >> 4, h = i & 15;
      if (t < a.T) {
        cp_async4(s_raw + i, a.cpos + (static_cast<size_t>(bn) * a.T + t) * kMaxHeads + h);
        if (!a.attn_only && a.pe != nullptr) cp_async4(s_raw + kTP * 16 + i, a.pe + (static_cast<size_t>(bn) * a.T + t) * kD + h);
      }
    }
  };
  // frames that are not read must hold zeros: warp w owns quad w % NQ of the frames w / NQ + k TSTEP
  auto zero_fill = [&](int buf, unsigned long long live) {
    unsigned char* slab = smem + S::oSlab + buf * S::kSlab;
    unsigned long long mine = 0;  // frames t = warp / NQ + k TSTEP
#pragma unroll
    for (int k = 0; k < kTP / TSTEP; ++k) mine |= 1ull << (k * TSTEP);
    unsigned long long dead = ~live & (mine << (warp / NQ));
    while (dead) {  // a full-length series leaves the frames T .. 63 only
      const int t = __ffsll(static_cast<long long>(dead)) - 1;
      dead &= dead - 1;
      *reinterpret_cast<uint4*>(slab + t * FB + (warp % NQ) * 512 + lane * 16) = make_uint4(0, 0, 0, 0);
    }
  };
  // warp 0 issues the copies of a tile.  The copy unit takes about one cycle per 16-byte row and blocks the issuing
  // thread once its queue is full, so the boxes are as large as the live frames allow (16, 4 or 1 frames): a regular
  // tile is 4-7 instructions instead of 61 and the issuing warp is not held at the next barrier by its own copies.
  // (A copy may complete before its group's bytes are announced: the phase still needs the announcing arrival.)
  auto issue_tile = [&](int tile, int buf, unsigned long long live) {
    const int b = tile / a.tiles_per_b;
    const int pix0 = (tile - b * a.tiles_per_b) * kPix;
    const uint32_t slab = s32(smem + S::oSlab + buf * S::kSlab);
    if (lane < 16) {  // lane = quad of frames 4 lane .. 4 lane + 3, in group lane / 4
      const int grp = lane >> 2, t4 = 4 * lane;
      const uint32_t m16 = static_cast<uint32_t>(live >> (16 * grp)) & 0xffffu;
      const uint32_t m4 = static_cast<uint32_t>(live >> t4) & 0xfu;
      const uint32_t bar = bars + 8 * (buf * 4 + grp);
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

  const int first = blockIdx.x, stride = gridDim.x;
  unsigned long long live_q[NBUF], pad_q[NBUF];
#pragma unroll
  for (int s = 0; s < NBUF; ++s) {
    live_q[s] = 0, pad_q[s] = 0;
    const int tile = first + s * stride;
    if (tile < a.n_tiles) {
      const int b0 = tile / a.tiles_per_b;
      live_q[s] = __ldg(a.masks + 2 * b0), pad_q[s] = __ldg(a.masks + 2 * b0 + 1);
      zero_fill(s, live_q[s]);
      if (warp == 0) issue_tile(tile, s, live_q[s]);
    }
  }

  const bool store_attn = a.attn != nullptr && !a.skip_attn_store;
  int cur_b = -1;
  if (first < a.n_tiles) fetch_consts(first / a.tiles_per_b);

#pragma unroll 1
  for (int k = 0;; ++k) {
    const int tile = first + k * stride;
    if (tile >= a.n_tiles) break;
    const int buf = (NBUF == 2) ? (k & 1) : 0;
    const uint32_t par = static_cast<uint32_t>(k / NBUF) & 1u;
    const unsigned long long live = (NBUF == 2 && buf) ? live_q[NBUF - 1] : live_q[0];
    const unsigned long long padm = (NBUF == 2 && buf) ? pad_q[NBUF - 1] : pad_q[0];
#ifdef C2S_FA_TIMING
    const long long dbg_t0 = clock64();
#endif
    const int n_live = __popcll(live);
    const int b = tile / a.tiles_per_b;
    const int pix0 = (tile - b * a.tiles_per_b) * kPix;
    unsigned char* slab_ptr = smem + S::oSlab + buf * S::kSlab;
    const uint32_t slab = s32(slab_ptr);

    // ---- per-sample constants: copied into the raw staging during the previous tile ---------------------
    {
      const bool new_b = b != cur_b;  // CTA-uniform
      cur_b = b;
      cp_async_wait_all();
      if (new_b) {
#pragma unroll
        for (int q = 0; q < kTP * 16 / NT; ++q) {
          const int i = tid + q * NT, t = i >> 4, h = i & 15;
          // frames behind T never count; padded frames that are not read (rows of zeros) start from the mask
          // value and stay there (tae.py:831): the softmax below needs no per-value test for them
          float c0 = s_raw[i] * kLog2e;
          if (a.zero_padded && ((padm >> t) & 1ull)) c0 = -1e6f * kLog2e;
          if (t >= a.T) c0 = -INFINITY;
          s_cpos[h * kAP + t] = c0;
          if (!a.attn_only) {
            const float pe = s_raw[kTP * 16 + i];
            const __nv_bfloat16 hi = __float2bfloat16_rn(pe);
            s_pe_hi[h * kPeRow + t] = hi;
            s_pe_lo[h * kPeRow + t] = __float2bfloat16_rn(pe - __bfloat162float(hi));
          }
        }
      }
      const int nxt1 = tile + stride;          // this CTA's next tile: its sample's constants
      if (nxt1 < a.n_tiles) {
        const int bn = nxt1 / a.tiles_per_b;
        if (bn != b) fetch_consts(bn);
      }
      const int nxt2 = tile + NBUF * stride;   // the tile that will take over this slab: its frame masks
      if (tid == 0 && nxt2 < a.n_tiles) cp_async16(s_mask + 2 * (k & 1), a.masks + 2 * (nxt2 / a.tiles_per_b));
    }
    FA_DBG(1);

    // ---- transposition in place + GroupNorm sums (tae.py:461; all T frames count, padded ones as zeros) ----------
    // warp w owns quad w % NQ of the frames w / NQ + k TSTEP; shifted sums with the first live frame as the pivot
    {
      constexpr int SUB = S::kSub;
      const int t_first = n_live > 0 ? __ffsll(static_cast<long long>(live)) - 1 : 0;
      const __nv_bfloat16* x_first = a.x + (static_cast<size_t>(b) * a.T + t_first) * C * a.hw + pix0;
      float pv_fin = 0.f;  // pivot of (group tid / 8, pixel tid % 8): first live frame, first channel of the group
      if (tid < kH * kPix && n_live > 0) pv_fin = __bfloat162float(x_first[static_cast<size_t>((tid >> 3) * CPG) * a.hw + (tid & 7)]);
      const int q4 = warp % NQ;
      constexpr int FPG = 16 / TSTEP;  // frames of a 16-frame barrier group that this warp owns
      static_assert(16 % TSTEP == 0 && FPG * TSTEP == 16, "a warp owns whole frames of every barrier group");
      float s1[4], s2[4];
      unsigned long long s1p[4], s2p[4], npv[4];  // {even channel, odd channel} pairs: FADD2 / FFMA2
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        s1p[i] = 0ull, s2p[i] = 0ull;
        const int c0 = (4 * q4 + i) * 8 + (CPG == 4 ? 4 * (j >> 1) : 0);
        const float pv = n_live > 0 ? __bfloat162float(x_first[static_cast<size_t>(c0) * a.hw + g]) : 0.f;
        npv[i] = pack_f32x2(-pv, -pv);
      }
      const uint32_t blk0 = slab + q4 * 512 + mat * 128;
      const int f0 = warp / NQ;
#pragma unroll
      for (int grp = 0; grp < 4; ++grp) {
        const uint32_t gl = static_cast<uint32_t>(live >> (16 * grp)) & 0xffffu;  // warp-uniform
        if (gl == 0) continue;
        mbar_wait(bars + 8 * (buf * 4 + grp), par);  // once per group: a completed barrier still costs ~90 cycles
        uint32_t v[FPG][4];
#pragma unroll
        for (int q = 0; q < FPG; ++q)  // every load of the group goes out before the first use
          if ((gl >> (f0 + TSTEP * q)) & 1u) ldsm_x4_trans(v[q], blk0 + (16 * grp + f0 + TSTEP * q) * FB + mr * 16);
#pragma unroll
        for (int q = 0; q < FPG; ++q) {
          if (!((gl >> (f0 + TSTEP * q)) & 1u)) continue;
          const int t = 16 * grp + f0 + TSTEP * q;
          // v[q][i]: pixel g, channels 2j, 2j+1 of block 4 q4 + i; row = pixel, 8 channels; slot pixel ^ (t & 7)
          stsm_x4(blk0 + t * FB + ((mr ^ (t & 7)) << 4), v[q]);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const unsigned long long d = add_f32x2(pack_f32x2(bf16_lo(v[q][i]), bf16_hi(v[q][i])), npv[i]);
            s1p[i] = add_f32x2(s1p[i], d);
            s2p[i] = fma_f32x2(d, d, s2p[i]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float lo, hi;
        unpack_f32x2(s1p[i], lo, hi);
        s1[i] = lo + hi;
        unpack_f32x2(s2p[i], lo, hi);
        s2[i] = lo + hi;
      }
      FA_DBG(2);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], 1);
        s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], 1);
        if (CPG == 8) {
          s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], 2);
          s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], 2);
        }
        const bool writer = (CPG == 8) ? (j == 0) : ((j & 1) == 0);
        if (writer) s_part[((warp * 4 + i) * SUB + (CPG == 4 ? (j >> 1) : 0)) * kPix + g] = make_float2(s1[i], s2[i]);
      }
      FA_DBG(3);
      __syncthreads();
      FA_DBG(4);
      if (tid < kH * kPix) {
        const int grp = tid >> 3, px = tid & 7;
        const int cb = (CPG == 8) ? grp : (grp >> 1), sub = (CPG == 8) ? 0 : (grp & 1);
        const int qq = cb >> 2, ii = cb & 3;
        float t1 = 0.f, t2 = 0.f;
#pragma unroll
        for (int m = 0; m < TSTEP; ++m) {
          const float2 v = s_part[(((qq + NQ * m) * 4 + ii) * SUB + sub) * kPix + px];
          t1 += v.x, t2 += v.y;
        }
        const float n_all = static_cast<float>(a.T) * CPG;
        const float n_skip = n_all - static_cast<float>(n_live) * CPG;  // frames known to be zero
        t1 -= n_skip * pv_fin;
        t2 = fmaf(n_skip * pv_fin, pv_fin, t2);
        const float m = t1 / n_all;
        float var = t2 / n_all - m * m;
        var = var < 0.f ? 0.f : var;
        const float rstd = rsqrtf(var + a.gn_eps);
        s_rstd[grp * kPix + px] = rstd;
        s_mu[grp * kPix + px] = (m + pv_fin) * rstd;
      }
      __syncthreads();
    }

    FA_DBG(5);
    // ---- scores S^T[h, t] for the frames 32 half .. 32 half + 31 of pixel p ---------------- tae.py:827-831
    float sacc[FN][4];
#pragma unroll
    for (int nt = 0; nt < FN; ++nt) {
      const int t = (FN * half + nt) * 8 + 2 * j;
      const float2 c0 = *reinterpret_cast<const float2*>(s_cpos + g * kAP + t);
      const float2 c1 = *reinterpret_cast<const float2*>(s_cpos + (g + 8) * kAP + t);
      sacc[nt][0] = c0.x, sacc[nt][1] = c0.y, sacc[nt][2] = c1.x, sacc[nt][3] = c1.y;
    }
    const unsigned long long live_w = (WPP == 1) ? live : ((live >> (FPW * half)) & 0xffffffffull);  // this warp's frames
    {
      const uint32_t xrow = slab + ((p ^ mr) << 4) + (mat & 1) * 128 + (FPW * half + (mat >> 1) * 8 + mr) * FB;
#pragma unroll 2
      for (int ks = 0; ks < KS; ++ks) {
        const float4 u0 = s_uf[ks * 64 + lane], u1 = s_uf[ks * 64 + 32 + lane];
        const int c_lo = ks * 16 + 2 * j;
        const float r0 = s_rstd[(c_lo / CPG) * kPix + p], r1 = s_rstd[((c_lo + 8) / CPG) * kPix + p];
        uint32_t ahi[4], alo[4];
        split_bf16(u0.x * r0, u0.y * r0, ahi[0], alo[0]);  // (row g,     k 2j, 2j+1)
        split_bf16(u0.z * r0, u0.w * r0, ahi[1], alo[1]);  // (row g + 8, k 2j, 2j+1)
        split_bf16(u1.x * r1, u1.y * r1, ahi[2], alo[2]);  // (row g,     k 2j+8, 2j+9)
        split_bf16(u1.z * r1, u1.w * r1, ahi[3], alo[3]);  // (row g + 8, k 2j+8, 2j+9)
        // every fragment of the k-step is requested before the first product (one ldmatrix latency per k-step instead
        // of one per pair of frame blocks); bfr[ntp]: (block 2 ntp, channels 16 ks..+7), (.., +8..15), (block 2 ntp + 1, ..)
        uint32_t bfr[FN / 2][4];
#pragma unroll
        for (int ntp = 0; ntp < FN / 2; ++ntp)
          if (((live_w >> (16 * ntp)) & 0xffffull) != 0) ldsm_x4(bfr[ntp], xrow + ntp * 16 * FB + ks * 256);
        // hi pass over every frame block, then the lo pass: FN products between two that share an accumulator
#pragma unroll
        for (int ntp = 0; ntp < FN / 2; ++ntp) {
          if (((live_w >> (16 * ntp)) & 0xffffull) == 0) continue;  // both frame blocks hold zeros
          mma_bf16(sacc[2 * ntp], ahi, bfr[ntp][0], bfr[ntp][1]);
          mma_bf16(sacc[2 * ntp + 1], ahi, bfr[ntp][2], bfr[ntp][3]);
        }
#pragma unroll
        for (int ntp = 0; ntp < FN / 2; ++ntp) {
          if (((live_w >> (16 * ntp)) & 0xffffull) == 0) continue;
          mma_bf16(sacc[2 * ntp], alo, bfr[ntp][0], bfr[ntp][1]);
          mma_bf16(sacc[2 * ntp + 1], alo, bfr[ntp][2], bfr[ntp][3]);
        }
      }
    }

    FA_DBG(6);
    // ---- softmax over t for rows h = g and g + 8 (base 2: the scores carry log2 e) --------- tae.py:831-836
    float sa0 = 0.f, sa1 = 0.f;  // sum_t a of this warp's frames, rows g and g + 8
    {
      float* red = s_red + (p * 2 + half) * 2 * kH;
      const float* red_other = s_red + (p * 2 + (half ^ 1)) * 2 * kH;
      const unsigned long long pad_w = (WPP == 1) ? padm : ((padm >> (FPW * half)) & 0xffffffffull);
      float mx0 = -INFINITY, mx1 = -INFINITY;
      if (!a.zero_padded && pad_w != 0) {  // padded frames were read: their scores are replaced here (tae.py:831)
#pragma unroll
        for (int nt = 0; nt < FN; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            if ((pad_w >> (nt * 8 + 2 * j + e)) & 1ull) sacc[nt][e] = -1e6f * kLog2e, sacc[nt][2 + e] = -1e6f * kLog2e;
      }
#pragma unroll
      for (int nt = 0; nt < FN; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(sacc[nt][0], sacc[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(sacc[nt][2], sacc[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      if constexpr (WPP == 2) {
        if (j == 0) red[g] = mx0, red[g + 8] = mx1;
        asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
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
      float inv0, inv1;
      if constexpr (WPP == 2) {
        if (j == 0) red[kH + g] = d0, red[kH + g + 8] = d1;
        asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
        // the sum is formed in the same order by both warps so that they normalise identically
        const float lo0 = half ? red_other[kH + g] : d0, hi0 = half ? d0 : red_other[kH + g];
        const float lo1 = half ? red_other[kH + g + 8] : d1, hi1 = half ? d1 : red_other[kH + g + 8];
        inv0 = 1.f / (lo0 + hi0), inv1 = 1.f / (lo1 + hi1);
      } else {
        inv0 = 1.f / d0, inv1 = 1.f / d1;
      }
      sa0 = 0.f, sa1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < FN; ++nt) {
        sacc[nt][0] *= inv0, sacc[nt][1] *= inv0, sacc[nt][2] *= inv1, sacc[nt][3] *= inv1;
        if (a.attn_keep != nullptr) {  // training: dropout acts on the attention that is returned (tae.py:837)
          const int t = (FN * half + nt) * 8 + 2 * j;
          const uint8_t* k0 = a.attn_keep + ((static_cast<size_t>(g) * a.B + b) * a.T + t) * a.hw + pix0 + p;
          const uint8_t* k1 = a.attn_keep + ((static_cast<size_t>(g + 8) * a.B + b) * a.T + t) * a.hw + pix0 + p;
          const float sc = a.attn_keep_scale;
          sacc[nt][0] = (t < a.T && k0[0]) ? sacc[nt][0] * sc : 0.f;
          sacc[nt][1] = (t + 1 < a.T && k0[a.hw]) ? sacc[nt][1] * sc : 0.f;
          sacc[nt][2] = (t < a.T && k1[0]) ? sacc[nt][2] * sc : 0.f;
          sacc[nt][3] = (t + 1 < a.T && k1[a.hw]) ? sacc[nt][3] * sc : 0.f;
        }
        sa0 += sacc[nt][0] + sacc[nt][1];
        sa1 += sacc[nt][2] + sacc[nt][3];
      }
      sa0 += __shfl_xor_sync(0xffffffffu, sa0, 1);
      sa0 += __shfl_xor_sync(0xffffffffu, sa0, 2);
      sa1 += __shfl_xor_sync(0xffffffffu, sa1, 1);
      sa1 += __shfl_xor_sync(0xffffffffu, sa1, 2);
      if (WPP == 2 && j == 0) s_sap[(p * 2 + half) * kH + g] = sa0, s_sap[(p * 2 + half) * kH + g + 8] = sa1;
    }

    FA_DBG(7);
    // ---- values: partial z[h, c] over this warp's frames, all channels (+ 16 positional columns) --- tae.py:839
    float zacc[C / 8][4];
    float pacc[2][4];
    if (!a.attn_only) {
#pragma unroll
      for (int nt = 0; nt < C / 8; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) zacc[nt][i] = 0.f;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) pacc[nt][i] = 0.f;
      // lane's row of the transposed loads: frame (mat >> 1) * 8 + mr of the k-step, channel block mat & 1 of the pair
      const uint32_t xrow = slab + ((p ^ mr) << 4) + (mat & 1) * 128 + (FPW * half + (mat >> 1) * 8 + mr) * FB;
      const uint32_t pe_row = s32((mat >> 1) ? s_pe_lo : s_pe_hi) + static_cast<uint32_t>(mr * kPeRow + FPW * half + (mat & 1) * 8) * 2u;
#pragma unroll
      for (int ksl = 0; ksl < FN / 2; ++ksl) {
        uint32_t ahi[4], alo[4];
        split_bf16(sacc[2 * ksl][0], sacc[2 * ksl][1], ahi[0], alo[0]);
        split_bf16(sacc[2 * ksl][2], sacc[2 * ksl][3], ahi[1], alo[1]);
        split_bf16(sacc[2 * ksl + 1][0], sacc[2 * ksl + 1][1], ahi[2], alo[2]);
        split_bf16(sacc[2 * ksl + 1][2], sacc[2 * ksl + 1][3], ahi[3], alo[3]);
        if (((live_w >> (16 * ksl)) & 0xffffull) != 0) {
          constexpr int CB = (C == 64) ? 4 : 2;  // channel-block pairs whose fragments are requested together (registers)
#pragma unroll
          for (int cb0 = 0; cb0 < C / 16; cb0 += CB) {
            uint32_t v[CB][4];  // (frames 0-7, block 2 cbp), (0-7, 2 cbp + 1), (8-15, 2 cbp), (8-15, 2 cbp + 1)
#pragma unroll
            for (int q = 0; q < CB; ++q) ldsm_x4_trans(v[q], xrow + ksl * 16 * FB + (cb0 + q) * 256);
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
        if (a.pe != nullptr) {  // matrices (hi, frames 0-7), (hi, 8-15), (lo, 0-7), (lo, 8-15) of 8 table columns
#pragma unroll
          for (int nt2 = 0; nt2 < 2; ++nt2) {
            uint32_t bp[4];
            ldsm_x4(bp, pe_row + static_cast<uint32_t>(nt2 * 8 * kPeRow + ksl * 16) * 2u);
            mma_bf16(pacc[nt2], ahi, bp[0], bp[1]);
            mma_bf16(pacc[nt2], alo, bp[0], bp[1]);
            mma_bf16(pacc[nt2], ahi, bp[2], bp[3]);
          }
        }
      }
    }
    FA_DBG(8);
    __syncthreads();  // every warp is done with x: the slab becomes epilogue scratch

    FA_DBG(9);
    float* s_stage = reinterpret_cast<float*>(slab_ptr + (S::kStageApart ? S::oStage : 0));
    if (store_attn) {
      float* as = s_stage + p * kAsP;
#pragma unroll
      for (int nt = 0; nt < FN; ++nt) {
        const int t = (FN * half + nt) * 8 + 2 * j;
        *reinterpret_cast<float2*>(as + g * kAP + t) = make_float2(sacc[nt][0], sacc[nt][1]);
        *reinterpret_cast<float2*>(as + (g + 8) * kAP + t) = make_float2(sacc[nt][2], sacc[nt][3]);
      }
    }
    auto store_attention = [&]() {  // attn[h, b, t, pix0 .. pix0 + 7]: 32-byte segments            tae.py:490-493
      const int pp = lane & 7, tq = lane >> 3;
#pragma unroll
      for (int h = warp; h < kH; h += NW) {
        float* dst = a.attn + ((static_cast<size_t>(h) * a.B + b) * a.T + tq) * a.hw + pix0 + pp;
        const float* src = s_stage + pp * kAsP + h * kAP + tq;
        const size_t step = static_cast<size_t>(4) * a.hw;
        float v[kTP / 4];
#pragma unroll
        for (int u = 0; u < kTP / 4; ++u) v[u] = src[4 * u];  // t = tq + 4 u <= 63: inside the staging rows
#pragma unroll
        for (int u = 0; u < kTP / 4; ++u)
          if (tq + 4 * u < a.T) dst[u * step] = v[u];
      }
    };
    if (store_attn && (!S::kStageApart || a.attn_only)) {  // the staging area shares its space with the exchange
      __syncthreads();
      store_attention();
      __syncthreads();
    }

    FA_DBG(10);
    uint4 wlo[(WPP == 2 && !S::kLoResident) ? KS : 1];  // lo fragments of head `warp` of the in-projection weights (C = 128)
    if (!a.attn_only) {
      // GroupNorm affine on the weighted sums -> fp16 hi/lo tiles zn[p][h][c] (tae.py:461) for the channel tiles
      // FIRST .. FIRST + COUNT - 1, the positional sums of the 8-column tiles PFIRST .. PFIRST + PCOUNT - 1
      auto write_zn = [&](auto first_, auto count_, auto pfirst_, auto pcount_, float sa_lo, float sa_hi) {
        constexpr int FIRST = decltype(first_)::value, COUNT = decltype(count_)::value;
        constexpr int PFIRST = decltype(pfirst_)::value, PCOUNT = decltype(pcount_)::value;
        unsigned char* zb = slab_ptr + p * S::PB;
#pragma unroll
        for (int i = 0; i < COUNT; ++i) {
          const int c = (FIRST + i) * 8 + 2 * j;
          const int grp = c / CPG;
          const float r = s_rstd[grp * kPix + p], m = s_mu[grp * kPix + p];
          const float gm0 = s_gam[c], gm1 = s_gam[c + 1], bt0 = s_gam[C + c], bt1 = s_gam[C + c + 1];
          const float(&z)[4] = zacc[FIRST + i];
          // sum_t a (x rstd - mean rstd) gamma + beta sum_t a
          const float z00 = fmaf(gm0, fmaf(z[0], r, -m * sa_lo), bt0 * sa_lo);
          const float z01 = fmaf(gm1, fmaf(z[1], r, -m * sa_lo), bt1 * sa_lo);
          const float z10 = fmaf(gm0, fmaf(z[2], r, -m * sa_hi), bt0 * sa_hi);
          const float z11 = fmaf(gm1, fmaf(z[3], r, -m * sa_hi), bt1 * sa_hi);
          uint32_t hi, lo;
          split_f16(z00, z01, hi, lo);
          *reinterpret_cast<uint32_t*>(zb + (g * (C + 8) + c) * 2) = hi;
          *reinterpret_cast<uint32_t*>(zb + S::kZn + (g * (C + 8) + c) * 2) = lo;
          split_f16(z10, z11, hi, lo);
          *reinterpret_cast<uint32_t*>(zb + ((g + 8) * (C + 8) + c) * 2) = hi;
          *reinterpret_cast<uint32_t*>(zb + S::kZn + ((g + 8) * (C + 8) + c) * 2) = lo;
        }
        float* s_pa = reinterpret_cast<float*>(slab_ptr + S::oPa);
#pragma unroll
        for (int q = 0; q < PCOUNT; ++q) {
          const int i0 = (PFIRST + q) * 8 + 2 * j;
          s_pa[(g * 16 + i0) * kPix + p] = pacc[PFIRST + q][0];
          s_pa[(g * 16 + i0 + 1) * kPix + p] = pacc[PFIRST + q][1];
          s_pa[((g + 8) * 16 + i0) * kPix + p] = pacc[PFIRST + q][2];
          s_pa[((g + 8) * 16 + i0 + 1) * kPix + p] = pacc[PFIRST + q][3];
        }
        if (j == 0 && PFIRST == 0) s_sa[g * kPix + p] = sa_lo, s_sa[(g + 8) * kPix + p] = sa_hi;
      };
      using std::integral_constant;
      if constexpr (WPP == 1) {  // the warp holds the complete sums
        FA_DBG(11);
        write_zn(integral_constant<int, 0>{}, integral_constant<int, C / 8>{}, integral_constant<int, 0>{},
                 integral_constant<int, 2>{}, sa0, sa1);
      } else {
        // ---- the two partial sums of a pixel meet: each warp finalises half of the channel tiles ----------
        float* ex = reinterpret_cast<float*>(slab_ptr + p * S::PB);
        auto meet = [&](auto hf_) {  // generic over the half so that every register index is static
          constexpr int HF = decltype(hf_)::value;
          {
            float* mine = ex + (HF * NR) * 32 + lane;
#pragma unroll
            for (int i = 0; i < ZH; ++i)
#pragma unroll
              for (int e = 0; e < 4; ++e) mine[(i * 4 + e) * 32] = zacc[(1 - HF) * ZH + i][e];
#pragma unroll
            for (int e = 0; e < 4; ++e) mine[(ZH * 4 + e) * 32] = pacc[1 - HF][e];
          }
          asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
          {
            const float* theirs = ex + ((1 - HF) * NR) * 32 + lane;
#pragma unroll
            for (int i = 0; i < ZH; ++i)
#pragma unroll
              for (int e = 0; e < 4; ++e) zacc[HF * ZH + i][e] += theirs[(i * 4 + e) * 32];
#pragma unroll
            for (int e = 0; e < 4; ++e) pacc[HF][e] += theirs[(ZH * 4 + e) * 32];
          }
          const float st0 = s_sap[(p * 2) * kH + g] + s_sap[(p * 2 + 1) * kH + g];
          const float st1 = s_sap[(p * 2) * kH + g + 8] + s_sap[(p * 2 + 1) * kH + g + 8];
          asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");  // the exchange is read: zn may overwrite it
          if constexpr (!S::kLoResident) {  // in flight while zn is finalised
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) wlo[ks] = __ldg(a.wc16 + S::kWcHalf / 16 + (warp * KS + ks) * 32 + lane);
          }
          FA_DBG(11);
          write_zn(integral_constant<int, HF * ZH>{}, integral_constant<int, ZH>{}, integral_constant<int, HF>{},
                   integral_constant<int, 1>{}, st0, st1);
        };
        if (half == 0) meet(integral_constant<int, 0>{});
        else meet(integral_constant<int, 1>{});
      }
    }
    FA_DBG(12);
    __syncthreads();

    FA_DBG(13);
    if (store_attn && S::kStageApart && !a.attn_only) store_attention();

    FA_DBG(14);
    if (!a.attn_only) {
      // ---- in-projection of head `warp`: o[16 h + i, px] = Wc[16 h + i, :] . zn[px, h, :] + sa bc + sum_t a PE
      //                                                                              tae.py:463, 479, 839
      // The heads of a warp run side by side and every term has its own accumulator: HPW x 3 independent chains of KS
      // products instead of one chain of 3 KS (an mma.sync result comes back after ~30 cycles).
      constexpr int HPW = kH / NW;  // heads per warp
      float acc[HPW][3][4];
#pragma unroll
      for (int hh = 0; hh < HPW; ++hh)
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[hh][q][e] = 0.f;
      uint4 wha[HPW][S::kHiResident ? 1 : KS], wla[HPW][S::kHiResident ? 1 : KS];
      if constexpr (!S::kHiResident) {  // streamed from L2: every load goes out before the first product
#pragma unroll
        for (int hh = 0; hh < HPW; ++hh) {
          const uint4* wc = a.wc16 + ((warp + hh * NW) * KS) * 32 + lane;
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) wha[hh][ks] = __ldg(wc + ks * 32), wla[hh][ks] = __ldg(wc + S::kWcHalf / 16 + ks * 32);
        }
      }
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
        for (int hh = 0; hh < HPW; ++hh) {
          const int h = warp + hh * NW;
          const unsigned char* zb = slab_ptr + g * S::PB + (h * (C + 8) + 2 * j) * 2;  // B[k = c][n = pixel g]
          uint4 wa, wl;
          if constexpr (!S::kHiResident) {
            wa = wha[hh][ks], wl = wla[hh][ks];
          } else {
            const uint4* wc = reinterpret_cast<const uint4*>(smem + S::oWc) + (h * KS) * 32 + lane;
            wa = wc[ks * 32];
            if constexpr (S::kLoResident) wl = wc[S::kWcHalf / 16 + ks * 32];
            else wl = wlo[ks];
          }
          const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(zb + ks * 32);
          const uint32_t bh1 = *reinterpret_cast<const uint32_t*>(zb + ks * 32 + 16);
          const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(zb + S::kZn + ks * 32);
          const uint32_t bl1 = *reinterpret_cast<const uint32_t*>(zb + S::kZn + ks * 32 + 16);
          mma_f16(acc[hh][0], wa, bh0, bh1);
          mma_f16(acc[hh][1], wl, bh0, bh1);
          mma_f16(acc[hh][2], wa, bl0, bl1);
        }
      }
#pragma unroll
      for (int hh = 0; hh < HPW; ++hh) {
        const int h = warp + hh * NW;
        const float* s_pa = reinterpret_cast<const float*>(slab_ptr + S::oPa);
        uint16_t* os_hi = reinterpret_cast<uint16_t*>(slab_ptr + S::oOsHi);
        uint16_t* os_lo = reinterpret_cast<uint16_t*>(slab_ptr + S::oOsLo);
        // accumulator: rows i = g, g + 8; columns pixel 2j, 2j + 1
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = g + (e >> 1) * 8, pp = 2 * j + (e & 1);
          const int d = h * 16 + i;
          const float sum = acc[hh][0][e] + (acc[hh][1][e] + acc[hh][2][e]);
          const float v = fmaf(sum, inv_sc, fmaf(s_sa[h * kPix + pp], __ldg(a.bc + d), s_pa[(h * 16 + i) * kPix + pp]));
          const __nv_bfloat16 hi = __float2bfloat16_rn(v);
          const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
          os_hi[pp * kOsRow + d] = *reinterpret_cast<const uint16_t*>(&hi);
          os_lo[pp * kOsRow + d] = *reinterpret_cast<const uint16_t*>(&lo);
          if (a.save_o != nullptr) a.save_o[(static_cast<size_t>(b) * a.hw + pix0 + pp) * kD + d] = v;
        }
      }
      FA_DBG(15);
      __syncthreads();

      FA_DBG(16);
      {  // the MLP, BatchNorm, ReLU and output GroupNorm run as a tcgen05 row GEMM (c2s_ltae_mlp_tc.cu)
        const size_t row0 = static_cast<size_t>(b) * a.hw + pix0;
        const uint16_t* os_hi = reinterpret_cast<const uint16_t*>(slab_ptr + S::oOsHi);
        const uint16_t* os_lo = reinterpret_cast<const uint16_t*>(slab_ptr + S::oOsLo);
        for (int i = tid; i < 2 * kPix * (kD / 8); i += NT) {  // 16-byte pieces of the 8 rows, hi then lo
          const int plane = i / (kPix * (kD / 8)), r = i - plane * (kPix * (kD / 8));
          const int pp = r / (kD / 8), q = r - pp * (kD / 8);
          const uint16_t* src = (plane ? os_lo : os_hi) + pp * kOsRow + q * 8;
          __nv_bfloat16* dst = (plane ? a.o_lo : a.o_hi) + (row0 + pp) * kD + q * 8;
          *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
        }
      }
    }

    FA_DBG(17);
    // ---- the slab is free: bring the tile after next (NBUF = 2) / the next tile (NBUF = 1) -------------------
    fence_proxy_async();  // generic writes above, bulk-copy writes below
    if (tid == 0) cp_async_wait_all();  // the masks of the slab's next tile have landed long ago
    __syncthreads();
    FA_DBG(18);
    {
      const int nxt = tile + NBUF * stride;
      unsigned long long lv = 0, pd = 0;
      if (nxt < a.n_tiles) {
        lv = s_mask[2 * (k & 1)], pd = s_mask[2 * (k & 1) + 1];
        zero_fill(buf, lv);
        if (warp == 0) issue_tile(nxt, buf, lv);
      }
      if (NBUF == 2 && buf) live_q[NBUF - 1] = lv, pad_q[NBUF - 1] = pd;
      else live_q[0] = lv, pad_q[0] = pd;
    }
    FA_DBG(19);
#ifdef C2S_FA_TIMING
    if (a.dbg != nullptr && tid == 32 && blockIdx.x == 0) a.dbg[0] += 1;
#endif
  }
}

// ---- weights in fragment order (built per call on the device) -----------------------------------------------
// ufrag[ks][lane][8]: fp32 U (in_norm.weight folded) * log2(e) in A-fragment order, rows = heads
__global__ void fa_build_ufrag_kernel(const float* __restrict__ u /*[C][16]*/, float* __restrict__ uf, int C) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (C / 16) * 32 * 8) return;
  const int e = i & 7, lane = (i >> 3) & 31, ks = i >> 8;
  const int j = lane & 3, r8 = lane >> 2;
  const int row = r8 + ((e >> 1) & 1) * 8;
  const int k = 2 * j + (e & 1) + (e >> 2) * 8;
  uf[i] = u[(ks * 16 + k) * kMaxHeads + row] * kLog2e;
}

// masks[b] = {frames the kernel reads, padded frames} as bit sets over t < T <= 64
__global__ void fa_masks_kernel(const uint8_t* __restrict__ pad, unsigned long long* __restrict__ masks, int B, int T,
                                int zero_padded) {
  // one warp per sample: two coalesced byte loads and two ballots instead of T dependent loads per thread
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const bool p0 = pad != nullptr && lane < T && pad[b * T + lane] != 0;
  const bool p1 = pad != nullptr && lane + 32 < T && pad[b * T + 32 + lane] != 0;
  const unsigned long long pd = static_cast<unsigned long long>(__ballot_sync(0xffffffffu, p0)) |
                                (static_cast<unsigned long long>(__ballot_sync(0xffffffffu, p1)) << 32);
  const unsigned long long all = T >= 64 ? ~0ull : ((1ull << T) - 1ull);
  if (lane == 0) masks[2 * b] = zero_padded ? (all & ~pd) : all, masks[2 * b + 1] = pd;
}

// out = {s, 1/s} with s the power of two that brings max |w| into [1, 2)
__global__ void fa_weight_scale_kernel(const float* __restrict__ w, int n, float* __restrict__ out) {
  __shared__ float red[32];
  float m = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, fabsf(w[i]));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < static_cast<int>(blockDim.x >> 5); ++i) m = fmaxf(m, red[i]);
    float s = 1.f;
    if (m > 0.f && m < INFINITY) s = exp2f(-floorf(log2f(m)));
    out[0] = s, out[1] = 1.f / s;
  }
}

// fp16 hi and lo A fragments of W[rows][cols] * scale, tiled (rows/16) x (cols/16): wf[hi | lo][tile][lane][4] pairs
__global__ void fa_build_w16_kernel(const float* __restrict__ w, const float* __restrict__ scale,
                                    uint32_t* __restrict__ wf, int rows, int cols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // one (tile, lane, reg)
  const int n = (rows / 16) * (cols / 16) * 32 * 4;
  if (i >= n) return;
  const int reg = i & 3, lane = (i >> 2) & 31, tile = i >> 7;
  const int ks = tile % (cols / 16), mt = tile / (cols / 16);
  const int j = lane & 3, r8 = lane >> 2;
  const int row = mt * 16 + r8 + (reg & 1) * 8;
  const int k = ks * 16 + 2 * j + (reg >> 1) * 8;
  const float s = scale[0];
  const float v0 = w[static_cast<size_t>(row) * cols + k] * s, v1 = w[static_cast<size_t>(row) * cols + k + 1] * s;
  uint32_t hi, lo;
  split_f16(v0, v1, hi, lo);
  wf[i] = hi;
  wf[n + i] = lo;
}

template <int C, int WPP>
int fa_launch(const CUtensorMap& map16, const CUtensorMap& map4, const CUtensorMap& map1, const FaArgs& a,
              cudaStream_t stream, const char* name) {
  using S = FaSmem<C, WPP>;
  C2S_SMEM_ATTR((ltae_fa_kernel<C, WPP>), S::kTotal);
  const int slots = sm_count() * (WPP == 1 ? 2 : 1);  // persistent CTAs: one per SM, two for the single-warp tiles
  const int grid = a.n_tiles < slots ? a.n_tiles : slots;
  ltae_fa_kernel<C, WPP><<<static_cast<unsigned>(grid), 256 * WPP, S::kTotal, stream>>>(map16, map4, map1, a);
  C2S_LAUNCH_CHECK(name);
  return C2S_OK;
}

}  // namespace

bool ltae_fa_eligible(const c2s_ltae_desc& d, const void* x, const void* out) {
  const bool attn_only = (d.flags & C2S_LTAE_ATTN_ONLY) != 0;
  if (d.dtype != C2S_BF16 || d.n_head != kH || d.d_model != kD || !d.has_inconv) return false;
  if (d.C != 64 && d.C != 128) return false;
  if (d.T > kTP || (d.H * d.W) % kPix != 0) return false;
  if (d.pe_mode == C2S_PE_SINUSOID_LINEAR) return false;  // table differs per head chunk
  if (!attn_only && (d.c_out % 16 != 0 || d.c_out > 256)) return false;
  if (reinterpret_cast<uintptr_t>(x) % 16 != 0 || reinterpret_cast<uintptr_t>(out) % 16 != 0) return false;
  return true;
}

size_t ltae_fa_workspace_floats(const c2s_ltae_desc& d) {
  // ufrag, Wc fragments (fp16 hi + lo), scale
  return align64(static_cast<size_t>(d.C) * 16) + align64(static_cast<size_t>(kD) * d.C) + align64(2) +
         align64(static_cast<size_t>(d.B) * 4);
}

int ltae_fa_forward(const c2s_ltae_desc& d, const c2s_ltae_params& p, const void* x, const uint8_t* pad_mask, void* out,
                    float* attn, float* ws, const LtaeWorkspace& lay, float* fa_ws, cudaStream_t stream) {
  const int C = d.C, hw = d.H * d.W;
  const bool attn_only = (d.flags & C2S_LTAE_ATTN_ONLY) != 0;
  const bool train = (d.flags & C2S_LTAE_BN_BATCH_STATS) != 0 && !attn_only;
  float* ufrag = fa_ws;
  uint32_t* wc16 = reinterpret_cast<uint32_t*>(ufrag + align64(static_cast<size_t>(C) * 16));
  float* wscale = reinterpret_cast<float*>(wc16 + align64(static_cast<size_t>(kD) * C));
  unsigned long long* masks = reinterpret_cast<unsigned long long*>(wscale + align64(2));

  const bool reuse = (d.flags & C2S_LTAE_REUSE_FOLDED) != 0;
  if (!reuse) {
    fa_build_ufrag_kernel<<<ceil_div((C / 16) * 256, 256), 256, 0, stream>>>(ws + lay.u, ufrag, C);
    C2S_LAUNCH_CHECK("ltae_fa_build_ufrag");
  }
  fa_masks_kernel<<<ceil_div(d.B, 4), 128, 0, stream>>>(pad_mask, masks, d.B, d.T, (d.flags & C2S_LTAE_ZERO_PADDED) != 0);
  C2S_LAUNCH_CHECK("ltae_fa_masks");
  if (!attn_only && !reuse) {
    fa_weight_scale_kernel<<<1, 1024, 0, stream>>>(p.inconv_weight, kD * C, wscale);
    C2S_LAUNCH_CHECK("ltae_fa_weight_scale");
    fa_build_w16_kernel<<<ceil_div((kD / 16) * (C / 16) * 128, 256), 256, 0, stream>>>(p.inconv_weight, wscale, wc16, kD, C);
    C2S_LAUNCH_CHECK("ltae_fa_build_wc16");
  }

  CUtensorMap map16, map4, map1;
  const cuuint64_t dims[3] = {static_cast<cuuint64_t>(hw), static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(d.B) * d.T};
  const cuuint64_t strides[2] = {static_cast<cuuint64_t>(hw) * 2, static_cast<cuuint64_t>(C) * hw * 2};
  CUtensorMap* maps[3] = {&map16, &map4, &map1};
  const cuuint32_t frames[3] = {16, 4, 1};
  const char* what[3] = {"features, 16 frames per box", "features, 4 frames per box", "features, 1 frame per box"};
  for (int i = 0; i < 3; ++i) {
    const cuuint32_t box[3] = {kPix, static_cast<cuuint32_t>(C), frames[i]};
    const int status = encode_tensor_map(maps[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, x, dims, strides, box,
                                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, what[i]);
    if (status != C2S_OK) return status;
  }

  FaArgs a{};
  a.x = static_cast<const __nv_bfloat16*>(x);
  a.pad = pad_mask;
  a.masks = masks;
  a.out = static_cast<__nv_bfloat16*>(out);
  a.attn = attn;
  a.ufrag = ufrag;
  a.wc16 = reinterpret_cast<const uint4*>(wc16);
  a.wscale = wscale;
  a.cpos = ws + lay.cpos;
  a.pe = d.pe_mode != C2S_PE_NONE ? ws + lay.pe : nullptr;
  a.bc = p.inconv_bias, a.bm = p.mlp_bias;
  a.gamma = p.in_norm_weight, a.beta = p.in_norm_bias;
  a.bnf = (attn_only || train) ? nullptr : ws + lay.bnf;
  a.on_w = p.out_norm_weight, a.on_b = p.out_norm_bias;
  a.ypre = train ? (p.save_y != nullptr ? p.save_y : ws + lay.ypre) : nullptr;
  a.attn_keep = p.attn_keep, a.mlp_keep = p.mlp_keep;
  a.save_o = p.save_o;
  a.attn_keep_scale = d.attn_keep_scale, a.mlp_keep_scale = d.mlp_keep_scale;
  a.B = d.B, a.T = d.T, a.hw = hw;
  a.attn_only = attn_only;
  a.skip_attn_store = (d.flags & C2S_LTAE_SKIP_ATTN_STORE) != 0;
  a.zero_padded = (d.flags & C2S_LTAE_ZERO_PADDED) != 0;
  a.gn_eps = d.gn_eps;
  a.tiles_per_b = hw / kPix;
  if (static_cast<long long>(d.B) * a.tiles_per_b > 0x3fffffffll) C2S_UNSUPPORTED("c2s_ltae_forward: too many pixel tiles");
  a.n_tiles = d.B * a.tiles_per_b;
#if defined(C2S_FA_TIMING) || defined(C2S_TEAM_TIMING)
  static unsigned long long* dbg = nullptr;
  if (getenv("C2S_FA_DBG") != nullptr) {
    if (dbg == nullptr) cudaMalloc(&dbg, 32 * 8);
    unsigned long long h[32];
    cudaMemcpy(h, dbg, sizeof(h), cudaMemcpyDeviceToHost);
    if (h[0] > 0) {
      fprintf(stderr, "[fa dbg] %llu tiles in CTA 0; mean cycles since the tile started at each checkpoint:", h[0]);
      for (int k = 1; k < 20; ++k) fprintf(stderr, " %d:%.0f", k, double(h[k]) / h[0]);
      fprintf(stderr, "\n");
    }
    cudaMemset(dbg, 0, sizeof(h));
    a.dbg = dbg;
  }
#endif
  if (!attn_only) {
    __nv_bfloat16 *w_hi, *w_lo;
    ltae_mlp_tc_buffers(d, ws + lay.tc, &a.o_hi, &a.o_lo, &w_hi, &w_lo);
  }
  int status;
  if (option(C2S_OPT_LTAE_KERNEL) != C2S_LTAE_KERNEL_SLAB && ltae_team_eligible(C, a))
    status = ltae_team_launch(C, map16, map4, map1, a, stream);
  else if (C == 128)
    status = fa_launch<128, 2>(map16, map4, map1, a, stream, "ltae_forward<fa,C=128>");
  else
    status = fa_launch<64, 1>(map16, map4, map1, a, stream, "ltae_forward<fa,C=64>");
  if (status != C2S_OK) return status;
  if (!attn_only)
    return ltae_mlp_tc_forward(d, p, ws + lay.tc, a.bnf, a.ypre, out, stream);
  return C2S_OK;
}

}  // namespace c2s
