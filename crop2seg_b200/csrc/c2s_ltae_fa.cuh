// Shared pieces of the tensor-core L-TAE forward kernels (c2s_ltae_fa.cu: whole-slab kernel with CTA-wide phases;
// c2s_ltae_team.cu: the same slab processed by independent 8-warp teams with early refill): launch arguments, constants,
// PTX wrappers (packed fp32, hi/lo splits, cp.async).  sm_100a.
#pragma once

#include <cuda_fp16.h>

#include "c2s_ltae_prep.cuh"
#include "c2s_sm100.cuh"

namespace c2s {

struct FaArgs {
  const __nv_bfloat16* x;
  const uint8_t* pad;
  const unsigned long long* masks;  // [B][2]: frames to read, padded frames (bit t)
  __nv_bfloat16* out;
  float* attn;
  const float* ufrag;     // [C/16][32][8] fp32, A-fragment order, times log2(e)
  const uint4* wc16;      // [hi | lo][16 heads][C/16][32] fp16 A fragments of inconv.weight * scale
  const float* wscale;    // {scale, 1 / scale}
  const float* cpos;      // [B, T, 16]
  const float* pe;        // [B, T, 256] or nullptr
  const float* bc;        // [256]
  const float* bm;        // [c_out]
  const float* gamma;
  const float* beta;
  const float* bnf;       // [2, c_out] or nullptr (training)
  const float* on_w;
  const float* on_b;
  float* ypre;
  const uint8_t* attn_keep;  // [16, B, T, hw] dropout keep mask or nullptr
  const uint8_t* mlp_keep;   // [B, c_out, hw] or nullptr
  float attn_keep_scale, mlp_keep_scale;
  __nv_bfloat16* o_hi;       // [B*hw][256] rows for the tcgen05 MLP kernel
  __nv_bfloat16* o_lo;
  float* save_o;             // [B*hw][256] fp32 copy of the same rows for the backward, or nullptr
  int B, T, hw;
  int attn_only, skip_attn_store, zero_padded;
  float gn_eps;
  int tiles_per_b;
  int n_tiles;
  unsigned long long* dbg;
};

namespace {

constexpr int kPix = 8;            // pixels per tile; WPP warps (2 for C = 128, 1 for C = 64) share a pixel
constexpr int kTP = 64;            // frames in the slab
constexpr int kH = 16;             // heads
constexpr int kD = 256;            // d_model
constexpr int kAP = 72;            // pitch of the [h][t] fp32 tiles
constexpr int kAsP = kH * kAP + 4;  // attention staging: floats per pixel
constexpr int kPeRow = kTP + 8;    // positional table rows [d][t] (bf16), 144 B pitch
constexpr int kOsRow = kD + 8;     // o rows [pixel][d] (16-bit), pitch in elements
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
// v = hi + lo with hi, lo bf16: ~16 mantissa bits survive.  The residual v - hi is formed by mixed-precision adds that read
// the 16-bit halves of the packed register in place (FHADD.BF16): 5 instructions per pair instead of 6.
__device__ __forceinline__ void split_bf16(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16(v0, v1);
  uint32_t nh;
  uint16_t l, h;
  float r0, r1;
  asm("neg.bf16x2 %0, %1;" : "=r"(nh) : "r"(hi));
  asm("mov.b32 {%0, %1}, %2;" : "=h"(l), "=h"(h) : "r"(nh));
  asm("add.rn.f32.bf16 %0, %1, %2;" : "=f"(r0) : "h"(l), "f"(v0));
  asm("add.rn.f32.bf16 %0, %1, %2;" : "=f"(r1) : "h"(h), "f"(v1));
  lo = pack_bf16(r0, r1);
}
// same with fp16 halves: ~22 mantissa bits survive (|v| must stay below 65504); the negation folds into FHADD: 4 instructions
__device__ __forceinline__ void split_f16(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  uint32_t nh;
  uint16_t l, h;
  float r0, r1;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(v1), "f"(v0));
  asm("neg.f16x2 %0, %1;" : "=r"(nh) : "r"(hi));
  asm("mov.b32 {%0, %1}, %2;" : "=h"(l), "=h"(h) : "r"(nh));
  asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(r0) : "h"(l), "f"(v0));
  asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(r1) : "h"(h), "f"(v1));
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
}
// packed fp32 pairs (FADD2 / FFMA2 on sm_100): two lanes of arithmetic per issue slot
__device__ __forceinline__ unsigned long long pack_f32x2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long add_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long fma_f32x2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
// {lo, hi} halves of a packed bf16 pair plus an fp32 constant, as one f32x2: two mixed-precision adds (FHADD.BF16 reads
// the 16-bit halves in place, no unpacking)
__device__ __forceinline__ unsigned long long bf16x2_plus_f32(uint32_t w, float c) {
  uint16_t l, h;
  float lo, hi;
  asm("mov.b32 {%0, %1}, %2;" : "=h"(l), "=h"(h) : "r"(w));
  asm("add.rn.f32.bf16 %0, %1, %2;" : "=f"(lo) : "h"(l), "f"(c));
  asm("add.rn.f32.bf16 %0, %1, %2;" : "=f"(hi) : "h"(h), "f"(c));
  return pack_f32x2(lo, hi);
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float ex2(float v) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

}  // namespace

// c2s_ltae_bwd_tc.cu: stage A of the backward on the tensor cores
struct BwdTcArgs {
  const __nv_bfloat16* x;
  const float* g_o;     // [N][256]
  const float* g_attn;  // [16][B][T][hw] or nullptr
  const float* u;       // [C][16]  (in_norm.weight folded in)
  const float* cpos;    // [B][T][16]
  const float* wct;     // [C][256]
  const float* wb;      // [256]  bc + Wc beta
  const float* pe;      // [B][T][256] or nullptr (the 16 columns of a head repeat)
  const float* gamma;
  const float* beta;
  const uint8_t* pad;
  const uint8_t* attn_keep;
  float attn_keep_scale;
  float* g_u;
  float* g_cpos;
  float* g_gamma;
  float* g_beta;
  float* zn_rows;
  float* sa_rows;
  int B, T, hw, tiles_per_b, n_tiles;
  float gn_eps;
};
bool ltae_bwd_tc_eligible(const c2s_ltae_desc& d, const void* x, const c2s_ltae_bwd_io& io);
int ltae_bwd_tc_launch(const c2s_ltae_desc& d, const BwdTcArgs& a, void* grad_x, cudaStream_t stream);

// c2s_ltae_team.cu
bool ltae_team_eligible(int C, const FaArgs& a);
int ltae_team_launch(int C, const CUtensorMap& map16, const CUtensorMap& map4, const CUtensorMap& map1, const FaArgs& a,
                     cudaStream_t stream);

}  // namespace c2s
