// Shared convolutional encoder over the (batch x time) frames (SURVEY.md section 8f, rank 4), sm_100a.
// Reference: ConvLayer = Conv2d(k, padding_mode='reflect') -> GroupNorm(n_groups) -> ReLU, src/backbones/conv.py:29-96;
// ConvBlock (conv.py:164-200), DownConvBlock (conv.py:238-296) and their smart_forward over B*T frames
// (src/backbones/temp_shared_block.py:18-47).
//
//   c2s_conv2d_forward   3x3 / stride 1 / reflect padding as an implicit GEMM on the 5th-generation tensor cores:
//                        D[pixel, c_out] = sum_{tap, c} X[pixel + tap, c] * W[c_out, tap, c]      (bf16 x bf16 -> fp32)
//     * one persistent CTA per SM walks over (frame, band of image rows) units; M = one image row of 128 pixels,
//       N = 64 output channels, K = 9 taps x C_in;
//     * the input row y of a frame is brought in ONCE: four producer warps read the NCHW rows (16-byte loads, the next
//       row's loads in flight while the current one is stored),
//       transpose 8 channel x 8 pixel blocks in registers (PRMT) and store them pixel-major into a ring slot
//       [130 pixels][64 channels] in the K-major 128-byte-swizzled layout tcgen05 reads (chunk ^ (row & 7); the two halo
//       pixels are the reflected ones, so the padding costs nothing);
//     * the nine taps of an output row are nine START ADDRESSES into three ring slots (rows y-1, y, y+1 -- reflected at the
//       frame edges -- shifted by 0 / 1 / 2 pixel rows of 128 bytes; tools/ubench/umma_rowshift.cu shows that the matrix
//       descriptor accepts any 128-byte-aligned start when the swizzle follows the absolute address), so shared memory is
//       filled at 1x the input bytes instead of 9x;
//     * the prepared weights [64][9 * C_in] (bf16, K-major, 64-wide swizzled chunks) stay resident in shared memory;
//     * one elected thread issues the tcgen05 products (umma_bf16: M 128, N 64, K 16) into one of two TMEM accumulators;
//       umma_commit frees ring slots and hands the accumulator to eight epilogue warps (tmem_ld32), which add the bias,
//       store the raw (pre-normalisation) row as bf16 NCHW and keep the GroupNorm sums of their frame in registers (one
//       atomic per warp and quarter of the channels per unit).
//                        The same contract on whole 16-pixel-wide frames with 64 or 128 channels in and out
//                        (conv3x3_w16_tc_kernel: padded frame resident, weights streamed by TMA, N = c_out; see there);
//                        and the strided 4x4 layer of DownConvBlock (conv4x4s2_tc_kernel).
//   c2s_group_stats      per-(frame, group) sum / sum of squares of a raw NCHW tensor (layers whose convolution ran elsewhere)
//   c2s_group_norm_relu  y = relu((x - mean) * rstd * gamma + beta) [+ residual]: the second, element-wise pass
//                        (GroupNorm needs the statistics of the whole frame before the first output element).
// Forward only (inference).  bf16 features; the statistics and the normalisation are fp32.
#include "c2s_sm100.cuh"

namespace c2s {
namespace {

constexpr int kCN = 64;              // output channels = UMMA N
// one ring slot = one image row [W + 2 pixels][128 B], rounded up to the 1024-byte swizzle atom (W = 128: 17408, W = 64: 9216)
__host__ __device__ constexpr int slot_bytes(int w) { return ((w + 2) * 128 + 1023) / 1024 * 1024; }
constexpr int kRing = 8;             // input rows in flight
constexpr int kAccBufs = 4;          // TMEM accumulators (64 columns each)
constexpr int kConvThreads = 416;    // warp 0: MMA issuer, warps 1-4: producers, warps 5-12: epilogue (2 per TMEM lane quarter)
constexpr int kStatQuarters = 4;     // statistics granularity of the tensor-core kernel: 16 channels

struct ConvArgs {
  const __nv_bfloat16* x;    // [frames][c_in][H][128]
  __nv_bfloat16* y;          // [frames][64][H][128] raw convolution output (bias added)
  const float* bias;         // [64] or nullptr
  float* stats;              // [frames][4][2] sum, sum of squares per 16-channel quarter (accumulated), or nullptr
  const __nv_bfloat16* wp;   // [64][chunks * 64] prepared weights, k = tap * CK + c
  int frames, c_in, H, rows_per_unit, units_per_frame, n_units;
  // optional normalisation of the INPUT on the fly: x is the raw output of the previous layer, the producers apply
  // relu(GroupNorm(x)) while they transpose it (the previous layer's second pass never touches HBM)
  const float* in_stats;     // [frames][in_sub][2] or nullptr
  const float* in_gamma;
  const float* in_beta;
  int in_groups, in_sub, in_relu;
  float in_eps;
};

// the low-word shortcut of umma_desc_k_sw128: ((address >> 4) | leading byte offset 1 << 16) with the constant high word
__device__ __forceinline__ uint64_t desc_from(uint32_t lo) { return (static_cast<uint64_t>(kUmmaDescHiSw128) << 32) | lo; }

// the unit -> (frame, rows) arithmetic shared by the three roles
struct Unit {
  int f, y0, y1, lo, hi;  // output rows [y0, y1), input rows [lo, hi]
};
__device__ __forceinline__ Unit unit_of(const ConvArgs& a, int u) {
  Unit t;
  t.f = u / a.units_per_frame;
  const int band = u - t.f * a.units_per_frame;
  t.y0 = band * a.rows_per_unit;
  t.y1 = min(t.y0 + a.rows_per_unit, a.H);
  t.lo = max(t.y0 - 1, 0);
  t.hi = min(t.y1, a.H - 1);
  return t;
}

// W = image width: 128 = UMMA M (one accumulator row per TMEM lane), 64 (an M = 64 accumulator lives in lanes 0-15 of every
// 32-lane quarter, tools/ubench/umma_rowshift.cu) or 32 (M = 64 products whose rows 32-63 read whatever follows the slot --
// the rows of a product are independent, their accumulator lanes are never stored; the tensor pipe is not what limits
// these kernels, the issue rate of the products is)
template <int CK, bool NORM, int W>
__global__ void __launch_bounds__(kConvThreads, 1) conv3x3_tc_kernel(const ConvArgs a) {
  constexpr int kCW = W;
  constexpr int kM = W < 64 ? 64 : W;              // UMMA M
  constexpr int kSlotBytes = slot_bytes(W);
  constexpr int KS = CK / 16;                      // k-steps (MMA instructions) per tap
  constexpr int NCHUNK = (9 * CK + 63) / 64;       // 64-wide K chunks of the resident weights
  constexpr int CB = CK / 8;                       // 8-channel blocks per pixel row
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long bars[2 * kRing + 2 * kAccBufs];  // full[R], empty[R], tfull[A], tempty[A]
  __shared__ uint32_t tmem_s;
  __shared__ float s_bias[kCN];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t base = (s32(smem_raw) + 1023u) & ~1023u;
  unsigned char* sm = smem_raw + (base - s32(smem_raw));
  const uint32_t ring = base + NCHUNK * 8192;
  unsigned char* ring_ptr = sm + NCHUNK * 8192;
  const uint32_t bar0 = s32(&bars[0]);
  auto full = [&](int s) { return bar0 + 8u * s; };
  auto empty = [&](int s) { return bar0 + 8u * (kRing + s); };
  auto tfull = [&](int b) { return bar0 + 8u * (2 * kRing + b); };
  auto tempty = [&](int b) { return bar0 + 8u * (2 * kRing + kAccBufs + b); };

  if (tid == 0) {
    constexpr int kRowBlocks = (CK / 8) * (W / 8);  // producer threads of a row (see the producer role): whole warps -> groups
    constexpr int kRowWarps = (kRowBlocks < 128 && kRowBlocks % 32 == 0) ? kRowBlocks / 32 : 4;
    for (int s = 0; s < kRing; ++s) mbar_init(full(s), kRowWarps), mbar_init(empty(s), 1);   // one arrival per warp serving the row
    for (int b = 0; b < kAccBufs; ++b) mbar_init(tfull(b), 1), mbar_init(tempty(b), 8);       // one arrival per epilogue warp
    fence_mbarrier_init();
  }
  if (warp == 0) {
    tmem_alloc(s32(&tmem_s), 256);
    tmem_relinquish();
  }
  if (tid < kCN) s_bias[tid] = a.bias != nullptr ? a.bias[tid] : 0.f;
  // resident weights: [chunk][64 rows n][128 B], 16-byte pieces at chunk position c16 ^ (n & 7)
  for (int i = tid; i < kCN * NCHUNK * 8; i += kConvThreads) {
    const int c16 = i & 7, j = (i >> 3) % NCHUNK, n = i / (8 * NCHUNK);
    const uint4 v = *reinterpret_cast<const uint4*>(a.wp + static_cast<size_t>(n) * (NCHUNK * 64) + j * 64 + c16 * 8);
    *reinterpret_cast<uint4*>(sm + j * 8192 + n * 128 + ((c16 ^ (n & 7)) << 4)) = v;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tacc = tmem_s;

  if (warp == 0) {
    // ---- MMA issuer ----------------------------------------------------------------------------------------------
    // The issuing thread is the pipeline's clock: umma_bf16 blocks it while the (shallow) queue is full, so every scalar
    // instruction between the last product of a row and the first one of the next row is tensor-pipe idle time.  The
    // bookkeeping is therefore incremental (no divisions, one barrier wait and one release per row in the steady state)
    // and the tap loops stay rolled: the descriptor arithmetic of a tap sits between the products, not in front of them.
    if (elect_one()) {
      static constexpr uint32_t idesc = umma_idesc_bf16(kM, kCN);
      const uint32_t b_lo0 = ((base >> 4) & 0x3fffu) | (1u << 16);
      uint32_t in_slot = 0, in_phase = 0;      // ring slot of the next input row to wait for; bit s = parity of slot s
      uint32_t free_slot = 0;                  // ring slot of the next input row to release
      uint32_t o = 0;                          // output rows issued
      auto slot_lo = [&](uint32_t slot) { return (((ring + slot * kSlotBytes) >> 4) & 0x3fffu) | (1u << 16); };
#ifdef C2S_CONV_TIMING
      long long dbg_full = 0, dbg_tempty = 0, dbg_mma = 0, dbg_rows = 0;
      const long long dbg_start = clock64();
#endif
      auto take_row = [&]() {                  // wait for the next input row, return the descriptor word of its slot
#ifdef C2S_CONV_TIMING
        const long long dbg_t = clock64();
#endif
        mbar_wait(full(in_slot), (in_phase >> in_slot) & 1u);
#ifdef C2S_CONV_TIMING
        dbg_full += clock64() - dbg_t;
#endif
        const uint32_t lo = slot_lo(in_slot);
        in_phase ^= 1u << in_slot;
        in_slot = in_slot + 1 == kRing ? 0 : in_slot + 1;
        return lo;
      };
      auto release_row = [&]() {               // the oldest resident input row is dead once the products issued so far are done
        umma_commit(empty(free_slot));
        free_slot = free_slot + 1 == kRing ? 0 : free_slot + 1;
      };
      for (int u = blockIdx.x; u < a.n_units; u += gridDim.x) {
        const Unit t = unit_of(a, u);
        // descriptor words of the slots holding rows y - 1, y, y + 1 (reflected at the frame edges, conv.py:76)
        uint32_t dm, d0, dp;
        int resident;                          // input rows of this unit waited for and not yet released
        if (t.y0 == 0) {
          d0 = take_row(), dp = take_row(), dm = dp, resident = 2;   // row -1 = row 1
        } else {
          dm = take_row(), d0 = take_row(), resident = 2;
          if (t.y0 + 1 <= t.hi) dp = take_row(), ++resident;
          else dp = dm;                                               // y0 = H - 1: row H = row H - 2
        }
        for (int y = t.y0; y < t.y1; ++y) {
          const uint32_t buf = o & (kAccBufs - 1);
#ifdef C2S_CONV_TIMING
          const long long dbg_t0 = clock64();
#endif
          if (o >= kAccBufs) mbar_wait(tempty(buf), ((o / kAccBufs) - 1u) & 1u);
#ifdef C2S_CONV_TIMING
          const long long dbg_t1 = clock64();
          dbg_tempty += dbg_t1 - dbg_t0;
#endif
          tc_fence_after();
          const uint32_t d_tmem = tacc + buf * kCN;
          uint32_t b_lo = b_lo0;
#pragma unroll 1
          for (int dyi = 0; dyi < 3; ++dyi) {
            const uint32_t row_lo = dyi == 0 ? dm : (dyi == 1 ? d0 : dp);
#pragma unroll 1
            for (int dxi = 0; dxi < 3; ++dxi) {
              const uint32_t a_lo = row_lo + dxi * 8;   // pixel x + dx sits in row 1 + x + dx of the slot: start (1 + dx) * 128 B
              if (KS == 4) {
#pragma unroll
                for (int ks = 0; ks < KS; ++ks)
                  umma_bf16(d_tmem, desc_from(a_lo + ks * 2), desc_from(b_lo + ks * 2), idesc, (dyi | dxi | ks) != 0);
                b_lo += 512;                            // next tap = next 64-wide chunk of the weights (8192 B)
              } else {                                  // CK = 16: four taps share a chunk
                const int tap = dyi * 3 + dxi;
                umma_bf16(d_tmem, desc_from(a_lo), desc_from(b_lo0 + (tap >> 2) * 512 + (tap & 3) * 2), idesc, tap != 0);
              }
            }
          }
          umma_commit(tfull(buf));
#ifdef C2S_CONV_TIMING
          dbg_mma += clock64() - dbg_t1, ++dbg_rows;
#endif
          ++o;
          // row y - 1 is not needed by later output rows (the first output row of a frame has no row above it)
          if (y > t.lo) release_row(), --resident;
          // slide the window: rows y, y + 1, y + 2
          if (y + 1 < t.y1) {
            dm = d0, d0 = dp;
            if (y + 2 <= t.hi) dp = take_row(), ++resident;
            else dp = dm;                                             // y + 2 = H: reflected onto row H - 2 = the new row y - 1... see below
          }
        }
        while (resident > 0) release_row(), --resident;
      }
#ifdef C2S_CONV_TIMING
      if (blockIdx.x == 0)
        printf("[conv3x3 W=%d CK=%d] issuer of CTA 0: %lld rows, %lld cycles total; per row: wait full %lld, wait tempty %lld, "
               "issue %lld\n", kCW, CK, dbg_rows, clock64() - dbg_start, dbg_full / dbg_rows, dbg_tempty / dbg_rows, dbg_mma / dbg_rows);
#endif
    }
  } else if (warp <= 4) {
    // ---- producers: one 8 channel x 8 pixel block per thread and input row -------------------------------------------
    // A row has BPR = CB * W / 8 blocks.  When that is a whole number of warps below 128 threads (64- and 32-pixel rows, the
    // 16-channel first layer), the 128 producer threads form NG = 128 / BPR groups that take the rows of the (unit, row)
    // sequence in turn, each filling its own ring slots; otherwise all four warps serve every row (spare threads idle).
    constexpr int BPR0 = CB * (kCW / 8);
    constexpr int NG = (BPR0 < 128 && BPR0 % 32 == 0) ? 128 / BPR0 : 1;
    constexpr int BPR = NG > 1 ? BPR0 : 128;
    if constexpr (NG == 1) {
      // every producer thread serves every row (the nested unit / row loops schedule measurably better than the cursor
      // form below when there is nothing to skip: 2.25 vs 2.96 ms for the 64 -> 64 layer with the input normalisation)
      const int ptid = tid - 32;
      const int cb = ptid % CB, pb = ptid / CB;
      const bool active = pb < kCW / 8;
      unsigned g = 0;
      const size_t plane = static_cast<size_t>(a.H) * kCW;
      auto load_row = [&](uint4 (&v)[8], int f, int r) {
        const __nv_bfloat16* src = a.x + (static_cast<size_t>(f) * a.c_in + cb * 8) * plane + static_cast<size_t>(r) * kCW + pb * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          v[i] = (active && cb * 8 + i < a.c_in) ? __ldg(reinterpret_cast<const uint4*>(src + i * plane)) : make_uint4(0, 0, 0, 0);
      };
      // (unit, row) cursor of the newest row whose loads are in flight: two rows ahead of the row being stored (one row of
      // latency hiding was measured as not enough: the producers sat on the long scoreboard)
      int nu = blockIdx.x, nr = 0;
      Unit nt{};
      auto advance = [&]() {  // next (unit, row) in the order every role walks
        if (++nr > nt.hi) {
          nu += gridDim.x;
          if (nu < a.n_units) nt = unit_of(a, nu), nr = nt.lo;
        }
      };
      uint4 vn0[8], vn1[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) vn0[i] = vn1[i] = make_uint4(0, 0, 0, 0);
      if (nu < a.n_units) {
        nt = unit_of(a, nu);
        nr = nt.lo;
        load_row(vn0, nt.f, nr);
        advance();
        if (nu < a.n_units) load_row(vn1, nt.f, nr);
      }
      float sc[8], sh[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) sc[i] = 1.f, sh[i] = 0.f;
      int norm_f = -1;
      for (int u = blockIdx.x; u < a.n_units; u += gridDim.x) {
        const Unit t = unit_of(a, u);
        if (NORM && t.f != norm_f && active) {  // scale / shift of this thread's 8 channels in frame t.f
          norm_f = t.f;
          const int cpg = a.c_in / a.in_groups, spg = a.in_sub / a.in_groups;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int c = cb * 8 + i;
            if (c >= a.c_in) continue;
            const int grp = c / cpg;
            double t1 = 0.0, t2 = 0.0;
            for (int k = 0; k < spg; ++k) {
              t1 += a.in_stats[(static_cast<size_t>(t.f) * a.in_sub + grp * spg + k) * 2];
              t2 += a.in_stats[(static_cast<size_t>(t.f) * a.in_sub + grp * spg + k) * 2 + 1];
            }
            const double n = static_cast<double>(cpg) * a.H * kCW;
            const double mean = t1 / n;
            double var = t2 / n - mean * mean;
            var = var < 0.0 ? 0.0 : var;
            sc[i] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(a.in_eps))) * a.in_gamma[c];
            sh[i] = a.in_beta[c] - static_cast<float>(mean) * sc[i];
          }
        }
        for (int r = t.lo; r <= t.hi; ++r, ++g) {
          uint4 v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = vn0[i], vn0[i] = vn1[i];
          if (NORM) {  // the same arithmetic as group_norm_relu_kernel: fma in fp32, ReLU, round to bf16
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float f[8];
              Elem<__nv_bfloat16>::unpack(v[i], f);
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                f[e] = fmaf(f[e], sc[i], sh[i]);
                if (a.in_relu) f[e] = fmaxf(f[e], 0.f);
              }
              v[i] = Elem<__nv_bfloat16>::pack(f);
            }
          }
          // issue the loads of the row after next: they fly during two rows of waits and stores
          if (nu < a.n_units) {
            advance();
            if (nu < a.n_units) load_row(vn1, nt.f, nr);
          }
          const unsigned slot = g % kRing;
          if (g >= kRing) mbar_wait(empty(slot), ((g / kRing) - 1u) & 1u);
          if (active) {
            unsigned char* sl = ring_ptr + slot * kSlotBytes;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;
              // word j / 2 of channel i holds pixels (j & ~1, j | 1) of that channel
              auto word = [&](int i) -> uint32_t {
                return (j >> 1) == 0 ? v[i].x : ((j >> 1) == 1 ? v[i].y : ((j >> 1) == 2 ? v[i].z : v[i].w));
              };
              uint4 w;
              w.x = __byte_perm(word(0), word(1), sel);
              w.y = __byte_perm(word(2), word(3), sel);
              w.z = __byte_perm(word(4), word(5), sel);
              w.w = __byte_perm(word(6), word(7), sel);
              const int row = pb * 8 + j + 1;
              *reinterpret_cast<uint4*>(sl + row * 128 + ((cb ^ (row & 7)) << 4)) = w;
              if (pb == 0 && j == 1) *reinterpret_cast<uint4*>(sl + ((cb ^ 0) << 4)) = w;                       // pixel -1 = pixel 1
              if (pb == kCW / 8 - 1 && j == 6) *reinterpret_cast<uint4*>(sl + (kCW + 1) * 128 + ((cb ^ ((kCW + 1) & 7)) << 4)) = w;  // pixel W = pixel W - 2
            }
          }
          fence_proxy_async();  // generic stores -> tensor-core (async proxy) reads
          __syncwarp();
          if (lane == 0) mbar_arrive(full(slot));  // hundreds of per-thread arrivals on one mbarrier cost ~1000 cycles per row
        }
      }
    } else {
      const int ptid = tid - 32;
      const int grp = ptid / BPR, btid = ptid % BPR;
      const int cb = btid % CB, pb = btid / CB;
      const bool active = pb < kCW / 8;
      const size_t plane = static_cast<size_t>(a.H) * kCW;
      auto load_row = [&](uint4 (&v)[8], int f, int r) {
        const __nv_bfloat16* src = a.x + (static_cast<size_t>(f) * a.c_in + cb * 8) * plane + static_cast<size_t>(r) * kCW + pb * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          v[i] = (active && cb * 8 + i < a.c_in) ? __ldg(reinterpret_cast<const uint4*>(src + i * plane)) : make_uint4(0, 0, 0, 0);
      };
      // cursors over the (unit, row) sequence every role walks: `cs` the row being stored, `cl` the newest row whose loads
      // are in flight -- two of this group's rows ahead (one row of latency hiding was measured as not enough)
      struct Cursor {
        int u, r, hi, f;  // unit, row, last row of the unit, frame; u >= n_units: behind the end
      };
      auto enter = [&](Cursor& c) {
        if (c.u < a.n_units) {
          const Unit t = unit_of(a, c.u);
          c.r = t.lo, c.hi = t.hi, c.f = t.f;
        }
      };
      auto step = [&](Cursor& c, int n) {
        for (int i = 0; i < n && c.u < a.n_units; ++i)
          if (++c.r > c.hi) c.u += gridDim.x, enter(c);
      };
      Cursor cs{};
      cs.u = blockIdx.x;
      enter(cs);
      step(cs, grp);
      Cursor cl = cs;
      uint4 vn0[8], vn1[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) vn0[i] = vn1[i] = make_uint4(0, 0, 0, 0);
      if (cl.u < a.n_units) load_row(vn0, cl.f, cl.r);
      step(cl, NG);
      if (cl.u < a.n_units) load_row(vn1, cl.f, cl.r);
      float sc[8], sh[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) sc[i] = 1.f, sh[i] = 0.f;
      int norm_f = -1;
      for (unsigned g = grp; cs.u < a.n_units; g += NG, step(cs, NG)) {
        if (NORM && cs.f != norm_f && active) {  // scale / shift of this thread's 8 channels in frame cs.f
          norm_f = cs.f;
          const int cpg = a.c_in / a.in_groups, spg = a.in_sub / a.in_groups;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int c = cb * 8 + i;
            if (c >= a.c_in) continue;
            const int gq = c / cpg;
            double t1 = 0.0, t2 = 0.0;
            for (int k = 0; k < spg; ++k) {
              t1 += a.in_stats[(static_cast<size_t>(norm_f) * a.in_sub + gq * spg + k) * 2];
              t2 += a.in_stats[(static_cast<size_t>(norm_f) * a.in_sub + gq * spg + k) * 2 + 1];
            }
            const double n = static_cast<double>(cpg) * a.H * kCW;
            const double mean = t1 / n;
            double var = t2 / n - mean * mean;
            var = var < 0.0 ? 0.0 : var;
            sc[i] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(a.in_eps))) * a.in_gamma[c];
            sh[i] = a.in_beta[c] - static_cast<float>(mean) * sc[i];
          }
        }
        uint4 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = vn0[i], vn0[i] = vn1[i];
        if (NORM) {  // the same arithmetic as group_norm_relu_kernel: fma in fp32, ReLU, round to bf16
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float f[8];
            Elem<__nv_bfloat16>::unpack(v[i], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              f[e] = fmaf(f[e], sc[i], sh[i]);
              if (a.in_relu) f[e] = fmaxf(f[e], 0.f);
            }
            v[i] = Elem<__nv_bfloat16>::pack(f);
          }
        }
        // issue the loads of this group's row after next: they fly during two rows of waits and stores
        step(cl, NG);
        if (cl.u < a.n_units) load_row(vn1, cl.f, cl.r);
        const unsigned slot = g % kRing;
        if (g >= kRing) mbar_wait(empty(slot), ((g / kRing) - 1u) & 1u);
        if (active) {
          unsigned char* sl = ring_ptr + slot * kSlotBytes;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;
            // word j / 2 of channel i holds pixels (j & ~1, j | 1) of that channel
            auto word = [&](int i) -> uint32_t {
              return (j >> 1) == 0 ? v[i].x : ((j >> 1) == 1 ? v[i].y : ((j >> 1) == 2 ? v[i].z : v[i].w));
            };
            uint4 w;
            w.x = __byte_perm(word(0), word(1), sel);
            w.y = __byte_perm(word(2), word(3), sel);
            w.z = __byte_perm(word(4), word(5), sel);
            w.w = __byte_perm(word(6), word(7), sel);
            const int row = pb * 8 + j + 1;
            *reinterpret_cast<uint4*>(sl + row * 128 + ((cb ^ (row & 7)) << 4)) = w;
            if (pb == 0 && j == 1) *reinterpret_cast<uint4*>(sl + ((cb ^ 0) << 4)) = w;                       // pixel -1 = pixel 1
            if (pb == kCW / 8 - 1 && j == 6) *reinterpret_cast<uint4*>(sl + (kCW + 1) * 128 + ((cb ^ ((kCW + 1) & 7)) << 4)) = w;  // pixel W = pixel W - 2
          }
        }
        fence_proxy_async();  // generic stores -> tensor-core (async proxy) reads
        __syncwarp();
        if (lane == 0) mbar_arrive(full(slot));  // hundreds of per-thread arrivals on one mbarrier cost ~1000 cycles per row
      }
    }
  } else {
    // ---- epilogue: TMEM lanes 32 q .. 32 q + 31 = pixels of the row; the two warps of a quarter split the channels ------
    const int q = warp & 3, half = (warp - 5) >> 2;
    const int x = kM == 128 ? q * 32 + lane : q * 16 + (lane & 15);  // M = 64: rows 16 q .. 16 q + 15 in lanes 0-15
    const bool valid = (kM == 128 || lane < 16) && x < kCW;
    float bias_r[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) bias_r[c] = s_bias[half * 32 + c];
    unsigned o = 0;
    for (int u = blockIdx.x; u < a.n_units; u += gridDim.x) {
      const Unit t = unit_of(a, u);
      float s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f};  // the two 16-channel quarters of this warp's 32 channels
      for (int y = t.y0; y < t.y1; ++y, ++o) {
        const unsigned buf = o & (kAccBufs - 1);
        mbar_wait(tfull(buf), (o / kAccBufs) & 1u);
        tc_fence_after();
        uint32_t r0[32];
        tmem_ld32(tacc + (static_cast<uint32_t>(q * 32) << 16) + buf * kCN + half * 32, r0);
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty(buf));  // the accumulator is in registers: the next row but one may overwrite it
        // 2-byte stores, 64 contiguous bytes per warp instruction.  (Staging the tile in shared memory for 16-byte stores was
        // measured and is SLOWER, 2.17 vs 1.56 ms: with N = 64 the products read 6 KB of shared memory per 48 cycles, i.e. they
        // saturate its bandwidth, and every other shared-memory access -- the staging, even a bias read per channel -- is
        // taken from them.  The bias therefore lives in registers.)
        const size_t cstride = static_cast<size_t>(a.H) * kCW;
        __nv_bfloat16* dst = a.y + ((static_cast<size_t>(t.f) * kCN + half * 32) * a.H + y) * kCW + x;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const float v0 = valid ? __uint_as_float(r0[c]) + bias_r[c] : 0.f;
          if (valid) dst[c * cstride] = __float2bfloat16_rn(v0);
          s1[c >> 4] += v0, s2[c >> 4] = fmaf(v0, v0, s2[c >> 4]);
        }
      }
      if (a.stats != nullptr) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float t1 = warp_sum(s1[k]), t2 = warp_sum(s2[k]);
          if (lane == 0) {
            atomicAdd(a.stats + (static_cast<size_t>(t.f) * kStatQuarters + half * 2 + k) * 2, t1);
            atomicAdd(a.stats + (static_cast<size_t>(t.f) * kStatQuarters + half * 2 + k) * 2 + 1, t2);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tacc, 256);
}

// ---------------------------------------------------------------------------------------------------------------------
// 4x4 / stride 2 / reflect padding 1 (the strided layer of DownConvBlock, conv.py:252-263) from 128-pixel rows, 64 -> 64:
//     y[o, Y, X] = b[o] + sum_{c, ky, kx} W[o, c, ky, kx] x[c, reflect(2 Y + ky - 1), reflect(2 X + kx - 1)]
// The same machinery with three changes:
//   * an input row is stored PARITY-SPLIT: even pixels [0, 2, .., 126, 126'] and odd pixels [1', 1, 3, .., 127] in two
//     halves of the slot (primes: the reflected halo pixels 128 -> 126, -1 -> 1).  Output pixel X reads input pixel
//     2 X + kx - 1, i.e. row X (kx = 0, 1) or X + 1 (kx = 2, 3) of the odd (kx even) / even (kx odd) half: the 16 taps are
//     again start addresses, M = 64 output pixels per product;
//   * the loop is INPUT-stationary: every input row is used by two output rows (three at the reflected frame edges), so a
//     row's 32 products are issued when it arrives -- into the accumulators of those output rows -- and the row is
//     released at once.  The ring needs 5 rows instead of the 6+ an output-stationary order would hold, which is what lets
//     the 128 KB of weights (16 taps x 64 x 64 bf16) stay resident beside it;
//   * an accumulator is handed to the epilogue when the last input row of its output row (2 Y + 2, or H - 1) is through.
// Input rows of 64 or 32 pixels (the second and third down block) run the same M = 64 products with 32 / 16 live rows.
__host__ __device__ constexpr int dsub_bytes(int win) { return ((win / 2 + 1) * 128 + 1023) / 1024 * 1024; }  // one parity half
constexpr int kDRing = 5;
constexpr int kDChunks = 16;       // 16 taps x 64 channels, 64-wide K chunks

__device__ __forceinline__ Unit dunit_of(const ConvArgs& a, int u) {  // a.H = input rows; output rows [y0, y1), input rows [lo, hi]
  Unit t;
  t.f = u / a.units_per_frame;
  const int band = u - t.f * a.units_per_frame;
  t.y0 = band * a.rows_per_unit;
  t.y1 = min(t.y0 + a.rows_per_unit, a.H >> 1);
  t.lo = max(2 * t.y0 - 1, 0);
  t.hi = min(2 * t.y1, a.H - 1);
  return t;
}

template <int WIN>
__global__ void __launch_bounds__(kConvThreads, 1) conv4x4s2_tc_kernel(const ConvArgs a) {
  constexpr int kDW = WIN, kDWo = WIN / 2;
  constexpr int kDSub = dsub_bytes(WIN);  // WIN = 128: 65 pixel rows x 128 B -> 9216
  constexpr int kDSlot = 2 * kDSub;       // [even | odd]
  constexpr int CB = 8;  // 8-channel blocks per pixel
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long bars[2 * kDRing + 2 * kAccBufs];  // full[R], empty[R], tfull[A], tempty[A]
  __shared__ uint32_t tmem_s;
  __shared__ float s_bias[kCN];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t base = (s32(smem_raw) + 1023u) & ~1023u;
  unsigned char* sm = smem_raw + (base - s32(smem_raw));
  const uint32_t ring = base + kDChunks * 8192;
  unsigned char* ring_ptr = sm + kDChunks * 8192;
  const uint32_t bar0 = s32(&bars[0]);
  auto full = [&](int s) { return bar0 + 8u * s; };
  auto empty = [&](int s) { return bar0 + 8u * (kDRing + s); };
  auto tfull = [&](int b) { return bar0 + 8u * (2 * kDRing + b); };
  auto tempty = [&](int b) { return bar0 + 8u * (2 * kDRing + kAccBufs + b); };
  const int Ho = a.H >> 1;

  if (tid == 0) {
    for (int s = 0; s < kDRing; ++s) mbar_init(full(s), 4), mbar_init(empty(s), 1);
    for (int b = 0; b < kAccBufs; ++b) mbar_init(tfull(b), 1), mbar_init(tempty(b), 8);
    fence_mbarrier_init();
  }
  if (warp == 0) {
    tmem_alloc(s32(&tmem_s), 256);
    tmem_relinquish();
  }
  if (tid < kCN) s_bias[tid] = a.bias != nullptr ? a.bias[tid] : 0.f;
  for (int i = tid; i < kCN * kDChunks * 8; i += kConvThreads) {  // resident weights, as in conv3x3_tc_kernel
    const int c16 = i & 7, j = (i >> 3) % kDChunks, n = i / (8 * kDChunks);
    const uint4 v = *reinterpret_cast<const uint4*>(a.wp + static_cast<size_t>(n) * (kDChunks * 64) + j * 64 + c16 * 8);
    *reinterpret_cast<uint4*>(sm + j * 8192 + n * 128 + ((c16 ^ (n & 7)) << 4)) = v;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tacc = tmem_s;

  if (warp == 0) {
    // ---- MMA issuer ----------------------------------------------------------------------------------------------
    if (elect_one()) {
      static constexpr uint32_t idesc = umma_idesc_bf16(64, kCN);  // M = 64 (kDWo live rows)
      const uint32_t b_lo0 = ((base >> 4) & 0x3fffu) | (1u << 16);
      uint32_t in_slot = 0, in_phase = 0;
      uint32_t o = 0;  // output rows handed out so far (accumulator = o & 3)
#ifdef C2S_CONV_TIMING
      long long dbg_full = 0, dbg_tempty = 0, dbg_rows = 0;
      const long long dbg_start = clock64();
#endif
      for (int u = blockIdx.x; u < a.n_units; u += gridDim.x) {
        const Unit t = dunit_of(a, u);
        const uint32_t obase = o;
        int started = 0;  // output rows of this unit that have received their first product
        for (int r = t.lo; r <= t.hi; ++r) {
#ifdef C2S_CONV_TIMING
          const long long dbg_t = clock64();
#endif
          mbar_wait(full(in_slot), (in_phase >> in_slot) & 1u);
#ifdef C2S_CONV_TIMING
          dbg_full += clock64() - dbg_t, ++dbg_rows;
#endif
          tc_fence_after();
          const uint32_t row_lo = (((ring + in_slot * kDSlot) >> 4) & 0x3fffu) | (1u << 16);
          // the output rows fed by input row v (v = r, or the row r stands in for at a reflected frame edge)
          auto contribute = [&](int v) {
#pragma unroll 1
            for (int ky = 0; ky < 4; ++ky) {
              const int num = v + 1 - ky;  // = 2 Y
              if (num & 1) continue;
              const int Y = num >> 1;
              if (Y < t.y0 || Y >= t.y1) continue;
              const int rel = Y - t.y0;
              const uint32_t oi = obase + rel, buf = oi & (kAccBufs - 1);
              const bool fresh = rel == started;
              if (fresh) {
                ++started;
#ifdef C2S_CONV_TIMING
                const long long dbg_t2 = clock64();
#endif
                if (oi >= kAccBufs) mbar_wait(tempty(buf), ((oi / kAccBufs) - 1u) & 1u);
#ifdef C2S_CONV_TIMING
                dbg_tempty += clock64() - dbg_t2;
#endif
                tc_fence_after();
              }
              const uint32_t d_tmem = tacc + buf * kCN;
              // 16 products with compile-time offsets from three bases (even half, odd half, the tap row of the weights):
              // input pixel 2 X + kx - 1 = odd half for even kx, even half for odd kx; row X (+ 1 for kx >= 2)
              const uint32_t a_even = row_lo, a_odd = row_lo + static_cast<uint32_t>(kDSub >> 4);
              const uint32_t b_row = b_lo0 + ky * 2048;
#pragma unroll
              for (int kx = 0; kx < 4; ++kx) {
                const uint32_t a_lo = ((kx & 1) ? a_even : a_odd) + (kx >> 1) * 8;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  umma_bf16(d_tmem, desc_from(a_lo + ks * 2), desc_from(b_row + kx * 512 + ks * 2), idesc,
                            (kx | ks) != 0 ? 1u : (fresh ? 0u : 1u));
              }
            }
          };
          contribute(r);
          if (r == 1) contribute(-1);           // row -1 = row 1
          if (r == a.H - 2) contribute(a.H);    // row H = row H - 2
          umma_commit(empty(in_slot));          // the row is dead once the products issued so far are done
          in_phase ^= 1u << in_slot;
          in_slot = in_slot + 1 == kDRing ? 0 : in_slot + 1;
          // output rows whose last input row this was
          if (!(r & 1) && r >= 2) {
            const int yc = (r - 2) >> 1;
            if (yc >= t.y0 && yc < t.y1) umma_commit(tfull((obase + yc - t.y0) & (kAccBufs - 1)));
          }
          if (r == a.H - 1 && t.y1 == Ho) umma_commit(tfull((obase + Ho - 1 - t.y0) & (kAccBufs - 1)));
        }
        o += t.y1 - t.y0;
      }
#ifdef C2S_CONV_TIMING
      if (blockIdx.x == 0)
        printf("[conv4x4s2 W=%d] issuer of CTA 0: %lld input rows, %lld cycles total = %lld per row; per row: wait full %lld, "
               "wait tempty %lld\n", kDW, dbg_rows, clock64() - dbg_start, (clock64() - dbg_start) / dbg_rows, dbg_full / dbg_rows,
               dbg_tempty / dbg_rows);
#endif
    }
  } else if (warp <= 4) {
    // ---- producers: one 8 channel x 8 pixel block per thread and input row, stored parity-split ---------------------------
    const int ptid = tid - 32;
    const int cb = ptid % CB, pb = ptid / CB;  // 8 x 16 blocks = 128 threads
    const bool active = pb < kDW / 8;
    unsigned g = 0;
    const size_t plane = static_cast<size_t>(a.H) * kDW;
    auto load_row = [&](uint4 (&v)[8], int f, int r) {
      const __nv_bfloat16* src = a.x + (static_cast<size_t>(f) * a.c_in + cb * 8) * plane + static_cast<size_t>(r) * kDW + pb * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = active ? __ldg(reinterpret_cast<const uint4*>(src + i * plane)) : make_uint4(0, 0, 0, 0);
    };
    int nu = blockIdx.x, nr = 0;
    Unit nt{};
    auto advance = [&]() {
      if (++nr > nt.hi) {
        nu += gridDim.x;
        if (nu < a.n_units) nt = dunit_of(a, nu), nr = nt.lo;
      }
    };
    uint4 vn0[8], vn1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) vn0[i] = vn1[i] = make_uint4(0, 0, 0, 0);
    if (nu < a.n_units) {
      nt = dunit_of(a, nu);
      nr = nt.lo;
      load_row(vn0, nt.f, nr);
      advance();
      if (nu < a.n_units) load_row(vn1, nt.f, nr);
    }
    for (int u = blockIdx.x; u < a.n_units; u += gridDim.x) {
      const Unit t = dunit_of(a, u);
      for (int r = t.lo; r <= t.hi; ++r, ++g) {
        uint4 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = vn0[i], vn0[i] = vn1[i];
        if (nu < a.n_units) {
          advance();
          if (nu < a.n_units) load_row(vn1, nt.f, nr);
        }
        const unsigned slot = g % kDRing;
        if (g >= kDRing) mbar_wait(empty(slot), ((g / kDRing) - 1u) & 1u);
        unsigned char* sl = ring_ptr + slot * kDSlot;
        if (active) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;
            auto word = [&](int i) -> uint32_t {
              return (j >> 1) == 0 ? v[i].x : ((j >> 1) == 1 ? v[i].y : ((j >> 1) == 2 ? v[i].z : v[i].w));
            };
            uint4 w;
            w.x = __byte_perm(word(0), word(1), sel);
            w.y = __byte_perm(word(2), word(3), sel);
            w.z = __byte_perm(word(4), word(5), sel);
            w.w = __byte_perm(word(6), word(7), sel);
            // pixel 8 pb + j: even -> row (8 pb + j) / 2 of the even half, odd -> row (8 pb + j + 1) / 2 of the odd half
            const int row = 4 * pb + ((j + 1) >> 1);
            unsigned char* half = sl + ((j & 1) ? kDSub : 0);
            *reinterpret_cast<uint4*>(half + row * 128 + ((cb ^ (row & 7)) << 4)) = w;
            if (pb == 0 && j == 1) *reinterpret_cast<uint4*>(sl + kDSub + ((cb ^ 0) << 4)) = w;  // pixel -1 = pixel 1
            if (pb == kDW / 8 - 1 && j == 6)                                                       // pixel W = pixel W - 2
              *reinterpret_cast<uint4*>(sl + kDWo * 128 + ((cb ^ (kDWo & 7)) << 4)) = w;
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(full(slot));
      }
    }
  } else {
    // ---- epilogue: an M = 64 accumulator keeps rows 16 q .. 16 q + 15 in lanes 0-15 of TMEM quarter q ---------------------
    const int q = warp & 3, half = (warp - 5) >> 2;
    const int x = q * 16 + (lane & 15);
    const bool valid = lane < 16 && x < kDWo;
    float bias_r[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) bias_r[c] = s_bias[half * 32 + c];
    unsigned o = 0;
    for (int u = blockIdx.x; u < a.n_units; u += gridDim.x) {
      const Unit t = dunit_of(a, u);
      float s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f};
      for (int y = t.y0; y < t.y1; ++y, ++o) {
        const unsigned buf = o & (kAccBufs - 1);
        mbar_wait(tfull(buf), (o / kAccBufs) & 1u);
        tc_fence_after();
        uint32_t r0[32];
        tmem_ld32(tacc + (static_cast<uint32_t>(q * 32) << 16) + buf * kCN + half * 32, r0);
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty(buf));
        const size_t cstride = static_cast<size_t>(Ho) * kDWo;
        __nv_bfloat16* dst = a.y + ((static_cast<size_t>(t.f) * kCN + half * 32) * Ho + y) * kDWo + x;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const float v0 = valid ? __uint_as_float(r0[c]) + bias_r[c] : 0.f;
          if (valid) dst[c * cstride] = __float2bfloat16_rn(v0);
          s1[c >> 4] += v0, s2[c >> 4] = fmaf(v0, v0, s2[c >> 4]);
        }
      }
      if (a.stats != nullptr) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float t1 = warp_sum(s1[k]), t2 = warp_sum(s2[k]);
          if (lane == 0) {
            atomicAdd(a.stats + (static_cast<size_t>(t.f) * kStatQuarters + half * 2 + k) * 2, t1);
            atomicAdd(a.stats + (static_cast<size_t>(t.f) * kStatQuarters + half * 2 + k) * 2 + 1, t2);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tacc, 256);
}

// ---------------------------------------------------------------------------------------------------------------------
// 3x3 / stride 1 / reflect padding 1 on 16-pixel-wide frames (conv1 / conv2 of U-TAE's last down block, 16 x 16 pixels),
// c_in and c_out in {64, 128}.  A 16-pixel row is too narrow for one image row per product, so a unit is a whole frame:
//   * four producer warps store the frame reflect-padded to (H + 2) x 18 pixels, pixel-major, one slot [pixel][64 channels]
//     per 64-channel K chunk, in the K-major 128-byte-swizzled layout of conv3x3_tc_kernel.  Two frame buffers: the next
//     frame is staged while the current one computes;
//   * output pixel (y, x) is accumulator row p = 18 y + x and tap (ky, kx) reads the same slot from row p + 18 ky + kx, so
//     every tap is a start address.  M = 128 tiles cover p in [0, 18 H): tile t starts at min(128 t, 18 H - 128) -- the
//     last tile overlaps the one before it rather than reading past the slot; the two junk columns of a row and the
//     overlapped rows are computed and not stored;
//   * the weights (c_out x 9 c_in bf16, 295 KB at 128 -> 128: too large to stay resident) stream from L2 by TMA, one
//     [c_out][64] box per (tap, K chunk) through a ring of kWStages.  The loop is weight-stationary: each box serves every
//     tile of the frame before the next one is waited for;
//   * N = c_out (M 128 x N 128 x K 16 products for the 128-channel layers).  Tensor memory holds 512 / c_out tile
//     accumulators in a ring; the issuer waits for a tile's accumulator just before its first product, so the products
//     of a frame start while the epilogue still drains the previous one.
constexpr int kW16Threads = 448;     // warp 0: MMA issuer, warp 1: weight TMA, warps 2-5: producers, warps 6-13: epilogue
constexpr int kW16Rows = 18;         // padded row pitch in pixels
constexpr int kW16MaxH = 16;
// one K-chunk slot: (16 + 2) x 18 pixel rows of 128 B; the last tile reads up to row 18 H + 37 (325 at H = 16), below the
// 328 rows of the slot
constexpr int kW16Slot = ((kW16MaxH + 2) * kW16Rows * 128 + 1023) / 1024 * 1024;
constexpr int kWStages = 3;
constexpr int kW16AccCols = 512;

__host__ __device__ constexpr size_t w16_smem_bytes(int kc, int n) {
  return static_cast<size_t>(2) * kc * kW16Slot + static_cast<size_t>(kWStages) * n * 128 + 1024;
}

template <int KC, int N, bool NORM>
__global__ void __launch_bounds__(kW16Threads, 1) conv3x3_w16_tc_kernel(const __grid_constant__ CUtensorMap wmap, const ConvArgs a) {
  constexpr int CIN = KC * 64;
  constexpr int kAccN = kW16AccCols / N;   // tile accumulators in tensor memory (4 or 8)
  constexpr int kWBox = N * 128;           // one weight box [N][64] bf16
  constexpr int kJ = 9 * KC;               // weight boxes per frame
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long bars[4 + 2 * kWStages + 2 * kAccN];  // in_full[2], in_empty[2], wfull, wempty, tfull, tempty
  __shared__ uint32_t tmem_s;
  __shared__ __align__(16) float s_bias[N];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t base = (s32(smem_raw) + 1023u) & ~1023u;
  unsigned char* sm = smem_raw + (base - s32(smem_raw));
  const uint32_t wring = base + 2 * KC * kW16Slot;
  const uint32_t bar0 = s32(&bars[0]);
  auto in_full = [&](int b) { return bar0 + 8u * b; };
  auto in_empty = [&](int b) { return bar0 + 8u * (2 + b); };
  auto wfull = [&](int s) { return bar0 + 8u * (4 + s); };
  auto wempty = [&](int s) { return bar0 + 8u * (4 + kWStages + s); };
  auto tfull = [&](int b) { return bar0 + 8u * (4 + 2 * kWStages + b); };
  auto tempty = [&](int b) { return bar0 + 8u * (4 + 2 * kWStages + kAccN + b); };
  const int P = a.H * kW16Rows;                  // accumulator rows that hold outputs
  const int n_tiles = (P + 127) / 128;
  const int last_start = P > 128 ? P - 128 : 0;

  if (tid == 0) {
    for (int b = 0; b < 2; ++b) mbar_init(in_full(b), 4), mbar_init(in_empty(b), 1);   // one arrival per producer warp
    for (int s = 0; s < kWStages; ++s) mbar_init(wfull(s), 1), mbar_init(wempty(s), 1);
    for (int b = 0; b < kAccN; ++b) mbar_init(tfull(b), 1), mbar_init(tempty(b), 8);   // one arrival per epilogue warp
    fence_mbarrier_init();
  }
  if (warp == 0) {
    tmem_alloc(s32(&tmem_s), kW16AccCols);
    tmem_relinquish();
  }
  if (tid < N) s_bias[tid] = a.bias != nullptr ? a.bias[tid] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tacc = tmem_s;

  if (warp == 0) {
    // ---- MMA issuer ----------------------------------------------------------------------------------------------
    if (elect_one()) {
      static constexpr uint32_t idesc = umma_idesc_bf16(128, N);
      const uint32_t w_lo0 = ((wring >> 4) & 0x3fffu) | (1u << 16);
      uint32_t ws = 0, wphase = 0;             // weight stage of the next box; bit s = parity of stage s
      uint32_t o = 0;                          // tiles issued
#ifdef C2S_CONV_TIMING
      long long dbg_in = 0, dbg_w = 0, dbg_tempty = 0, dbg_frames = 0;
      const long long dbg_start = clock64();
#endif
      int i = 0;
      for (int f = blockIdx.x; f < a.frames; f += gridDim.x, ++i) {
        const uint32_t fb = i & 1;
#ifdef C2S_CONV_TIMING
        long long dbg_t = clock64();
#endif
        mbar_wait(in_full(fb), (i >> 1) & 1);
#ifdef C2S_CONV_TIMING
        dbg_in += clock64() - dbg_t;
#endif
        tc_fence_after();
        const uint32_t a_lo0 = (((base + fb * KC * kW16Slot) >> 4) & 0x3fffu) | (1u << 16);
        int j = 0;
#pragma unroll 1
        for (int ky = 0; ky < 3; ++ky) {
#pragma unroll 1
          for (int kx = 0; kx < 3; ++kx) {
#pragma unroll 1
            for (int kc = 0; kc < KC; ++kc, ++j) {
#ifdef C2S_CONV_TIMING
              dbg_t = clock64();
#endif
              mbar_wait(wfull(ws), (wphase >> ws) & 1u);
#ifdef C2S_CONV_TIMING
              dbg_w += clock64() - dbg_t;
#endif
              tc_fence_after();
              const uint32_t b_lo = w_lo0 + ws * (kWBox >> 4);
              // tap (ky, kx) = start row 18 ky + kx of the K chunk's slot (8 x 16 B per pixel row)
              const uint32_t a_lo = a_lo0 + kc * (kW16Slot >> 4) + (ky * kW16Rows + kx) * 8;
#pragma unroll 1
              for (int t = 0; t < n_tiles; ++t) {
                const uint32_t ot = o + t, buf = ot % kAccN;
                if (j == 0) {
#ifdef C2S_CONV_TIMING
                  dbg_t = clock64();
#endif
                  if (ot >= kAccN) mbar_wait(tempty(buf), ((ot / kAccN) - 1u) & 1u);
#ifdef C2S_CONV_TIMING
                  dbg_tempty += clock64() - dbg_t;
#endif
                  tc_fence_after();
                }
                const uint32_t d_tmem = tacc + buf * N;
                const uint32_t at = a_lo + min(t * 128, last_start) * 8;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  umma_bf16(d_tmem, desc_from(at + ks * 2), desc_from(b_lo + ks * 2), idesc, (j | ks) != 0);
                if (j == kJ - 1) umma_commit(tfull(buf));
              }
              umma_commit(wempty(ws));         // the box is dead once the products issued so far are done
              wphase ^= 1u << ws;
              ws = ws + 1 == kWStages ? 0 : ws + 1;
            }
          }
        }
        umma_commit(in_empty(fb));
        o += n_tiles;
#ifdef C2S_CONV_TIMING
        ++dbg_frames;
#endif
      }
#ifdef C2S_CONV_TIMING
      if (blockIdx.x == 0 && dbg_frames > 0)
        printf("[conv3x3 W=16 c_in=%d c_out=%d H=%d] issuer of CTA 0: %lld frames, %lld cycles per frame; per frame: wait input "
               "%lld, wait weights %lld, wait tempty %lld\n", CIN, N, a.H, dbg_frames, (clock64() - dbg_start) / dbg_frames,
               dbg_in / dbg_frames, dbg_w / dbg_frames, dbg_tempty / dbg_frames);
#endif
    }
  } else if (warp == 1) {
    // ---- weight boxes: TMA from the prepared weights [N][9 CIN], box (tap, K chunk) = columns 64 j .. 64 j + 63 ---------
    if (elect_one()) {
      uint32_t s = 0, round = 0;               // stage of the next box, passes through the ring so far
      for (int f = blockIdx.x; f < a.frames; f += gridDim.x) {
        for (int j = 0; j < kJ; ++j) {
          if (round > 0) mbar_wait(wempty(s), (round - 1u) & 1u);
          mbar_expect_tx(wfull(s), kWBox);
          tma_load_2d(wring + s * kWBox, &wmap, j * 64, 0, wfull(s));
          if (++s == kWStages) s = 0, ++round;
        }
      }
    }
  } else if (warp <= 5) {
    // ---- producers: one 8 channel x 8 pixel block per thread and step; thread = (channel block, first pixel block) ------
    constexpr int CB = CIN / 8;
    constexpr int TPB = 128 / CB;               // threads sharing a channel block (16 or 8)
    const int ptid = tid - 64;
    const int cb = ptid % CB, p0 = ptid / CB;   // pixel block pb = (row pb / 2, half pb & 1); this thread: p0, p0 + TPB, ..
    const int piece = cb & 7;
    const int nblk = 2 * a.H;
    const bool active = p0 < nblk;
    const size_t plane = static_cast<size_t>(a.H) * 16;
    auto load_blk = [&](uint4 (&v)[8], int f, int pb) {
      const __nv_bfloat16* src = a.x + (static_cast<size_t>(f) * CIN + cb * 8) * plane + (pb >> 1) * 16 + (pb & 1) * 8;
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = __ldg(reinterpret_cast<const uint4*>(src + k * plane));
    };
    // the next block to load: one block of latency hiding, across frame boundaries
    int lf = blockIdx.x, lp = p0;
    uint4 vn[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) vn[k] = make_uint4(0, 0, 0, 0);
    if (active && lf < a.frames) load_blk(vn, lf, lp);
    float sc[8], sh[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) sc[k] = 1.f, sh[k] = 0.f;
    int i = 0;
    for (int f = blockIdx.x; f < a.frames; f += gridDim.x, ++i) {
      const uint32_t fb = i & 1;
      if (NORM && active) {  // scale / shift of this thread's 8 channels in frame f, as in conv3x3_tc_kernel
        const int cpg = CIN / a.in_groups, spg = a.in_sub / a.in_groups;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = cb * 8 + k;
          const int grp = c / cpg;
          double t1 = 0.0, t2 = 0.0;
          for (int s = 0; s < spg; ++s) {
            t1 += a.in_stats[(static_cast<size_t>(f) * a.in_sub + grp * spg + s) * 2];
            t2 += a.in_stats[(static_cast<size_t>(f) * a.in_sub + grp * spg + s) * 2 + 1];
          }
          const double n = static_cast<double>(cpg) * a.H * 16;
          const double mean = t1 / n;
          double var = t2 / n - mean * mean;
          var = var < 0.0 ? 0.0 : var;
          sc[k] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(a.in_eps))) * a.in_gamma[c];
          sh[k] = a.in_beta[c] - static_cast<float>(mean) * sc[k];
        }
      }
      if (i >= 2) mbar_wait(in_empty(fb), ((i >> 1) - 1) & 1);
      unsigned char* sl = sm + (fb * KC + (cb >> 3)) * kW16Slot;
      for (int pb = p0; active && pb < nblk; pb += TPB) {
        uint4 v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = vn[k];
        lp += TPB;
        if (lp >= nblk) lf += gridDim.x, lp = p0;
        if (lf < a.frames) load_blk(vn, lf, lp);
        if (NORM) {  // the same arithmetic as group_norm_relu_kernel: fma in fp32, ReLU, round to bf16
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float e[8];
            Elem<__nv_bfloat16>::unpack(v[k], e);
#pragma unroll
            for (int m = 0; m < 8; ++m) {
              e[m] = fmaf(e[m], sc[k], sh[k]);
              if (a.in_relu) e[m] = fmaxf(e[m], 0.f);
            }
            v[k] = Elem<__nv_bfloat16>::pack(e);
          }
        }
        const int y = pb >> 1, h = pb & 1;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;
          // word j / 2 of channel k holds pixels (j & ~1, j | 1) of that channel
          auto word = [&](int k) -> uint32_t {
            return (j >> 1) == 0 ? v[k].x : ((j >> 1) == 1 ? v[k].y : ((j >> 1) == 2 ? v[k].z : v[k].w));
          };
          uint4 w;
          w.x = __byte_perm(word(0), word(1), sel);
          w.y = __byte_perm(word(2), word(3), sel);
          w.z = __byte_perm(word(4), word(5), sel);
          w.w = __byte_perm(word(6), word(7), sel);
          // pixel (y, 8 h + j) -> padded (y + 1, 8 h + j + 1); reflected copies: column 0 = column 2, column 17 = column 15,
          // row 0 = row 2, row H + 1 = row H - 1 (padded coordinates)
          auto put_row = [&](int R) {
            auto st = [&](int col) {
              const int r = R * kW16Rows + col;
              *reinterpret_cast<uint4*>(sl + r * 128 + ((piece ^ (r & 7)) << 4)) = w;
            };
            st(8 * h + j + 1);
            if (h == 0 && j == 1) st(0);
            if (h == 1 && j == 6) st(17);
          };
          put_row(y + 1);
          if (y == 1) put_row(0);
          if (y == a.H - 2) put_row(a.H + 1);
        }
      }
      fence_proxy_async();  // generic stores -> tensor-core (async proxy) reads
      __syncwarp();
      if (lane == 0) mbar_arrive(in_full(fb));
    }
  } else {
    // ---- epilogue: TMEM lanes 32 q .. 32 q + 31 = accumulator rows of a tile; the two warps of a quarter split the channels
    constexpr int NH = N / 2, NCH = NH / 32, QW = N / 4;  // channels per warp, 32-column loads, channels per stats quarter
    const int q = warp & 3, half = (warp - 6) >> 2;
    const size_t cstride = static_cast<size_t>(a.H) * 16;
    unsigned o = 0;
    for (int f = blockIdx.x; f < a.frames; f += gridDim.x) {
      float s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f};  // the two stats quarters of this warp's channels
      for (int t = 0; t < n_tiles; ++t, ++o) {
        const unsigned buf = o % kAccN;
        mbar_wait(tfull(buf), (o / kAccN) & 1u);
        tc_fence_after();
        uint32_t r[NCH][32];
#pragma unroll
        for (int cc = 0; cc < NCH; ++cc)
          tmem_ld32(tacc + (static_cast<uint32_t>(q * 32) << 16) + buf * N + half * NH + cc * 32, r[cc]);
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty(buf));  // the accumulator is in registers
        const int p = min(t * 128, last_start) + q * 32 + lane;
        const int y = p / kW16Rows, x = p - y * kW16Rows;
        const bool valid = x < 16 && p < P && p >= t * 128;  // junk columns, tail rows, rows the previous tile stored
        __nv_bfloat16* dst = a.y + ((static_cast<size_t>(f) * N + half * NH) * a.H + y) * 16 + x;
#pragma unroll
        for (int cc = 0; cc < NCH; ++cc) {
#pragma unroll
          for (int c4 = 0; c4 < 8; ++c4) {
            const float4 b4 = *reinterpret_cast<const float4*>(&s_bias[half * NH + cc * 32 + c4 * 4]);
            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = cc * 32 + c4 * 4 + e;
              const float v0 = valid ? __uint_as_float(r[cc][c4 * 4 + e]) + bb[e] : 0.f;
              if (valid) dst[c * cstride] = __float2bfloat16_rn(v0);
              s1[c / QW] += v0, s2[c / QW] = fmaf(v0, v0, s2[c / QW]);
            }
          }
        }
      }
      if (a.stats != nullptr) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float t1 = warp_sum(s1[k]), t2 = warp_sum(s2[k]);
          if (lane == 0) {
            atomicAdd(a.stats + (static_cast<size_t>(f) * kStatQuarters + half * 2 + k) * 2, t1);
            atomicAdd(a.stats + (static_cast<size_t>(f) * kStatQuarters + half * 2 + k) * 2 + 1, t2);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tacc, kW16AccCols);
}

// weight[c_out][c_in][3][3] fp32 -> wp[c_out][chunks * 64] bf16 with k = tap * CK + c (zero for c >= c_in and behind 9 CK)
__global__ void conv_weight_prep_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wp, int c_out, int c_in, int ck,
                                        int k_total, int taps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c_out * k_total) return;
  const int n = i / k_total, k = i - n * k_total;
  const int tap = k / ck, c = k - tap * ck;
  float v = 0.f;
  if (tap < taps && c < c_in) v = w[(static_cast<size_t>(n) * c_in + c) * taps + tap];
  wp[i] = __float2bfloat16_rn(v);
}

// ---- GroupNorm over (channels of the group) x H x W of one frame -----------------------------------------------------
constexpr int kStatThreads = 512;

template <typename T>
__global__ void __launch_bounds__(kStatThreads) group_stats_kernel(const T* __restrict__ x, float* __restrict__ stats, size_t span) {
  // block (g, f): the group's channels are contiguous in NCHW: one span of cpg * H * W elements
  const size_t blk = static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x;
  const T* p = x + blk * span;
  float s1 = 0.f, s2 = 0.f;
  for (size_t i = threadIdx.x; i < span; i += kStatThreads) {
    const float v = Elem<T>::load(p + i);
    s1 += v, s2 = fmaf(v, v, s2);
  }
  __shared__ double r1[kStatThreads / 32], r2[kStatThreads / 32];
  s1 = warp_sum(s1), s2 = warp_sum(s2);
  if ((threadIdx.x & 31) == 0) r1[threadIdx.x >> 5] = s1, r2[threadIdx.x >> 5] = s2;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int i = 0; i < kStatThreads / 32; ++i) t1 += r1[i], t2 += r2[i];
    stats[blk * 2] = static_cast<float>(t1), stats[blk * 2 + 1] = static_cast<float>(t2);
  }
}

struct NormArgs {
  const void* x;         // raw [frames][C][hw]
  const void* residual;  // [frames][C][hw] or nullptr
  void* out;
  const float* stats;    // [frames][n_sub][2]
  const float* gamma;
  const float* beta;
  int C, hw, n_groups, n_sub, relu;
  float eps;
};

// kNormItems 16-byte vectors per thread: four independent loads in flight, 16 KB (bf16) per block; 1 for tiny planes
template <typename T, int kNormItems>
__global__ void __launch_bounds__(256) group_norm_relu_kernel(const NormArgs a) {
  constexpr int VEC = Elem<T>::kVec;
  constexpr uint32_t SPAN = 256 * kNormItems * VEC;  // elements per block
  __shared__ float s_sc[256], s_sh[256];  // scale / shift of the channels this block touches (the host checks <= 256)
  const int f = blockIdx.y;
  // 32-bit arithmetic inside a frame (the host checks C * hw < 2^31): 64-bit divisions cost ~100 instructions per vector
  const uint32_t hw = static_cast<uint32_t>(a.hw), per_frame = static_cast<uint32_t>(a.C) * hw;
  const uint32_t e0 = blockIdx.x * SPAN;
  const uint32_t c_first = e0 / hw;
  uint32_t e_last = e0 + SPAN - 1;
  e_last = e_last < per_frame ? e_last : per_frame - 1;
  const int n_ch = static_cast<int>(e_last / hw - c_first) + 1;
  if (static_cast<int>(threadIdx.x) < n_ch) {
    const int c = static_cast<int>(c_first) + threadIdx.x;
    const int cpg = a.C / a.n_groups, g = c / cpg, spg = a.n_sub / a.n_groups;
    double t1 = 0.0, t2 = 0.0;
    for (int k = 0; k < spg; ++k) {
      t1 += a.stats[(static_cast<size_t>(f) * a.n_sub + g * spg + k) * 2];
      t2 += a.stats[(static_cast<size_t>(f) * a.n_sub + g * spg + k) * 2 + 1];
    }
    const double n = static_cast<double>(cpg) * a.hw;
    const double mean = t1 / n;
    double var = t2 / n - mean * mean;
    var = var < 0.0 ? 0.0 : var;
    const float sc = static_cast<float>(1.0 / sqrt(var + static_cast<double>(a.eps))) * a.gamma[c];
    s_sc[threadIdx.x] = sc;
    s_sh[threadIdx.x] = a.beta[c] - static_cast<float>(mean) * sc;
  }
  // the loads go out before the barrier: they travel while the scale / shift of the block is formed
  const size_t base = static_cast<size_t>(f) * per_frame;
  uint4 xv[kNormItems], rv[kNormItems];
  uint32_t e[kNormItems];
#pragma unroll
  for (int k = 0; k < kNormItems; ++k) {
    e[k] = e0 + (static_cast<uint32_t>(k) * 256 + threadIdx.x) * VEC;
    xv[k] = rv[k] = make_uint4(0, 0, 0, 0);
    if (e[k] < per_frame) {
      xv[k] = *reinterpret_cast<const uint4*>(static_cast<const T*>(a.x) + base + e[k]);  // plain load: out may alias x
      if (a.residual != nullptr) rv[k] = ld_stream_v4(static_cast<const T*>(a.residual) + base + e[k]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kNormItems; ++k) {
    if (e[k] >= per_frame) continue;
    const uint32_t ci = e[k] / hw - c_first;  // hw % VEC == 0: the vector stays inside one channel
    const float sc = s_sc[ci], sh = s_sh[ci];
    float v[VEC];
    Elem<T>::unpack(xv[k], v);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      v[i] = fmaf(v[i], sc, sh);
      if (a.relu) v[i] = fmaxf(v[i], 0.f);
    }
    if (a.residual != nullptr) {
      float r[VEC];
      Elem<T>::unpack(rv[k], r);
#pragma unroll
      for (int i = 0; i < VEC; ++i) v[i] += r[i];
    }
    *reinterpret_cast<uint4*>(static_cast<T*>(a.out) + base + e[k]) = Elem<T>::pack(v);
  }
}

int conv_ck(int c_in) { return c_in <= 16 ? 16 : 64; }
int conv_chunks(int ck) { return (9 * ck + 63) / 64; }
// the strided layer of DownConvBlock on the tensor cores: 4x4 / stride 2 / padding 1 from 128-pixel rows, 64 -> 64 channels
bool conv_is_down(const c2s_conv_desc& d) {
  return d.kernel == 4 && d.stride == 2 && d.padding == 1 && (d.W == 128 || d.W == 64 || d.W == 32) && d.H >= 4 && d.H % 2 == 0 && d.c_in == 64 &&
         d.c_out == kCN && d.dtype == C2S_BF16 && d.frames > 0;
}
// 3x3 / stride 1 / padding 1 on whole 16-pixel-wide frames, 64 or 128 channels in and out (conv3x3_w16_tc_kernel)
bool conv_is_w16(const c2s_conv_desc& d) {
  return d.kernel == 3 && d.stride == 1 && d.padding == 1 && d.W == 16 && d.H >= 2 && d.H <= kW16MaxH &&
         (d.c_in == 64 || d.c_in == 128) && (d.c_out == 64 || d.c_out == 128) && d.dtype == C2S_BF16 && d.frames > 0;
}

}  // namespace
}  // namespace c2s

extern "C" {

int c2s_conv2d_supported(const c2s_conv_desc* d) {
  if (d == nullptr) return 0;
  if (c2s::conv_is_down(*d) || c2s::conv_is_w16(*d)) return 1;
  return d->kernel == 3 && d->stride == 1 && d->padding == 1 && (d->W == 128 || d->W == 64 || d->W == 32) && d->H >= 2 && d->c_out == c2s::kCN &&
         (d->c_in <= 16 || d->c_in == 64) && d->c_in >= 1 && d->dtype == C2S_BF16 && d->frames > 0;
}

size_t c2s_conv2d_workspace_bytes(const c2s_conv_desc* d) {
  if (!c2s_conv2d_supported(d)) return 0;
  if (c2s::conv_is_down(*d)) return static_cast<size_t>(c2s::kCN) * c2s::kDChunks * 64 * sizeof(__nv_bfloat16);
  if (c2s::conv_is_w16(*d)) return static_cast<size_t>(d->c_out) * 9 * d->c_in * sizeof(__nv_bfloat16);
  return static_cast<size_t>(c2s::kCN) * c2s::conv_chunks(c2s::conv_ck(d->c_in)) * 64 * sizeof(__nv_bfloat16);
}

int c2s_conv2d_forward(const c2s_conv_desc* desc, const void* x, const c2s_conv_input_norm* in_norm, const float* weight,
                       const float* bias, void* y, float* stats, void* workspace, size_t workspace_bytes, void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(desc != nullptr && x != nullptr && weight != nullptr && y != nullptr, "c2s_conv2d_forward: NULL argument");
  const c2s_conv_desc& d = *desc;
  if (!c2s_conv2d_supported(desc))
    C2S_UNSUPPORTED("c2s_conv2d_forward: serves 3x3 / stride 1 / reflect padding 1, W = 128, 64 or 32, c_out = 64, c_in <= 16 or 64; "
                    "3x3 / stride 1 / reflect padding 1, W = 16, H <= 16, c_in and c_out 64 or 128; "
                    "and 4x4 / stride 2 / padding 1, W = 128, 64 or 32, even H, 64 -> 64 channels; bf16 "
                    "(got k=%d s=%d p=%d H=%d W=%d c_in=%d c_out=%d dtype=%d)", d.kernel, d.stride, d.padding, d.H, d.W, d.c_in,
                    d.c_out, d.dtype);
  C2S_CHECK_ARG(reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(y) % 16 == 0,
                "c2s_conv2d_forward: x and y must be 16-byte aligned");
  const size_t need = c2s_conv2d_workspace_bytes(desc);
  C2S_CHECK_ARG(workspace != nullptr && workspace_bytes >= need, "c2s_conv2d_forward: workspace of %zu bytes needed, %zu given",
                need, workspace_bytes);
  int status = check_device();
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  const bool down = conv_is_down(d), w16 = conv_is_w16(d);
  const int c_out = w16 ? d.c_out : kCN;
  const int ck = w16 ? d.c_in : conv_ck(d.c_in), chunks = down ? kDChunks : conv_chunks(ck), k_total = chunks * 64;
  __nv_bfloat16* wp = static_cast<__nv_bfloat16*>(workspace);
  if (w16)  // the weight boxes are loaded by TMA
    C2S_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 16 == 0, "c2s_conv2d_forward: the workspace must be 16-byte aligned");
  conv_weight_prep_kernel<<<ceil_div(c_out * k_total, 256), 256, 0, stream>>>(weight, wp, c_out, d.c_in, ck, k_total, down ? 16 : 9);
  C2S_LAUNCH_CHECK("conv_weight_prep");
  if (stats != nullptr) C2S_CUDA(cudaMemsetAsync(stats, 0, static_cast<size_t>(d.frames) * kStatQuarters * 2 * sizeof(float), stream));
  const int sms = sm_count();
  ConvArgs a{};
  a.x = static_cast<const __nv_bfloat16*>(x), a.y = static_cast<__nv_bfloat16*>(y), a.bias = bias, a.stats = stats, a.wp = wp;
  a.frames = d.frames, a.c_in = d.c_in, a.H = d.H;
  if (in_norm != nullptr) {
    C2S_CHECK_ARG(in_norm->stats != nullptr && in_norm->gamma != nullptr && in_norm->beta != nullptr && in_norm->n_groups > 0 &&
                      d.c_in % in_norm->n_groups == 0 && in_norm->n_sub > 0 && in_norm->n_sub % in_norm->n_groups == 0,
                  "c2s_conv2d_forward: bad input normalisation (groups=%d, sub-groups=%d, c_in=%d)", in_norm->n_groups,
                  in_norm->n_sub, d.c_in);
    a.in_stats = in_norm->stats, a.in_gamma = in_norm->gamma, a.in_beta = in_norm->beta;
    a.in_groups = in_norm->n_groups, a.in_sub = in_norm->n_sub, a.in_relu = in_norm->relu, a.in_eps = in_norm->eps;
  }
  if (w16) {  // one unit per frame
    CUtensorMap wmap;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(k_total), static_cast<cuuint64_t>(c_out)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(k_total) * sizeof(__nv_bfloat16)};
    const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(c_out)};
    status = encode_tensor_map(&wmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, wp, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "prepared conv weights");
    if (status != C2S_OK) return status;
    const int grid_w = d.frames < sms ? d.frames : sms;
    const size_t smem_w = w16_smem_bytes(d.c_in / 64, c_out);
#define C2S_CONV_W16_LAUNCH(KC_, N_, NORM_)                                                       \
  do {                                                                                            \
    C2S_SMEM_ATTR((conv3x3_w16_tc_kernel<KC_, N_, NORM_>), smem_w);                               \
    conv3x3_w16_tc_kernel<KC_, N_, NORM_><<<grid_w, kW16Threads, smem_w, stream>>>(wmap, a);      \
  } while (0)
    const bool norm = in_norm != nullptr;
    if (d.c_in == 64 && c_out == 64) {
      if (norm) C2S_CONV_W16_LAUNCH(1, 64, true);
      else C2S_CONV_W16_LAUNCH(1, 64, false);
    } else if (d.c_in == 64) {
      if (norm) C2S_CONV_W16_LAUNCH(1, 128, true);
      else C2S_CONV_W16_LAUNCH(1, 128, false);
    } else if (c_out == 64) {
      if (norm) C2S_CONV_W16_LAUNCH(2, 64, true);
      else C2S_CONV_W16_LAUNCH(2, 64, false);
    } else {
      if (norm) C2S_CONV_W16_LAUNCH(2, 128, true);
      else C2S_CONV_W16_LAUNCH(2, 128, false);
    }
#undef C2S_CONV_W16_LAUNCH
    C2S_LAUNCH_CHECK("conv3x3_reflect_w16<tcgen05>");
    return C2S_OK;
  }
  if (down) {  // units are bands of OUTPUT rows
    C2S_CHECK_ARG(in_norm == nullptr, "c2s_conv2d_forward: the strided layer reads a normalised input (no in_norm)");
    const int ho = d.H / 2;
    a.rows_per_unit = ho;
    while (a.rows_per_unit > 8 && static_cast<long long>(d.frames) * ceil_div(ho, a.rows_per_unit) < 4LL * sms) a.rows_per_unit /= 2;
    a.units_per_frame = ceil_div(ho, a.rows_per_unit);
    a.n_units = d.frames * a.units_per_frame;
    const int grid_d = a.n_units < sms ? a.n_units : sms;
    // narrow rows: the M = 64 products read 65 pixel rows from a half of 33 / 17; the ring is followed by what they run into
    const size_t smem_d = static_cast<size_t>(kDChunks) * 8192 + static_cast<size_t>(kDRing) * 2 * dsub_bytes(d.W) + 1024 +
                          (d.W == 128 ? 0 : 8192);
    if (d.W == 128) {
      C2S_SMEM_ATTR(conv4x4s2_tc_kernel<128>, smem_d);
      conv4x4s2_tc_kernel<128><<<grid_d, kConvThreads, smem_d, stream>>>(a);
    } else if (d.W == 64) {
      C2S_SMEM_ATTR(conv4x4s2_tc_kernel<64>, smem_d);
      conv4x4s2_tc_kernel<64><<<grid_d, kConvThreads, smem_d, stream>>>(a);
    } else {
      C2S_SMEM_ATTR(conv4x4s2_tc_kernel<32>, smem_d);
      conv4x4s2_tc_kernel<32><<<grid_d, kConvThreads, smem_d, stream>>>(a);
    }
    C2S_LAUNCH_CHECK("conv4x4s2_reflect<tcgen05>");
    return C2S_OK;
  }
  // whole frames per unit when there are enough of them to balance the SMs, bands of rows otherwise
  a.rows_per_unit = d.H;
  while (a.rows_per_unit > 16 && static_cast<long long>(d.frames) * ceil_div(d.H, a.rows_per_unit) < 4LL * sms) a.rows_per_unit /= 2;
  a.units_per_frame = ceil_div(d.H, a.rows_per_unit);
  a.n_units = d.frames * a.units_per_frame;
  const int grid = a.n_units < sms ? a.n_units : sms;
  // W = 32: the products read 66 pixel rows from a slot of 40; the ring is followed by what the last slot's reads run into
  const size_t smem = static_cast<size_t>(chunks) * 8192 + static_cast<size_t>(kRing) * slot_bytes(d.W) + 1024 + (d.W == 32 ? 4096 : 0);
  if (ck == 16)  // the first layer of a block reads the model input: no normalisation on the fly
    C2S_CHECK_ARG(in_norm == nullptr, "c2s_conv2d_forward: input normalisation needs c_in = 64");
#define C2S_CONV_LAUNCH(CK_, NORM_, W_)                                                   \
  do {                                                                                    \
    C2S_SMEM_ATTR((conv3x3_tc_kernel<CK_, NORM_, W_>), smem);                             \
    conv3x3_tc_kernel<CK_, NORM_, W_><<<grid, kConvThreads, smem, stream>>>(a);           \
  } while (0)
  if (d.W == 128) {
    if (ck == 16) C2S_CONV_LAUNCH(16, false, 128);
    else if (in_norm != nullptr) C2S_CONV_LAUNCH(64, true, 128);
    else C2S_CONV_LAUNCH(64, false, 128);
  } else if (d.W == 64) {
    if (ck == 16) C2S_CONV_LAUNCH(16, false, 64);
    else if (in_norm != nullptr) C2S_CONV_LAUNCH(64, true, 64);
    else C2S_CONV_LAUNCH(64, false, 64);
  } else {
    if (ck == 16) C2S_CONV_LAUNCH(16, false, 32);
    else if (in_norm != nullptr) C2S_CONV_LAUNCH(64, true, 32);
    else C2S_CONV_LAUNCH(64, false, 32);
  }
#undef C2S_CONV_LAUNCH
  C2S_LAUNCH_CHECK("conv3x3_reflect<tcgen05>");
  return C2S_OK;
}

int c2s_group_stats(const void* x, int32_t dtype, int64_t frames, int32_t channels, int64_t hw, int32_t n_groups, float* stats,
                    void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(x != nullptr && stats != nullptr, "c2s_group_stats: NULL argument");
  C2S_CHECK_ARG(frames > 0 && channels > 0 && hw > 0 && n_groups > 0 && channels % n_groups == 0,
                "c2s_group_stats: bad shape frames=%lld C=%d hw=%lld groups=%d", static_cast<long long>(frames), channels,
                static_cast<long long>(hw), n_groups);
  C2S_CHECK_ARG(dtype == C2S_F32 || dtype == C2S_BF16, "c2s_group_stats: unknown dtype %d", dtype);
  int status = check_device();
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  const size_t span = static_cast<size_t>(channels / n_groups) * hw;
  dim3 grid(n_groups, static_cast<unsigned>(frames));
  if (dtype == C2S_BF16)
    group_stats_kernel<__nv_bfloat16><<<grid, kStatThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), stats, span);
  else
    group_stats_kernel<float><<<grid, kStatThreads, 0, stream>>>(static_cast<const float*>(x), stats, span);
  C2S_LAUNCH_CHECK("group_stats");
  return C2S_OK;
}

int c2s_group_norm_relu(const void* x, const float* stats, int32_t n_sub, const float* gamma, const float* beta,
                        const void* residual, void* out, int32_t dtype, int64_t frames, int32_t channels, int64_t hw,
                        int32_t n_groups, float eps, int32_t relu, void* stream_ptr) {
  using namespace c2s;
  C2S_CHECK_ARG(x != nullptr && stats != nullptr && gamma != nullptr && beta != nullptr && out != nullptr,
                "c2s_group_norm_relu: NULL argument");
  C2S_CHECK_ARG(frames > 0 && channels > 0 && hw > 0 && n_groups > 0 && channels % n_groups == 0 && n_sub > 0 &&
                    n_sub % n_groups == 0,
                "c2s_group_norm_relu: bad shape");
  C2S_CHECK_ARG(dtype == C2S_F32 || dtype == C2S_BF16, "c2s_group_norm_relu: unknown dtype %d", dtype);
  const int vec = dtype == C2S_BF16 ? 8 : 4;
  if (static_cast<long long>(channels) * hw >= (1ll << 31)) C2S_UNSUPPORTED("c2s_group_norm_relu: a frame of %lld elements is too large",
                                                                              static_cast<long long>(channels) * hw);
  C2S_CHECK_ARG(hw % vec == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0 &&
                    reinterpret_cast<uintptr_t>(residual) % 16 == 0,
                "c2s_group_norm_relu: planes must be whole, aligned 16-byte vectors");
  int status = check_device();
  if (status != C2S_OK) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  NormArgs a{};
  a.x = x, a.residual = residual, a.out = out, a.stats = stats, a.gamma = gamma, a.beta = beta;
  a.C = channels, a.hw = static_cast<int>(hw), a.n_groups = n_groups, a.n_sub = n_sub, a.relu = relu, a.eps = eps;
  // four vectors per thread unless the planes are so small that a block would touch more than 256 channels
  const int items = (256LL * 4 * vec / hw + 2 <= 256) ? 4 : 1;
  dim3 grid(ceil_div(static_cast<long long>(channels) * hw, 256LL * items * vec), static_cast<unsigned>(frames));
  if (dtype == C2S_BF16) {
    if (items == 4) group_norm_relu_kernel<__nv_bfloat16, 4><<<grid, 256, 0, stream>>>(a);
    else group_norm_relu_kernel<__nv_bfloat16, 1><<<grid, 256, 0, stream>>>(a);
  } else {
    if (items == 4) group_norm_relu_kernel<float, 4><<<grid, 256, 0, stream>>>(a);
    else group_norm_relu_kernel<float, 1><<<grid, 256, 0, stream>>>(a);
  }
  C2S_LAUNCH_CHECK("group_norm_relu");
  return C2S_OK;
}

}  // extern "C"
