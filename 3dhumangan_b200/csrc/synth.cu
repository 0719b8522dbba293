// SPADE synthesis backbone: one kernel launch per SPADE half-block
//     x_out = Conv1x1_SN( lrelu_0.2( BN(x) * (1 + gamma) + beta ) ) + b  [+ x_skip]  [-> ToRGB accumulate]
// (SPADE2d.forward lib/components/map3d_layers.py:176-190, SPADEBlock.forward :218-238,
//  ToRGB :346-352, SynthesisNetwork.forward lib/generators/map3d_generator.py:58-97.)
//
// Activations live in HBM as fp32 in a tile-blocked planar layout [B, T, C=256, 128] (T = ceil(HW/128)
// tiles of 128 consecutive pixels): the 128 KB a CTA reads / writes per tile are CONTIGUOUS, and every
// 32-channel slice of a tile is one contiguous 16 KB block (one cp.async.bulk).
//
// Per CTA (512 threads), persistent over tiles of 128 pixels of one image:
//   warps 0-7   operand team: build the bf16 hi/lo A operand of the NEXT tile in a 2-slot ring of
//               [128 x 64] K-major SW128 chunks (BN scale/shift, SPADE modulation, LeakyReLU fused)
//   warps 8-11  epilogue team: drain the fp32 accumulator of the PREVIOUS tile from TMEM (warp 8+q owns lanes
//               32q..32q+31, all 256 columns): bias, residual, ToRGB, per-channel sum / sum-of-squares for the
//               next BatchNorm (so SyncBN statistics never need their own pass), plane stores
//   warp 12     MMA issuer: the warp walks the tile / chunk loops in convergent code, its elected lane issues tcgen05.mma
//               (M=128, N=256, K=16; bf16x3 split or plain bf16)
//   warp 13     one thread streams the packed weight tiles from L2 (cp.async.bulk, 2 x 32 KB stages)
//   warp 14     one thread streams activation slices (ring slots 0-2, operand team) from HBM with cp.async.bulk
//   warp 15     one thread streams residual slices (ring slots 3-4, epilogue team).  Two threads, not one: with a
//               single producer the two rings are coupled by program order, and in the pixel-style variant
//               (gamma/beta GEMM of tile t+1 waits for the epilogue of tile t) that coupling deadlocks.
// The two TMEM halves (2 x 256 columns) alternate between tiles, so the epilogue of tile t, the MMAs of tile
// t+1 and the operand production of tile t+1/t+2 overlap.
//
// Two variants:
//   const-style : gamma/beta are per-sample vectors (blocks whose style map is spatially constant, 12 of 18
//                 half-blocks in 'mixed'/'isolated' mode).
//   pixel-style : gamma/beta come from a second GEMM on relu(bilinear_up(P_lr)) where
//                 P_lr = W_shared . feature_maps + b at RENDER resolution (W_shared commutes with the bilinear
//                 up-sample), so the 28x larger up-sampled style map of map3d_generator.py:244-245 is never
//                 materialised.  TMEM plan per tile t (R = half t&1, R' = the other, still being drained):
//                 G1(gamma|beta, channels 0-127) -> R, G1(channels 128-255) -> R' once the epilogue of t-1 is
//                 done, y chunks 0,1 <- R, conv accumulator -> R, y chunks 2,3 <- R'.
//
// The const-style kernel doubles as the library's blocked 1x1-convolution engine (runtime fields at the end of SpadeArgs):
// K of 64..512 input channels from one or two sources, LeakyReLU / sine / identity operand transform, and -- template
// flag kBwd -- the data-gradient form: the operand is the incoming gradient (optionally scaled per sample and channel),
// the weight image is W^T and the epilogue multiplies by the activation derivative rebuilt from the forward input that
// arrives through the residual ring, adds a rank-k term (the renderer's sigma / rgb heads) and accumulates the
// per-(sample, channel) sums the BatchNorm / FiLM gradients need (DESIGN.md "Backward").
//
// Ring protocol note: every consumer warp of a staging ring waits for and releases EVERY slice in order
// (only the owning column half reads it).  With per-half arrivals a slot of an odd-sized ring alternates
// between halves, a fast half gets two phases ahead and the parity wait succeeds on a stale phase -- that race
// produced launch failures in an earlier version (DESIGN.md "Pitfalls").
#include "common.cuh"
#include "umma.cuh"

namespace hg {

constexpr int kC = 256;             // channels (hidden_dim == feature_dim == 256)
constexpr int kSynThreads = 512;
constexpr int kSynStages = 2;       // weight stages
constexpr int kASlots = 2;          // operand ring
constexpr int kXSlots = 5;          // staging slots in total
constexpr int kXs = 3;              //   slots 0..2: activation slices (operand team)
constexpr int kSs = 2;              //   slots 3..4: residual slices (epilogue team)
constexpr uint32_t kAChunk = 128 * 128;   // [128 x 64] bf16
constexpr uint32_t kBStage = 256 * 128;   // [256 x 64] bf16
constexpr uint32_t kXSlice = 32 * 128 * 4;  // 32 channels x 128 pixels fp32

struct SpadeArgs {
  const float* x;        // [B or 1, T, C, 128] tile-blocked
  long x_bstride;        // T*C*128, or 0 when x is shared by the whole batch (synthesis input)
  const float* mod;      // const-style: [B,2,C] (g1, g0): y = lrelu(x*g1 + g0)
  const float* scsh;     // pixel-style: [2,C] BN scale, shift
  const float* p_lr;     // pixel-style: [B, Rh*Rw, p_stride>=128] pre-activation of mlp_shared at render res
  long p_stride;         //              row stride of p_lr in floats (multiple of 4)
  const float* p_bias;   // pixel-style: [B,128] per-sample constant added after interpolation (or null)
  const uint8_t* wgb;    // pixel-style: packed [512 x 128] gamma/beta weights (2 N-blocks, interleaved)
  const float* bgb;      // pixel-style: [512] bias in the same interleaved order (gamma part includes +1)
  const uint8_t* wimg;   // packed conv weight [256 x 256] (already divided by sigma)
  const float* bias;     // [C]
  const float* skip;     // [B,T,C,128] residual or null   (backward: the forward input x of the half-block)
  long skip_bstride;     // T*C*128, or 0 when shared by the whole batch
  float* out;            // [B,T,C,128]
  double* stats;         // [2,C] accumulated sum / sumsq of out, or null
  const float* rgb_w;    // [3,C] or null
  const float* rgb_b;    // [3]
  const float* rgb_in;   // [B,3,HW] or null
  float* rgb_out;        // [B,3,HW]
  int B, HW, Hg, Wg, Rh, Rw;
  // generalisations used by the backward schedule (defaults reproduce the forward half-block):
  int nkc;               // K chunks of 64 input channels per tile: 1, 2, 4 or 8
  int xC;                // channels per source tile (128 or 256); chunks beyond xC/64 come from x2
  const float* x2;       // second source [B,T,xC,128] (K = 512 products) or null
  float slope;           // operand LeakyReLU slope (1 = identity); backward epilogue: slope of the mask (0.2 / 0 = ReLU)
  int cout;              // output channels written by the epilogue: 256 or 128 (the MMA always runs N = 256)
  int out_pm;            // backward epilogue: write pixel-major [B,HW,cout] instead of tile-blocked
  int act;               // 0: LeakyReLU(slope) (SPADE), 1: sine (FiLM-SIREN layers of the renderer: y = sin(x*g1 + g0))
  const float* ascale;   // backward operand: per-(b,c) scale [B,C] applied to the incoming gradient, or null
  const float* rk_v;     // backward epilogue: rank-k term  acc += sum_j rgb_w[j][c] * rk_v[b][j][pixel]  (k = rk_n <= 3)
  int rk_n;
  const float* mod2;     // forward, K = 512: [B,2,C] table of the SECOND source's channels (null: the first table serves both,
                         // as for the renderer's first FiLM layer); lets a 512-channel layer (hidden_dim 384 / 420 zero-padded
                         // to 2 x 256) be modulated per channel
};

struct SynSmem {
  uint8_t* a_hi;   // [kASlots] chunks
  uint8_t* a_lo;
  uint8_t* b_st;
  float* x_st;     // [kXSlots][32][128]
  float* tab_g1;   // [C]  (const: g1 | pixel: bn scale)
  float* tab_g0;   // [C]  (const: g0 | pixel: bn shift)
  float* tab_bias; // [C]
  float* tab_rgbw; // [3*C]
  float* tab_bgb;  // [512]
  float* tab_as;   // [C]  backward operand scale
  float* st_sum;   // [C]
  float* st_sq;    // [C]
  uint64_t* bars;
  uint32_t* tmem_slot;
};

__device__ __forceinline__ SynSmem carve(uint8_t* raw) {
  uint8_t* s = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
  SynSmem m;
  m.a_hi = s;
  m.a_lo = s + kASlots * kAChunk;
  m.b_st = s + 2 * kASlots * kAChunk;
  m.x_st = reinterpret_cast<float*>(m.b_st + kSynStages * kBStage);
  float* f = m.x_st + kXSlots * (kXSlice / 4);
  m.tab_g1 = f; f += kC;
  m.tab_g0 = f; f += kC;
  m.tab_bias = f; f += kC;
  m.tab_rgbw = f; f += 3 * kC;
  m.tab_bgb = f; f += 512;
  m.tab_as = f; f += kC;
  m.st_sum = f; f += kC;
  m.st_sq = f; f += kC;
  m.bars = reinterpret_cast<uint64_t*>(f);
  m.tmem_slot = reinterpret_cast<uint32_t*>(m.bars + 40);
  return m;
}
constexpr uint32_t kSynSmemBytes = 2 * kASlots * kAChunk + kSynStages * kBStage + kXSlots * kXSlice +
                                   (kC * 9 + 512) * 4 + 40 * 8 + 16 + 1024;
static_assert(kSynSmemBytes <= 232448, "shared memory budget");

// barrier slots
enum { A_FULL = 0 /*2*/, A_EMPTY = 2 /*2*/, B_FULL = 4 /*2*/, B_EMPTY = 6 /*2*/, ACC_FULL = 8 /*2*/,
       ACC_EMPTY = 10 /*2*/, G1A_FULL = 12, G1B_FULL = 13, A1_FULL = 14, X_FULL = 16 /*5*/, X_EMPTY = 24 /*5*/ };

__device__ __forceinline__ void rows_barrier() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__device__ __forceinline__ float lrelu02(float v) { return v > 0.f ? v : 0.2f * v; }

// sin / cos for |t| up to a few thousand: two-term Cody-Waite reduction by 2*pi, then the SFU (abs error ~2^-21);
// the same evaluation as the fused renderer (csrc/render.cu), so that forward and backward agree.
__device__ __forceinline__ float reduce_2pi(float t) {
  const float y = t * 0.15915494309189535f;
  const float k = (y + 12582912.f) - 12582912.f;
  float r = fmaf(-k, 6.2831854820251465f, t);
  return fmaf(-k, -1.7484555314695172e-07f, r);
}
__device__ __forceinline__ float sin_red(float t) { return __sinf(reduce_2pi(t)); }
__device__ __forceinline__ float cos_red(float t) { return __cosf(reduce_2pi(t)); }
// the same reduction on a pair (packed fp32: identical operations per lane)
__device__ __forceinline__ float2 reduce_2pi2(float2 t) {
  const float2 y = __fmul2_rn(t, make_float2(0.15915494309189535f, 0.15915494309189535f));
  const float2 k = __fadd2_rn(__fadd2_rn(y, make_float2(12582912.f, 12582912.f)), make_float2(-12582912.f, -12582912.f));
  const float2 r = __ffma2_rn(k, make_float2(-6.2831854820251465f, -6.2831854820251465f), t);
  return __ffma2_rn(k, make_float2(1.7484555314695172e-07f, 1.7484555314695172e-07f), r);
}
__device__ __forceinline__ float2 sin_red2(float2 t) { const float2 r = reduce_2pi2(t); return make_float2(__sinf(r.x), __sinf(r.y)); }
__device__ __forceinline__ float2 cos_red2(float2 t) { const float2 r = reduce_2pi2(t); return make_float2(__cosf(r.x), __cosf(r.y)); }

// 32 lanes x 32 values: after the call lane j holds sum over lanes of v[j].
__device__ __forceinline__ float transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
    const bool upper = (lane & w) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float send = upper ? v[i] : v[i + w];
      const float keep = upper ? v[i + w] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
    }
  }
  return v[0];
}

struct TileMap {
  int T, first, stride, count;
  __device__ __forceinline__ void get(int it, int& b, int& ti) const {
    const int tile = first + it * stride;
    b = tile / T;
    ti = tile - b * T;
  }
};

// ------------------------------------------------------------------------------------------
// common setup
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void init_common(const SpadeArgs& a, const SynSmem& m, int warp) {
  for (int i = threadIdx.x; i < kC; i += blockDim.x) {
    m.tab_bias[i] = a.bias[i];
    m.st_sum[i] = 0.f;
    m.st_sq[i] = 0.f;
  }
  if (a.rgb_w)
    for (int i = threadIdx.x; i < 3 * kC; i += blockDim.x) m.tab_rgbw[i] = a.rgb_w[i];
  if (threadIdx.x == 0) {
    for (int i = 0; i < kASlots; ++i) {
      mbar_init(m.bars + A_FULL + i, 8);
      mbar_init(m.bars + A_EMPTY + i, 1);
    }
    for (int i = 0; i < kSynStages; ++i) {
      mbar_init(m.bars + B_FULL + i, 1);
      mbar_init(m.bars + B_EMPTY + i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(m.bars + ACC_FULL + i, 1);
      mbar_init(m.bars + ACC_EMPTY + i, 4);     // the 4 epilogue warps
    }
    mbar_init(m.bars + G1A_FULL, 1);
    mbar_init(m.bars + G1B_FULL, 1);
    mbar_init(m.bars + A1_FULL, 8);
    for (int i = 0; i < kXSlots; ++i) {
      mbar_init(m.bars + X_FULL + i, 1);
      mbar_init(m.bars + X_EMPTY + i, i < kXs ? 8 : 4);   // operand team: 8 warps, epilogue team: 4 warps
    }
    fence_mbar_init();
  }
  if (warp == 12) tmem_alloc<512>(m.tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
}

// ------------------------------------------------------------------------------------------
// warp 13: weight stages.  Every tile consumes the same sequence: for each image `nstages` tiles of [256 x 64]
// in storage order (kc-major, hi then lo); the lo tiles are skipped in 1-pass mode.
// ------------------------------------------------------------------------------------------
template <int kPasses>
__device__ __forceinline__ void weight_producer_loop(const SynSmem& m, const uint8_t* const* imgs, const int* nstages,
                                                     int nimgs, int num_my_tiles) {
  uint32_t st = 0, ph = 0;
  for (int t = 0; t < num_my_tiles; ++t)
    for (int g = 0; g < nimgs; ++g)
      for (int s = 0; s < nstages[g]; ++s) {
        if (kPasses == 1 && (s & 1)) continue;
        mbar_wait_backoff(m.bars + B_EMPTY + st, ph ^ 1);
        mbar_arrive_expect_tx(m.bars + B_FULL + st, kBStage);
        bulk_g2s(m.b_st + st * kBStage, imgs[g] + static_cast<size_t>(s) * kBStage, kBStage, m.bars + B_FULL + st);
        if (++st == kSynStages) { st = 0; ph ^= 1; }
      }
}

struct MmaPipe {
  uint32_t st = 0, ph = 0;
};

// One K=64 chunk of a 3-pass (or 1-pass) product against the next weight stage(s).
// `leader`: the elected lane of the (converged) MMA warp -- the whole warp walks the issue loops (umma.cuh: elect_one_sync).
template <int kPasses>
__device__ __forceinline__ void mma_chunk(const SynSmem& m, MmaPipe& p, bool leader, uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo,
                                          uint32_t idesc, bool accumulate) {
  mbar_wait(m.bars + B_FULL + p.st, p.ph);
  tc_fence_after();
  umma_k64_if(leader, tmem_d, a_hi, smem_u32(m.b_st + p.st * kBStage), idesc, accumulate);
  if (kPasses == 3) umma_k64_if(leader, tmem_d, a_lo, smem_u32(m.b_st + p.st * kBStage), idesc, true);
  umma_commit_if(leader, m.bars + B_EMPTY + p.st);
  if (++p.st == kSynStages) { p.st = 0; p.ph ^= 1; }
  if (kPasses == 3) {
    mbar_wait(m.bars + B_FULL + p.st, p.ph);
    tc_fence_after();
    umma_k64_if(leader, tmem_d, a_hi, smem_u32(m.b_st + p.st * kBStage), idesc, true);
    umma_commit_if(leader, m.bars + B_EMPTY + p.st);
    if (++p.st == kSynStages) { p.st = 0; p.ph ^= 1; }
  }
}

// ------------------------------------------------------------------------------------------
// warp 14: activation slices (slots 0..2), warp 15: residual slices (slots 3..4): two independent rings.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void ring_emit(const SynSmem& m, uint32_t& g, int base, int slots, const float* src) {
  const uint32_t slot = base + g % slots;
  mbar_wait_backoff(m.bars + X_EMPTY + slot, ((g / slots) & 1) ^ 1);
  mbar_arrive_expect_tx(m.bars + X_FULL + slot, kXSlice);
  bulk_g2s(m.x_st + slot * (kXSlice / 4), src, kXSlice, m.bars + X_FULL + slot);
  ++g;
}
__device__ __forceinline__ void x_producer_loop(const SpadeArgs& a, const SynSmem& m, const TileMap& tm) {
  uint32_t g = 0;
  for (int it = 0; it < tm.count; ++it) {
    int b, ti;
    tm.get(it, b, ti);
    const int per_src = a.xC / 32;                 // 32-channel slices per source tile
    const float* base = a.x + static_cast<long>(b) * a.x_bstride + static_cast<long>(ti) * a.xC * 128;
    const float* base2 = a.x2 ? a.x2 + (static_cast<long>(b) * tm.T + ti) * a.xC * 128 : nullptr;
    for (int j = 0; j < 2 * a.nkc; ++j)
      ring_emit(m, g, 0, kXs, (j < per_src ? base : base2 - per_src * 32 * 128) + j * 32 * 128);
  }
}
__device__ __forceinline__ void skip_producer_loop(const SpadeArgs& a, const SynSmem& m, const TileMap& tm) {
  if (!a.skip) return;
  uint32_t g = 0;
  for (int it = 0; it < tm.count; ++it) {
    int b, ti;
    tm.get(it, b, ti);
    const float* base = a.skip + static_cast<long>(b) * a.skip_bstride + static_cast<long>(ti) * a.cout * 128;
    for (int j = 0; j < a.cout / 32; ++j) ring_emit(m, g, kXs, kSs, base + j * 32 * 128);
  }
}

// Operand-team side of the activation ring: every warp walks both slices of a chunk, half h reads slice 2kc+h.
__device__ __forceinline__ void take_x_pair(const SynSmem& m, uint32_t& xg, int h, int row, int lane, float (&dst)[32]) {
#pragma unroll
  for (int hh = 0; hh < 2; ++hh, ++xg) {
    const uint32_t xslot = xg % kXs;
    mbar_wait_sleep(m.bars + X_FULL + xslot, (xg / kXs) & 1);
    if (hh == h) {
      const uint32_t xs = smem_u32(m.x_st + xslot * (kXSlice / 4)) + row * 4;
#pragma unroll
      for (int j = 0; j < 32; ++j) dst[j] = lds_f32(xs + j * 512);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(m.bars + X_EMPTY + xslot);
  }
}

// ------------------------------------------------------------------------------------------
// warps 8-11: epilogue team (identical for both variants): tile `it` lives in TMEM half it&1.
// The four epilogue warps -- one per scheduler, each a single instruction stream -- are the critical path of these
// kernels (ncu: never waiting, ~5 cycles per instruction), so the per-element work is straight-line code: residual /
// ToRGB / statistics are compile-time variants and rows past the image are handled by one warp-uniform branch per
// 32-column group (with run-time flags inside the unrolled loop the plain half-block spent 391 instructions per group,
// 45 % of them selects, zero-adds, register clears and branches).
// ------------------------------------------------------------------------------------------
template <bool kSkip, bool kRgb, bool kStats>
__device__ __forceinline__ void epilogue_team_variant(const SpadeArgs& a, const SynSmem& m, const TileMap& tm, uint32_t tmem,
                                                      int q, int lane) {
  const int row = q * 32 + lane;
  uint32_t sg = 0;   // residual slices consumed
  uint32_t tbias = smem_u32(m.tab_bias), trgb = smem_u32(m.tab_rgbw);   // constant tables, written before init's barrier
  opaque(tbias);
  opaque(trgb);
  // without a residual the 2 residual staging slots (32 KB) are free: per-warp [32][33] transpose scratch for the
  // statistics (32 STS + 32 LDS + 64 FP instead of a 248-instruction shuffle tree)
  const uint32_t scratch = smem_u32(m.x_st + kXs * (kXSlice / 4) + q * (32 * 33));
  const int HW = a.HW, cout = a.cout, ncg = a.cout >> 5;
  float* const outp = a.out;
  for (int it = 0; it < tm.count; ++it) {
    int b, ti;
    tm.get(it, b, ti);
    const uint32_t buf = it & 1;
    const int pix = ti * 128 + row;
    const bool valid = pix < HW;
    const bool full = ti * 128 + 128 <= HW;      // warp-uniform: every row of the tile is a pixel
    float* const orow = outp + (static_cast<long>(b) * tm.T + ti) * cout * 128 + row;
    mbar_wait_sleep(m.bars + ACC_FULL + buf, (it >> 1) & 1);
    tc_fence_after();
    float2 r0 = make_float2(0.f, 0.f), r1 = r0, r2 = r0;
#pragma unroll 1
    for (int cg = 0; cg < ncg; ++cg) {
      const int c0 = cg * 32;
      uint32_t raw[32];
      tmem_ld32(tmem + buf * 256 + (static_cast<uint32_t>(q * 32) << 16) + c0, raw);
      float sk[32];
      if (kSkip) {
        const uint32_t sslot = kXs + sg % kSs;
        mbar_wait_sleep(m.bars + X_FULL + sslot, (sg / kSs) & 1);
        const uint32_t xs = smem_u32(m.x_st + sslot * (kXSlice / 4)) + row * 4;
#pragma unroll
        for (int j = 0; j < 32; ++j) sk[j] = lds_f32(xs + j * 512);
        __syncwarp();
        if (lane == 0) mbar_arrive(m.bars + X_EMPTY + sslot);
        ++sg;
      }
      tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float bs[8];
        lds8(tbias + (c0 + g * 8) * 4, bs);
#pragma unroll
        for (int jj = 0; jj < 8; jj += 2) {      // packed fp32 adds on channel pairs (same operations, half the instructions)
          const int j = g * 8 + jj;
          float2 p = __fadd2_rn(make_float2(__uint_as_float(raw[j]), __uint_as_float(raw[j + 1])), make_float2(bs[jj], bs[jj + 1]));
          if (kSkip) p = __fadd2_rn(p, make_float2(sk[j], sk[j + 1]));
          v[j] = p.x;
          v[j + 1] = p.y;
        }
      }
      float* const o = orow + c0 * 128;
      if (full) {
#pragma unroll
        for (int j = 0; j < 32; ++j) o[j * 128] = v[j];
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (valid) o[j * 128] = v[j];
          else v[j] = 0.f;
        }
      }
      if (kRgb) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float w0[8], w1[8], w2[8];
          lds8(trgb + (c0 + g * 8) * 4, w0);
          lds8(trgb + (kC + c0 + g * 8) * 4, w1);
          lds8(trgb + (2 * kC + c0 + g * 8) * 4, w2);
#pragma unroll
          for (int jj = 0; jj < 8; jj += 2) {      // even / odd channels in the two lanes of a packed accumulator
            const float2 vv = make_float2(v[g * 8 + jj], v[g * 8 + jj + 1]);
            r0 = __ffma2_rn(vv, make_float2(w0[jj], w0[jj + 1]), r0);
            r1 = __ffma2_rn(vv, make_float2(w1[jj], w1[jj + 1]), r1);
            r2 = __ffma2_rn(vv, make_float2(w2[jj], w2[jj + 1]), r2);
          }
        }
      }
      if (kStats) {
        float t1, t2;
        if (kSkip) {
          float s2[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) s2[j] = v[j] * v[j];
          t1 = transpose_reduce32(v, lane);
          t2 = transpose_reduce32(s2, lane);
        } else {
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; ++j) asm volatile("st.shared.f32 [%0], %1;" ::"r"(scratch + (lane * 33 + j) * 4), "f"(v[j]) : "memory");
          __syncwarp();
          float2 ts = make_float2(0.f, 0.f), qs = make_float2(0.f, 0.f);      // two chains each, as one packed pair
#pragma unroll
          for (int r = 0; r < 32; r += 2) {
            const float2 x = make_float2(lds_f32(scratch + (r * 33 + lane) * 4), lds_f32(scratch + ((r + 1) * 33 + lane) * 4));
            ts = __fadd2_rn(ts, x);
            qs = __ffma2_rn(x, x, qs);
          }
          t1 = ts.x + ts.y;
          t2 = qs.x + qs.y;
        }
        atomicAdd(m.st_sum + c0 + lane, t1);
        atomicAdd(m.st_sq + c0 + lane, t2);
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(m.bars + ACC_EMPTY + buf);
    if (kRgb && valid) {   // this thread saw all 256 channels of its pixel
      const float r[3] = {r0.x + r0.y, r1.x + r1.y, r2.x + r2.y};
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const long idx = (static_cast<long>(b) * 3 + j) * HW + pix;
        float o = r[j] + a.rgb_b[j];
        if (a.rgb_in) o += a.rgb_in[idx];
        a.rgb_out[idx] = o;
      }
    }
  }
  asm volatile("bar.sync 2, 128;" ::: "memory");
  if (kStats) {
    for (int c = threadIdx.x - 256; c < kC; c += 128) {
      atomicAdd(a.stats + c, static_cast<double>(m.st_sum[c]));
      atomicAdd(a.stats + kC + c, static_cast<double>(m.st_sq[c]));
    }
  }
}

// warp-uniform dispatch on the launch's flags
__device__ __forceinline__ void epilogue_team_loop(const SpadeArgs& a, const SynSmem& m, const TileMap& tm, uint32_t tmem,
                                                   int q, int lane) {
  const int sel = (a.skip ? 4 : 0) | (a.rgb_w ? 2 : 0) | (a.stats ? 1 : 0);
  switch (sel) {
    case 0: epilogue_team_variant<false, false, false>(a, m, tm, tmem, q, lane); break;
    case 1: epilogue_team_variant<false, false, true>(a, m, tm, tmem, q, lane); break;
    case 2: epilogue_team_variant<false, true, false>(a, m, tm, tmem, q, lane); break;
    case 3: epilogue_team_variant<false, true, true>(a, m, tm, tmem, q, lane); break;
    case 4: epilogue_team_variant<true, false, false>(a, m, tm, tmem, q, lane); break;
    case 5: epilogue_team_variant<true, false, true>(a, m, tm, tmem, q, lane); break;
    case 6: epilogue_team_variant<true, true, false>(a, m, tm, tmem, q, lane); break;
    default: epilogue_team_variant<true, true, true>(a, m, tm, tmem, q, lane); break;
  }
}


// ------------------------------------------------------------------------------------------
// warps 8-11 of the BACKWARD (data-gradient) variant.  The accumulator holds dL/dy = W^T dL/dout for the 128
// pixels of the tile; the forward input x of the half-block arrives through the residual ring, so that
//     pre = x*g1[b,c] + g0[b,c]            (the folded BatchNorm + SPADE modulation of the forward pass)
//     dpre = dL/dy * lrelu'(pre)           -> stored (tile-blocked, like every activation)
//     S1[b,c] += dpre,  S2[b,c] += dpre*x  -> everything BatchNorm / gamma / beta need (DESIGN.md "Backward")
// ------------------------------------------------------------------------------------------
// Compile-time variants (the per-element work must be straight-line code: with run-time flags inside the 32-wide unrolled
// loop the compiler emitted ~4 branches, 4 address LEAs and several constant reloads per element, and the four epilogue
// warps -- one instruction stream per scheduler -- became the critical path of the kernel at 5.7 cycles per instruction):
//   kSine  activation derivative cos(pre) (FiLM-SIREN) instead of the LeakyReLU / ReLU mask
//   kRk    rank-3 term from the renderer's heads (rows beyond rk_n of the [3,C] weight table are zero)
//   kPm    pixel-major [B,HW,cout] output
template <bool kSine, bool kRk, bool kPm>
__device__ __forceinline__ void epilogue_bwd_loop(const SpadeArgs& a, const SynSmem& m, const TileMap& tm, uint32_t tmem,
                                                  int q, int lane) {
  const int row = q * 32 + lane;
  const int et = threadIdx.x - 256;   // 0..127 within the epilogue team
  uint32_t sg = 0;
  int cur_b = -1;
  const int cout = a.cout;
  double* const stats = a.stats;
  auto flush = [&](int b) {
    for (int c = et; c < cout; c += 128) {
      atomicAdd(stats + (static_cast<long>(b) * 2 + 0) * cout + c, static_cast<double>(m.st_sum[c]));
      atomicAdd(stats + (static_cast<long>(b) * 2 + 1) * cout + c, static_cast<double>(m.st_sq[c]));
      m.st_sum[c] = 0.f;
      m.st_sq[c] = 0.f;
    }
  };
  const float mslope = a.slope;
  const int ncg = cout >> 5;
  const int HW = a.HW, rk_n = a.rk_n;
  const float* const modp = a.mod;
  const float* const rkv = a.rk_v;
  float* const outp = a.out;
  uint32_t trk = smem_u32(m.tab_rgbw);     // rank-k weights (loaded by init_common through a.rgb_w)
  opaque(trk);
  for (int it = 0; it < tm.count; ++it) {
    int b, ti;
    tm.get(it, b, ti);
    if (b != cur_b) {   // per-sample tables and per-sample sums
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (cur_b >= 0) flush(cur_b);
      for (int c = et; c < cout; c += 128) {
        m.tab_g1[c] = modp ? modp[(static_cast<long>(b) * 2 + 0) * cout + c] : 1.f;
        m.tab_g0[c] = modp ? modp[(static_cast<long>(b) * 2 + 1) * cout + c] : 0.f;
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      cur_b = b;
    }
    uint32_t tg1 = smem_u32(m.tab_g1), tg0 = smem_u32(m.tab_g0);
    opaque(tg1);   // no table load may move above the refresh
    opaque(tg0);
    const uint32_t buf = it & 1;
    const bool valid = ti * 128 + row < HW;
    float* const orow = kPm ? outp + (static_cast<long>(b) * HW + ti * 128 + row) * cout
                            : outp + (static_cast<long>(b) * tm.T + ti) * cout * 128 + row;
    float rv0 = 0.f, rv1 = 0.f, rv2 = 0.f;
    if (kRk && valid) {
      const float* r = rkv + static_cast<long>(b) * rk_n * HW + ti * 128 + row;
      rv0 = r[0];
      if (rk_n > 1) rv1 = r[HW];
      if (rk_n > 2) rv2 = r[2 * static_cast<long>(HW)];
    }
    mbar_wait_sleep(m.bars + ACC_FULL + buf, (it >> 1) & 1);
    tc_fence_after();
#pragma unroll 1
    for (int cg = 0; cg < ncg; ++cg) {
      const int c0 = cg * 32;
      uint32_t raw[32];
      tmem_ld32(tmem + buf * 256 + (static_cast<uint32_t>(q * 32) << 16) + c0, raw);
      float xs_[32];
      {
        const uint32_t sslot = kXs + sg % kSs;
        mbar_wait_sleep(m.bars + X_FULL + sslot, (sg / kSs) & 1);
        const uint32_t xs = smem_u32(m.x_st + sslot * (kXSlice / 4)) + row * 4;
#pragma unroll
        for (int j = 0; j < 32; ++j) xs_[j] = lds_f32(xs + j * 512);
        __syncwarp();
        if (lane == 0) mbar_arrive(m.bars + X_EMPTY + sslot);
        ++sg;
      }
      if (!valid) {      // rows past the image (last, partial tile only): the staged slice holds whatever the padding holds
#pragma unroll
        for (int j = 0; j < 32; ++j) xs_[j] = 0.f;
      }
      tmem_ld_wait();
      float v[32], w[32];
      float* const o = kPm ? orow + c0 : orow + c0 * 128;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float t1[8], t0[8], k0[8], k1[8], k2[8];
        lds8(tg1 + (c0 + g * 8) * 4, t1);
        lds8(tg0 + (c0 + g * 8) * 4, t0);
        if (kRk) {
          lds8(trk + (c0 + g * 8) * 4, k0);
          lds8(trk + (kC + c0 + g * 8) * 4, k1);
          lds8(trk + (2 * kC + c0 + g * 8) * 4, k2);
        }
#pragma unroll
        for (int jj = 0; jj < 8; jj += 2) {      // channel pairs on packed fp32 (same operations)
          const int j = g * 8 + jj;
          const float2 x2 = make_float2(xs_[j], xs_[j + 1]);
          const float2 pre = __ffma2_rn(x2, make_float2(t1[jj], t1[jj + 1]), make_float2(t0[jj], t0[jj + 1]));
          float2 acc = make_float2(__uint_as_float(raw[j]), __uint_as_float(raw[j + 1]));   // 0 for rows past the image
          if (kRk) {
            const float2 a0 = make_float2(rv0, rv0), a1 = make_float2(rv1, rv1), a2 = make_float2(rv2, rv2);
            acc = __ffma2_rn(a2, make_float2(k2[jj], k2[jj + 1]),
                             __ffma2_rn(a1, make_float2(k1[jj], k1[jj + 1]), __ffma2_rn(a0, make_float2(k0[jj], k0[jj + 1]), acc)));
          }
          const float2 mask = kSine ? cos_red2(pre)
                                    : make_float2(pre.x > 0.f ? 1.f : mslope, pre.y > 0.f ? 1.f : mslope);
          const float2 d = __fmul2_rn(acc, mask);
          const float2 dx = __fmul2_rn(d, x2);
          if (!kPm && valid) {
            o[j * 128] = d.x;
            o[(j + 1) * 128] = d.y;
          }
          v[j] = d.x;
          v[j + 1] = d.y;
          w[j] = dx.x;
          w[j + 1] = dx.y;
        }
      }
      if (kPm && valid) {
        float4* o4 = reinterpret_cast<float4*>(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) o4[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
      const float s1 = transpose_reduce32(v, lane);
      const float s2 = transpose_reduce32(w, lane);
      atomicAdd(m.st_sum + c0 + lane, s1);
      atomicAdd(m.st_sq + c0 + lane, s2);
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(m.bars + ACC_EMPTY + buf);
  }
  asm volatile("bar.sync 2, 128;" ::: "memory");
  if (cur_b >= 0) flush(cur_b);
}

// ------------------------------------------------------------------------------------------
// const-style variant.  kBwd: data gradient of the same half-block: the operand is dL/dout passed through
// unchanged, the weight image is W^T, the epilogue is `epilogue_bwd_loop`.
// ------------------------------------------------------------------------------------------
template <int kPasses, bool kBwd>
__global__ void __launch_bounds__(kSynThreads, 1) spade_const_kernel(SpadeArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const SynSmem m = carve(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  init_common(a, m, warp);
  const uint32_t tmem = *m.tmem_slot;
  TileMap tm;
  tm.T = (a.HW + 127) / 128;
  tm.first = blockIdx.x;
  tm.stride = gridDim.x;
  tm.count = (a.B * tm.T - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp < 8) {
    // ------------------------------------------------------------------ operand team
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    int cur_b = -1;
    uint32_t acnt = 0;   // operand chunks produced (2-slot ring)
    uint32_t xg = 0;     // activation slices walked
    for (int it = 0; it < tm.count; ++it) {
      int b, ti;
      tm.get(it, b, ti);
      if (b != cur_b && (!kBwd || a.ascale)) {  // refresh the per-sample tables of the operand team
        rows_barrier();
        for (int i = threadIdx.x; i < kC; i += 256) {
          if (kBwd) {
            m.tab_as[i] = a.ascale[static_cast<long>(b) * kC + i];
          } else {   // no table = identity (plain 1x1 convolution)
            m.tab_g1[i] = a.mod ? a.mod[(static_cast<long>(b) * 2 + 0) * kC + i] : 1.f;
            m.tab_g0[i] = a.mod ? a.mod[(static_cast<long>(b) * 2 + 1) * kC + i] : 0.f;
            if (a.mod2) {      // second source's table lives in the (otherwise pixel-style only) gamma/beta bias table
              m.tab_bgb[i] = a.mod2[(static_cast<long>(b) * 2 + 0) * kC + i];
              m.tab_bgb[kC + i] = a.mod2[(static_cast<long>(b) * 2 + 1) * kC + i];
            }
          }
        }
        rows_barrier();
        cur_b = b;
      }
      const bool valid = ti * 128 + row < a.HW;
      uint32_t tg1a = smem_u32(kBwd ? m.tab_as : m.tab_g1), tg0a = smem_u32(m.tab_g0);
      uint32_t tg1b = smem_u32(m.tab_bgb), tg0b = smem_u32(m.tab_bgb + kC);
      opaque(tg1a);   // the tables may just have been refreshed: no table load may move above this point
      opaque(tg0a);
      opaque(tg1b);
      opaque(tg0b);
      const float slope = a.slope;
      const bool sine = a.act == 1, scaled = kBwd && a.ascale != nullptr;
      const bool two_tables = !kBwd && a.mod2 != nullptr;
#pragma unroll 1
      for (int kc = 0; kc < a.nkc; ++kc, ++acnt) {
        const int c0 = (kc * 64 + h * 32) & (kC - 1);
        const bool second = two_tables && kc * 64 >= kC;
        const uint32_t tg1 = second ? tg1b : tg1a, tg0 = second ? tg0b : tg0a;
        float cur[32];
        take_x_pair(m, xg, h, row, lane, cur);
        const uint32_t slot = acnt & 1;
        mbar_wait_sleep(m.bars + A_EMPTY + slot, ((acnt >> 1) & 1) ^ 1);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float y[8], t1[8], t0[8];
          if (!kBwd || scaled) lds8(tg1 + (c0 + g * 8) * 4, t1);
          if (!kBwd) lds8(tg0 + (c0 + g * 8) * 4, t0);
          if (kBwd) {
#pragma unroll
            for (int j = 0; j < 8; ++j) y[j] = scaled ? cur[g * 8 + j] * t1[j] : cur[g * 8 + j];
          } else if (sine) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
              const float2 sv = sin_red2(__ffma2_rn(make_float2(cur[g * 8 + j], cur[g * 8 + j + 1]), make_float2(t1[j], t1[j + 1]),
                                                    make_float2(t0[j], t0[j + 1])));
              y[j] = sv.x;
              y[j + 1] = sv.y;
            }
          } else {
            affine_lrelu8(cur + g * 8, t1, t0, slope, y);
          }
          if (!valid) {   // only the last, partial tile of an image
#pragma unroll
            for (int j = 0; j < 8; ++j) y[j] = 0.f;
          }
          store_a8<kPasses == 3>(m.a_hi + slot * kAChunk, m.a_lo + slot * kAChunk, row, h * 32 + g * 8, y);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(m.bars + A_FULL + slot);
      }
    }
  } else if (warp < 12) {
    if (kBwd) {      // warp-uniform dispatch to a straight-line variant (the host side rejects the other combinations)
      if (a.act == 1) {
        if (a.rk_v) epilogue_bwd_loop<true, true, false>(a, m, tm, tmem, warp - 8, lane);
        else epilogue_bwd_loop<true, false, false>(a, m, tm, tmem, warp - 8, lane);
      } else {
        if (a.out_pm) epilogue_bwd_loop<false, false, true>(a, m, tm, tmem, warp - 8, lane);
        else epilogue_bwd_loop<false, false, false>(a, m, tm, tmem, warp - 8, lane);
      }
    } else {
      epilogue_team_loop(a, m, tm, tmem, warp - 8, lane);
    }
  } else if (warp == 12) {
    {
      const bool leader = elect_one_sync();
      const uint32_t idesc = umma_idesc_bf16(128, 256);
      MmaPipe p;
      uint32_t acnt = 0;
      for (int it = 0; it < tm.count; ++it) {
        const uint32_t buf = it & 1;
        mbar_wait_sleep(m.bars + ACC_EMPTY + buf, ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int kc = 0; kc < a.nkc; ++kc, ++acnt) {
          const uint32_t slot = acnt & 1;
          mbar_wait_sleep(m.bars + A_FULL + slot, (acnt >> 1) & 1);
          tc_fence_after();
          mma_chunk<kPasses>(m, p, leader, tmem + buf * 256, smem_u32(m.a_hi + slot * kAChunk), smem_u32(m.a_lo + slot * kAChunk),
                             idesc, kc > 0);
          umma_commit_if(leader, m.bars + A_EMPTY + slot);
        }
        umma_commit_if(leader, m.bars + ACC_FULL + buf);
      }
    }
  } else if (warp == 13) {
    if (lane == 0) {
      const uint8_t* imgs[1] = {a.wimg};
      const int ns[1] = {2 * a.nkc};
      weight_producer_loop<kPasses>(m, imgs, ns, 1, tm.count);
    }
  } else if (warp == 14) {
    if (lane == 0) x_producer_loop(a, m, tm);
  } else {
    if (lane == 0) skip_producer_loop(a, m, tm);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 12) tmem_dealloc<512>(tmem);
}

// ------------------------------------------------------------------------------------------
// pixel-style variant
// ------------------------------------------------------------------------------------------
// PyTorch's bilinear source index (align_corners=False): src = max(scale*(dst+0.5)-0.5, 0)
__device__ __forceinline__ void bilin(int dst, int in_size, float scale, int& i0, int& i1, float& l0, float& l1) {
  float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = static_cast<int>(src);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - static_cast<float>(i0);
  l0 = 1.f - l1;
}

template <int kPasses>
__global__ void __launch_bounds__(kSynThreads, 1) spade_pixel_kernel(SpadeArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const SynSmem m = carve(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kC; i += blockDim.x) {
    m.tab_g1[i] = a.scsh[i];
    m.tab_g0[i] = a.scsh[kC + i];
  }
  for (int i = threadIdx.x; i < 512; i += blockDim.x) m.tab_bgb[i] = a.bgb[i];
  init_common(a, m, warp);
  const uint32_t tmem = *m.tmem_slot;
  TileMap tm;
  tm.T = (a.HW + 127) / 128;
  tm.first = blockIdx.x;
  tm.stride = gridDim.x;
  tm.count = (a.B * tm.T - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const float sy = static_cast<float>(a.Rh) / static_cast<float>(a.Hg);
  const float sx = static_cast<float>(a.Rw) / static_cast<float>(a.Wg);

  if (warp < 8) {
    // ------------------------------------------------------------------ operand team
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    uint32_t acnt = 0, xg = 0;
    uint32_t tg1 = smem_u32(m.tab_g1), tg0 = smem_u32(m.tab_g0), tbgb = smem_u32(m.tab_bgb);   // constant tables
    opaque(tg1);
    opaque(tg0);
    opaque(tbgb);
    for (int it = 0; it < tm.count; ++it) {
      int b, ti;
      tm.get(it, b, ti);
      const int pix = ti * 128 + row;
      const bool valid = pix < a.HW;
      const uint32_t R = (it & 1) * 256, Rp = 256 - R;      // TMEM halves of this tile
      // ---- phase 0: A1 = relu(bilinear(P_lr) + c): column half h builds K chunk h into ring slot h.
      // Both slots must have been consumed by the previous tile's conv (its chunks 2 and 3).
      if (it > 0) mbar_wait_sleep(m.bars + A_EMPTY + h, 1);
      {
        const int py = valid ? pix / a.Wg : 0, px = valid ? pix % a.Wg : 0;
        int y0, y1, x0, x1;
        float ly0, ly1, lx0, lx1;
        bilin(py, a.Rh, sy, y0, y1, ly0, ly1);
        bilin(px, a.Rw, sx, x0, x1, lx0, lx1);
        const float* base = a.p_lr + static_cast<long>(b) * a.Rh * a.Rw * a.p_stride;
        const float4* n00 = reinterpret_cast<const float4*>(base + (static_cast<long>(y0) * a.Rw + x0) * a.p_stride);
        const float4* n01 = reinterpret_cast<const float4*>(base + (static_cast<long>(y0) * a.Rw + x1) * a.p_stride);
        const float4* n10 = reinterpret_cast<const float4*>(base + (static_cast<long>(y1) * a.Rw + x0) * a.p_stride);
        const float4* n11 = reinterpret_cast<const float4*>(base + (static_cast<long>(y1) * a.Rw + x1) * a.p_stride);
        const float4* pb = a.p_bias ? reinterpret_cast<const float4*>(a.p_bias + static_cast<long>(b) * 128) : nullptr;
        const float2 lx0p = make_float2(lx0, lx0), lx1p = make_float2(lx1, lx1), ly0p = make_float2(ly0, ly0), ly1p = make_float2(ly1, ly1);
#pragma unroll 2
        for (int g = 0; g < 8; ++g) {
          float y[8];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int f4 = h * 16 + g * 2 + u;
            const float4 v00 = __ldg(n00 + f4), v01 = __ldg(n01 + f4), v10 = __ldg(n10 + f4), v11 = __ldg(n11 + f4);
            // same association as upsample_bilinear2d: ly0*(lx0*a + lx1*b) + ly1*(lx0*c + lx1*d), on channel pairs (packed fp32:
            // this loop is on the critical chain of the tile -- the gamma/beta GEMM cannot start before it)
            auto lerp2 = [&](float2 a, float2 b, float2 c, float2 d) {
              const float2 top = __ffma2_rn(b, lx1p, __fmul2_rn(a, lx0p));
              const float2 bot = __ffma2_rn(d, lx1p, __fmul2_rn(c, lx0p));
              return __ffma2_rn(top, ly0p, __fmul2_rn(bot, ly1p));
            };
            float2 lo2 = lerp2(make_float2(v00.x, v00.y), make_float2(v01.x, v01.y), make_float2(v10.x, v10.y), make_float2(v11.x, v11.y));
            float2 hi2 = lerp2(make_float2(v00.z, v00.w), make_float2(v01.z, v01.w), make_float2(v10.z, v10.w), make_float2(v11.z, v11.w));
            if (pb) {
              const float4 c4 = __ldg(pb + f4);
              lo2 = __fadd2_rn(lo2, make_float2(c4.x, c4.y));
              hi2 = __fadd2_rn(hi2, make_float2(c4.z, c4.w));
            }
            y[u * 4 + 0] = lo2.x; y[u * 4 + 1] = lo2.y; y[u * 4 + 2] = hi2.x; y[u * 4 + 3] = hi2.y;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] = valid ? fmaxf(y[j], 0.f) : 0.f;
          store_a8<kPasses == 3>(m.a_hi + h * kAChunk, m.a_lo + h * kAChunk, row, g * 8, y);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(m.bars + A1_FULL);
      }
      // ---- phase 1: y = lrelu(BN(x)*(1+gamma)+beta), chunks 0,1 from half R, chunks 2,3 from half R'
#pragma unroll 1
      for (int kc = 0; kc < 4; ++kc, ++acnt) {
        const int c0 = kc * 64 + h * 32;
        const uint32_t col = (kc >> 1) * 256 + (kc & 1) * 128 + h * 32;      // index into the bias table
        const uint32_t tcol = (kc < 2 ? R : Rp) + (kc & 1) * 128 + h * 32;   // TMEM column
        float cur[32];
        take_x_pair(m, xg, h, row, lane, cur);
        if (kc == 0) {   // gamma/beta of channels 0..127 ready; A1 may be overwritten only after BOTH gamma/beta GEMMs
          mbar_wait_sleep(m.bars + G1A_FULL, it & 1);
          mbar_wait_sleep(m.bars + G1B_FULL, it & 1);
          tc_fence_after();
        }
        uint32_t gr[32], br[32];
        tmem_ld32(tmem + (static_cast<uint32_t>(q * 32) << 16) + tcol, gr);
        tmem_ld32(tmem + (static_cast<uint32_t>(q * 32) << 16) + tcol + 64, br);
        tmem_ld_wait();
        const uint32_t slot = acnt & 1;
        // chunks 0,1 overwrite A1 (free: G1B_FULL); chunks 2,3 wait for the conv to have consumed chunks 0,1
        mbar_wait_sleep(m.bars + A_EMPTY + slot, ((acnt >> 1) & 1) ^ 1);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float y[8], bg[8], bb[8], t1[8], t0[8];
          lds8(tbgb + (col + g * 8) * 4, bg);
          lds8(tbgb + (col + 64 + g * 8) * 4, bb);
          lds8(tg1 + (c0 + g * 8) * 4, t1);
          lds8(tg0 + (c0 + g * 8) * 4, t0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int jj = g * 8 + j;
            const float gam = __uint_as_float(gr[jj]) + bg[j];        // 1 + gamma
            const float bet = __uint_as_float(br[jj]) + bb[j];        // beta
            const float xn = fmaf(cur[jj], t1[j], t0[j]);
            const float v = fmaf(xn, gam, bet);
            y[j] = valid ? fmaxf(v, 0.2f * v) : 0.f;
          }
          store_a8<kPasses == 3>(m.a_hi + slot * kAChunk, m.a_lo + slot * kAChunk, row, h * 32 + g * 8, y);
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(m.bars + A_FULL + slot);
      }
    }
  } else if (warp < 12) {
    epilogue_team_loop(a, m, tm, tmem, warp - 8, lane);
  } else if (warp == 12) {
    {
      const bool leader = elect_one_sync();
      const uint32_t idesc = umma_idesc_bf16(128, 256);
      MmaPipe p;
      uint32_t acnt = 0;
      for (int it = 0; it < tm.count; ++it) {
        const uint32_t R = (it & 1) * 256, Rp = 256 - R;
        auto a1_hi = [&](int kc) { return smem_u32(m.a_hi + kc * kAChunk); };
        auto a1_lo = [&](int kc) { return smem_u32(m.a_lo + kc * kAChunk); };
        mbar_wait_sleep(m.bars + A1_FULL, it & 1);
        tc_fence_after();
        // gamma|beta of channels 0..127 -> half R: free since the previous tile read its chunks 2,3 from it
        // (that tile's A_FULL arrivals for chunks 2,3 precede this tile's A1_FULL)
        for (int kc = 0; kc < 2; ++kc) mma_chunk<kPasses>(m, p, leader, tmem + R, a1_hi(kc), a1_lo(kc), idesc, kc > 0);
        umma_commit_if(leader, m.bars + G1A_FULL);
        // gamma|beta of channels 128..255 -> half R': holds the previous tile's conv accumulator until drained
        if (it > 0) mbar_wait_sleep(m.bars + ACC_EMPTY + ((it - 1) & 1), ((it - 1) >> 1) & 1);
        tc_fence_after();
        for (int kc = 0; kc < 2; ++kc) mma_chunk<kPasses>(m, p, leader, tmem + Rp, a1_hi(kc), a1_lo(kc), idesc, kc > 0);
        umma_commit_if(leader, m.bars + G1B_FULL);
        // conv -> half R: y chunks 0 and 1 must BOTH exist first (their gamma/beta live in R)
        const uint32_t ph0 = (acnt >> 1) & 1;
        mbar_wait_sleep(m.bars + A_FULL + 0, ph0);
        mbar_wait_sleep(m.bars + A_FULL + 1, ph0);
        tc_fence_after();
        for (int kc = 0; kc < 4; ++kc, ++acnt) {
          const uint32_t slot = acnt & 1;
          if (kc >= 2) {
            mbar_wait_sleep(m.bars + A_FULL + slot, (acnt >> 1) & 1);
            tc_fence_after();
          }
          mma_chunk<kPasses>(m, p, leader, tmem + R, smem_u32(m.a_hi + slot * kAChunk), smem_u32(m.a_lo + slot * kAChunk), idesc, kc > 0);
          umma_commit_if(leader, m.bars + A_EMPTY + slot);
        }
        umma_commit_if(leader, m.bars + ACC_FULL + (it & 1));
      }
    }
  } else if (warp == 13) {
    if (lane == 0) {
      // gamma/beta image: [2 nblocks][2 kchunks][hi,lo] = 8 stages, then the conv image: 8 stages
      const uint8_t* imgs[2] = {a.wgb, a.wimg};
      const int ns[2] = {8, 8};
      weight_producer_loop<kPasses>(m, imgs, ns, 2, tm.count);
    }
  } else if (warp == 14) {
    if (lane == 0) x_producer_loop(a, m, tm);
  } else {
    if (lane == 0) skip_producer_loop(a, m, tm);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 12) tmem_dealloc<512>(tmem);
}

// ------------------------------------------------------------------------------------------
// BatchNorm finalisation: batch (or running) statistics -> scale/shift (+ fused per-sample modulation)
// ------------------------------------------------------------------------------------------
// nn.SyncBatchNorm semantics (map3d_layers.py:162): biased variance for normalisation, unbiased for
// the running estimate, momentum 0.1, eps 1e-5.
__global__ void bn_finalize_kernel(const double* __restrict__ stats, double count_in, const double* __restrict__ count_ptr,
                                   const float* __restrict__ weight,
                                   const float* __restrict__ bias, float* running_mean, float* running_var,
                                   int training, float eps, float momentum, const float* __restrict__ gb, int B,
                                   float* __restrict__ scsh, float* __restrict__ mod) {
  const int c = threadIdx.x;
  float mean, var;
  const double count = count_ptr ? count_ptr[0] : count_in;
  if (training) {
    const double mu = stats[c] / count;
    double v = stats[kC + c] / count - mu * mu;
    v = v < 0 ? 0 : v;
    mean = static_cast<float>(mu);
    var = static_cast<float>(v);
    if (running_mean) {
      const double unb = count > 1 ? v * count / (count - 1) : v;
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unb);
    }
  } else {
    mean = running_mean[c];
    var = running_var[c];
  }
  const float sc = weight[c] * rsqrtf(var + eps);
  const float sh = bias[c] - mean * sc;
  if (scsh) {
    scsh[c] = sc;
    scsh[kC + c] = sh;
  }
  if (mod && gb) {
    for (int b = 0; b < B; ++b) {
      const float G = gb[(static_cast<long>(b) * 2 + 0) * kC + c];   // 1 + gamma
      const float Bt = gb[(static_cast<long>(b) * 2 + 1) * kC + c];  // beta
      mod[(static_cast<long>(b) * 2 + 0) * kC + c] = sc * G;
      mod[(static_cast<long>(b) * 2 + 1) * kC + c] = fmaf(sh, G, Bt);
    }
  }
}

// ------------------------------------------------------------------------------------------
// synthesis input x0 = sin(W [i, j]^T + b)  (map3d_layers.py:260-275), shared by the whole batch,
// written in the tile-blocked layout [T, C, 128], with its BatchNorm statistics.
// ------------------------------------------------------------------------------------------
__global__ void synth_input_kernel(const float* __restrict__ w, const float* __restrict__ bias,
                                   const float* __restrict__ ic, const float* __restrict__ jc, int Hg, int Wg,
                                   float* __restrict__ x0, double* __restrict__ stats, double batch_mult) {
  // grid: (ceil(HW/256), C); one channel per blockIdx.y
  const int c = blockIdx.y;
  const int HW = Hg * Wg;
  const float w0 = w[c * 2 + 0], w1 = w[c * 2 + 1], bb = bias[c];
  float s1 = 0.f, s2 = 0.f;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += gridDim.x * blockDim.x) {
    const float v = sinf(fmaf(w1, jc[p % Wg], fmaf(w0, ic[p / Wg], bb)));
    x0[(static_cast<long>(p >> 7) * kC + c) * 128 + (p & 127)] = v;
    s1 += v;
    s2 += v * v;
  }
  __shared__ float r1[8], r2[8];
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0 && stats) {
    float t1 = 0.f, t2 = 0.f;
    for (int i = 0; i < static_cast<int>(blockDim.x >> 5); ++i) { t1 += r1[i]; t2 += r2[i]; }
    atomicAdd(stats + c, static_cast<double>(t1) * batch_mult);
    atomicAdd(stats + kC + c, static_cast<double>(t2) * batch_mult);
  }
}

}  // namespace hg

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int hg_spade_conv(const float* x, long x_bstride, const float* mod, const float* scsh, const float* p_lr,
                  long p_stride, const float* p_bias, const void* wgb, const float* bgb, const void* wimg, const float* bias, const float* skip,
                  float* out, double* stats, const float* rgb_w, const float* rgb_b, const float* rgb_in,
                  float* rgb_out, int B, int C, int Hg, int Wg, int Rh, int Rw, int passes, void* stream) {
  HG_REQUIRE(C == hg::kC, "hg_spade_conv: only %d channels are supported (got %d)", hg::kC, C);
  HG_REQUIRE(x && wimg && bias && out, "hg_spade_conv: null pointer");
  HG_REQUIRE((mod != nullptr) != (p_lr != nullptr), "hg_spade_conv: give exactly one of mod (const style) / p_lr (pixel style)");
  HG_REQUIRE(passes == 1 || passes == 3, "hg_spade_conv: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_spade_conv: bad shape");
  HG_REQUIRE(!rgb_w || (rgb_b && rgb_out), "hg_spade_conv: rgb_b / rgb_out missing");
  if (p_lr) {
    HG_REQUIRE(scsh && wgb && bgb && Rh > 0 && Rw > 0, "hg_spade_conv: pixel-style arguments missing");
    HG_REQUIRE((reinterpret_cast<uintptr_t>(p_lr) & 15) == 0 && p_stride >= 128 && (p_stride & 3) == 0,
               "hg_spade_conv: p_lr must be 16-byte aligned with a row stride >= 128 that is a multiple of 4");
    HG_REQUIRE(!p_bias || (reinterpret_cast<uintptr_t>(p_bias) & 15) == 0, "hg_spade_conv: p_bias must be 16-byte aligned");
  }
  hg::SpadeArgs a{x, x_bstride, mod, scsh, p_lr, p_stride, p_bias, static_cast<const uint8_t*>(wgb), bgb,
                  static_cast<const uint8_t*>(wimg), bias, skip,
                  static_cast<long>((Hg * Wg + 127) / 128) * hg::kC * 128, out, stats, rgb_w, rgb_b, rgb_in, rgb_out,
                  B, Hg * Wg, Hg, Wg, Rh, Rw};
  a.nkc = 4; a.xC = hg::kC; a.x2 = nullptr; a.slope = 0.2f; a.cout = hg::kC; a.out_pm = 0;
  const int tiles = B * ((Hg * Wg + 127) / 128);
  const int grid = tiles < hg::num_sms() ? tiles : hg::num_sms();
  auto st = static_cast<cudaStream_t>(stream);
#define HG_LAUNCH(KERNEL, THREADS)                                                                                \
  do {                                                                                                            \
    cudaError_t e = cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, hg::kSynSmemBytes); \
    if (e != cudaSuccess) { hg::set_error("hg_spade_conv: smem opt-in failed: %s", cudaGetErrorString(e)); return 2; } \
    KERNEL<<<grid, THREADS, hg::kSynSmemBytes, st>>>(a);                                                          \
  } while (0)
  if (mod) {
    if (passes == 3) HG_LAUNCH((hg::spade_const_kernel<3, false>), hg::kSynThreads); else HG_LAUNCH((hg::spade_const_kernel<1, false>), hg::kSynThreads);
  } else {
    if (passes == 3) HG_LAUNCH(hg::spade_pixel_kernel<3>, hg::kSynThreads); else HG_LAUNCH(hg::spade_pixel_kernel<1>, hg::kSynThreads);
  }
#undef HG_LAUNCH
  return hg::check_launch("hg_spade_conv");
}

static int launch_blocked_gemm(const hg::SpadeArgs& a, int passes, bool bwd, cudaStream_t st, const char* who) {
  const int tiles = a.B * ((a.HW + 127) / 128);
  const int grid = tiles < hg::num_sms() ? tiles : hg::num_sms();
  cudaError_t e;
#define HG_LAUNCH_G(KERNEL)                                                                             \
  do {                                                                                                  \
    e = cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, hg::kSynSmemBytes);   \
    if (e == cudaSuccess) KERNEL<<<grid, hg::kSynThreads, hg::kSynSmemBytes, st>>>(a);                   \
  } while (0)
  if (bwd) {
    if (passes == 3) HG_LAUNCH_G((hg::spade_const_kernel<3, true>)); else HG_LAUNCH_G((hg::spade_const_kernel<1, true>));
  } else {
    if (passes == 3) HG_LAUNCH_G((hg::spade_const_kernel<3, false>)); else HG_LAUNCH_G((hg::spade_const_kernel<1, false>));
  }
#undef HG_LAUNCH_G
  if (e != cudaSuccess) { hg::set_error("%s: smem opt-in failed: %s", who, cudaGetErrorString(e)); return 2; }
  return hg::check_launch(who);
}

int hg_spade_bwd_dgrad(const float* dout, const float* x, long x_bstride, const float* mod, const void* wimg_t, float* dpre,
                       double* sums, int B, int C, int Hg, int Wg, int passes, void* stream) {
  HG_REQUIRE(C == hg::kC, "hg_spade_bwd_dgrad: only %d channels are supported (got %d)", hg::kC, C);
  HG_REQUIRE(dout && x && mod && wimg_t && dpre && sums, "hg_spade_bwd_dgrad: null pointer");
  HG_REQUIRE(passes == 1 || passes == 3, "hg_spade_bwd_dgrad: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_spade_bwd_dgrad: bad shape");
  const long T = (Hg * Wg + 127) / 128;
  hg::SpadeArgs a{};
  a.x = dout;
  a.x_bstride = T * hg::kC * 128;
  a.mod = mod;
  a.wimg = static_cast<const uint8_t*>(wimg_t);
  a.bias = mod;            // unused by the backward epilogue; init_common reads C floats
  a.skip = x;
  a.skip_bstride = x_bstride;
  a.out = dpre;
  a.stats = sums;
  a.B = B; a.HW = Hg * Wg; a.Hg = Hg; a.Wg = Wg;
  a.nkc = 4; a.xC = hg::kC; a.slope = 0.2f; a.cout = hg::kC;
  return launch_blocked_gemm(a, passes, true, static_cast<cudaStream_t>(stream), "hg_spade_bwd_dgrad");
}

int hg_conv1x1_blocked(const float* x, int Cin, const void* wimg, const float* bias, float* out, int B, int Hg, int Wg,
                       int passes, void* stream) {
  HG_REQUIRE(x && wimg && bias && out, "hg_conv1x1_blocked: null pointer");
  HG_REQUIRE(Cin == 64 || Cin == 128 || Cin == 256, "hg_conv1x1_blocked: Cin must be 64, 128 or 256 (got %d)", Cin);
  HG_REQUIRE(passes == 1 || passes == 3, "hg_conv1x1_blocked: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_conv1x1_blocked: bad shape");
  const long T = (Hg * Wg + 127) / 128;
  hg::SpadeArgs a{};
  a.x = x;
  a.x_bstride = T * Cin * 128;
  a.wimg = static_cast<const uint8_t*>(wimg);
  a.bias = bias;
  a.skip_bstride = T * hg::kC * 128;
  a.out = out;
  a.B = B; a.HW = Hg * Wg; a.Hg = Hg; a.Wg = Wg;
  a.nkc = Cin / 64; a.xC = Cin; a.slope = 1.f; a.cout = hg::kC;
  return launch_blocked_gemm(a, passes, false, static_cast<cudaStream_t>(stream), "hg_conv1x1_blocked");
}

int hg_act_conv1x1_blocked(const float* x, const float* x2, const float* mod, int act, const void* wimg, const float* bias,
                           float* out, int B, int Hg, int Wg, int passes, void* stream) {
  HG_REQUIRE(x && mod && wimg && bias && out, "hg_act_conv1x1_blocked: null pointer");
  HG_REQUIRE(act == 0 || act == 1, "hg_act_conv1x1_blocked: act must be 0 (LeakyReLU 0.2) or 1 (sine)");
  HG_REQUIRE(passes == 1 || passes == 3, "hg_act_conv1x1_blocked: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_act_conv1x1_blocked: bad shape");
  const long T = (Hg * Wg + 127) / 128;
  hg::SpadeArgs a{};
  a.x = x;
  a.x_bstride = T * hg::kC * 128;
  a.x2 = x2;
  a.mod = mod;
  a.wimg = static_cast<const uint8_t*>(wimg);
  a.bias = bias;
  a.skip_bstride = T * hg::kC * 128;
  a.out = out;
  a.B = B; a.HW = Hg * Wg; a.Hg = Hg; a.Wg = Wg;
  a.nkc = x2 ? 8 : 4; a.xC = hg::kC; a.slope = 0.2f; a.cout = hg::kC; a.act = act;
  return launch_blocked_gemm(a, passes, false, static_cast<cudaStream_t>(stream), "hg_act_conv1x1_blocked");
}

int hg_blocked_conv_wide(const float* x, const float* x2, const float* mod, const float* mod2, int act, float slope,
                         const void* wimg, const float* bias, const float* skip, float* out, double* stats,
                         const float* rgb_w, const float* rgb_b, const float* rgb_in, float* rgb_out, int B, int Hg, int Wg,
                         int passes, void* stream) {
  HG_REQUIRE(x && wimg && bias && out, "hg_blocked_conv_wide: null pointer");
  HG_REQUIRE(act == 0 || act == 1, "hg_blocked_conv_wide: act must be 0 (LeakyReLU(slope)) or 1 (sine)");
  HG_REQUIRE(slope >= 0.f && slope <= 1.f, "hg_blocked_conv_wide: the operand computes LeakyReLU as max(v, slope*v), "
             "which needs 0 <= slope <= 1 (got %g)", static_cast<double>(slope));
  HG_REQUIRE(!mod2 || (mod && x2), "hg_blocked_conv_wide: mod2 needs mod and a second source");
  HG_REQUIRE(!rgb_w || (rgb_b && rgb_out), "hg_blocked_conv_wide: rgb_b / rgb_out missing");
  HG_REQUIRE(passes == 1 || passes == 3, "hg_blocked_conv_wide: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_blocked_conv_wide: bad shape");
  const long T = (Hg * Wg + 127) / 128;
  hg::SpadeArgs a{};
  a.x = x;
  a.x_bstride = T * hg::kC * 128;
  a.x2 = x2;
  a.mod = mod;
  a.mod2 = mod2;
  a.wimg = static_cast<const uint8_t*>(wimg);
  a.bias = bias;
  a.skip = skip;
  a.skip_bstride = T * hg::kC * 128;
  a.out = out;
  a.stats = stats;
  a.rgb_w = rgb_w; a.rgb_b = rgb_b; a.rgb_in = rgb_in; a.rgb_out = rgb_out;
  a.B = B; a.HW = Hg * Wg; a.Hg = Hg; a.Wg = Wg;
  a.nkc = x2 ? 8 : 4; a.xC = hg::kC; a.slope = slope; a.cout = hg::kC; a.act = act;
  return launch_blocked_gemm(a, passes, false, static_cast<cudaStream_t>(stream), "hg_blocked_conv_wide");
}

int hg_conv1x1_blocked_bwd(const float* g, const float* g2, const float* aux, const float* mod, const void* wimg_t,
                           float* out, double* sums, int Cout, float slope, int pixel_major, int act, const float* ascale,
                           const float* rk_w, const float* rk_v, int rk_n, int B, int Hg, int Wg, int passes,
                           void* stream) {
  HG_REQUIRE(act == 0 || act == 1, "hg_conv1x1_blocked_bwd: act must be 0 (LeakyReLU/ReLU mask) or 1 (cosine)");
  HG_REQUIRE(!ascale || !g2, "hg_conv1x1_blocked_bwd: the operand scale is built for K = 256");
  HG_REQUIRE(!rk_v || (rk_w && rk_n >= 1 && rk_n <= 3 && Cout == 256), "hg_conv1x1_blocked_bwd: bad rank-k term");
  HG_REQUIRE(g && aux && wimg_t && out && sums, "hg_conv1x1_blocked_bwd: null pointer");
  HG_REQUIRE(Cout == 128 || Cout == 256, "hg_conv1x1_blocked_bwd: Cout must be 128 or 256 (got %d)", Cout);
  HG_REQUIRE(!pixel_major || Cout == 128, "hg_conv1x1_blocked_bwd: the pixel-major output is built for Cout == 128");
  HG_REQUIRE(!(act == 1 && pixel_major) && !(act == 0 && rk_v),
             "hg_conv1x1_blocked_bwd: compiled epilogues are sine [+ rank-k term] / LeakyReLU [+ pixel-major output]");
  HG_REQUIRE(passes == 1 || passes == 3, "hg_conv1x1_blocked_bwd: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_conv1x1_blocked_bwd: bad shape");
  const long T = (Hg * Wg + 127) / 128;
  hg::SpadeArgs a{};
  a.x = g;
  a.x_bstride = T * hg::kC * 128;
  a.x2 = g2;
  a.mod = mod;
  a.wimg = static_cast<const uint8_t*>(wimg_t);
  a.bias = static_cast<const float*>(wimg_t);   // unused by the backward epilogue; init_common reads C floats
  a.skip = aux;
  a.skip_bstride = T * Cout * 128;
  a.out = out;
  a.stats = sums;
  a.B = B; a.HW = Hg * Wg; a.Hg = Hg; a.Wg = Wg;
  a.nkc = g2 ? 8 : 4; a.xC = hg::kC; a.slope = slope; a.cout = Cout; a.out_pm = pixel_major;
  a.act = act; a.ascale = ascale; a.rgb_w = rk_v ? rk_w : nullptr; a.rk_v = rk_v; a.rk_n = rk_n;
  return launch_blocked_gemm(a, passes, true, static_cast<cudaStream_t>(stream), "hg_conv1x1_blocked_bwd");
}

int hg_bn_finalize(const double* stats, double count, const double* count_dev, const float* weight, const float* bias, float* running_mean,
                   float* running_var, int training, float eps, float momentum, const float* gb, int B, int C,
                   float* scsh, float* mod, void* stream) {
  HG_REQUIRE(C == hg::kC, "hg_bn_finalize: only %d channels are supported (got %d)", hg::kC, C);
  HG_REQUIRE(weight && bias && (scsh || mod), "hg_bn_finalize: null pointer");
  HG_REQUIRE(training ? (stats != nullptr && (count > 0 || count_dev)) : (running_mean && running_var),
             "hg_bn_finalize: statistics missing");
  hg::bn_finalize_kernel<<<1, hg::kC, 0, static_cast<cudaStream_t>(stream)>>>(
      stats, count, count_dev, weight, bias, running_mean, running_var, training, eps, momentum, gb, B, scsh, mod);
  return hg::check_launch("hg_bn_finalize");
}

int hg_synth_input(const float* w, const float* bias, const float* ic, const float* jc, int C, int Hg, int Wg,
                   float* x0, double* stats, int batch, void* stream) {
  HG_REQUIRE(C == hg::kC, "hg_synth_input: only %d channels are supported (got %d)", hg::kC, C);
  HG_REQUIRE(w && bias && ic && jc && x0, "hg_synth_input: null pointer");
  const int HW = Hg * Wg;
  int bx = (HW + 255) / 256;
  if (bx > 32) bx = 32;
  dim3 grid(bx, C);
  hg::synth_input_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(w, bias, ic, jc, Hg, Wg, x0, stats,
                                                                              static_cast<double>(batch));
  return hg::check_launch("hg_synth_input");
}

}  // extern "C"
