// Backward of one const-style SPADE half-block (forward: csrc/synth.cu; reference: autograd through
// SPADE2d.forward lib/components/map3d_layers.py:176-190 and SPADEBlock.forward :218-238).
//
// With the folded forward  pre = x*g1[b,c] + g0[b,c],  y = lrelu_0.2(pre),  out = W y + bias (+ skip) the
// gradients split into three streaming kernels over the tile-blocked activations [B, T, C=256, 128]:
//
//   hg_spade_bwd_dgrad   (csrc/synth.cu, tcgen05)   dpre = (W^T dout) * lrelu'(pre);  S1[b,c] = sum dpre,
//                                                   S2[b,c] = sum dpre*x
//   hg_spade_bwd_wgrad   (here, tcgen05)            dW[co,ci] = sum_{b,p} dout[b,co,p] * y[b,ci,p]  (y recomputed),
//                                                   dbias[co] = sum dout
//   hg_spade_bwd_combine (here, streaming)          dL/dx = dpre*g1[b,c] + a[c] + k[c]*x  (+ skip gradient)
//                                                   (+ W_rgb^T drgb), and the ToRGB weight gradient
//
// a[c], k[c] carry the gradient that reaches x through the batch statistics (d/dx of sum x and sum x^2); they
// and every other [B,C]/[C]-sized quantity are computed on the host side from S1, S2 (modules/synthesis_bwd.py).
//
// wgrad layout.  Both operands of dW = dout . y^T are K-major in the blocked layout as stored (K = pixels, 128
// contiguous per channel row), so the operand warps only convert rows (coalesced 256 B row segments -> bf16 hi/lo
// SW128 images); per-row constants (g1, g0) instead of per-column ones.  The [256 x 256] fp32 accumulator fills
// the whole TMEM (two M=128 halves x 256 columns) for the CTA's lifetime and is written once, as a per-CTA
// partial, then reduced deterministically by `wgrad_reduce_kernel`.
#include "common.cuh"
#include "umma.cuh"

namespace hg {

constexpr int kWC = 256;
constexpr int kWgThreads = 512;                 // 16 operand warps; warp 0 also issues the MMAs (one elected lane)
constexpr uint32_t kWgImg = 256 * 128;          // [256 rows x 64 px] bf16 = 32 KB
// dout image (hi, lo) double-buffered, x image (hi, lo) single: 6 x 32 KB
constexpr uint32_t kWgSmemBytes = 6 * kWgImg + 8 * 8 + 16 + 1024;

struct WgradArgs {
  const float* dout;     // [B,T,C,128]
  const float* x;        // [B or 1,T,C,128]
  long x_bstride;
  const float* mod;      // [B,2,C] g1, g0
  float* part_w;         // [grid, C, nq]
  float* part_b;         // [grid, C]
  int B, HW;
  int nq;                // rows (channels) of the second operand x: 256, or 128 (gamma/beta weight gradients)
  int act;               // y = 0: lrelu_0.2(x*g1+g0), 1: sin(x*g1+g0), 2: x (identity)
  const float* pscale;   // [B,C] per-(b,row) scale of dout, or null
};

enum { WG_FULL = 0, WG_EMPTY = 1, WG_DONE = 2 };

// the renderer's sine (csrc/render.cu `sin_reduced`): Cody-Waite reduction by 2*pi + SFU
__device__ __forceinline__ float wg_red(float t) {
  const float y = t * 0.15915494309189535f;
  const float k = (y + 12582912.f) - 12582912.f;
  float r = fmaf(-k, 6.2831854820251465f, t);
  return fmaf(-k, -1.7484555314695172e-07f, r);
}
__device__ __forceinline__ float wg_sin(float t) { return __sinf(wg_red(t)); }
__device__ __forceinline__ float wg_cos(float t) { return __cosf(wg_red(t)); }

// Schedule (chunk c = 64 pixels of a tile; a thread owns 8 pixels of 4 rows per operand):
//     convert x(c) -> B image      needs MMA(c-1) done (single buffer)
//     arrive FULL(c); lane 0 of warp 0 issues MMA(c) on (A[c&1], B)
//     convert dout(c+1) -> A[(c+1)&1]   while MMA(c) runs (that slot was read last by MMA(c-1))
// and the global loads of chunk c+1 (x) / c+2 (dout) are issued as soon as their registers are free, so HBM latency is
// hidden behind the conversions and the MMA wait.  (The first version had 8 operand warps, one image of each operand and
// loaded x only after converting dout: ncu showed 29 % of the samples waiting for MMA(c-1) and 14 % on the exposed x loads.)
template <int kPasses, int kAct>
__global__ void __launch_bounds__(kWgThreads, 1) spade_wgrad_kernel(WgradArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* s = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_img = s;                      // [slot][hi, lo]
  uint8_t* b_hi = s + 4 * kWgImg;
  uint8_t* b_lo = s + 5 * kWgImg;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s + 6 * kWgImg);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    mbar_init(bars + WG_FULL, 16);
    mbar_init(bars + WG_EMPTY, 1);
    mbar_init(bars + WG_DONE, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int T = (a.HW + 127) / 128;
  const int total = a.B * T;
  const int count = (total - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int nchunks = 2 * count;
  const int nq = a.nq, HW = a.HW;
  const int nst = nq >> 6;                    // row steps of the x operand: 4 (256 rows) or 2 (128)
  const bool leader = warp == 0 && elect_one_sync();     // warp-uniform condition first: only warp 0 executes the elect
  const uint32_t idesc = umma_idesc_bf16(128, nq);

  const int sub = threadIdx.x & 7;            // which 8-pixel group of the 64-pixel chunk
  const int rsub = threadIdx.x >> 3;          // 0..63: row within a 64-row step
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
  float4 va[8], vb[8];

  // chunk c -> sample, tile, first pixel of this thread, pixels of the image left from there
  auto locate = [&](int c, int& b, int& ti, int& p0, int& nvalid) {
    const int tile = blockIdx.x + (c >> 1) * gridDim.x;
    b = tile / T;
    ti = tile - b * T;
    p0 = (c & 1) * 64 + sub * 8;
    nvalid = HW - (ti * 128 + p0);
  };
  auto load_d = [&](int c) {
    int b, ti, p0, nv;
    locate(c, b, ti, p0, nv);
    const float* base = a.dout + (static_cast<long>(b) * T + ti) * kWC * 128 + rsub * 128 + p0;
#pragma unroll
    for (int st = 0; st < 4; ++st) {
      const float4* src = reinterpret_cast<const float4*>(base + st * 64 * 128);
      va[2 * st] = __ldcs(src);
      va[2 * st + 1] = __ldcs(src + 1);
    }
  };
  auto load_x = [&](int c) {
    int b, ti, p0, nv;
    locate(c, b, ti, p0, nv);
    const float* base = a.x + static_cast<long>(b) * a.x_bstride + static_cast<long>(ti) * nq * 128 + rsub * 128 + p0;
#pragma unroll
    for (int st = 0; st < 4; ++st) {
      if (st < nst) {
        const float4* src = reinterpret_cast<const float4*>(base + st * 64 * 128);
        vb[2 * st] = __ldcs(src);
        vb[2 * st + 1] = __ldcs(src + 1);
      }
    }
  };
  auto convert_d = [&](int c) {      // dout rows of chunk c -> A[c & 1]; bias partial sums
    int b, ti, p0, nvalid;
    locate(c, b, ti, p0, nvalid);
    uint8_t* hi = a_img + (c & 1) * 2 * kWgImg;
    uint8_t* lo = hi + kWgImg;
#pragma unroll
    for (int st = 0; st < 4; ++st) {
      const int row = st * 64 + rsub;
      float y[8] = {va[2 * st].x, va[2 * st].y, va[2 * st].z, va[2 * st].w,
                    va[2 * st + 1].x, va[2 * st + 1].y, va[2 * st + 1].z, va[2 * st + 1].w};
      if (nvalid < 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = j < nvalid ? y[j] : 0.f;
      }
      if (a.pscale) {
        const float ps = __ldg(a.pscale + static_cast<long>(b) * kWC + row);
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] *= ps;
      }
      bsum[st] += ((y[0] + y[1]) + (y[2] + y[3])) + ((y[4] + y[5]) + (y[6] + y[7]));
      store_a8<kPasses == 3>(hi, lo, row, sub * 8, y);
    }
  };
  auto convert_x = [&](int c) {      // x rows of chunk c -> act(x*g1 + g0) -> B
    int b, ti, p0, nvalid;
    locate(c, b, ti, p0, nvalid);
#pragma unroll
    for (int st = 0; st < 4; ++st) {
      if (st < nst) {
        const int row = st * 64 + rsub;
        float g1 = 1.f, g0 = 0.f;               // no table: y = act(x)
        if (a.mod) {
          g1 = __ldg(a.mod + (static_cast<long>(b) * 2 + 0) * kWC + row);
          g0 = __ldg(a.mod + (static_cast<long>(b) * 2 + 1) * kWC + row);
        }
        float y[8] = {vb[2 * st].x, vb[2 * st].y, vb[2 * st].z, vb[2 * st].w,
                      vb[2 * st + 1].x, vb[2 * st + 1].y, vb[2 * st + 1].z, vb[2 * st + 1].w};
        if (kAct == 1) {
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] = wg_sin(fmaf(y[j], g1, g0));
        } else {      // packed fp32 on pixel pairs: affine (+ LeakyReLU as max(v, 0.2 v))
          const float2 g1p = make_float2(g1, g1), g0p = make_float2(g0, g0);
#pragma unroll
          for (int j = 0; j < 8; j += 2) {
            const float2 v = __ffma2_rn(make_float2(y[j], y[j + 1]), g1p, g0p);
            if (kAct == 2) {
              y[j] = v.x;
              y[j + 1] = v.y;
            } else {
              const float2 sv = __fmul2_rn(v, make_float2(0.2f, 0.2f));
              y[j] = fmaxf(v.x, sv.x);
              y[j + 1] = fmaxf(v.y, sv.y);
            }
          }
        }
        if (nvalid < 8) {
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] = j < nvalid ? y[j] : 0.f;
        }
        store_a8<kPasses == 3>(b_hi, b_lo, row, sub * 8, y);
      }
    }
  };

  if (nchunks > 0) {
    load_d(0);
    load_x(0);
    convert_d(0);
    if (nchunks > 1) load_d(1);
    for (int c = 0; c < nchunks; ++c) {
      if (c > 0) mbar_wait_sleep(bars + WG_EMPTY, (c - 1) & 1);      // MMA(c-1) done: B and A[(c-1)&1] are free
      convert_x(c);
      if (c + 1 < nchunks) load_x(c + 1);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + WG_FULL);
      if (warp == 0) {      // the whole warp waits; its elected lane issues (convergent code: descriptors in uniform registers)
        mbar_wait_sleep(bars + WG_FULL, c & 1);
        tc_fence_after();
        const uint32_t ah0 = smem_u32(a_img + (c & 1) * 2 * kWgImg), al0 = ah0 + kWgImg;
#pragma unroll
        for (uint32_t mh = 0; mh < 2; ++mh) {
          const uint32_t d = tmem + mh * 256;
          const uint32_t ah = ah0 + mh * (kWgImg / 2), al = al0 + mh * (kWgImg / 2);
          umma_k64_if(leader, d, ah, smem_u32(b_hi), idesc, c > 0);
          if (kPasses == 3) {
            umma_k64_if(leader, d, al, smem_u32(b_hi), idesc, true);
            umma_k64_if(leader, d, ah, smem_u32(b_lo), idesc, true);
          }
        }
        umma_commit_if(leader, bars + WG_EMPTY);
        if (c + 1 == nchunks) umma_commit_if(leader, bars + WG_DONE);
      }
      if (c + 1 < nchunks) {
        convert_d(c + 1);
        if (c + 2 < nchunks) load_d(c + 2);
      }
    }
  }
  // bias-gradient partials: row (st*64 + rsub) is shared by the 8 `sub` lanes
#pragma unroll
  for (int st = 0; st < 4; ++st) {
    float v = bsum[st];
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    if (sub == 0) a.part_b[static_cast<long>(blockIdx.x) * kWC + st * 64 + rsub] = v;
  }
  // ---- drain: warps 0-3 own TMEM lanes 32w..32w+31 (co within the half), 2 x 256 columns (ci)
  if (warp < 4) {
    float* dst = a.part_w + static_cast<long>(blockIdx.x) * kWC * a.nq;
    if (count > 0) {
      mbar_wait_sleep(bars + WG_DONE, 0);
      tc_fence_after();
      for (int mh = 0; mh < 2; ++mh) {
        const int co = mh * 128 + warp * 32 + lane;
        for (int cg = 0; cg < (a.nq >> 5); ++cg) {
          uint32_t raw[32];
          tmem_ld32(tmem + mh * 256 + (static_cast<uint32_t>(warp * 32) << 16) + cg * 32, raw);
          tmem_ld_wait();
          float4* o = reinterpret_cast<float4*>(dst + static_cast<long>(co) * a.nq + cg * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            o[j] = make_float4(__uint_as_float(raw[4 * j]), __uint_as_float(raw[4 * j + 1]), __uint_as_float(raw[4 * j + 2]),
                               __uint_as_float(raw[4 * j + 3]));
        }
      }
    } else {
      for (int i = threadIdx.x; i < kWC * a.nq; i += 128) dst[i] = 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

// dW[i] = sum over CTAs of part[cta][i] (fp64 accumulation, fixed order -> deterministic), likewise the bias.
__global__ void wgrad_reduce_kernel(const float* __restrict__ part_w, const float* __restrict__ part_b, int nparts,
                                    int nw, float* __restrict__ dw, float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nw) {
    double acc = 0.0;
    for (int p = 0; p < nparts; ++p) acc += static_cast<double>(part_w[static_cast<long>(p) * nw + i]);
    dw[i] = static_cast<float>(acc);
  }
  if (db && i < kWC) {
    double acc = 0.0;
    for (int p = 0; p < nparts; ++p) acc += static_cast<double>(part_b[static_cast<long>(p) * kWC + i]);
    db[i] = static_cast<float>(acc);
  }
}

// ------------------------------------------------------------------------------------------
// combine: the gradient that reaches the INPUT x of a half-block (= the output of the previous one)
//   dx[b,c,p] = dpre[b,c,p]*g1[b,c] + a[c] + k[c]*x[b,c,p]  (+ dskip[b,c,p])  (+ sum_j W_rgb[j,c]*drgb[b,j,p])
// plus, when x is also the input of a ToRGB layer, dW_rgb[j,c] = sum_{b,p} drgb[b,j,p]*x[b,c,p].
// Pure streaming: warp w owns channels w, w+8, ...; a lane owns 4 consecutive pixels of the 128-pixel tile.
// ------------------------------------------------------------------------------------------
struct CombineArgs {
  const float* dpre;     // [B,T,C,128] or null (then only the skip / rgb terms)
  const float* x;        // [B or 1,T,C,128] (needed when k or rgb_w is given)
  long x_bstride;
  const float* g1;       // [B,2,C] (row 0 used) or null
  const float* ak;       // [2,C]: a, k or null
  const float* dskip;    // [B,T,C,128] or null
  const float* drgb;     // [B,3,HW] or null
  const float* rgb_w;    // [3,C]
  float* dx;             // [B,T,C,128]
  double* dwrgb;         // [3,C] accumulated, or null
  int B, HW;
};

__global__ void __launch_bounds__(256) spade_combine_kernel(CombineArgs a) {
  __shared__ float s_wrgb[3 * kWC];
  __shared__ float s_acc[3 * kWC];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 3 * kWC; i += blockDim.x) {
    s_wrgb[i] = a.drgb ? a.rgb_w[i] : 0.f;
    s_acc[i] = 0.f;
  }
  __syncthreads();
  const int T = (a.HW + 127) / 128;
  const int total = a.B * T;
  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const int b = tile / T, ti = tile - b * T;
    const int p = ti * 128 + lane * 4;
    const long off = (static_cast<long>(b) * T + ti) * kWC * 128 + lane * 4;
    const long xoff = static_cast<long>(b) * a.x_bstride + static_cast<long>(ti) * kWC * 128 + lane * 4;
    float4 r[3];
    if (a.drgb) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const float* src = a.drgb + (static_cast<long>(b) * 3 + j) * a.HW + p;
        r[j] = p + 3 < a.HW ? *reinterpret_cast<const float4*>(src)
                            : make_float4(p < a.HW ? src[0] : 0.f, p + 1 < a.HW ? src[1] : 0.f, p + 2 < a.HW ? src[2] : 0.f, 0.f);
      }
    }
    // padding rows (past HW) are SELECTED away, not multiplied by 0: the producers never write them, so they may hold NaN
    const bool m0 = p < a.HW, m1 = p + 1 < a.HW, m2 = p + 2 < a.HW, m3 = p + 3 < a.HW;
#pragma unroll 4
    for (int c = warp; c < kWC; c += 8) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.ak || a.drgb) xv = __ldcs(reinterpret_cast<const float4*>(a.x + xoff + c * 128));
      xv = make_float4(m0 ? xv.x : 0.f, m1 ? xv.y : 0.f, m2 ? xv.z : 0.f, m3 ? xv.w : 0.f);
      if (a.dpre) {
        const float4 d = __ldcs(reinterpret_cast<const float4*>(a.dpre + off + c * 128));
        const float g = a.g1[static_cast<long>(b) * 2 * kWC + c];
        v = make_float4(d.x * g, d.y * g, d.z * g, d.w * g);
      }
      if (a.ak) {
        const float aa = a.ak[c], kk = a.ak[kWC + c];
        v.x += fmaf(kk, xv.x, aa); v.y += fmaf(kk, xv.y, aa); v.z += fmaf(kk, xv.z, aa); v.w += fmaf(kk, xv.w, aa);
      }
      if (a.dskip) {
        const float4 d = __ldcs(reinterpret_cast<const float4*>(a.dskip + off + c * 128));
        v.x += d.x; v.y += d.y; v.z += d.z; v.w += d.w;
      }
      if (a.drgb) {
        float t[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const float w = s_wrgb[j * kWC + c];
          v.x = fmaf(w, r[j].x, v.x); v.y = fmaf(w, r[j].y, v.y); v.z = fmaf(w, r[j].z, v.z); v.w = fmaf(w, r[j].w, v.w);
          t[j] = (r[j].x * xv.x + r[j].y * xv.y) + (r[j].z * xv.z + r[j].w * xv.w);
        }
        if (a.dwrgb) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            t[0] += __shfl_xor_sync(0xffffffffu, t[0], o);
            t[1] += __shfl_xor_sync(0xffffffffu, t[1], o);
            t[2] += __shfl_xor_sync(0xffffffffu, t[2], o);
          }
          if (lane == 0) {   // channel c belongs to this warp alone: no atomics
            s_acc[c] += t[0];
            s_acc[kWC + c] += t[1];
            s_acc[2 * kWC + c] += t[2];
          }
        }
      }
      v = make_float4(m0 ? v.x : 0.f, m1 ? v.y : 0.f, m2 ? v.z : 0.f, m3 ? v.w : 0.f);
      __stcs(reinterpret_cast<float4*>(a.dx + off + c * 128), v);
    }
  }
  __syncthreads();
  if (a.dwrgb)
    for (int i = threadIdx.x; i < 3 * kWC; i += blockDim.x) atomicAdd(a.dwrgb + i, static_cast<double>(s_acc[i]));
}


// ------------------------------------------------------------------------------------------
// synthesis input backward: x0[c,p] = sin(w[c,0]*i(p) + w[c,1]*j(p) + b[c]) is shared by the batch, so
//   darg[c,p] = cos(arg) * sum_b dx[b,c,p];  dw[c,0] = sum_p darg*i,  dw[c,1] = sum_p darg*j,  db[c] = sum_p darg
// (autograd through SynthesisInput.forward, map3d_layers.py:260-275).  One block per channel.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) synth_input_bwd_kernel(const float* __restrict__ dx, const float* __restrict__ w,
                                                              const float* __restrict__ bias, const float* __restrict__ ic,
                                                              const float* __restrict__ jc, int B, int Hg, int Wg,
                                                              float* __restrict__ dw, float* __restrict__ db) {
  const int c = blockIdx.x;
  const int HW = Hg * Wg, T = (HW + 127) / 128;
  const float w0 = w[c * 2 + 0], w1 = w[c * 2 + 1], bb = bias[c];
  double a0 = 0.0, a1 = 0.0, a2 = 0.0;
  for (int p = threadIdx.x; p < HW; p += blockDim.x) {
    const float iv = ic[p / Wg], jv = jc[p % Wg];
    float g = 0.f;
    for (int b = 0; b < B; ++b) g += dx[((static_cast<long>(b) * T + (p >> 7)) * kWC + c) * 128 + (p & 127)];
    const float d = g * cosf(fmaf(w1, jv, fmaf(w0, iv, bb)));
    a0 += static_cast<double>(d * iv);
    a1 += static_cast<double>(d * jv);
    a2 += static_cast<double>(d);
  }
  __shared__ double red[3][8];
  for (int o = 16; o > 0; o >>= 1) {
    a0 += __shfl_xor_sync(0xffffffffu, a0, o);
    a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    a2 += __shfl_xor_sync(0xffffffffu, a2, o);
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a0; red[1][threadIdx.x >> 5] = a1; red[2][threadIdx.x >> 5] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t0 = 0, t1 = 0, t2 = 0;
    for (int i = 0; i < 8; ++i) { t0 += red[0][i]; t1 += red[1][i]; t2 += red[2][i]; }
    dw[c * 2 + 0] = static_cast<float>(t0);
    dw[c * 2 + 1] = static_cast<float>(t1);
    db[c] = static_cast<float>(t2);
  }
}


// ------------------------------------------------------------------------------------------
// Pixel-style half-blocks (gamma/beta per pixel).  Forward, per pixel p of sample b:
//   A1 = relu(bilinear_up(P_lr)[p] + c[b])            [128]   (P_lr = W_shared . feature_maps at render resolution)
//   gam = Wg A1 + bg + 1,  bet = Wb A1 + bb           [256]
//   pre = (x*sc + sh)*gam + bet,  y = lrelu(pre),  out = W y + bias
// The backward schedule (modules/synthesis_train.py) recomputes A1, gam, bet, pre with the kernels below + the
// generic blocked 1x1 convolution, then re-uses the const-style dgrad / wgrad / combine kernels on `pre`.
// ------------------------------------------------------------------------------------------
// PyTorch's bilinear source index (align_corners=False): src = max(scale*(dst+0.5)-0.5, 0)
__device__ __forceinline__ void bilin_src(int dst, int in_size, float scale, int& i0, int& i1, float& l0, float& l1) {
  float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = static_cast<int>(src);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - static_cast<float>(i0);
  l0 = 1.f - l1;
}

// A1 in the tile-blocked layout [B,T,128,128]; one block = one tile, one thread = one pixel.
__global__ void __launch_bounds__(128) a1_gather_kernel(const float* __restrict__ p_lr, long p_stride,
                                                        const float* __restrict__ p_bias, float* __restrict__ a1, int B,
                                                        int Hg, int Wg, int Rh, int Rw) {
  const int HW = Hg * Wg, T = (HW + 127) / 128;
  const int tile = blockIdx.x, b = tile / T, ti = tile - b * T;
  const int pix = ti * 128 + threadIdx.x;
  const bool valid = pix < HW;
  const int py = valid ? pix / Wg : 0, px = valid ? pix % Wg : 0;
  int y0, y1, x0, x1;
  float ly0, ly1, lx0, lx1;
  bilin_src(py, Rh, static_cast<float>(Rh) / static_cast<float>(Hg), y0, y1, ly0, ly1);
  bilin_src(px, Rw, static_cast<float>(Rw) / static_cast<float>(Wg), x0, x1, lx0, lx1);
  const float* base = p_lr + static_cast<long>(b) * Rh * Rw * p_stride;
  const float4* n00 = reinterpret_cast<const float4*>(base + (static_cast<long>(y0) * Rw + x0) * p_stride);
  const float4* n01 = reinterpret_cast<const float4*>(base + (static_cast<long>(y0) * Rw + x1) * p_stride);
  const float4* n10 = reinterpret_cast<const float4*>(base + (static_cast<long>(y1) * Rw + x0) * p_stride);
  const float4* n11 = reinterpret_cast<const float4*>(base + (static_cast<long>(y1) * Rw + x1) * p_stride);
  const float4* pb = p_bias ? reinterpret_cast<const float4*>(p_bias + static_cast<long>(b) * 128) : nullptr;
  float* dst = a1 + static_cast<long>(tile) * 128 * 128 + threadIdx.x;
#pragma unroll 4
  for (int f4 = 0; f4 < 32; ++f4) {
    const float4 v00 = __ldg(n00 + f4), v01 = __ldg(n01 + f4), v10 = __ldg(n10 + f4), v11 = __ldg(n11 + f4);
    // the SAME packed operation sequence as the forward kernel (csrc/synth.cu phase 0), so that the recomputed A1 and its ReLU mask
    // are bit-identical to what the forward multiplied with
    const float2 lx0p = make_float2(lx0, lx0), lx1p = make_float2(lx1, lx1), ly0p = make_float2(ly0, ly0), ly1p = make_float2(ly1, ly1);
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
    const float4 y = make_float4(lo2.x, lo2.y, hi2.x, hi2.y);
    dst[(f4 * 4 + 0) * 128] = valid ? fmaxf(y.x, 0.f) : 0.f;
    dst[(f4 * 4 + 1) * 128] = valid ? fmaxf(y.y, 0.f) : 0.f;
    dst[(f4 * 4 + 2) * 128] = valid ? fmaxf(y.z, 0.f) : 0.f;
    dst[(f4 * 4 + 3) * 128] = valid ? fmaxf(y.w, 0.f) : 0.f;
  }
}

// pre = (x*sc[c] + sh[c])*gam + bet, written over bet.  All tensors tile-blocked [B,T,C,128].
__global__ void __launch_bounds__(256) pixel_pre_kernel(const float* __restrict__ x, long x_bstride, const float* __restrict__ scsh,
                                                        const float* __restrict__ gam, float* __restrict__ bet_pre, int B,
                                                        int T) {
  const long per_b = static_cast<long>(T) * kWC * 32;     // float4 per sample
  const long n4 = per_b * B;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>((i >> 5) & (kWC - 1));
    const long b = i / per_b;
    const float sc = scsh[c], sh = scsh[kWC + c];
    const float4 xv = __ldcs(reinterpret_cast<const float4*>(x + b * x_bstride) + (i - b * per_b));
    const float4 g = __ldcs(reinterpret_cast<const float4*>(gam) + i);
    float4 t = __ldcs(reinterpret_cast<const float4*>(bet_pre) + i);
    t.x = fmaf(fmaf(xv.x, sc, sh), g.x, t.x);
    t.y = fmaf(fmaf(xv.y, sc, sh), g.y, t.y);
    t.z = fmaf(fmaf(xv.z, sc, sh), g.z, t.z);
    t.w = fmaf(fmaf(xv.w, sc, sh), g.w, t.w);
    __stcs(reinterpret_cast<float4*>(bet_pre) + i, t);
  }
}

// dxn = dpre*gam (over `pre_dxn`), dgam = dpre*(x*sc+sh) (over `gam_dgam`); per-channel sums
//   sums[0][c] = sum dxn*x, sums[1][c] = sum dxn, sums[2][c] = sum dgam     (fp64, accumulated)
// over the valid pixels only: the padding rows of the last tile hold whatever the producers left there (dpre comes from
// the data-gradient engine, which never writes them), so they are selected away and written back as zeros.
// Same mapping as the combine kernel: warp w owns channels w, w+8, ..., a lane owns 4 pixels of the tile.
__global__ void __launch_bounds__(256) pixel_mod_bwd_kernel(const float* __restrict__ dpre, const float* __restrict__ x,
                                                            long x_bstride, const float* __restrict__ scsh,
                                                            float* __restrict__ gam_dgam, float* __restrict__ dxn,
                                                            double* __restrict__ sums, int B, int T, int HW) {
  __shared__ float s_acc[3 * kWC];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 3 * kWC; i += blockDim.x) s_acc[i] = 0.f;
  __syncthreads();
  const int total = B * T;
  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const int b = tile / T, ti = tile - b * T;
    const long off = static_cast<long>(tile) * kWC * 128 + lane * 4;
    const long xoff = static_cast<long>(b) * x_bstride + static_cast<long>(ti) * kWC * 128 + lane * 4;
    const int p = ti * 128 + lane * 4;
    const bool v0 = p < HW, v1 = p + 1 < HW, v2 = p + 2 < HW, v3 = p + 3 < HW;
    auto valid4 = [&](float4 t) { return make_float4(v0 ? t.x : 0.f, v1 ? t.y : 0.f, v2 ? t.z : 0.f, v3 ? t.w : 0.f); };
#pragma unroll 4
    for (int c = warp; c < kWC; c += 8) {
      const float sc = scsh[c], sh = scsh[kWC + c];
      const float4 d = valid4(__ldcs(reinterpret_cast<const float4*>(dpre + off + c * 128)));
      const float4 xv = valid4(__ldcs(reinterpret_cast<const float4*>(x + xoff + c * 128)));
      const float4 g = valid4(__ldcs(reinterpret_cast<const float4*>(gam_dgam + off + c * 128)));
      const float4 dx = make_float4(d.x * g.x, d.y * g.y, d.z * g.z, d.w * g.w);
      const float4 dg = make_float4(d.x * fmaf(xv.x, sc, sh), d.y * fmaf(xv.y, sc, sh), d.z * fmaf(xv.z, sc, sh),
                                    d.w * fmaf(xv.w, sc, sh));
      __stcs(reinterpret_cast<float4*>(dxn + off + c * 128), dx);
      __stcs(reinterpret_cast<float4*>(gam_dgam + off + c * 128), dg);
      float t0 = (dx.x * xv.x + dx.y * xv.y) + (dx.z * xv.z + dx.w * xv.w);
      float t1 = (dx.x + dx.y) + (dx.z + dx.w);
      float t2 = (dg.x + dg.y) + (dg.z + dg.w);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        t0 += __shfl_xor_sync(0xffffffffu, t0, o);
        t1 += __shfl_xor_sync(0xffffffffu, t1, o);
        t2 += __shfl_xor_sync(0xffffffffu, t2, o);
      }
      if (lane == 0) {
        s_acc[c] += t0;
        s_acc[kWC + c] += t1;
        s_acc[2 * kWC + c] += t2;
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * kWC; i += blockDim.x) atomicAdd(sums + i, static_cast<double>(s_acc[i]));
}

// Adjoint of the bilinear up-sample: dP[b, s, :] = sum over the output pixels whose footprint contains texel s of
// weight * dA1[b, p, :].  Gather form (deterministic, no atomics): one block per texel, one thread per channel;
// the candidate pixels are enumerated from the inverse of the source-index formula and checked with the forward one.
__global__ void __launch_bounds__(128) bilinear_adjoint_kernel(const float* __restrict__ da1 /* [B,HW,128] */,
                                                               float* __restrict__ dp, long dp_stride, int B, int Hg,
                                                               int Wg, int Rh, int Rw) {
  const int s = blockIdx.x;                       // b*Rh*Rw + sy*Rw + sx
  const int b = s / (Rh * Rw), r = s - b * Rh * Rw, sy = r / Rw, sx = r - sy * Rw;
  const float ry = static_cast<float>(Rh) / static_cast<float>(Hg), rx = static_cast<float>(Rw) / static_cast<float>(Wg);
  int ylo = static_cast<int>(floorf((static_cast<float>(sy) - 0.5f) / ry - 0.5f)) - 1;
  int yhi = static_cast<int>(ceilf((static_cast<float>(sy) + 1.5f) / ry - 0.5f)) + 1;
  int xlo = static_cast<int>(floorf((static_cast<float>(sx) - 0.5f) / rx - 0.5f)) - 1;
  int xhi = static_cast<int>(ceilf((static_cast<float>(sx) + 1.5f) / rx - 0.5f)) + 1;
  ylo = ylo < 0 ? 0 : ylo; xlo = xlo < 0 ? 0 : xlo;
  yhi = yhi > Hg - 1 ? Hg - 1 : yhi; xhi = xhi > Wg - 1 ? Wg - 1 : xhi;
  const float* src = da1 + static_cast<long>(b) * Hg * Wg * 128 + threadIdx.x;
  float acc = 0.f;
  // The footprint weights depend on the row / column only: 2 x <= 64 of them are computed once per block (the first version
  // evaluated both source-index formulas per candidate pixel in every one of the 128 channel threads: ~10 K instructions per
  // thread for ~120 useful loads).  Same candidates, same order, same products: bit-identical sums.
  __shared__ float s_wy[64], s_wx[64];
  const int ny = yhi - ylo + 1, nx = xhi - xlo + 1;
  if (ny <= 64 && nx <= 64) {
    if (threadIdx.x < 64) {
      const int k = threadIdx.x;
      float w = 0.f;
      if (k < ny) {
        int y0, y1;
        float ly0, ly1;
        bilin_src(ylo + k, Rh, ry, y0, y1, ly0, ly1);
        w = (y0 == sy ? ly0 : 0.f) + (y1 == sy ? ly1 : 0.f);
      }
      s_wy[k] = w;
    } else {
      const int k = threadIdx.x - 64;
      float w = 0.f;
      if (k < nx) {
        int x0, x1;
        float lx0, lx1;
        bilin_src(xlo + k, Rw, rx, x0, x1, lx0, lx1);
        w = (x0 == sx ? lx0 : 0.f) + (x1 == sx ? lx1 : 0.f);
      }
      s_wx[k] = w;
    }
    __syncthreads();
    for (int ky = 0; ky < ny; ++ky) {
      const float wy = s_wy[ky];
      if (wy == 0.f) continue;
      const float* row = src + (static_cast<long>(ylo + ky) * Wg + xlo) * 128;
      for (int kx = 0; kx < nx; ++kx) {
        const float wx = s_wx[kx];
        if (wx == 0.f) continue;
        acc = fmaf(wy * wx, row[static_cast<long>(kx) * 128], acc);
      }
    }
  } else {
    for (int py = ylo; py <= yhi; ++py) {
      int y0, y1;
      float ly0, ly1;
      bilin_src(py, Rh, ry, y0, y1, ly0, ly1);
      const float wy = (y0 == sy ? ly0 : 0.f) + (y1 == sy ? ly1 : 0.f);
      if (wy == 0.f) continue;
      for (int px = xlo; px <= xhi; ++px) {
        int x0, x1;
        float lx0, lx1;
        bilin_src(px, Rw, rx, x0, x1, lx0, lx1);
        const float wx = (x0 == sx ? lx0 : 0.f) + (x1 == sx ? lx1 : 0.f);
        if (wx == 0.f) continue;
        acc = fmaf(wy * wx, src[(static_cast<long>(py) * Wg + px) * 128], acc);
      }
    }
  }
  dp[static_cast<long>(s) * dp_stride + threadIdx.x] = acc;
}

}  // namespace hg

extern "C" {

int hg_wgrad_blocked(const float* dout, const float* x, long x_bstride, int Cx, const float* mod, float* dw, float* dbias,
                     void* workspace, int B, int C, int Hg, int Wg, int passes, void* stream);
int hg_act_wgrad_blocked(const float* dout, const float* pscale, const float* x, long x_bstride, int Cx, const float* mod,
                         int act, float* dw, float* dbias, void* workspace, int B, int C, int Hg, int Wg, int passes,
                         void* stream);

size_t hg_spade_bwd_wgrad_workspace_bytes(void) {
  return static_cast<size_t>(hg::num_sms()) * (hg::kWC * hg::kWC + hg::kWC) * sizeof(float);
}

int hg_spade_bwd_wgrad(const float* dout, const float* x, long x_bstride, const float* mod, float* dw, float* dbias,
                       void* workspace, int B, int C, int Hg, int Wg, int passes, void* stream) {
  return hg_wgrad_blocked(dout, x, x_bstride, C, mod, dw, dbias, workspace, B, C, Hg, Wg, passes, stream);
}

int hg_wgrad_blocked(const float* dout, const float* x, long x_bstride, int Cx, const float* mod, float* dw, float* dbias,
                     void* workspace, int B, int C, int Hg, int Wg, int passes, void* stream) {
  return hg_act_wgrad_blocked(dout, nullptr, x, x_bstride, Cx, mod, 0, dw, dbias, workspace, B, C, Hg, Wg, passes, stream);
}

int hg_act_wgrad_blocked(const float* dout, const float* pscale, const float* x, long x_bstride, int Cx, const float* mod,
                         int act, float* dw, float* dbias, void* workspace, int B, int C, int Hg, int Wg, int passes,
                         void* stream) {
  HG_REQUIRE(act >= 0 && act <= 2, "hg_act_wgrad_blocked: act must be 0 (LeakyReLU 0.2), 1 (sine) or 2 (identity)");
  HG_REQUIRE(C == hg::kWC, "hg_wgrad_blocked: only %d gradient channels are supported (got %d)", hg::kWC, C);
  HG_REQUIRE(Cx == 128 || Cx == 256, "hg_wgrad_blocked: the second operand must have 128 or 256 channels (got %d)", Cx);
  HG_REQUIRE(dout && x && dw && workspace, "hg_wgrad_blocked: null pointer");
  HG_REQUIRE(passes == 1 || passes == 3, "hg_wgrad_blocked: passes must be 1 or 3");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_wgrad_blocked: bad shape");
  HG_REQUIRE(((reinterpret_cast<uintptr_t>(dout) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(workspace)) & 15) == 0,
             "hg_wgrad_blocked: tensors must be 16-byte aligned");
  const int T = (Hg * Wg + 127) / 128;
  const int tiles = B * T;
  const int grid = tiles < hg::num_sms() ? tiles : hg::num_sms();
  float* part_w = static_cast<float*>(workspace);
  float* part_b = part_w + static_cast<size_t>(hg::num_sms()) * hg::kWC * hg::kWC;
  hg::WgradArgs a{dout, x, x_bstride, mod, part_w, part_b, B, Hg * Wg, Cx, act, pscale};
  auto st = static_cast<cudaStream_t>(stream);
  cudaError_t e;
#define HG_WG_LAUNCH(P, A)                                                                                              \
  do {                                                                                                                  \
    e = cudaFuncSetAttribute(hg::spade_wgrad_kernel<P, A>, cudaFuncAttributeMaxDynamicSharedMemorySize, hg::kWgSmemBytes); \
    if (e == cudaSuccess) hg::spade_wgrad_kernel<P, A><<<grid, hg::kWgThreads, hg::kWgSmemBytes, st>>>(a);              \
  } while (0)
  if (passes == 3) {
    if (act == 0) HG_WG_LAUNCH(3, 0); else if (act == 1) HG_WG_LAUNCH(3, 1); else HG_WG_LAUNCH(3, 2);
  } else {
    if (act == 0) HG_WG_LAUNCH(1, 0); else if (act == 1) HG_WG_LAUNCH(1, 1); else HG_WG_LAUNCH(1, 2);
  }
#undef HG_WG_LAUNCH
  if (e != cudaSuccess) { hg::set_error("hg_spade_bwd_wgrad: smem opt-in failed: %s", cudaGetErrorString(e)); return 2; }
  int rc = hg::check_launch("hg_spade_bwd_wgrad");
  if (rc) return rc;
  hg::wgrad_reduce_kernel<<<(hg::kWC * Cx + 255) / 256, 256, 0, st>>>(part_w, part_b, grid, hg::kWC * Cx, dw, dbias);
  return hg::check_launch("hg_spade_bwd_wgrad(reduce)");
}

int hg_spade_bwd_combine(const float* dpre, const float* x, long x_bstride, const float* g1, const float* ak,
                         const float* dskip, const float* drgb, const float* rgb_w, float* dx, double* dwrgb, int B, int C,
                         int Hg, int Wg, void* stream) {
  HG_REQUIRE(C == hg::kWC, "hg_spade_bwd_combine: only %d channels are supported (got %d)", hg::kWC, C);
  HG_REQUIRE(dx, "hg_spade_bwd_combine: null output");
  HG_REQUIRE(!dpre || g1, "hg_spade_bwd_combine: dpre needs its g1 table");
  HG_REQUIRE(!(ak || drgb) || x, "hg_spade_bwd_combine: x is needed for the statistics / ToRGB terms");
  HG_REQUIRE(!drgb || rgb_w, "hg_spade_bwd_combine: drgb needs rgb_w");
  HG_REQUIRE(!drgb || ((Hg * Wg) % 4 == 0 && (reinterpret_cast<uintptr_t>(drgb) & 15) == 0),
             "hg_spade_bwd_combine: drgb must be 16-byte aligned with H*W a multiple of 4");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_spade_bwd_combine: bad shape");
  const int T = (Hg * Wg + 127) / 128;
  const int tiles = B * T;
  int grid = hg::num_sms() * 4;
  if (grid > tiles) grid = tiles;
  hg::CombineArgs a{dpre, x, x_bstride, g1, ak, dskip, drgb, rgb_w, dx, dwrgb, B, Hg * Wg};
  hg::spade_combine_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  return hg::check_launch("hg_spade_bwd_combine");
}

int hg_synth_input_bwd(const float* dx, const float* w, const float* bias, const float* ic, const float* jc, int B, int C,
                       int Hg, int Wg, float* dw, float* db, void* stream) {
  HG_REQUIRE(C == hg::kWC, "hg_synth_input_bwd: only %d channels are supported (got %d)", hg::kWC, C);
  HG_REQUIRE(dx && w && bias && ic && jc && dw && db, "hg_synth_input_bwd: null pointer");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0, "hg_synth_input_bwd: bad shape");
  hg::synth_input_bwd_kernel<<<C, 256, 0, static_cast<cudaStream_t>(stream)>>>(dx, w, bias, ic, jc, B, Hg, Wg, dw, db);
  return hg::check_launch("hg_synth_input_bwd");
}

int hg_spade_a1(const float* p_lr, long p_stride, const float* p_bias, float* a1, int B, int Hg, int Wg, int Rh, int Rw,
                void* stream) {
  HG_REQUIRE(p_lr && a1, "hg_spade_a1: null pointer");
  HG_REQUIRE((reinterpret_cast<uintptr_t>(p_lr) & 15) == 0 && p_stride >= 128 && (p_stride & 3) == 0,
             "hg_spade_a1: p_lr must be 16-byte aligned with a row stride >= 128 that is a multiple of 4");
  HG_REQUIRE(!p_bias || (reinterpret_cast<uintptr_t>(p_bias) & 15) == 0, "hg_spade_a1: p_bias must be 16-byte aligned");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0 && Rh > 0 && Rw > 0, "hg_spade_a1: bad shape");
  const int tiles = B * ((Hg * Wg + 127) / 128);
  hg::a1_gather_kernel<<<tiles, 128, 0, static_cast<cudaStream_t>(stream)>>>(p_lr, p_stride, p_bias, a1, B, Hg, Wg, Rh, Rw);
  return hg::check_launch("hg_spade_a1");
}

int hg_spade_pixel_pre(const float* x, long x_bstride, const float* scsh, const float* gam, float* bet_pre, int B, int C,
                       int Hg, int Wg, void* stream) {
  HG_REQUIRE(C == hg::kWC, "hg_spade_pixel_pre: only %d channels are supported (got %d)", hg::kWC, C);
  HG_REQUIRE(x && scsh && gam && bet_pre, "hg_spade_pixel_pre: null pointer");
  const int T = (Hg * Wg + 127) / 128;
  hg::pixel_pre_kernel<<<hg::num_sms() * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, x_bstride, scsh, gam, bet_pre, B, T);
  return hg::check_launch("hg_spade_pixel_pre");
}

int hg_spade_pixel_mod_bwd(const float* dpre, const float* x, long x_bstride, const float* scsh, float* gam_dgam, float* dxn,
                           double* sums, int B, int C, int Hg, int Wg, void* stream) {
  HG_REQUIRE(C == hg::kWC, "hg_spade_pixel_mod_bwd: only %d channels are supported (got %d)", hg::kWC, C);
  HG_REQUIRE(dpre && x && scsh && gam_dgam && dxn && sums, "hg_spade_pixel_mod_bwd: null pointer");
  const int T = (Hg * Wg + 127) / 128;
  int grid = hg::num_sms() * 4;
  if (grid > B * T) grid = B * T;
  hg::pixel_mod_bwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(dpre, x, x_bstride, scsh, gam_dgam, dxn, sums, B, T,
                                                                               Hg * Wg);
  return hg::check_launch("hg_spade_pixel_mod_bwd");
}

int hg_bilinear_adjoint(const float* da1, float* dp, long dp_stride, int B, int Hg, int Wg, int Rh, int Rw, void* stream) {
  HG_REQUIRE(da1 && dp && dp_stride >= 128, "hg_bilinear_adjoint: bad arguments");
  HG_REQUIRE(B > 0 && Hg > 0 && Wg > 0 && Rh > 0 && Rw > 0, "hg_bilinear_adjoint: bad shape");
  hg::bilinear_adjoint_kernel<<<B * Rh * Rw, 128, 0, static_cast<cudaStream_t>(stream)>>>(da1, dp, dp_stride, B, Hg, Wg, Rh, Rw);
  return hg::check_launch("hg_bilinear_adjoint");
}

}  // extern "C"
