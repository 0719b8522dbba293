// Z-buffer rasteriser of the preprocessor's segmentation targets (SURVEY.md 8f-2).  Reference:
// `SHHQPreprocessor._forward_rasterize` (lib/data/preprocessor.py:138-176), which rasterises the posed SMPL mesh with pytorch3d
// 0.6.2's MeshRasterizer (faces_per_pixel = 1, blur_radius = 0, no culling, perspective-correct barycentrics) and turns the
// result into the label map `rasterized_segments` and the T-pose coordinate map `rasterized_semantics`.
//
// The arithmetic is the contract restated in oracle/raster_port.py, one IEEE fp32 operation per step (__fmul_rn / __fadd_rn /
// __fsub_rn / __fdiv_rn: nothing that decides coverage or depth may be contracted into an FMA), so pix_to_face, zbuf and the
// barycentrics are bit-identical to the oracle's.  Three steps on one stream, no host synchronisation:
//   clear    key buffer [B,H,W] (uint64) = all ones
//   splat    one thread per (image, face): project the three vertices, reject (zmax < 0, zero area), walk the pixels of the
//            face's bounding box (conservative by 1 pixel; the exact closed-box test is part of the per-pixel test) and
//            atomicMin key = (bits(pz) << 32) | face.  pz >= 0 after the pz < 0 rejection (-0.0 canonicalised to +0.0), so the
//            float bits order like the values; min is order-independent (deterministic) and the lowest face wins equal pz.
//            Faces with more than kSmallBox box pixels (most SMPL faces at 512 x 256 and up: a median box of 55 pixels at
//            512 x 256, 100 at 512 x 512) are walked by the whole warp, one after the other.
//   resolve  one thread per pixel: recompute the winner's barycentrics with the same device function, write the outputs.
// Face indices are validated against V by the caller (raster.py, once per face tensor): the kernels do not bounds-check.
#include "common.cuh"

namespace hg {

constexpr float kRasterEps = 1e-8f;     // pytorch3d's kEpsilon
constexpr int kSmallBox = 16;           // box pixels a thread walks alone (sub-pixel and clipped faces)
constexpr unsigned long long kNoFace = ~0ull;

struct RasterTri {
  float x[3], y[3], z[3];
};

struct RasterView {
  int H, W;
  float rx, ox, sx;     // PixToNonSquareNdc parameters of the columns (r, o, S1 = W)
  float ry, oy, sy;     // ... and of the rows (S1 = H)
};

__device__ __forceinline__ float edge_fn(float px, float py, float ax, float ay, float bx, float by) {
  return __fsub_rn(__fmul_rn(__fsub_rn(px, ax), __fsub_rn(by, ay)), __fmul_rn(__fsub_rn(py, ay), __fsub_rn(bx, ax)));
}

// -o + (r * i + o) / S1
__device__ __forceinline__ float pix_to_ndc(int i, float r, float o, float S1) {
  return __fadd_rn(-o, __fdiv_rn(__fadd_rn(__fmul_rn(r, static_cast<float>(i)), o), S1));
}

// view = X @ R + T (row vectors), NDC = (f * view.xy) / view.z, z = view.z
__device__ __forceinline__ void load_face(const float* __restrict__ verts, const int* __restrict__ faces, int f,
                                          const float* __restrict__ R, const float* __restrict__ T, float focal, RasterTri& t) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float* v = verts + 3l * faces[3l * f + k];
    const float X = v[0], Y = v[1], Z = v[2];
    float c[3];
#pragma unroll
    for (int j = 0; j < 3; ++j)
      c[j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(X, R[j]), __fmul_rn(Y, R[3 + j])), __fmul_rn(Z, R[6 + j])), T[j]);
    t.x[k] = __fdiv_rn(__fmul_rn(focal, c[0]), c[2]);
    t.y[k] = __fdiv_rn(__fmul_rn(focal, c[1]), c[2]);
    t.z[k] = c[2];
  }
}

__device__ __forceinline__ bool face_rejected(const RasterTri& t) {
  const float zmax = fmaxf(fmaxf(t.z[0], t.z[1]), t.z[2]);
  const float area = edge_fn(t.x[0], t.y[0], t.x[1], t.y[1], t.x[2], t.y[2]);
  return zmax < 0.f || fabsf(area) <= kRasterEps;
}

// The per-pixel test of the contract: closed box, barycentrics, perspective correction, pz >= 0, strictly inside.
__device__ __forceinline__ bool pixel_test(const RasterTri& t, float px, float py, float& w0, float& w1, float& w2, float& pz) {
  const float xmin = fminf(fminf(t.x[0], t.x[1]), t.x[2]), xmax = fmaxf(fmaxf(t.x[0], t.x[1]), t.x[2]);
  const float ymin = fminf(fminf(t.y[0], t.y[1]), t.y[2]), ymax = fmaxf(fmaxf(t.y[0], t.y[1]), t.y[2]);
  const bool inbox = !(px > xmax || px < xmin || py > ymax || py < ymin);
  const float area = __fadd_rn(edge_fn(t.x[2], t.y[2], t.x[0], t.y[0], t.x[1], t.y[1]), kRasterEps);
  const float b0 = __fdiv_rn(edge_fn(px, py, t.x[1], t.y[1], t.x[2], t.y[2]), area);
  const float b1 = __fdiv_rn(edge_fn(px, py, t.x[2], t.y[2], t.x[0], t.y[0]), area);
  const float b2 = __fdiv_rn(edge_fn(px, py, t.x[0], t.y[0], t.x[1], t.y[1]), area);
  const float t0 = __fmul_rn(__fmul_rn(b0, t.z[1]), t.z[2]);
  const float t1 = __fmul_rn(__fmul_rn(t.z[0], b1), t.z[2]);
  const float t2 = __fmul_rn(__fmul_rn(t.z[0], t.z[1]), b2);
  const float d = fmaxf(__fadd_rn(__fadd_rn(t0, t1), t2), kRasterEps);
  w0 = __fdiv_rn(t0, d);
  w1 = __fdiv_rn(t1, d);
  w2 = __fdiv_rn(t2, d);
  pz = __fadd_rn(__fadd_rn(__fmul_rn(w0, t.z[0]), __fmul_rn(w1, t.z[1])), __fmul_rn(w2, t.z[2]));
  return inbox && !(pz < 0.f) && w0 > 0.f && w1 > 0.f && w2 > 0.f;
}

// Conservative index range [i0, i1] of PixToNonSquareNdc(i) over [lo, hi] (i = S1 - 1 - pixel): the fp32 inversion below is
// off by far less than a pixel, so one pixel of margin on each side is enough.  Non-finite: the whole axis.
__device__ __forceinline__ void index_range(float lo, float hi, float r, float o, int S1, int& i0, int& i1) {
  if (!isfinite(lo) || !isfinite(hi)) {
    i0 = 0;
    i1 = S1 - 1;
    return;
  }
  const float a = fminf(fmaxf(((lo + o) * S1 - o) / r, -4.f), S1 + 4.f);
  const float b = fminf(fmaxf(((hi + o) * S1 - o) / r, -4.f), S1 + 4.f);
  i0 = max(static_cast<int>(floorf(a)) - 1, 0);
  i1 = min(static_cast<int>(ceilf(b)) + 1, S1 - 1);
}

__device__ __forceinline__ void splat_pixel(const RasterTri& t, int f, int xi, int yi, const RasterView& vw,
                                            unsigned long long* __restrict__ keys) {
  const float px = pix_to_ndc(vw.W - 1 - xi, vw.rx, vw.ox, vw.sx);
  const float py = pix_to_ndc(vw.H - 1 - yi, vw.ry, vw.oy, vw.sy);
  float w0, w1, w2, pz;
  if (!pixel_test(t, px, py, w0, w1, w2, pz)) return;
  if (pz == 0.f) pz = 0.f;        // -0.0 -> +0.0
  const unsigned long long key = (static_cast<unsigned long long>(__float_as_uint(pz)) << 32) | static_cast<unsigned>(f);
  atomicMin(keys + static_cast<long>(yi) * vw.W + xi, key);
}

__global__ void __launch_bounds__(256) raster_splat_kernel(const float* __restrict__ verts, const int* __restrict__ faces,
                                                           const float* __restrict__ R, const float* __restrict__ T, float focal,
                                                           int B, int V, int F, RasterView vw, unsigned long long* __restrict__ keys) {
  const long gid = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool live = gid < static_cast<long>(B) * F;
  const int b = live ? static_cast<int>(gid / F) : 0, f = live ? static_cast<int>(gid % F) : 0;
  RasterTri t;
  int x0 = 0, x1 = -1, y0 = 0, y1 = -1;       // pixel column / row ranges (inclusive)
  if (live) {
    load_face(verts + static_cast<long>(b) * V * 3, faces, f, R + b * 9, T + b * 3, focal, t);
    if (!face_rejected(t)) {
      int i0, i1;
      index_range(fminf(fminf(t.x[0], t.x[1]), t.x[2]), fmaxf(fmaxf(t.x[0], t.x[1]), t.x[2]), vw.rx, vw.ox, vw.W, i0, i1);
      x0 = vw.W - 1 - i1;
      x1 = vw.W - 1 - i0;
      index_range(fminf(fminf(t.y[0], t.y[1]), t.y[2]), fmaxf(fmaxf(t.y[0], t.y[1]), t.y[2]), vw.ry, vw.oy, vw.H, i0, i1);
      y0 = vw.H - 1 - i1;
      y1 = vw.H - 1 - i0;
    }
  }
  const int nx = max(x1 - x0 + 1, 0), n = nx * max(y1 - y0 + 1, 0);
  unsigned long long* img = keys + static_cast<long>(b) * vw.H * vw.W;
  const bool big = n > kSmallBox;
  if (!big)
    for (int p = 0; p < n; ++p) splat_pixel(t, f, x0 + p % nx, y0 + p / nx, vw, img);
  unsigned mask = __ballot_sync(0xffffffffu, big);
  while (mask) {                  // large faces: the warp walks each box together
    const int src = __ffs(mask) - 1;
    mask &= mask - 1;
    RasterTri s;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      s.x[k] = __shfl_sync(0xffffffffu, t.x[k], src);
      s.y[k] = __shfl_sync(0xffffffffu, t.y[k], src);
      s.z[k] = __shfl_sync(0xffffffffu, t.z[k], src);
    }
    const int sf = __shfl_sync(0xffffffffu, f, src), sb = __shfl_sync(0xffffffffu, b, src);
    const int sx0 = __shfl_sync(0xffffffffu, x0, src), sy0 = __shfl_sync(0xffffffffu, y0, src);
    const int snx = __shfl_sync(0xffffffffu, nx, src), sn = __shfl_sync(0xffffffffu, n, src);
    unsigned long long* simg = keys + static_cast<long>(sb) * vw.H * vw.W;
    for (int p = lane; p < sn; p += 32) splat_pixel(s, sf, sx0 + p % snx, sy0 + p / snx, vw, simg);
  }
}

__global__ void __launch_bounds__(256) raster_resolve_kernel(const float* __restrict__ verts, const int* __restrict__ faces,
                                                             const float* __restrict__ R, const float* __restrict__ T, float focal,
                                                             int B, int V, int F, RasterView vw,
                                                             const unsigned long long* __restrict__ keys,
                                                             const long* __restrict__ labels, const float* __restrict__ sem_verts,
                                                             long* __restrict__ pix_to_face, float* __restrict__ zbuf,
                                                             float* __restrict__ bary, long* __restrict__ segments,
                                                             float* __restrict__ semantics) {
  const long HW = static_cast<long>(vw.H) * vw.W;
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  const int b = static_cast<int>(i / HW);
  const long hw = i - b * HW;
  const unsigned long long key = keys[i];
  if (key == kNoFace) {
    if (pix_to_face) pix_to_face[i] = -1;
    if (zbuf) zbuf[i] = -1.f;
    if (bary) bary[3 * i] = bary[3 * i + 1] = bary[3 * i + 2] = -1.f;
    if (segments) segments[i] = 1;
    if (semantics)
      for (int c = 0; c < 3; ++c) semantics[(static_cast<long>(b) * 3 + c) * HW + hw] = 0.f;
    return;
  }
  const int f = static_cast<int>(key & 0xffffffffull);
  const int yi = static_cast<int>(hw / vw.W), xi = static_cast<int>(hw - static_cast<long>(yi) * vw.W);
  RasterTri t;
  load_face(verts + static_cast<long>(b) * V * 3, faces, f, R + b * 9, T + b * 3, focal, t);
  float w0, w1, w2, pz;
  pixel_test(t, pix_to_ndc(vw.W - 1 - xi, vw.rx, vw.ox, vw.sx), pix_to_ndc(vw.H - 1 - yi, vw.ry, vw.oy, vw.sy), w0, w1, w2, pz);
  if (pix_to_face) pix_to_face[i] = static_cast<long>(b) * F + f;        // packed, as pytorch3d returns it
  if (zbuf) zbuf[i] = pz;
  if (bary) {
    bary[3 * i] = w0;
    bary[3 * i + 1] = w1;
    bary[3 * i + 2] = w2;
  }
  if (segments) segments[i] = labels[f] + 2;
  if (semantics) {
    const int k = w1 > w0 ? (w2 > w1 ? 2 : 1) : (w2 > w0 ? 2 : 0);      // torch.argmax: the first maximum
    const float* s = sem_verts + 3l * faces[3l * f + k];
    for (int c = 0; c < 3; ++c) semantics[(static_cast<long>(b) * 3 + c) * HW + hw] = s[c];
  }
}

// PixToNonSquareNdc's range and offset in fp32: r = 2, or (S1 * 2) / S2 when S1 > S2; o = r / 2
static void ndc_params(int S1, int S2, float& r, float& o) {
  float range = 2.0f;
  if (S1 > S2) range = (static_cast<float>(S1) * range) / static_cast<float>(S2);
  r = range;
  o = range / 2.0f;
}

}  // namespace hg

extern "C" {

// See include/hg3d.h.
int hg_mesh_raster(const float* verts, const int* faces, const float* R, const float* T, float focal, int B, int V, int F, int H,
                   int W, unsigned long long* keys, const long* faces_to_labels, const float* sem_verts, long* pix_to_face,
                   float* zbuf, float* bary, long* segments, float* semantics, void* stream) {
  HG_REQUIRE(verts && faces && R && T && keys, "hg_mesh_raster: null pointer");
  HG_REQUIRE(B > 0 && V > 0 && F > 0 && H > 0 && W > 0, "hg_mesh_raster: bad sizes");
  // one splat thread per (image, face) and one resolve thread per pixel: both grids must fit gridDim.x (2^31 - 1 blocks of 256)
  HG_REQUIRE(static_cast<long>(B) * F < (1l << 31) && static_cast<long>(H) * W < (1l << 28) &&
                 static_cast<long>(B) * H * W < (1l << 38),
             "hg_mesh_raster: too large (B * F < 2^31, H * W < 2^28, B * H * W < 2^38)");
  HG_REQUIRE(!segments || faces_to_labels, "hg_mesh_raster: segments need faces_to_labels");
  HG_REQUIRE(!semantics || sem_verts, "hg_mesh_raster: semantics need sem_verts");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  hg::RasterView vw;
  vw.H = H;
  vw.W = W;
  hg::ndc_params(W, H, vw.rx, vw.ox);
  hg::ndc_params(H, W, vw.ry, vw.oy);
  vw.sx = static_cast<float>(W);
  vw.sy = static_cast<float>(H);
  const long n = static_cast<long>(B) * H * W;
  if (cudaMemsetAsync(keys, 0xff, n * sizeof(unsigned long long), s) != cudaSuccess) return hg::check_launch("hg_mesh_raster (clear)");
  const long nf = static_cast<long>(B) * F;
  hg::raster_splat_kernel<<<static_cast<unsigned>((nf + 255) / 256), 256, 0, s>>>(verts, faces, R, T, focal, B, V, F, vw, keys);
  int rc = hg::check_launch("hg_mesh_raster (splat)");
  if (rc) return rc;
  hg::raster_resolve_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(verts, faces, R, T, focal, B, V, F, vw, keys,
                                                                                 faces_to_labels, sem_verts, pix_to_face, zbuf,
                                                                                 bary, segments, semantics);
  return hg::check_launch("hg_mesh_raster (resolve)");
}

}  // extern "C"
