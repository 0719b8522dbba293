/* hg3d.h -- C ABI of lib3dhg_sm100a.so: the B200-native (sm_100a) kernels behind the 3DHumanGAN
 * generator / discriminator hot path.
 *
 * Boundary contract (SURVEY.md section 8b; the reference's own native boundary is the pybind11
 * plugin loader lib/components/custom_ops.py:46-110 with bias_act.cpp:32, upfirdn2d.cpp:16):
 *   - plain C: raw DEVICE pointers, sizes, enums; no C++ or torch types cross the boundary;
 *   - ownership: the caller allocates every input, output and workspace tensor and keeps it alive;
 *     the library never allocates device memory and never synchronises the device;
 *   - stream: every launch takes the CUDA stream explicitly (`void* stream` = cudaStream_t);
 *     the default stream is never touched implicitly;
 *   - errors: return 0 on success, non-zero otherwise; `hg_last_error()` returns a thread-local
 *     message (the Python shim raises RuntimeError, mirroring TORCH_CHECK in bias_act.cpp:34-51);
 *   - threading: re-entrant; call from the rank's Python thread and from autograd's backward thread;
 *   - all floating-point tensors are fp32 and densely packed unless a stride argument says otherwise.
 *
 * "passes" selects the tensor-core precision mode of every GEMM-shaped kernel:
 *     3 = bf16x3 split (A_hi.B_hi + A_lo.B_hi + A_hi.B_lo, fp32 accumulate): meets the 1e-3-of-fp32 contract
 *     1 = plain bf16 operands (the analogue of the reference's autocast training mode)
 */
#ifndef HG3D_H_
#define HG3D_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library state -------------------------------------------------------------------------- */
const char* hg_last_error(void);
int hg_abi_version(void);
int hg_check_device(void); /* 0 iff the current device is an sm_100 part */

/* ---- packed tensor-core weights --------------------------------------------------------------
 * W [N,K] fp32 (row stride ldw) * scale (* *scale_dev when non-null, a DEVICE scalar such as the
 * 1/sigma of spectral normalisation, map3d_layers.py:205-206) -> bf16 hi/lo operand image:
 * [N/Nb blocks][ceil(K/64) chunks][hi, lo][Nb x 64, K-major, 128B-swizzled].  Nb multiple of 16, <= 256. */
size_t hg_packed_weight_bytes(int N, int K, int Nb);
int hg_pack_weight(const float* W, int N, int K, int ldw, const float* scale_dev, float scale, int Nb,
                   void* out_img, size_t out_bytes, void* stream);

/* Y[M,N] = X[M,K] . W^T + bias   (K <= 256).  Used for mlp_shared at render resolution
 * (SPADE2d.forward, map3d_layers.py:178) and as the primitive self-test. */
int hg_linear(const float* X, int ldx, int M, int K, const void* Wimg, int Nb, int N, const float* bias, float* Y,
              int ldy, int passes, void* stream);

/* ---- renderer -------------------------------------------------------------------------------- */
/* vertex_ik[b,v,:] = sum_j lbs[b,v,j] * inverse(fk[b,j])      replaces smpl.py:217-218.
 * fk [B,24,4,4], lbs [B,V,24] -> vertex_ik [B,V,16] (16-byte aligned). */
int hg_vertex_ik(const float* fk, const float* lbs, int B, int V, float* vertex_ik, void* stream);

/* Exact-KNN acceleration structure: Morton-sorted vertices (x,y,z,index) + one box per cluster of 32.
 * vertices [B,V,3] (V <= 8192) -> sorted [B,Vp] float4, boxes [B,Vp/32,2] float4, Vp = hg_knn_padded(V). */
int hg_knn_padded(int V);
int hg_knn_prep(const float* vertices, int B, int V, void* sorted, void* boxes, void* stream);

/* Ray sampling + jitter + camera transform + K=1 nearest posed vertex + 31-d geometry feature.
 * Replaces vr.get_initial_rays_weak_perspective (volume_rendering.py:86-110), vr.perturb_points /
 * transform_sampled_points (:124-170) and get_geo_features (smpl.py:210-249, incl. pytorch3d knn_points).
 *   xs [Rw], ys [Rh], zs [S]: the three torch.linspace tables of the ray grid;
 *   focals, scales [B]; cam2world [B,4,4]; jitter [B,Rw*Rh*S] uniform draws or NULL;
 *   points_in [B,n_points,3] or NULL: when given, the ray stage is skipped (staged / test use);
 *   skeletons [B,24,3], vertices [B,V,3], tpose [B,V,3], vertex_ik [B,V,16];
 *   knn_sorted / knn_boxes: outputs of hg_knn_prep, or both NULL for the brute-force scan (same result);
 *   rec [B,n_points,36] out: xyz*input_scaler (3), features (31, order per legacy_mode), 2 zeros;
 *   z_vals [B,n_points], points [B,n_points,3], nearest [B,n_points] (int32), nearest_d2: optional outs.
 * Nearest index is bit-exact w.r.t. d2 = (dx*dx + dy*dy) + dz*dz in fp32, lowest index on ties. */
int hg_geo_features(const float* xs, const float* ys, const float* zs, const float* focals, const float* scales,
                    const float* cam2world, const float* jitter, const float* points_in, const float* skeletons,
                    const float* vertices, const float* tpose, const float* vertex_ik, const void* knn_sorted,
                    const void* knn_boxes, int B, int Rw, int Rh, int S, int V, int n_points, float input_scaler,
                    int legacy_mode, float* rec, float* z_vals, float* points, int* nearest, float* nearest_d2,
                    void* stream);

/* Fused FiLM-SIREN MLP + volume integration.  Replaces COORDCONCATSIREN.forward (modulated.py:41-75)
 * and vr.ray_integration (volume_rendering.py:12-56).
 *   rec [B,R*S,36]; z_vals [B,R*S]; noise [B,R*S] N(0,1) draws or NULL;
 *   film [B,7,2,256]: per layer (F, P) with layer output sin(F*acc + P) (host folds bias, x30, 15*freq+30);
 *   wblob: hg_render_weight_blob_bytes() bytes, the 7 packed matrices in kernel schedule order;
 *   w_sigma [256], w_rgb [3,256], b_feat [256], heads_b [4] = {b_sigma, b_rgb[3]};
 *   ray_out [B,R,260] out: 256 composited features, 3 composited rgb (before *2-1), depth;
 *   weights_out [B,R*S] optional; raw_out [B,R*S,260] optional: per-point (rgb, feat, sigma) INSTEAD of compositing.
 *   S: samples per ray, power of two in [2,128]; hidden must be 256. */
size_t hg_render_weight_blob_bytes(void);
int hg_render_mlp(const float* rec, const float* z_vals, const float* noise, const float* film, const void* wblob,
                  const float* w_sigma, const float* w_rgb, const float* b_feat, const float* heads_b, float* ray_out,
                  float* weights_out, float* raw_out, int B, int R, int S, int hidden, float noise_std, int white_back,
                  int last_back, int clamp_softplus, int passes, void* stream);

/* ---- synthesis backbone ---------------------------------------------------------------------- */
/* Synthesis activations use a tile-blocked planar layout [B, T, C, 128] with T = ceil(Hg*Wg/128): element
 * (b, c, pixel p) lives at ((b*T + p/128)*C + c)*128 + p%128, so the 128 KB a CTA touches per tile are contiguous.
 *
 * x0[T,C,128] = sin(w[:,0]*ic[i] + w[:,1]*jc[j] + b) (SynthesisInput, map3d_layers.py:260-275); when stats
 * is non-null adds batch * (sum, sumsq) per channel to stats[0:C], stats[C:2C] (double). */
int hg_synth_input(const float* w, const float* bias, const float* ic, const float* jc, int C, int Hg, int Wg,
                   float* x0, double* stats, int batch, void* stream);

/* BatchNorm statistics -> scale/shift (+ running-stat update, + fused per-sample SPADE modulation).
 * nn.SyncBatchNorm semantics (map3d_layers.py:162).  stats [2,C] double (already all-reduced across ranks),
 * count from `count_dev` (device double) when non-null else `count`.  training=0 uses the running stats.
 * gb [B,2,C] = (1+gamma, beta) per sample -> mod [B,2,C] = (sc*G, sh*G+beta); scsh [2,C] = (sc, sh). */
int hg_bn_finalize(const double* stats, double count, const double* count_dev, const float* weight, const float* bias,
                   float* running_mean, float* running_var, int training, float eps, float momentum, const float* gb,
                   int B, int C, float* scsh, float* mod, void* stream);

/* One SPADE half-block: out = Conv1x1_SN(lrelu(BN(x)*(1+gamma)+beta)) + bias [+ skip], optional ToRGB
 * accumulation and the (sum, sumsq) statistics of `out` for the next BatchNorm.
 * Replaces SPADE2d.forward + SPADEBlock.forward + ToRGB.forward (map3d_layers.py:176-190, 218-238, 346-352)
 * and, in pixel-style mode, the F.interpolate of map3d_generator.py:244-245.
 *   x [B or 1,T,C,128] with batch stride x_bstride (T*C*128, or 0 = shared by the batch);  exactly one of
 *   mod  [B,2,C]                      const-style (per-sample gamma/beta), or
 *   p_lr [B,Rh*Rw,p_stride] (+ p_bias [B,128], scsh [2,C], wgb packed [512x128], bgb [512])  pixel-style;
 *   wimg packed [C x C] conv weight; bias [C]; skip [B,T,C,128] or NULL; out [B,T,C,128];
 *   stats [2,C] double or NULL; rgb_w [3,C], rgb_b [3], rgb_in [B,3,HW] or NULL, rgb_out [B,3,HW] (all NULL = no ToRGB).
 *   C must be 256. */
int hg_spade_conv(const float* x, long x_bstride, const float* mod, const float* scsh, const float* p_lr,
                  long p_stride, const float* p_bias, const void* wgb, const float* bgb, const void* wimg,
                  const float* bias, const float* skip, float* out, double* stats, const float* rgb_w,
                  const float* rgb_b, const float* rgb_in, float* rgb_out, int B, int C, int Hg, int Wg, int Rh, int Rw,
                  int passes, void* stream);

/* ---- backward of a const-style SPADE half-block (autograd through map3d_layers.py:176-190, 218-238) ----
 * Forward, folded:  pre = x*g1[b,c] + g0[b,c],  y = lrelu_0.2(pre),  out = W y + bias (+ skip);  mod = [B,2,C] (g1,g0).
 *
 * hg_spade_bwd_dgrad: dpre = (W^T dout) * lrelu'(pre) and sums[b,0,c] += sum_p dpre, sums[b,1,c] += sum_p dpre*x
 *   (fp64, caller zeroes).  dout, dpre [B,T,C,128]; x [B or 1,T,C,128] with batch stride x_bstride;
 *   wimg_t = hg_pack_weight of W^T (rows = ci, K = co).
 * hg_spade_bwd_wgrad: dw[co,ci] = sum_{b,p} dout[b,co,p] * y[b,ci,p] (y recomputed from x, mod) and
 *   dbias[co] = sum dout (NULL = skip).  workspace: hg_spade_bwd_wgrad_workspace_bytes() bytes of device memory.
 * hg_spade_bwd_combine: dx = dpre*g1[b,c] + a[c] + k[c]*x (+ dskip) (+ rgb_w^T drgb), the gradient w.r.t. the
 *   half-block input; ak = [2,C] (a, k) carries the terms that reach x through the batch statistics.  dwrgb [3,C]
 *   (fp64, accumulated; NULL = skip) += sum_{b,p} drgb[b,j,p]*x[b,c,p].  Any of dpre/ak/dskip/drgb may be NULL. */
int hg_spade_bwd_dgrad(const float* dout, const float* x, long x_bstride, const float* mod, const void* wimg_t,
                       float* dpre, double* sums, int B, int C, int Hg, int Wg, int passes, void* stream);
size_t hg_spade_bwd_wgrad_workspace_bytes(void);
int hg_spade_bwd_wgrad(const float* dout, const float* x, long x_bstride, const float* mod, float* dw, float* dbias,
                       void* workspace, int B, int C, int Hg, int Wg, int passes, void* stream);
/* ---- generic pieces of the backward schedule over tile-blocked activations [B,T,C,128] (csrc/synth.cu, synth_bwd.cu) ----
 * hg_conv1x1_blocked:      out[B,T,256,128] = W[256 x Cin] x + bias, Cin in {64,128,256} (wimg = hg_pack_weight of W).
 * hg_conv1x1_blocked_bwd:  out = (Wt [g; g2]) * mask(aux*g1+g0), mask = 1 where positive else `slope` (0.2 LeakyReLU,
 *                          0 ReLU); g, g2 (NULL = absent) [B,T,256,128]; aux, out, sums carry Cout in {128,256} channels;
 *                          mod [B,2,Cout] or NULL (g1 = 1, g0 = 0); sums [B,2,Cout] fp64 += (sum out, sum out*aux);
 *                          pixel_major: out is [B,HW,Cout] instead (Cout == 128 only).
 * hg_wgrad_blocked:        dw[256, Cx] = sum_{b,p} dout[b,:,p] (x) lrelu(x*g1+g0)[b,:,p], x with Cx in {128,256} channels
 *                          (mod [B,2,256] with rows past Cx unused, or NULL: g1 = 1, g0 = 0), dbias[256] = sum dout;
 *                          padding rows of both operands are ignored; workspace as hg_spade_bwd_wgrad.
 * hg_spade_a1:             A1[B,T,128,128] = relu(bilinear_up(p_lr) + p_bias), the hidden layer of the gamma/beta MLP.
 * hg_spade_pixel_pre:      bet_pre <- (x*sc + sh)*gam + bet_pre                (scsh = [2,C]).
 * hg_spade_pixel_mod_bwd:  dxn = dpre*gam, gam_dgam <- dpre*(x*sc+sh); sums[3,C] fp64 += (sum dxn*x, sum dxn, sum dgam)
 *                          over the valid pixels.
 * hg_bilinear_adjoint:     dp[b*Rh*Rw + s, 0:128] = adjoint of the align_corners=False bilinear up-sample applied to
 *                          da1 [B,HW,128] (pixel-major); dp rows have stride dp_stride floats.
 * Padding rows (pixels past HW in the last tile of a sample) may hold anything, NaN included: every kernel here ignores them
 * in its inputs, except hg_spade_pixel_pre, which computes them like valid rows.  The engine (conv1x1 forward / backward)
 * leaves them unwritten in its tile-blocked outputs; hg_spade_a1, hg_spade_pixel_mod_bwd and hg_spade_bwd_combine write
 * zeros there. */
int hg_conv1x1_blocked(const float* x, int Cin, const void* wimg, const float* bias, float* out, int B, int Hg, int Wg,
                       int passes, void* stream);
/* act (0 LeakyReLU/ReLU, 1 sine/cosine) selects the mask; ascale [B,256] scales g per (sample, channel) before the product
 * (K = 256 only); rk_* adds  sum_j rk_w[j][c]*rk_v[b][j][pixel]  (rk_w [3,256], rk_v [B,rk_n,HW], rk_n in 1..3) to the
 * product before the mask -- the sigma / rgb heads of the renderer (modulated.py:62-73) feed back that way. */
int hg_conv1x1_blocked_bwd(const float* g, const float* g2, const float* aux, const float* mod, const void* wimg_t,
                           float* out, double* sums, int Cout, float slope, int pixel_major, int act, const float* ascale,
                           const float* rk_w, const float* rk_v, int rk_n, int B, int Hg, int Wg, int passes,
                           void* stream);
/* out[B,T,256,128] = W [act(x*g1+g0); act(x2*g1+g0)] + bias with act = LeakyReLU 0.2 (0) or sine (1); mod [B,2,256];
 * x2 NULL = K 256.  One FiLM-SIREN layer of COORDCONCATSIREN (modulated.py:41-75) over tile-blocked points. */
int hg_act_conv1x1_blocked(const float* x, const float* x2, const float* mod, int act, const void* wimg, const float* bias,
                           float* out, int B, int Hg, int Wg, int passes, void* stream);
/* The same engine with every option exposed: K = 256 or 512 input channels from one or two tile-blocked sources, a
 * modulation table per source (mod / mod2 [B,2,256]; null = identity), act 0 = LeakyReLU(slope), 0 <= slope <= 1 / 1 = sine, residual add,
 * next-layer BatchNorm statistics, ToRGB accumulation -- one output half (256 channels) of a layer whose width was
 * zero-padded to 512: hidden_dim 384 (configs/map3d.py:61) and 420 (:254, the released checkpoint) run on it. */
int hg_blocked_conv_wide(const float* x, const float* x2, const float* mod, const float* mod2, int act, float slope,
                         const void* wimg, const float* bias, const float* skip, float* out, double* stats,
                         const float* rgb_w, const float* rgb_b, const float* rgb_in, float* rgb_out, int B, int Hg, int Wg,
                         int passes, void* stream);
/* hg_wgrad_blocked with y = act(x*g1+g0), act 0 LeakyReLU 0.2 / 1 sine / 2 identity, and dout scaled per (sample, row) by
 * pscale [B,256] (NULL = 1). */
int hg_act_wgrad_blocked(const float* dout, const float* pscale, const float* x, long x_bstride, int Cx, const float* mod,
                         int act, float* dw, float* dbias, void* workspace, int B, int C, int Hg, int Wg, int passes,
                         void* stream);
/* ---- renderer, training mode (csrc/render_train.cu): heads and volume integration over tile-blocked points ----
 * hg_render_heads:      sig[B,N] = w_sigma . sin(f*out3+phi) + b0; rgbp[B,3,N] = W_rgb . sin(f*linc+phi) + b1..3
 *                       (mod3 [B,2,256] = f, phi of the last FiLM slice; modulated.py:62-73).
 * hg_render_heads_bwd:  acc[4*256+4] fp64 += (d w_sigma, d W_rgb[0..2], d b[0..3]).
 * hg_render_composite(_bwd): vr.ray_integration (volume_rendering.py:12-56) and its gradient; ray_out / dray [B,R,260] =
 *                       feat(256) | rgb(3) | depth; last_back in the forward only; S in {8,16,32,64,128}. */
int hg_render_heads(const float* out3, const float* linc, const float* mod3, const float* w_sigma, const float* w_rgb,
                    const float* heads_b, float* sig, float* rgbp, int B, int N, void* stream);
int hg_render_heads_bwd(const float* out3, const float* linc, const float* mod3, const float* dsig, const float* drgbp,
                        double* acc, int B, int N, void* stream);
int hg_render_composite(const float* sig, const float* z, const float* noise, const float* rgbp, const float* feat,
                        float* ray_out, float* weights, int B, int R, int S, float noise_std, int white_back,
                        int clamp_softplus, int last_back /* forward only: eval_last_back of the sample app */, void* stream);
int hg_render_composite_bwd(const float* sig, const float* z, const float* noise, const float* rgbp, const float* feat,
                            const float* dray, float* dfeat, float* drgbp, float* dsig, int B, int R, int S,
                            float noise_std, int white_back, int clamp_softplus, void* stream);
int hg_wgrad_blocked(const float* dout, const float* x, long x_bstride, int Cx, const float* mod, float* dw, float* dbias,
                     void* workspace, int B, int C, int Hg, int Wg, int passes, void* stream);
int hg_spade_a1(const float* p_lr, long p_stride, const float* p_bias, float* a1, int B, int Hg, int Wg, int Rh, int Rw,
                void* stream);
int hg_spade_pixel_pre(const float* x, long x_bstride, const float* scsh, const float* gam, float* bet_pre, int B, int C,
                       int Hg, int Wg, void* stream);
int hg_spade_pixel_mod_bwd(const float* dpre, const float* x, long x_bstride, const float* scsh, float* gam_dgam, float* dxn,
                           double* sums, int B, int C, int Hg, int Wg, void* stream);
int hg_bilinear_adjoint(const float* da1, float* dp, long dp_stride, int B, int Hg, int Wg, int Rh, int Rw, void* stream);

/* Weight gradient of a stride-1 "same" convolution over NCHW planes (autograd through nn.Conv2d,
 * unet_discriminators.py:21-38), `ntaps` filter taps per launch:
 *   dw[t, r, c] = sum_{b,h,w} dy[b, co0+r, h, w] * x[b, ci0+c, h+oy[t], w+ox[t]]   (zero outside the image)
 * for r < nco <= 256, c < nci <= 256; dw is [ntaps, 256, ceil32(nci)] (unused rows / columns zero), dbias [256] = sum dy
 * (NULL = skip).  ntaps * (nco > 128 ? 2 : 1) * ceil32(nci) <= 512 (TMEM columns); oy / ox are HOST arrays of shifts in
 * -1..1; larger filters / channel counts are chunked by the caller (abi.conv2d_wgrad).
 * workspace: hg_conv2d_wgrad_workspace_bytes() bytes of device memory. */
size_t hg_conv2d_wgrad_workspace_bytes(void);
int hg_conv2d_wgrad_taps(const float* dy, const float* x, float* dw, float* dbias, void* workspace, int B, int H, int W,
                         int Cout, int Cin, int co0, int nco, int ci0, int nci, int ntaps, const int* oy, const int* ox,
                         int passes, void* stream);
/* The same gradient for a WHOLE layer in one launch: every (256-row chunk of dy, 256-row chunk of x, group of taps) is a
 * blockIdx.y of one grid, the partials are reduced straight into dW [Cout,Cin,k,k] and dbias [Cout] (NULL = skip).  k = 1 or 3.
 * workspace: hg_conv2d_wgrad_layer_workspace_bytes(B,H,W,Cout,Cin,k) bytes (its size is passed for the check). */
size_t hg_conv2d_wgrad_layer_workspace_bytes(int B, int H, int W, int Cout, int Cin, int ksize);
int hg_conv2d_wgrad_layer(const float* dy, const float* x, float* dW, float* dbias, void* workspace, size_t workspace_bytes, int B,
                          int H, int W, int Cout, int Cin, int ksize, int passes, void* stream);
/* 3x3 weight gradient on image rows of >= 128 pixels (W % 128 == 0): the input is converted once per image row into the
 * forward kernel's pixel-major operand image and read as an MN-major B operand, a tap being a row offset of the descriptor.
 * dw [ntaps,128,64] for output channels co0..co0+nco (<= 128) x input channels ci0..ci0+nci (<= 64), ntaps <= 8 taps with
 * shifts (tdy[t], tdx[t]) in {-1,0,1} (host arrays); dbias [128] or NULL.  Same autograd contract as above. */
size_t hg_conv3x3_wgrad_halo_workspace_bytes(void);
int hg_conv3x3_wgrad_halo(const float* dy, const float* x, float* dw, float* dbias, void* workspace, int B, int H, int W,
                          int Cout, int Cin, int co0, int nco, int ci0, int nci, int ntaps, const int* tdy, const int* tdx,
                          int passes, void* stream);
/* Backward of hg_synth_input: dx [B,T,C,128] (gradient w.r.t. the batch-shared x0, per sample) -> dw [C,2], db [C]. */
int hg_synth_input_bwd(const float* dx, const float* w, const float* bias, const float* ic, const float* jc, int B, int C,
                       int Hg, int Wg, float* dw, float* db, void* stream);
int hg_spade_bwd_combine(const float* dpre, const float* x, long x_bstride, const float* g1, const float* ak,
                         const float* dskip, const float* drgb, const float* rgb_w, float* dx, double* dwrgb, int B,
                         int C, int Hg, int Wg, void* stream);


/* ---- discriminator --------------------------------------------------------------------------- */
/* 3x3 (pad 1) / 1x1 convolution over NCHW fp32 planes as an implicit GEMM; replaces the conv2d calls of
 * ResBlock / UNetDiscriminator (unet_discriminators.py:7-72, 114-160) with the surrounding ops folded in:
 *   x1 [B,C1,Hs,Ws] (+ x2 [B,C2,Hs,Ws]: channel concat, :147); up2: nearest x2 up-sample in front (Hs=H/2);
 *   pre_lrelu: LeakyReLU(0.2) in front; wimg: hg_pack_weight of W permuted to [Cout, tap, Cin] (K = taps*Cin,
 *   or 64 when taps*Cin <= 64); bias [Cout] or NULL; residual [B,Cout,H,W] (or [B,Cout,H/2,W/2] with res_up2)
 *   added in the epilogue; out [B,Cout,H,W].  C1, C2 multiples of 64 (or taps*Cin <= 64); Cout <= 2*Nb. */
int hg_conv2d(const float* x1, int C1, const float* x2, int C2, int B, int H, int W, int up2, int pre_lrelu, int ksize,
              const void* wimg, int Cout, int Nb, const float* bias, const float* residual, int res_up2, float* out,
              int passes, void* stream);
/* out[planes,H,W] = P_a(a) + P_b(b); P = AvgPool2d(2) of a [planes,2H,2W] source when the flag is set (:42-44,52-54). */
int hg_pool_add(const float* a, int pool_a, const float* b, int pool_b, float* out, long planes, int H, int W,
                void* stream);
/* out[B,O] = x[B,K] . w[O,K]^T + bias: the full-extent `latent_layer` convolution (:117-118,135). */
int hg_dense(const float* x, const float* w, const float* bias, float* out, int B, int K, int O, void* stream);

/* Spectral normalisation of a list of weights in one launch: torch.nn.utils.spectral_norm's forward pre-hook as applied at
 * lib/components/map3d_layers.py:205-206 (18 synthesis convolutions) and lib/discriminators/unet_discriminators.py:18
 * (30 discriminator convolutions).  table: `count` entries of hg_spectral_entry_bytes() = 32 bytes
 * { const float* w [N,K]; float* u [N]; float* v [K]; int32 N; int32 K }.  training != 0: v <- normalize(W^T u),
 * u <- normalize(W v) written back in place; inv_sigma[i] = 1 / (u . W v).  max_n / max_k bound the table's shapes. */
int hg_spectral_entry_bytes(void);
int hg_spectral_norm(const void* table, int count, int max_n, int max_k, float* inv_sigma, int training, float eps,
                     void* stream);

/* ---- SMPL skinning in front of the path (SURVEY.md 8f-4) ------------------------------------------------------------------
 * `lbs` of lib/components/smpl.py:11-107 (smplx.lbs: blend shapes, joint regression, Rodrigues, kinematic chain, skinning) and
 * the re-skinning of SHHQDataset._preprocess_smpl_fix_body (lib/data/datasets.py:146-155).
 * hg_smpl_shape: v_shaped [B,V,3] = v_template + shapedirs [V,3,NB] . betas [B,NB]; jpart [B, hg_smpl_shape_blocks(V), J, 3].
 * hg_smpl_pose : pose [B,J,3] axis-angle (pose_is_rotmat 0) or [B,J,9]; joints [B,J,3], rot [B,J,9], feat [B,(J-1)*9] = R - I,
 *                A [B,J,16] = rest-pose-relative rigid transforms (the generator's fk_matrices), joints_posed [B,J,3].
 * hg_smpl_skin : verts = (sum_j w[v,j] A_j) [v_in + posedirs^T feat; 1]; feat / posedirs NULL = no pose blend shapes;
 *                v_bstride / w_bstride 0 = shared by the batch. */
int hg_smpl_shape_blocks(int V);
int hg_smpl_shape(const float* v_template, const float* shapedirs, const float* betas, const float* j_regressor, float* v_shaped,
                  float* jpart, int B, int V, int NB, int J, void* stream);
int hg_smpl_pose(const float* jpart, int nblk, const float* pose, int pose_is_rotmat, const int* parents, float* joints, float* rot,
                 float* feat, float* A, float* joints_posed, int B, int J, void* stream);
int hg_smpl_skin(const float* v_in, long v_bstride, const float* feat, const float* posedirs, int P, const float* lbs_weights,
                 long w_bstride, const float* A, float* verts, int B, int V, int J, void* stream);

/* ---- the preprocessor's mesh rasteriser (SURVEY.md 8f-2) --------------------------------------------------------------------
 * Replaces pytorch3d's MeshRasterizer (faces_per_pixel 1, blur_radius 0, no culling, perspective-correct) as called by
 * SHHQPreprocessor._forward_rasterize (lib/data/preprocessor.py:138-152) and the label / semantic look-ups after it (:154-174).
 * verts [B,V,3]; faces [F,3] int32 in [0,V) (NOT checked here), shared by the batch; R [B,3,3], T [B,3]: view = X @ R + T;
 * focal: in-NDC focal length (the reference passes -1/tan(0.5 deg)).  keys [B,H,W] uint64 workspace (cleared here).
 * Outputs, each optional (NULL = not written): pix_to_face [B,H,W] int64 packed b*F + face, -1 background; zbuf [B,H,W] and
 * bary [B,H,W,3] (perspective-correct), -1 background; segments [B,H,W] int64 = faces_to_labels[face] + 2, background 1;
 * semantics [B,3,H,W] = sem_verts[V,3] at the face vertex of the largest barycentric (first maximum), background 0.
 * The arithmetic is oracle/raster_port.py's, bit for bit; deterministic (lowest face on equal depth). */
int hg_mesh_raster(const float* verts, const int* faces, const float* R, const float* T, float focal, int B, int V, int F, int H,
                   int W, unsigned long long* keys, const long* faces_to_labels, const float* sem_verts, long* pix_to_face,
                   float* zbuf, float* bary, long* segments, float* semantics, void* stream);

/* ---- loss + optimiser tail of a training iteration (SURVEY.md 8f-1) ---------------------------------------------------
 * Class-balanced segmentation cross entropy, PhaseTrainer._calculate_segmentation_loss mode 'cross_entropy_balanced'
 * (lib/trainers/phase_trainer.py:203-256): histogram of the int64 labels -> per-class coefficients (numel / (occ * n_occ) *
 * prior / mean(prior); background and absent classes 0; all ones when no foreground label occurs) -> one pass over the
 * logits [B,L,HW] that writes loss[0] = mean_px coef[gt] * CE and, optionally, d loss / d logits.  L <= 32. */
int hg_label_histogram(const long* labels, long n, int L, int* hist, void* stream);
int hg_seg_ce_coef(const int* hist, const float* prior /* [L] or NULL */, int L, double numel, float* coef, void* stream);
int hg_seg_ce(const float* logits, const long* labels, const float* coef, float* dlogits /* or NULL */, float* loss,
              double* workspace /* >= 2 * #SMs doubles */, int B, int L, long HW, void* stream);
/* Multi-tensor global-norm clipping (torch.nn.utils.clip_grad_norm_, phase_trainer.py:314,336), torch.optim.Adam's update
 * with per-group scalars (phase_trainer.py:57-76) and the generator's EMA (lib/components/ema.py:29-48) over a device table
 * of tensors: entries { float* p, g, exp_avg, exp_avg_sq, ema; long n } (hg_mt_entry_bytes() = 48; g NULL = no gradient this
 * step, ema NULL = no shadow), chunks { int tensor; int group; long offset } (hg_mt_chunk_bytes() = 16, hg_mt_chunk_elems()
 * elements each).  norm_clip[0] = global norm, [1] = min(1, max_norm / (norm + 1e-6)).  scalars (HOST): 7 arrays of ngroups
 * floats: lr, beta1, beta2, eps, weight_decay, 1 - beta1^t, sqrt(1 - beta2^t). */
int hg_mt_entry_bytes(void);
int hg_mt_chunk_bytes(void);
int hg_mt_chunk_elems(void);
int hg_mt_grad_norm(const void* table, const void* chunks, int nchunks, float max_norm, double* partials, float* norm_clip,
                    void* stream);
int hg_mt_adam(const void* table, const void* chunks, int nchunks, const float* norm_clip /* or NULL */, const float* scalars,
               int ngroups, float ema_one_minus_decay, int write_clipped_grad, void* stream);

/* ---- StyleGAN3 native ops named by the reference ---------------------------------------------- */
/* y = clamp(act(x + b[(i / stepB) % sizeB]) * gain)   replaces bias_act.cpp:32 / bias_act.cu:24 (forward).
 * act: 1 linear 2 relu 3 lrelu 4 tanh 5 sigmoid 6 elu 7 selu 8 softplus 9 swish; clamp < 0 disables. */
int hg_bias_act(const float* x, const float* b, float* y, long n, int stepB, int sizeB, int act, float alpha,
                float gain, float clamp, void* stream);

/* Derivatives of bias_act   replaces the grad=1 / grad=2 modes of bias_act.cpp:32 (bias_act.cu:46-150).
 * out = g * gain * act'(xref + b)            (order 1; g = incoming gradient)
 * out = g * gain * act''(xref + b) * dy      (order 2; g = gradient of the first-order result, dy = its upstream)
 * both zeroed where the forward output was clamped.  yref (forward output) is needed by every activation
 * except linear and swish; swish needs xref (forward input, bias NOT added) and b.  Null = absent. */
int hg_bias_act_grad(const float* g, const float* b, const float* xref, const float* yref, const float* dy, float* out,
                     long n, int stepB, int sizeB, int order, int act, float alpha, float gain, float clamp,
                     void* stream);

/* 2x2 average pooling (up = 0: y[planes,H/2,W/2] = scale * sum of the 2x2 block) or nearest 2x up-sampling (up = 1:
 * y[planes,2H,2W] = scale * x) -- F.avg_pool2d(x, 2) is scale 0.25, nn.Upsample(scale_factor=2) scale 1
 * (unet_discriminators.py:30,60-70); each is the other's adjoint up to the scale. */
int hg_resample2x(const float* x, float* y, long planes, int inH, int inW, int up, float scale, void* stream);

/* Zero-insert up-sample, pad/crop, 2-D FIR, decimate   replaces upfirdn2d.cpp:16 / upfirdn2d.cu:29-375.
 * x [NC,inH,inW] -> y [NC,outH,outW]; f [fH,fW]; the filter is flipped unless flip_filter (conv2d is a correlation). */
int hg_upfirdn2d(const float* x, const float* f, float* y, int NC, int inH, int inW, int outH, int outW, int fH,
                 int fW, int upx, int upy, int downx, int downy, int padx0, int pady0, int flip_filter, float gain,
                 void* stream);
/* Both 1-D passes of a SEPARABLE 2x resampler in one kernel (intermediate in shared memory): the reference's only call
 * shapes, upsample2d / downsample2d with the 12-tap sym6 filter (augment.py:314,325; two passes at upfirdn2d.py:243-244).
 * f [taps] with taps in {4,6,8,12,16}; up != 0: up = 2, down = 1; up == 0: up = 1, down = 2 (both axes).  gain is the
 * total gain (sqrt per axis).  out size = (in * up + pad0 + pad1 - taps) / down + 1 (computed by the caller). */
int hg_upfirdn2d_sep2(const float* x, const float* f, float* y, long planes, int inH, int inW, int outH, int outW, int taps,
                      int up, int padx0, int pady0, int flip_filter, float gain, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HG3D_H_ */
