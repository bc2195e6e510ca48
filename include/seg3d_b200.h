/* seg3d_b200.h - C ABI of the B200-native volumetric-segmentation hot path.
 *
 * Drop-in boundary for qinliuliuqin/Medical-Segmentation3d-Toolkit (reference paths below are
 * relative to that repository).  The reference has no FFI of its own: its hot path is a chain
 * of torch.nn layer calls made from Python.  Each entry point here replaces one such call
 * site; the Python host package `segmentation3d` (same import paths, same signatures as the
 * reference) binds this library with ctypes and is the only caller.
 *
 * Conventions
 *  - Plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in
 *    `_host`.  Nothing is allocated, retained or freed by the library: the caller owns all
 *    buffers and workspaces.  Calls are asynchronous on `stream` (a cudaStream_t passed as
 *    void*), thread-compatible, and hold no global mutable state.
 *  - Return value: 0 on success, negative seg3d_status otherwise; seg3d_last_error() gives the
 *    message for the calling thread.  The Python binding raises RuntimeError on non-zero.
 *  - Activations are channels-last "NDHWC": element (n,z,y,x,c) of a tensor with channel pitch
 *    `ld` (elements, ld >= C) lives at base[(((n*D+z)*H+y)*W+x)*ld + c].  A pitch larger than C
 *    lets two producers write the two halves of a concat buffer (vnet_upblock.py:21) in place.
 *  - `dtype` selects the STORAGE type of activations (and, for the tensor-core path, the MMA
 *    operand type).  Accumulation, GroupNorm statistics, softmax and all reductions are fp32
 *    (fp64 for the per-sample sums).
 *  - GroupNorm(1,C) is split in two: the producing convolution adds per-sample sum(y), sum(y*y)
 *    of its fp32 results to `stats[n][2]` (doubles, zeroed by the caller), and the consumer
 *    (seg3d_gn_apply / the out-block tail) turns them into mean / rstd.
 */
#ifndef SEG3D_B200_H
#define SEG3D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum { SEG3D_OK = 0, SEG3D_EINVAL = -1, SEG3D_ECUDA = -2, SEG3D_EUNSUPPORTED = -3 } seg3d_status;
typedef enum { SEG3D_F32 = 0, SEG3D_F16 = 1, SEG3D_BF16 = 2 } seg3d_dtype;
/* OR-ed into `dtype` of seg3d_conv3d_fwd: operands stay f16/bf16 but the raw result y is stored as fp32
 * (pitch y_ld in fp32 elements; y_ld < Cout keeps only the first y_ld channels - used to drop zero-padded output
 * channels).  k3 on the tensor cores: the z-march kernel (Cin in {16,32,64}, W % 8 == 0, weights <= 112 KB), else the
 * generic kernel, which stores all Cout channels (needs y_ld >= Cout, y_ld % 4 == 0). */
#define SEG3D_OUT_F32 0x100
typedef enum {
  SEG3D_CONV_K3 = 0,   /* k=3 s=1 p=1   nn.Conv3d          conv_gn_relu3.py:10, vnet_inblock.py:9, vnet_outblock.py:13 */
  SEG3D_CONV_K2S2 = 1, /* k=2 s=2 p=0   nn.Conv3d          vnet_downblock.py:11 */
  SEG3D_CONV_T2S2 = 2, /* k=2 s=2       nn.ConvTranspose3d vnet_upblock.py:11   */
  SEG3D_CONV_K1 = 3    /* k=1           nn.Conv3d          vnet_outblock.py:16  */
} seg3d_conv_mode;
typedef enum { SEG3D_IMPL_AUTO = 0, SEG3D_IMPL_SIMT = 1, SEG3D_IMPL_TCGEN05 = 2 } seg3d_impl;
typedef enum { SEG3D_NORM_NONE = 0, SEG3D_NORM_FIXED = 1, SEG3D_NORM_ADAPTIVE = 2 } seg3d_norm;

/* ---- library ---------------------------------------------------------------------------- */
int seg3d_version(void);
const char* seg3d_last_error(void);
/* 0 if `device` is an sm_100 part this library can run on. */
int seg3d_device_check(int device);

/* ---- convolutions (replace nn.Conv3d / nn.ConvTranspose3d forward) ------------------------
 * x: [N,D,H,W,Cin] pitch x_ld.  y: raw conv result + bias, pitch y_ld:
 *   K3, K1 : [N,D,H,W,Cout]      K2S2 : [N,D/2,H/2,W/2,Cout]      T2S2 : [N,2D,2H,2W,Cout]
 * w (packed by the host from the reference's OIDHW / IODHW fp32 weights):
 *   SIMT path    (fp32)    : [taps][Cin][Cout]  (T2S2: [Cin][8*Cout], column = tap*Cout+co)
 *   TCGEN05 path (dtype)   : [taps][Cout][Cin]  (T2S2: [8*Cout][Cin])
 *   tap = (kd*k + kh)*k + kw.
 * bias: fp32 [Cout] (may be NULL).  stats: double [N][2] accumulated (may be NULL).
 * Supported shapes: SIMT any Cin with Cin==1 or Cin%8==0; TCGEN05 needs Cin%16==0, Cout%16==0,
 * Cout<=256, dtype f16/bf16.  AUTO picks TCGEN05 when it applies and dtype != f32.
 * Input block (K3, Cin == 1, Cout == 16, x_ld == 1): w is the fp32 SIMT layout [27][16] for both paths; AUTO with
 * f16/bf16 storage and W % 8 == 0 runs the im2col-in-shared-memory tensor-core kernel (csrc/conv_tc_cin1.cu), which
 * keeps the weights fp32-accurate through a hi/lo operand split. */
int seg3d_conv3d_fwd(int mode, int dtype, int impl,
                     const void* x, int x_ld, int Cin,
                     const void* w, const float* bias,
                     void* y, int y_ld, int Cout,
                     int N, int D, int H, int W,
                     double* stats, void* stream);

/* Input block on the tensor cores as a banded-Toeplitz GEMM fed by TMA (vnet_inblock.py:9-15; csrc/conv_tc_cin1t.cu).
 * xpad: the single-channel input in a row-padded layout [N][D][H][W + SEG3D_CIN1_PAD] (dtype f16/bf16, W % 8 == 0): x index i
 * of a row sits at column i + SEG3D_CIN1_LEFT, every other column is zero (seg3d_patch_gather_rows writes this layout).
 * w: fp32 [27][16] (tap-major, as the SIMT layout), rounded to `dtype` inside the kernel like every other tensor-core layer's
 * weights (environment SEG3D_CIN1_LO=1: split into two `dtype` terms, fp32-accurate, twice the MMAs); y: [N,D,H,W,16] pitch y_ld.
 * epi_mode 0: y = conv + bias, stats[n] += {sum, sum of squares};  1: the sums only, y is not touched;
 * 2: y = relu(GroupNorm(conv + bias)) with `stats` holding the FINISHED sums (written by a mode-1 call), gamma / beta
 * the GroupNorm affine.  1 then 2 is the inference schedule: the raw tensor and the GroupNorm-apply pass never reach HBM. */
#define SEG3D_CIN1_PAD 16
#define SEG3D_CIN1_LEFT 9
int seg3d_conv3d_cin1_fwd(int dtype, int epi_mode, const void* xpad, int x_pitch, const float* w, const float* bias,
                          void* y, int y_ld, int N, int D, int H, int W, double* stats,
                          const float* gamma, const float* beta, float eps, void* stream);

/* weight gradient of the input block with the operands of seg3d_conv3d_cin1_fwd: dw (fp32 [27][16], tap-major, accumulated -
 * the caller zeroes it) += sum over voxels of x[v + tap] * dy[v][co].  dy: [N,D,H,W,16] f16/bf16, DENSE (dy_ld must be 16). */
int seg3d_conv3d_cin1_wgrad(int dtype, const void* xpad, int x_pitch, const void* dy, int dy_ld, float* dw,
                            int N, int D, int H, int W, void* stream);

/* data gradient of the input block, written as the NCDHW fp32 input gradient: dx[n][0][z][y][x] (dense [N,1,D,H,W]) =
 * sum over taps (a,b,c) and co < 16 of w[(a*3+b)*3+c][co] * gy[n][z+1-a][y+1-b][x+1-c][co], zero outside the volume,
 * accumulated in fp32.  gy: [N,D,H,W,16] in `dtype` (f32/f16/bf16) with pitch ld (>= 16, ld * sizeof % 16 == 0);
 * w: fp32 [27][16] (tap-major, the layout seg3d_conv3d_cin1_fwd reads).  gy and w 16-byte aligned. */
int seg3d_conv3d_cin1_dgrad(int dtype, const void* gy, int ld, const float* w, float* dx,
                            int N, int D, int H, int W, void* stream);

/* k3 s1 p1 convolution with a narrow output (Cout = classes <= 7; vnet_outblock.py:13) on the tensor cores: the nine
 * in-plane taps are folded into the GEMM N dimension and summed in the epilogue (csrc/conv_tc_narrow.cu).
 * x: [N,D,H,W,Cin] f16/bf16, Cin in {16,32,64}, W % 8 == 0.  w (dtype): [3 kd][NP][Cin] with row (kh*3+kw)*Cout + co,
 * zero rows up to NP = seg3d_conv3d_k3_narrow_np(Cout) (9*Cout rounded up to 16).  y: fp32 [N,D,H,W,Cout] dense
 * (raw conv result + bias).  stats as in seg3d_conv3d_fwd. */
int seg3d_conv3d_k3_narrow_np(int Cout);
int seg3d_conv3d_k3_narrow_fwd(int dtype, const void* x, int x_ld, int Cin, const void* w, const float* bias,
                               float* y, int Cout, int N, int D, int H, int W, double* stats, void* stream);
/* the same convolution applied to x = relu(GroupNorm(raw) + res): the network's last GroupNorm + residual + ReLU
 * (residual_block3.py:24 of up_32.rblock, whose only consumer is vnet_outblock.py:13) is formed in shared memory between
 * the TMA loads and the MMAs, bit-identical to seg3d_gn_apply followed by seg3d_conv3d_k3_narrow_fwd.
 * raw, res: [N,D,H,W,32] f16/bf16 (Cin must be 32); gn_stats: finished {sum, sum of squares} of raw per sample. */
int seg3d_conv3d_k3_narrow_gn_fwd(int dtype, const void* raw, int raw_ld, const void* res, int res_ld, int Cin,
                                  const double* gn_stats, const float* gamma, const float* beta, float eps,
                                  const void* w, const float* bias, float* y, int Cout, int N, int D, int H, int W,
                                  double* stats, void* stream);

/* GroupNorm-apply folded into the CONSUMERS of the last up-block (vnet_upblock.py:19-22 -> residual_block3.py:21-26 ->
 * vnet_outblock.py:13).  The transposed convolution writes its RAW result into the lower half of the concat buffer; then
 *  - seg3d_conv3d_k3_gnin_fwd: k3 convolution (z-march kernel, Cin == 32) whose first gn_ch input channels become
 *    relu(GroupNorm(1, gn_ch)(x[:, :gn_ch])) in shared memory between the TMA loads and the MMAs (finished sums gn_stats);
 *  - seg3d_conv3d_k3_narrow_gn2_fwd: seg3d_conv3d_k3_narrow_gn_fwd whose residual gets the same treatment for its first
 *    res_gn_ch channels.
 * Both are bit-identical to seg3d_gn_apply(relu = 1) followed by the plain call; the apply pass never touches HBM. */
int seg3d_conv3d_k3_gnin_fwd(int dtype, const void* x, int x_ld, int Cin, int gn_ch, const double* gn_stats,
                             const float* gamma, const float* beta, float eps, const void* w, const float* bias,
                             void* y, int y_ld, int Cout, int N, int D, int H, int W, double* stats, void* stream);
int seg3d_conv3d_k3_narrow_gn2_fwd(int dtype, const void* raw, int raw_ld, const void* res, int res_ld, int Cin,
                                   const double* gn_stats, const float* gamma, const float* beta, float eps,
                                   int res_gn_ch, const double* res_gn_stats, const float* res_gamma, const float* res_beta,
                                   const void* w, const float* bias, float* y, int Cout, int N, int D, int H, int W,
                                   double* stats, void* stream);

/* the narrow-output convolution in the strict-parity mode (split operands, see seg3d_conv3d_split_fwd below): x rows are
 * [hi(32) | lo(32)] f16 halves of the activation (Cin must be 32, the lo half directly behind the hi half, pitch x_ld >= 64),
 * w is [3 kd][NP][whi(32) | wlo(32)] f16 (rows as in seg3d_conv3d_k3_narrow_fwd); accumulates hi*whi + lo*whi + hi*wlo in fp32. */
int seg3d_conv3d_k3_narrow_split_fwd(const void* x, int x_ld, int Cin, const void* w, const float* bias,
                                     float* y, int Cout, int N, int D, int H, int W, double* stats, void* stream);

/* conv -> GroupNorm(1,C) -> ReLU without the raw intermediate, as two launches of the same tensor-core convolution
 * (vnet_downblock.py:19, vnet_upblock.py:19: the stride-2 / transposed convolutions are HBM-bound and cheap to run twice).
 * pass 0: stats[n] += {sum, sum of squares} of conv + bias, nothing is stored;  pass 1: recompute and store
 * y = relu((conv + bias - mean) * rstd * gamma + beta) from the finished statistics.  TCGEN05 shapes only. */
int seg3d_conv3d_gn_relu_fwd(int mode, int dtype, int pass, const void* x, int x_ld, int Cin, const void* w,
                             const float* bias, void* y, int y_ld, int Cout, int N, int D, int H, int W,
                             double* stats, const float* gamma, const float* beta, float eps, void* stream);

/* ---- strict-parity mode on the tensor cores: split operands -------------------------------------------------------------
 * Activations are stored as two f16 halves per voxel row, x = hi + lo (hi at channel c, lo at channel lo_off + c; the
 * plan uses rows [hi(Ctot) | lo(Ctot)], lo_off = Ctot, so concat-in-place still works per half).  Weights are packed
 * [taps][Cout][whi(Cin) | wlo(Cin)] f16 (T2S2: [8*Cout][whi | wlo]).  The convolution accumulates hi*whi + lo*whi + hi*wlo
 * in fp32 (the dropped lo*wlo term is 2^-22 relative) and writes the fp32 result + bias (pitch y_ld floats) and the
 * GroupNorm sums; seg3d_gn_apply_split normalises it (+ReLU, + split residual) back into the split format. */
int seg3d_conv3d_split_fwd(int mode, const void* x, int x_ld, int lo_off, int Cin, const void* w, const float* bias,
                           float* y, int y_ld, int Cout, int N, int D, int H, int W, double* stats, void* stream);
int seg3d_gn_apply_split(const float* y, int y_ld, int C, const double* stats, const float* gamma, const float* beta,
                         float eps, const void* res, int res_ld, int res_lo, void* out, int out_ld, int out_lo,
                         int relu, int N, int64_t nvox, void* stream);

/* ---- GroupNorm(1,C) apply + ReLU + residual (replaces nn.GroupNorm, nn.ReLU, `input + output`,
 * torch.cat: conv_gn_relu3.py:17-19, residual_block3.py:24,46, vnet_upblock.py:20-21) ----------
 * out = [relu]( (y-mean)*rstd*gamma + beta [+ res] ), mean/rstd from stats over C*nvox elements
 * (biased variance, eps inside the sqrt).  C % 8 == 0.  out may alias y. */
int seg3d_gn_apply(int dtype, const void* y, int y_ld, int C,
                   const double* stats, const float* gamma, const float* beta, float eps,
                   const void* res, int res_ld,
                   void* out, int out_ld, int relu,
                   int N, int64_t nvox, void* stream);

/* ---- output-block tail (vnet_outblock.py:20-24 after conv1) --------------------------------
 * y1: raw conv1 output [N,nvox,C] pitch ld (C <= 8).  Pass 1 accumulates the statistics of
 * z = conv2(relu(gn1(y1))) into stats2; pass 2 recomputes z, applies gn2 and the channel softmax
 * and writes fp32 probabilities in the reference's NCDHW order: probs[n][c][vox]. */
int seg3d_outblock_tail_stats(int dtype, const void* y1, int ld, int C,
                              const double* stats1, const float* gamma1, const float* beta1,
                              const float* w2 /*[C][C] out,in*/, const float* bias2, float eps,
                              double* stats2, int N, int64_t nvox, void* stream);
int seg3d_outblock_tail_probs(int dtype, const void* y1, int ld, int C,
                              const double* stats1, const float* gamma1, const float* beta1,
                              const float* w2, const float* bias2,
                              const double* stats2, const float* gamma2, const float* beta2, float eps,
                              float* probs, int N, int64_t nvox, void* stream);
/* The same tail for 1 <= C <= 127 classes on the tensor cores (csrc/tail_wide.cu): the 1x1x1 conv runs as split-operand
 * f16 MMAs (h = hi + lo, w2 = whi + wlo; hi*whi + lo*whi + hi*wlo into an fp32 accumulator).  y1 is the fp32 raw conv1
 * result [N][nvox][ld] (16-byte aligned, ld >= C, ld % 4 == 0; channels >= C are never read).  pass 0 accumulates the
 * GN2 sums into stats2 (caller zeroes); pass 1 reads them and writes probs[n][c][vox] (gamma2, beta2, probs unused in
 * pass 0).  C outside 1..127 (the int8 label mask) or a misaligned y1 / ld: SEG3D_EUNSUPPORTED. */
int seg3d_outblock_tail_wide(int pass, const float* y1, int ld, int C,
                             const double* stats1, const float* gamma1, const float* beta1,
                             const float* w2, const float* bias2, float eps, double* stats2,
                             const float* gamma2, const float* beta2, float* probs, int N, int64_t nvox, void* stream);

/* ---- sliding window (core/seg_infer.py:208-246,313-339; utils/image_tools.py:221-238,435-469) -
 * Volumes are fp32 [Z][Y][X] (the reference's numpy order); voxel coordinates are (x,y,z) int32
 * triples like the reference's start_voxel lists. */
/* per-patch sum / sum-of-squares (double [N][2]) for the adaptive normaliser (normalizer.py:59) */
int seg3d_patch_stats(const float* vol, int Z, int Y, int X, const int32_t* starts, int N,
                      int pz, int py, int px, double* stats, void* stream);
/* crop N patches and normalise: out[n][z][y][x] (Cin == 1) stored as dtype.
 * FIXED: (v-mean)/stddev, optional clip to [clip_lo,clip_hi]; ADAPTIVE: mean/std from `stats`. */
int seg3d_patch_gather(const float* vol, int Z, int Y, int X, const int32_t* starts, int N,
                       int pz, int py, int px, int norm, float mean, float stddev, int clip,
                       float clip_lo, float clip_hi, const double* stats,
                       int dtype, void* out, void* stream);
/* the same crop written with a row pitch: out[((n*pz + z)*py + y)*row_pitch + x_off + x].  Elements of a row outside
 * [x_off, x_off+px) are either left untouched or written as ZERO (2-byte types with row_pitch % 8 == 0 write whole 16-byte
 * words) - the row-padded input layout of seg3d_conv3d_cin1_fwd (row_pitch = px + SEG3D_CIN1_PAD, x_off = SEG3D_CIN1_LEFT)
 * wants zeros there either way. */
int seg3d_patch_gather_rows(const float* vol, int Z, int Y, int X, const int32_t* starts, int N,
                            int pz, int py, int px, int norm, float mean, float stddev, int clip,
                            float clip_lo, float clip_hi, const double* stats,
                            int dtype, void* out, int row_pitch, int x_off, void* stream);
/* acc[c][z0+z][y0+y][x0+x] += probs[n][c][z][y][x]  (add_image_region).  starts_x_mult4 != 0: the caller guarantees every
 * start x is a multiple of 4 (the list lives on the device; the host that built it knows), which lets the kernel add four
 * voxels per red.global.add.v4.f32 when px and X are multiples of 4 too */
int seg3d_blend_accumulate(const float* probs, int N, int C, int pz, int py, int px,
                           const int32_t* starts, float* acc, int Z, int Y, int X, int starts_x_mult4, void* stream);
/* acc[c] *= float(1.0/count) with count = cx[x]*cy[y]*cz[z] (add_image_value, seg_infer.py:325-327),
 * then mask = first argmax over c (seg_infer.py:337), int8.  mask may be NULL. */
int seg3d_blend_finalize_argmax(float* acc, int C, int Z, int Y, int X,
                                const int32_t* cx, const int32_t* cy, const int32_t* cz,
                                int8_t* mask, void* stream);
/* same on the z planes [z0, z1) only: a z slab can be finished (and its mask copied out) as soon as no remaining patch
 * touches it, while later patches are still running */
int seg3d_blend_finalize_argmax_z(float* acc, int C, int Z, int Y, int X, int z0, int z1,
                                  const int32_t* cx, const int32_t* cy, const int32_t* cz,
                                  int8_t* mask, void* stream);

/* ---- resampling either side of the path (utils/image_tools.py:329-377: sitk.Resample with an identity transform) ------
 * src [sz][sy][sx] -> dst [dz][dy][dx], both fp32, same origin and direction: output index i reads the continuous input
 * index i * r (r = spacing_out / spacing_in per axis, double).  linear != 0: trilinear with the upper neighbour clamped;
 * else nearest (floor(c + 0.5)).  Voxels whose continuous index is not in [-0.5, size - 0.5) get default_value. */
int seg3d_resample(const float* src, int sz, int sy, int sx, float* dst, int dz, int dy, int dx,
                   double rz, double ry, double rx, int linear, float default_value, void* stream);

/* crop with resampling (utils/image_tools.py:111-146, the training data loader's call): output index i reads the continuous
 * input index o + i * r per axis (o = (crop origin - volume origin) in input voxels, r = crop spacing / volume spacing,
 * axes of the crop = axes of the volume).  Same ITK semantics; both neighbours of the linear interpolation are clamped to
 * the volume, so -0.5 <= c < 0 returns the edge value.  Not yet run on a GPU (added after round 1's GPU budget was spent). */
int seg3d_crop_resample(const float* src, int sz, int sy, int sx, float* dst, int dz, int dy, int dx,
                        double oz, double oy, double ox, double rz, double ry, double rx,
                        int linear, float default_value, void* stream);

/* ---- connected-component post-processing (utils/image_tools.py:380-432; 26-connectivity, one label per call) ------------
 * out[v] = label for the voxels of `label` that belong to the largest component (min_size == 0; ties: the component whose
 * first voxel comes first in raster order) or to any component with at least min_size voxels (min_size > 0).  out is
 * not cleared (the caller zeroes it once and calls this per label).  parent, size: int32 [Z*Y*X] scratch; best: 8 bytes. */
int seg3d_cc_filter(const int8_t* mask, int Z, int Y, int X, int label, int min_size,
                    int32_t* parent, int32_t* size, unsigned long long* best, int8_t* out, void* stream);

/* ---- losses on probabilities (loss/multi_dice_loss.py, loss/binary_dice_loss.py, loss/focal_loss.py) -
 * probs fp32 [B][C][n], target fp32 [B][n] (class index stored as float, dataloader/dataset.py:208). */
/* terms[b][c] = { sum q*t, sum q*q, sum t*t } with q = p*[p > 1/C], t = [target == c] (double) */
int seg3d_dice_terms(const float* probs, const float* target, int B, int C, int64_t n,
                     double* terms, void* stream);
/* grad[b][c][i] = coef[b][c][0]*t*m + coef[b][c][1]*q   (m = [p > 1/C]); coef computed by the host
 * from the terms (closed form of d loss / d p). */
int seg3d_dice_bwd(const float* probs, const float* target, int B, int C, int64_t n,
                   const float* coef, float* grad, void* stream);
/* focal: partial[0] += sum_i -alpha[t_i] * (1-p_t)^gamma * log(p_t + 1e-10) (double);
 * partial[1] += number of voxels whose label lies outside [0, C) - they contribute nothing and the caller raises (the
 * reference's one-hot gather, loss/focal_loss.py:46-48, raises an index error).  partial holds two doubles. */
int seg3d_focal_fwd(const float* probs, const float* target, int B, int C, int64_t n,
                    const float* alpha, float gamma, double* partial, void* stream);
int seg3d_focal_bwd(const float* probs, const float* target, int B, int C, int64_t n,
                    const float* alpha, float gamma, float scale, float* grad, void* stream);

/* cross entropy with the network output used as logits (loss/cross_entropy_loss.py:5-18 -> nn.CrossEntropyLoss):
 * loss_i = w[t_i] * (logsumexp_c x_c - x_t), nothing for voxels whose label is ignore_index (or outside [0, C)).
 * partial[0] += sum loss_i, partial[1] += sum w[t_i] (double; 'mean' = ratio, 'sum' = partial[0]); loss_map (fp32 [B][n],
 * may be NULL) receives loss_i for reduction 'none'.  weight: fp32 [C] or NULL (all ones). */
int seg3d_ce_fwd(const float* logits, const float* target, int B, int C, int64_t n, const float* weight,
                 int ignore_index, double* partial, float* loss_map, void* stream);
/* grad[b][c][i] = scale * g_i * w[t_i] * (softmax_c(x) - [c == t_i]); g_i = grad_map[b][i] or 1 when grad_map is NULL */
int seg3d_ce_bwd(const float* logits, const float* target, int B, int C, int64_t n, const float* weight,
                 int ignore_index, float scale, const float* grad_map, float* grad, void* stream);

/* ---- training: backward of the conv + GroupNorm + ReLU (+ residual) unit (core/seg_train.py:124, i.e. the
 * autograd of conv_gn_relu3.py:16-20 / residual_block3.py:24) -------------------------------------------------
 * Data gradients of the convolutions reuse seg3d_conv3d_fwd with transformed weights (k3: flipped taps and
 * swapped channels; k2s2 <-> transposed conv).
 * seg3d_gn_bwd, two passes over the same arguments:
 *   g0..g2 : up to three gradient contributions wrt `out` (g1/g2 may be NULL), each with its own pitch;
 *   out    : the unit's saved post-ReLU output (mask = out > 0), or NULL for a unit WITHOUT a residual: the mask is then
 *            recomputed from y as fma(y, rstd*gamma, beta - mean*rstd*gamma) > 0, the expression seg3d_gn_apply evaluated on
 *            the same stored y (beta must be given; `out` is not read, a third of pass 0's traffic);
 *   y      : saved raw conv output;  stats : forward sums.
 *   pass 0 : sums[n] += {sum gamma*dz, sum gamma*dz*xhat} (double), dgamma[c] += sum dz*xhat, dbeta[c] += sum dz.
 *   pass 1 : dy = rstd*(gamma*dz - mean(gamma dz) - xhat*mean(gamma dz xhat)) stored with pitch dy_ld;
 *            dres (optional) = dz (the residual branch's gradient); dbias[c] (optional) += sum dy.
 * C % 8 == 0, 256 % (C/8) == 0. */
int seg3d_gn_bwd(int dtype, int pass, const void* g0, int ld0, const void* g1, int ld1, const void* g2, int ld2,
                 const void* out, int out_ld, const void* y, int y_ld, int C, const double* stats,
                 const float* gamma, const float* beta, float eps, double* sums, float* dgamma, float* dbeta,
                 void* dy, int dy_ld, void* dres, int dres_ld, float* dbias, int N, int64_t nvox, void* stream);
/* dw (fp32, SIMT weight layout of seg3d_conv3d_fwd: [taps][Cin][Cout], T2S2 [Cin][8*Cout]) += x (*) dy; the caller
 * zeroes dw.  D,H,W are the spatial dims of x (the convolution's input). */
int seg3d_conv3d_wgrad(int mode, int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout,
                       float* dw, int N, int D, int H, int W, void* stream);
/* backward of seg3d_outblock_tail_*: pass 0 (softmax bwd, GN2 sums, dgamma2/dbeta2), pass 1 (dw2/db2, GN1 sums,
 * dgamma1/dbeta1), pass 2 (dy1 = gradient wrt the raw conv1 output, stored with pitch dy_ld; db1 += sum dy1).
 * dprobs is fp32 [N][C][nvox]; all gradient outputs are accumulated (caller zeroes). */
int seg3d_outblock_tail_bwd(int dtype, int pass, const void* y1, int ld, int C,
                            const double* stats1, const float* gamma1, const float* beta1,
                            const float* w2, const float* bias2,
                            const double* stats2, const float* gamma2, const float* beta2, float eps,
                            const float* dprobs, double* sums2, double* sums1,
                            float* dgamma2, float* dbeta2, float* dw2, float* db2,
                            float* dgamma1, float* dbeta1, float* db1,
                            void* dy1, int dy_ld, int N, int64_t nvox, void* stream);
/* seg3d_gn_bwd without the ReLU: the backward of a unit that ends in a plain GroupNorm (a standalone
 * ConvGnRelu3(..., do_act=False)).  Same two passes, arguments and outputs as seg3d_gn_bwd with dz = g0 + g1 + g2
 * (no mask: there is no `out` and no beta).  dres (optional) = dz.  C % 8 == 0, 256 % (C/8) == 0, pitches % 8 == 0. */
int seg3d_gn_bwd_noact(int dtype, int pass, const void* g0, int ld0, const void* g1, int ld1, const void* g2, int ld2,
                       const void* y, int y_ld, int C, const double* stats, const float* gamma, float eps,
                       double* sums, float* dgamma, float* dbeta, void* dy, int dy_ld, void* dres, int dres_ld,
                       float* dbias, int N, int64_t nvox, void* stream);
/* Layout boundary of the standalone modules' backward (NCDHW fp32 outside a module, NDHWC storage type inside).
 * seg3d_grad_to_ncdhw: out[n][c][v] (fp32, dense [N][C][nvox]) = g0 + g1 + g2 summed in fp32 in that order, where
 *   contribution k (k < n_contrib, 1..3) is the NDHWC window gk[(n*nvox + v)*ldk + offk + c], c < C, in the storage type
 *   `dtype` (ldk >= offk + C).  Unused contributions may be NULL.
 * seg3d_grad_from_ncdhw: out[(n*nvox + v)*ld + off + c] = in[n][c][v] rounded to the storage type; channels outside
 *   [off, off + C) of each row are not written.
 * 16-byte accesses on the NDHWC side need C, pitch and offset multiples of 16 / sizeof(storage type) and a 16-byte
 * aligned base; other layouts take a scalar path. */
int seg3d_grad_to_ncdhw(int dtype, int n_contrib, const void* g0, int ld0, int off0, const void* g1, int ld1, int off1,
                        const void* g2, int ld2, int off2, int C, int N, int64_t nvox, float* out, void* stream);
int seg3d_grad_from_ncdhw(int dtype, const float* in, int C, int N, int64_t nvox, void* out, int ld, int off, void* stream);

/* ---- training: the parameter side of the step (reference core/seg_train.py:83 `optim.Adam(net.parameters(), lr, betas)`,
 * :127 `opt.step()`; the per-step weight re-layout replaces what nn.Conv3d does implicitly by reading its own parameter) ----
 * seg3d_gather_pack: table-driven strided gather with a cast.  Entry e fills the logical 5-D index space size[0..4]
 * (row-major, unused dims = 1):
 *     dst[dst_base + sum_d i_d*dst_stride[d]]  =  (all i_d < limit[d]) ? src[src_base + sum_d i_d*src_stride[d]] : 0
 * stored as `dtype` (SEG3D_F32 / F16 / BF16).  kind SEG3D_PACK_SPLIT_HI / _LO store f16(w) / f16(w - f16(w)) (the split-operand
 * strict mode).  Strides are in elements and may be negative (flipped taps of the data-gradient convolution).  `table` is a
 * DEVICE array of entries (each < 2^31 elements); one launch serves them all: block b handles elements
 * [block_map[2b+1]*SEG3D_PACK_CHUNK, +SEG3D_PACK_CHUNK) of entry block_map[2b] (block_map: device int32 pairs, n_blocks of them).
 * Used for: every convolution's kernel-layout weights (forward and data-gradient) from the fp32 OIDHW / IODHW parameters, and
 * the kernel-layout weight gradients back to parameter layout. */
#define SEG3D_PACK_PLAIN 0
#define SEG3D_PACK_SPLIT_HI 1
#define SEG3D_PACK_SPLIT_LO 2
#define SEG3D_PACK_CHUNK 4096
typedef struct seg3d_pack_entry {
  const float* src;
  void* dst;
  int64_t src_base, dst_base;
  int64_t src_stride[5], dst_stride[5];
  int32_t size[5], limit[5];
  int32_t dtype, kind;
} seg3d_pack_entry;
int seg3d_gather_pack(const seg3d_pack_entry* table, const int32_t* block_map, int n_blocks, void* stream);
/* torch.optim.Adam's update (no amsgrad, no maximize) over one flat fp32 range of n elements, `step` = 1, 2, ...:
 *   g += weight_decay*p;  m += (1-beta1)*(g-m);  v = beta2*v + (1-beta2)*g*g;
 *   p -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps).       All pointers 16-byte aligned. */
int seg3d_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                    float lr, float beta1, float beta2, float eps, float weight_decay, int step, void* stream);
/* the same update over n_ranges sub-ranges of the flat buffers, range k covering elements [offset, offset + n) with its own
 * step count (its own bias corrections); elements outside every range are not touched.  `ranges` is HOST memory, read
 * before the call returns; offsets are multiples of 4, ranges do not overlap. */
typedef struct {
  int64_t offset, n, step;
} seg3d_adam_range;
int seg3d_adam_step_ranges(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                           const seg3d_adam_range* ranges, int n_ranges, float lr, float beta1, float beta2,
                           float eps, float weight_decay, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEG3D_B200_H */
