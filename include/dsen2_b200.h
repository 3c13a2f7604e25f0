/*
 * dsen2_b200 -- C ABI of the B200-native DSen2 / VDSen2 super-resolution hot path.
 *
 * The reference (ACMEAtronOmatic/DSen2) has no FFI layer: its hot path is Python
 * calling numpy / scikit-image / Keras.  Each entry point below replaces one of
 * those Python-level operations (file:line into the reference tree) and is what a
 * ctypes binding on the reference side would call (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; nothing is
 *     allocated or freed by the library and there is no global mutable state
 *     besides a thread-local error string;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued, not synchronised;
 *   - return value: 0 = ok, >0 = cudaError_t, <0 = DSEN2_E_* argument error;
 *     dsen2_last_error() returns a human-readable message for the calling thread.
 */
#ifndef DSEN2_B200_H_
#define DSEN2_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSEN2_ABI_VERSION 3

#define DSEN2_E_BADARG   (-1)  /* null pointer / non-positive size / unsupported combination */
#define DSEN2_E_ALIGN    (-2)  /* pointer or channel count not aligned as the kernel requires */
#define DSEN2_E_DRIVER   (-3)  /* cuTensorMapEncodeTiled unavailable or failed */
#define DSEN2_E_NOTSM100 (-4)  /* device is not compute capability 10.x */

int dsen2_abi_version(void);
const char* dsen2_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * Patch extraction -- utils/patches.py:19-80 (get_test_patches) and :83-156 (get_test_patches60).
 * One call per resolution.  d_img is (H, W, C) float32 HWC with H = grid_h*ratio, W = grid_w*ratio
 * where (grid_h, grid_w) is the size of the tiling grid (the 20 m grid for the 20 m path, the 60 m
 * grid for the 60 m path) and ratio in {1,2,3,6}.  Patches are patch_lr*ratio square with a
 * symmetric-padded border of border_lr*ratio; crop starts follow patches.py:45-53.  Writes patches
 * [first_patch, first_patch+num_patches) of the ALLOCATED (k_i+1)*(k_j+1) stack (surplus patches are
 * zero, patches.py:32-39) to d_out (num_patches, C, p, p) float32, each value divided by `divisor`
 * (IEEE division; 1.0f = bit-exact copy; 2000.0f fuses supres.py:23-24).
 * ------------------------------------------------------------------------------------------- */
int dsen2_extract_patches(const float* d_img, int grid_h, int grid_w, int C, int ratio,
                          int patch_lr, int border_lr, int first_patch, int num_patches,
                          float divisor, float* d_out, void* stream);

/* Number of allocated patches (k_i+1)*(k_j+1) and of filled patches n_i*n_j (patches.py:32-53). */
int dsen2_patch_counts(int grid_h, int grid_w, int patch_lr, int border_lr, int* allocated, int* filled);

/* ---------------------------------------------------------------------------------------------
 * Bilinear upsample with mirror boundary, per (patch, band) plane -- utils/patches.py:11-16
 * (skimage.transform.resize(order=1, mode='reflect')).  d_in (planes, p, p) -> d_out (planes, p*s, p*s);
 * the result is divided by `post_divisor` (1.0f = none; 2000.0f fuses supres.py:24 / :43-44).
 * ------------------------------------------------------------------------------------------- */
int dsen2_bilinear_mirror_up(const float* d_in, int planes, int p, int s, float post_divisor, float* d_out,
                             void* stream);

/* ---------------------------------------------------------------------------------------------
 * Stitching -- utils/patches.py:374-405 (recompose_images), sequential-overwrite semantics restated
 * as ownership: patch t writes exactly the output pixels whose LAST writer it is.  d_pred holds
 * patches [first_patch, first_patch+num_patches) of the (N, C, P, P) prediction; d_out is the whole
 * (H, W, C) float32 HWC canvas (the array the reference returns as a transposed view, :405);
 * values are multiplied by `mul` (2000.0f fuses supres.py:29).
 * ------------------------------------------------------------------------------------------- */
int dsen2_recompose(const float* d_pred, int first_patch, int num_patches, int C, int P, int border,
                    int H, int W, float mul, float* d_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * MATLAB-compatible bicubic imresize -- utils/imresize.py:50-74,80-112.  The tap tables
 * (weights float64 (out, taps), indices int32 (out, taps)) are the ones imresize.py:28-48
 * (`contributions`) produces; the kernel reproduces imresizemex's float64 products summed left to
 * right, first along `first_dim` then along the other, so results are bit-identical.
 * d_in (h, w, C) float32 or float64 (in_is_f64), d_out (out_h, out_w, C) float64.
 * ------------------------------------------------------------------------------------------- */
int dsen2_bicubic_imresize(const void* d_in, int in_is_f64, int h, int w, int C,
                           const double* d_wy, const int32_t* d_iy, int taps_y, int out_h,
                           const double* d_wx, const int32_t* d_ix, int taps_x, int out_w,
                           int first_dim, double* d_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training-data generation -- utils/patches.py:353-371 (downPixelAggr): per band scipy
 * gaussian_filter(sigma = 1/scale) -- axis 0 then axis 1, double arithmetic, float32 storage between the
 * passes, 'reflect' boundary, kernel radius int(4/scale + 0.5) -- followed by the scale x scale block mean.
 * d_weights: the 2*radius+1 normalised Gaussian weights (host, scipy's _gaussian_kernel1d); d_tmp (H,W,C)
 * float32 scratch; d_out (H/scale, W/scale, C) float64.
 * integer_input != 0: d_img holds the values of an INTEGER image (the uint16 digital numbers GDAL hands
 * training/create_patches.py:189-197) -- scipy then stores each pass in that dtype, i.e. truncates towards zero.
 * ------------------------------------------------------------------------------------------- */
int dsen2_down_pixel_aggr(const float* d_img, int integer_input, int H, int W, int C, int scale, const double* d_weights,
                          int radius, float* d_tmp, double* d_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Network (utils/DSen2Net.py:9-43): tcgen05 implicit-GEMM convolutions on CTA pairs (cta_group::2), fp16 operands,
 * fp32 accumulation in TMEM (csrc/conv_pair.cu).  Activations are NHWC fp16.  One TMA halo-box load per tile and
 * 64-channel k-block serves all nine taps; zero 'same' padding at the PATCH edge is TMA out-of-bounds fill.  The
 * first and last layer are computed at fp32-equivalent precision (operands split v = hi + lo, fp16 each); the
 * residual trunk between resblocks is held as fp16 + 8 bits (below).  feature_size 128 (DSen2: the layer's weights
 * stay resident in shared memory) or 256 (VDSen2: weights stream through a shared-memory ring).
 * ------------------------------------------------------------------------------------------- */

/* Keras HWIO kernel (3,3,cin,cout) fp32 -> [tap][cout_pad][cin_pad] fp16 (K-major B operand of a trunk layer). */
int dsen2_pack_conv_weights(const float* d_hwio, int cin, int cout, int cin_pad, int cout_pad, void* d_packed_f16,
                            void* stream);

/* First convolution of a resBlock (DSen2Net.py:10-11): d_out = f16(relu(conv3x3(d_in) + bias)).
 * d_in / d_out NHWC fp16 (n, H, W, F); d_w from dsen2_pack_conv_weights(cin_pad = cout_pad = F); d_bias fp32 (F).   */
int dsen2_conv_relu(const void* d_in, const void* d_w, const float* d_bias, int n, int H, int W, int feature_size,
                    void* d_out, void* stream);

/* Prepared network input of the TRAINING step (and of a network without resblocks), "x_in": two NHWC fp16 tensors
 * (n, P, P, 64), hi and lo (value = hi + lo).  Channel t*16 + c of pixel (y, x) holds input band c of pixel
 * (y, x + t - 1) (t = 0..2; zero outside the patch; bands in DSen2Net.py:24,26 concatenation order; at most 16 bands):
 * the first layer's weight-gradient GEMM wants 128-byte pixel rows.  Inference uses the 16-channel form below.   */

/* x_in from NCHW fp32 patch stacks -- the arrays model.predict receives (supres.py:27,47,65). */
int dsen2_prep_from_patches(const float* d_x0, int c0, const float* d_x1, int c1, const float* d_x2, int c2,
                            int n, int P, void* d_xin_hi, void* d_xin_lo, void* stream);

/* Prepared input of the inference path: x_in16 hi / lo, NHWC fp16 (n, P, P, 16), channel c = band c of the concatenated
 * inputs (DSen2Net.py:24,26), c >= sum(c_i) zero.  dsen2_conv_head16_q reads it with all nine taps;
 * dsen2_conv_tail16[_stitch] take the global skip from it.
 *   dsen2_prep16_from_patches: from the NCHW fp32 patch stacks model.predict receives (supres.py:27,47,65);
 *   dsen2_prep16_from_images:  straight from the HWC images -- fuses get_test_patches / get_test_patches60
 *       (utils/patches.py:19-156), interp_patches (:11-16) and the /SCALE of supres.py:23-24,42-44 for patches
 *       [first_patch, first_patch + num_patches).  d_img60 == NULL selects the 20 m path (tiling grid = 20 m pixels),
 *       otherwise the 60 m path.  patch / border are the 10 m values of supres.py:22,41 (128 / 8 and 192 / 12).   */
int dsen2_prep16_from_patches(const float* d_x0, int c0, const float* d_x1, int c1, const float* d_x2, int c2,
                              int n, int P, void* d_xin_hi, void* d_xin_lo, void* stream);
/* dsen2_prep16_from_images reads the images as float32 or, natively, as the uint16 digital numbers GDAL hands
 * testing/s2_tiles_supres.py:311-315 (half the bytes to upload; uint16 -> float is exact, so both give bit-identical
 * prepared inputs).                                                                                              */
#define DSEN2_IMG_F32 0
#define DSEN2_IMG_U16 1
int dsen2_prep16_from_images(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                             int patch, int border, int first_patch, int num_patches, float divisor,
                             void* d_xin_hi, void* d_xin_lo, void* stream);
/* First layer kernel (3,3,cin,F) fp32 HWIO -> [9 taps][2F rows = W_hi ; W_lo][16] fp16 (for dsen2_conv_head16_q). */
int dsen2_pack_head16_weights(const float* d_hwio, int cin, int feature_size, void* d_packed, void* stream);

/* First layer kernel (3,3,cin,F) fp32 HWIO -> [3 vertical taps][2F rows = W_hi ; W_lo][64] fp16. */
int dsen2_pack_head_weights(const float* d_hwio, int cin, int feature_size, void* d_packed, void* stream);
/* Last layer kernel (3,3,F,cout) fp32 HWIO -> [9 taps][32 rows = W_hi(16) ; W_lo(16)][F] fp16 (for dsen2_conv_tail). */
int dsen2_pack_tail_weights(const float* d_hwio, int feature_size, int cout, void* d_packed, void* stream);

/* Conv2D(F, 3x3, relu) on the concatenated inputs (DSen2Net.py:29), 64-channel x_in -> trunk; feature_size 128.
 *   d_out_hi   NHWC fp16 (n,H,W,F): fp16 rounding of the layer output (the next convolution's operand)
 *   d_out_lo   optional NHWC fp16: out - out_hi (a network without resblocks hands it to dsen2_conv_tail)
 *   d_trunk32  optional fp32 trunk in TILE-ROW-MAJOR layout (n, H, ceil(W/8), F/4, 8, 4): element (n,y,x,c) at
 *              ((((n*H + y)*ceil(W/8) + x/8)*(F/4) + c/4)*8 + x%8)*4 + c%4 -- the layout dsen2_conv_res32
 *              updates in place (a thread that owns one pixel reads/writes it coalesced; 4 KB DRAM bursts)   */
int dsen2_conv_head(const void* d_xin_hi, const void* d_xin_lo, const void* d_w, const float* d_bias,
                    int n, int H, int W, int feature_size, void* d_out_hi, void* d_out_lo,
                    float* d_trunk32, void* stream);

/* Second convolution of a resBlock with the residual update on the fp32 trunk (DSen2Net.py:12-15):
 *   trunk32 <- trunk32 + res_scale * (conv3x3(d_in) + bias)          (in place, tile-row-major fp32)
 *   d_out_hi <- fp16(trunk32) NHWC;  d_out_lo (optional) <- fp16(trunk32 - out_hi) NHWC
 * d_in is the NHWC fp16 output of the block's first convolution (dsen2_conv_relu); d_w from
 * dsen2_pack_conv_weights(cin_pad = cout_pad = feature_size).  feature_size 128 or 256 (weights streamed).   */
int dsen2_conv_res32(const void* d_in, const void* d_w, const float* d_bias, int n, int H, int W, int feature_size,
                     float res_scale, float* d_trunk32, void* d_out_hi, void* d_out_lo, void* stream);

/* The trunk of the inference path (fp16 + 8 bits, 19 significant bits):
 * the trunk value x is held as the NHWC fp16 tensor x_hi the next convolution reads anyway plus one signed
 * byte per element, lo, in tile-row-major layout (n, H, ceil(W/8), F/16, 8, 16): element (n,y,x,c) at
 *   ((((n*H + y)*ceil(W/8) + x/8)*(F/16) + c/16)*8 + x%8)*16 + c%16.
 * With s = bits(x) + 0x1010: x_hi = fp16 of s truncated (x rounded to the nearest fp16, ties away from zero),
 * lo = ((s >> 5) & 0xff) - 128, and a reader recovers bits(x) ~ bits(float(x_hi)) + (lo << 5) (|error| <= 16 fp32
 * ulps).  Below 2^-14 x_hi is an fp16 subnormal and the pair only keeps x to an absolute 2^-24; lo is 0 where x_hi
 * is zero.  A resblock then moves 1024 B/pixel through HBM instead of the 1536 of the fp32 trunk above.
 *   dsen2_conv_head16_q: x = relu(conv(x_in16) + bias)  ->  d_x_hi, d_trunk_lo8           (DSen2Net.py:29; below)
 *   dsen2_conv_resq:    x <- x + res_scale * (conv3x3(d_in) + bias), in place               (DSen2Net.py:12-15)
 *                       d_out_lo != NULL marks the LAST block: x_hi <- fp16(x) (round to nearest even) and
 *                       d_out_lo <- fp16(x - x_hi) NHWC for dsen2_conv_tail; d_trunk_lo8 is then only read.
 * d_in must not alias d_x_hi.  feature_size 128 only.                                                       */
int dsen2_conv_resq(const void* d_in, const void* d_w, const float* d_bias, int n, int H, int W,
                    float res_scale, void* d_x_hi, void* d_trunk_lo8, void* d_out_lo, void* stream);
/* The same resblock update for feature_size 256 (VDSen2; d_w from dsen2_pack_conv_weights(cin_pad = cout_pad = 256):
 * 1.18 MB of weights per layer stream through an 8-slot shared-memory ring instead of staying resident).         */
int dsen2_conv_resq256(const void* d_in, const void* d_w, const float* d_bias, int n, int H, int W,
                       float res_scale, void* d_x_hi, void* d_trunk_lo8, void* d_out_lo, void* stream);
/* First layer on the 16-channel prepared input (dsen2_prep16_*, weights from dsen2_pack_head16_weights), feature_size 128
 * or 256: nine taps as shifted descriptors into a 32-byte-row (SWIZZLE_32B) halo box; per tap the three products
 * hi*W_hi + hi*W_lo + lo*W_hi accumulate into ONE TMEM accumulator (fp32-equivalent first layer).               */
int dsen2_conv_head16_q(const void* d_xin_hi, const void* d_xin_lo, const void* d_w, const float* d_bias,
                        int n, int H, int W, int feature_size, void* d_x_hi, void* d_trunk_lo8, void* stream);
/* The same first layer for the training step of the 256-feature network (supres_train.py:129-130): relu -> d_out_hi NHWC
 * fp16 and the seed of the fp32 trunk d_trunk32 (layout as dsen2_conv_head).  feature_size 256.                  */
int dsen2_conv_head16_relu(const void* d_xin_hi, const void* d_xin_lo, const void* d_w, const float* d_bias,
                           int n, int H, int W, int feature_size, void* d_out_hi, float* d_trunk32, void* stream);

/* Conv2D(cout, 3x3) + Add(last input) (DSen2Net.py:35,38,41) on the trunk (hi, lo).  The global skip is
 * read from x_in (centre tap, bands skip_ch0 .. skip_ch0+cout).  Output: NCHW fp32 predictions
 * (n, cout, H, W) -- what model.predict returns.                                                  */
int dsen2_conv_tail(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                    const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                    int n, int H, int W, float* d_pred_nchw, void* stream);

/* The last layer of the inference path (csrc/conv_tail.cu): the same Conv2D(cout) + Add with the global skip read from
 * the 16-channel prepared input, feature_size 128 or 256, cout <= 7 (DSen2: 6 bands at 20 m, 2 at 60 m).  The GEMM runs
 * with the operands SWAPPED -- the 18 * cout weight rows (tap x {W_hi, W_lo} x band) on the M side, the 18 x 10 pixel halo
 * box of a tile on the N side -- so an activation crosses the shared-memory read port once instead of once per tap; the
 * 3x3 shifts are applied in the epilogue.  d_w from dsen2_pack_tail16_weights: [128 rows][feature_size] fp16.      */
int dsen2_pack_tail16_weights(const float* d_hwio, int feature_size, int cout, void* d_packed, void* stream);
int dsen2_conv_tail16(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                      const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                      int n, int H, int W, float* d_pred_nchw, void* stream);
/* Same, fused with recompose_images (utils/patches.py:374-405) and the x SCALE of supres.py:29,49: the
 * n patches are patches [first_patch, first_patch + n) of the canvas tiling; each writes the pixels of
 * the (img_h, img_w, cout) float32 HWC canvas whose LAST writer it is, multiplied by `mul`.          */
int dsen2_conv_tail16_stitch(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                             const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                             int n, int P, int first_patch, int border, int img_h, int img_w, float mul,
                             float* d_canvas, void* stream);
/* The same into a (img_h, img_w, cout) uint16 canvas of digital numbers: with f the float the entry above writes, the
 * value is 0 for NaN and otherwise rint(clip(f, 0, 65535)) (round half to even).  A value equal to `avoid` (the nodata
 * value of the run, -1 = none, otherwise in [0, 65535]) is written as avoid + 1 (65534 for 65535): a network output never
 * reads as nodata.                                                                                                  */
int dsen2_conv_tail16_stitch_u16(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                 const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                                 int n, int P, int first_patch, int border, int img_h, int img_w, float mul, int avoid,
                                 uint16_t* d_canvas, void* stream);

/* The same two steps for an arbitrary list of patches (the active patches of dsen2_nodata_patches): the arguments of
 * dsen2_prep16_from_images / dsen2_conv_tail16_stitch, with batch entry b = patch d_patch_ids[b] (absolute indices in the
 * filled patch list, device int32 array of n = num_patches entries) instead of first_patch + b.  An id outside the tiling
 * prepares a zero input and writes nothing.                                                                          */
int dsen2_prep16_from_images_ids(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                                 int patch, int border, const int* d_patch_ids, int num_patches, float divisor,
                                 void* d_xin_hi, void* d_xin_lo, void* stream);
int dsen2_conv_tail16_stitch_ids(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                 const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                                 int n, int P, const int* d_patch_ids, int border, int img_h, int img_w, float mul,
                                 float* d_canvas, void* stream);
/* dsen2_conv_tail16_stitch_u16 for a list of patches. */
int dsen2_conv_tail16_stitch_ids_u16(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                     const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                                     int n, int P, const int* d_patch_ids, int border, int img_h, int img_w, float mul,
                                     int avoid, uint16_t* d_canvas, void* stream);

/* Radiometric offset (an extension: Sentinel-2 products of processing baseline 04.00 and later store
 * DN = 10000 * reflectance - add_offset, with add_offset = RADIO_ADD_OFFSET / BOA_ADD_OFFSET = -1000 in their metadata, while
 * the network expects DN = 10000 * reflectance).  The two steps above with a finite `add_offset` (anything else:
 * DSEN2_E_BADARG):
 *   dsen2_prep16_from_images_offset: every band value x of the images, as stored (uint16 or float32), becomes
 *       fl32(x + add_offset) before any other arithmetic of the preparation (the bilinear round trip, the / divisor).
 *   dsen2_conv_tail16_stitch_offset: with f the float the stitching entry writes for those inputs, the canvas receives
 *       fl32(f - add_offset) -- the output is in the convention of the input product -- or, for a uint16 canvas, the
 *       digital number of that value as dsen2_conv_tail16_stitch_u16 computes it.
 * Both take the range form and the list form: d_patch_ids == NULL: patches [first_patch, first_patch + num_patches); else
 * the listed ids (first_patch ignored).  The nodata entry points take the stored values: v is the value the product holds. */
int dsen2_prep16_from_images_offset(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                                    int patch, int border, int first_patch, const int* d_patch_ids, int num_patches,
                                    float divisor, float add_offset, void* d_xin_hi, void* d_xin_lo, void* stream);
/* canvas_dtype DSEN2_IMG_F32 / DSEN2_IMG_U16; avoid as dsen2_conv_tail16_stitch_u16 (-1 for a float canvas). */
int dsen2_conv_tail16_stitch_offset(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                    const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                                    int n, int P, int first_patch, const int* d_patch_ids, int border, int img_h, int img_w,
                                    float mul, float add_offset, int canvas_dtype, int avoid, void* d_canvas, void* stream);

/* Chip stacks (an extension: datasets of many small same-size scenes, e.g. 120 x 120 or 256 x 256 chips).  The images are
 * stacks (num_chips, H, W, 4), (num_chips, H/2, W/2, 6) and, for the 60 m path, (num_chips, H/6, W/6, 2), contiguous; the
 * canvas is (num_chips, img_h, img_w, cout).  Patches are numbered over the whole stack, g = chip * ppc + p, with ppc the
 * FILLED patches of one chip (dsen2_patch_counts' second count, n_i * n_j) and p the patch's index in the chip's own tiling,
 * so one call can run [first_patch, first_patch + num_patches) across chip boundaries.  Each chip is tiled, prepared and
 * stitched exactly as the single-image entry points do it for that image (the same geometry is rejected), so the
 * prepared input of a patch and the pixels it writes are bit-identical to theirs; a patch writes only into its own chip.
 * The offset is an explicit switch: add = 0 runs the arithmetic of dsen2_prep16_from_images / dsen2_conv_tail16_stitch(_u16),
 * add = 1 that of the _offset entry points with the finite add_offset (-0 + 0 is +0, so an add of 0 is not "no offset").
 * DSEN2_E_BADARG also for num_chips < 0, add not 0 / 1, and a range outside [0, num_chips * ppc) (num_chips * ppc < 2^31).
 * There is no id-list form.                                                                                          */
int dsen2_prep16_from_chips(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int num_chips,
                            int H, int W, int patch, int border, int first_patch, int num_patches, float divisor, int add,
                            float add_offset, void* d_xin_hi, void* d_xin_lo, void* stream);
/* canvas_dtype DSEN2_IMG_F32 / DSEN2_IMG_U16; avoid as dsen2_conv_tail16_stitch_u16 (-1 for a float canvas). */
int dsen2_conv_tail16_stitch_chips(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                   const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                                   int n, int P, int first_patch, int border, int num_chips, int img_h, int img_w, float mul,
                                   int add, float add_offset, int canvas_dtype, int avoid, void* d_canvas, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Nodata (csrc/nodata.cu; an extension: the reference super-resolves nodata like data).  Images, img_dtype, H, W, patch
 * and border as dsen2_prep16_from_images (d_img60 == NULL: 20 m path); `nodata` is the fill value v (not NaN).  Output pixel
 * (y, x) is NODATA iff every band of img10[y, x], img20[y/2, x/2] and (60 m) img60[y/6, x/6] equals v in the images'
 * element type; any other pixel is valid.
 *   dsen2_nodata_patches: of the filled patches [first_patch, first_patch + num_patches), the ACTIVE ones -- those that
 *       own (last writer wins, as dsen2_conv_tail16_stitch) at least one valid pixel -- as ascending absolute ids in
 *       d_ids[0, *d_count).  d_ids holds num_patches ints (it is also the scan's scratch); d_count one int.
 *   dsen2_nodata_fill: writes v into all cout bands of every nodata pixel of the (H, W, cout) float32 canvas that the
 *       range owns.  Run it after the last layer: an active patch also stitches network values over its nodata pixels.
 *   dsen2_nodata_fill_u16: the same for the uint16 canvas of dsen2_conv_tail16_stitch[_ids]_u16; v must be an integer in
 *       [0, 65535].  With avoid = v there, nodata pixels are exactly those that hold v.
 * Running only the active patches (dsen2_*_ids) and then the fill leaves every valid pixel bit-identical to the whole
 * range run without nodata.                                                                                          */
int dsen2_nodata_patches(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                         int patch, int border, int first_patch, int num_patches, float nodata, int* d_ids, int* d_count,
                         void* stream);
int dsen2_nodata_fill(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                      int patch, int border, int first_patch, int num_patches, float nodata, int cout, float* d_canvas,
                      void* stream);
int dsen2_nodata_fill_u16(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                          int patch, int border, int first_patch, int num_patches, float nodata, int cout,
                          uint16_t* d_canvas, void* stream);

/* Whole s2model forward (model.predict on one batch, supres.py:65) for n patches of (P, P).
 * d_weights[i] / d_bias[i] are the packed layers in Keras topological order (2*num_layers+2 entries):
 *   [0] dsen2_pack_head16_weights (dsen2_pack_head_weights when num_layers == 0, feature_size 128 only),
 *   [1..2L] dsen2_pack_conv_weights(cin_pad = cout_pad = feature_size), [2L+1] dsen2_pack_tail16_weights
 *   (dsen2_pack_tail_weights when num_layers == 0);
 *   biases fp32 of length F / F / 16;
 *   pipeline: prep16_from_patches -> conv_head16_q -> L x (conv_relu, conv_resq[256]) -> conv_tail16
 *   for feature_size 128 (DSen2) and 256 (VDSen2) alike.
 * Workspace: see dsen2_s2model_workspace_bytes.  d_x[0..n_inputs) NCHW fp32 inputs; the last one is
 * the global skip. */
size_t dsen2_s2model_workspace_bytes(int n, int P, int in_channels, int feature_size);
int dsen2_s2model_forward(const float* const* d_x, const int* channels, int n_inputs,
                          int n, int P, int num_layers, int feature_size,
                          const void* const* d_weights, const float* const* d_bias,
                          void* d_workspace, size_t workspace_bytes,
                          float* d_out_f32, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training step -- training/supres_train.py:137-144 (Nadam, mean_absolute_error, mean_squared_error
 * metric) and :218-230 (model.fit inner step), feature_size 128 (DSen2) or 256 (VDSen2, supres_train.py:129-130).
 * Forward = the inference kernels with per-layer activation buffers.  Backward data path = the same convolution kernels on
 * dsen2_pack_dgrad_weights operands: dsen2_conv_relu_bwd (gradient through Conv2D + ReLU) and
 * dsen2_conv_res32 with scale 1 (gradient through the Add of resBlock, accumulated on an fp32
 * gradient trunk).  Weight gradients = dsen2_wgrad_nhwc, a tcgen05 GEMM over the pixel dimension.
 * Gradients carry a power-of-two loss scale chosen by the host (see dsen2_b200/train.py).
 * ------------------------------------------------------------------------------------------- */

/* backward-data operand of a layer: packed[t][i][o] = scale * hwio[8-t][i][o], fp16, (9, rows_pad, k_pad) */
int dsen2_pack_dgrad_weights(const float* d_hwio, int cin, int cout, int rows_pad, int k_pad, float scale,
                             void* d_packed, void* stream);

/* All F -> F layers in one launch: layer l's Keras kernel (3,3,F,F) fp32 at d_first_kernel + l * layer_stride (floats; the
 * flat Keras-order parameter vector puts them 9*F*F + F apart) -> forward operand d_fwd[l] (dsen2_pack_conv_weights layout)
 * and backward-data operand d_bwd[l] (dsen2_pack_dgrad_weights layout, scale = scale_second for odd l -- the second
 * convolution of a resBlock, whose Lambda(x * 0.1) is folded in -- and 1 otherwise).                                  */
int dsen2_pack_trunk_layers(const float* d_first_kernel, long long layer_stride, int num_layers, int feature_size,
                            float scale_second, void* d_fwd, void* d_bwd, void* stream);

/* d_out = conv3x3(d_in, d_w) * [d_fwd_act > 0]   (NHWC fp16, feature_size = 128 or 256 channels; d_bias must be zeros) */
int dsen2_conv_relu_bwd(const void* d_in, const void* d_w, const float* d_bias, const void* d_fwd_act,
                        int n, int H, int W, int feature_size, void* d_out, void* stream);

/* up to three NCHW fp32 inputs concatenated along channels -> NHWC fp16 (n,H,W,cpad), remaining channels zero */
int dsen2_nchw_to_nhwc_f16(const float* d_x0, int c0, const float* d_x1, int c1, const float* d_x2, int c2,
                           int n, int H, int W, int cpad, void* d_out, void* stream);
/* d_out = d_in where d_act > 0, else 0 (NHWC fp16, `total` elements, multiple of 8) */
int dsen2_relu_mask(const void* d_in, const void* d_act, long long total, void* d_out, void* stream);
/* Weight gradient straight from the NHWC fp16 tensors (C = channels = 128 or 256 each), MN-major tcgen05 operands:
 * d_dw (9,C,C) fp32 += scale * sum_px X[px + tap][ci] * dY[px][co]   (HWIO order; one CTA per vertical tap, pixel
 * slice and 128 x 128 block of the gradient).  d_db (optional, C floats): the bias gradient of the same layer,
 * d_db[co] += scale * sum_px dY[px][co], summed from the dY tiles the kernel stages anyway.                    */
int dsen2_wgrad_nhwc(const void* d_x, const void* d_dy, int n, int H, int W, int channels, float scale, float* d_dw,
                     float* d_db, void* stream);

/* mean_absolute_error: d_dpred = gscale * sign(pred - y); d_sums[0] += sum|pred-y|, d_sums[1] += sum (pred-y)^2 */
int dsen2_mae_grad(const float* d_pred, const float* d_y, long long total, float gscale, float* d_dpred,
                   double* d_sums, void* stream);

/* Keras-2 Nadam update of a flat fp32 parameter vector (gradient multiplied by grad_mul first: 1/loss_scale/world).
 * mu_t, mu_next, sched_new = prod(mu_1..mu_t), sched_next = sched_new*mu_next, bias2 = 1 - beta2^t (host).   */
int dsen2_nadam_step(float* d_p, const float* d_g, float* d_m, float* d_v, long long total, float grad_mul,
                     float lr, float beta1, float beta2, float eps, float mu_t, float mu_next,
                     float sched_new, float sched_next, float bias2, void* stream);

/* Same update, step-dependent scalars in device memory (replayable inside a captured CUDA graph):
 * d_hp = {grad_mul, lr, beta1, beta2, eps, mu_t, mu_next, sched_new, sched_next, bias2}.                     */
int dsen2_nadam_step_dev(float* d_p, const float* d_g, float* d_m, float* d_v, long long total,
                         const float* d_hp, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSEN2_B200_H_ */
