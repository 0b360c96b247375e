/*
 * aa_resize.h -- C ABI of the B200-native anti-aliased separable resize (libaa_resize_b200.so).
 *
 * This is the drop-in boundary for ONE hot path of vfdev-5/interpolate-antialiasing: everything
 * below the pybind functions of step_two_dot_two/extension_interpolate.cpp.  Each entry point
 * names the reference interface it replaces (file:line under /root/reference/step_two_dot_two/).
 *
 * Conventions
 *   - plain C types only; no torch / C++ types cross this boundary;
 *   - every function returns 0 (AA_OK) or a negative aa_status; aa_last_error() gives the
 *     thread-local message; no C++ exception ever crosses the ABI;
 *   - the caller owns every tensor buffer (torch allocates them); the library owns only the
 *     per-device table cache, which is thread-safe;
 *   - device entry points are asynchronous on the given stream and never synchronise, except on
 *     a table-cache MISS (one tiny D2H of table metadata; call aa_warm_tables before CUDA-graph
 *     capture);
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     AA_ERR_CUDA.
 */
#ifndef AA_RESIZE_H_
#define AA_RESIZE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AA_RESIZE_ABI_VERSION 2

typedef enum aa_status {
  AA_OK = 0,
  AA_ERR_INVALID = -1,     /* bad argument (shape, dtype, filter, null pointer)            */
  AA_ERR_UNSUPPORTED = -2, /* valid but not implemented layout/dtype combination            */
  AA_ERR_CUDA = -3,        /* CUDA runtime error (message has cudaGetErrorString)           */
  AA_ERR_NOMEM = -4
} aa_status;

/* filter ids follow the reference's three helpers */
typedef enum aa_filter {
  AA_FILTER_BOX = 0,      /* nearest_forward ("it's not nearest but box") extension_interpolate.cpp:26-33,48;
                             HelperInterpNearest aa_interpolation_impl.h:331-373 */
  AA_FILTER_TRIANGLE = 1, /* linear_forward  extension_interpolate.cpp:7-14;  HelperInterpLinear :285-329 */
  AA_FILTER_CUBIC = 2     /* cubic_forward   extension_interpolate.cpp:35-42; HelperInterpCubic  :375-425 */
} aa_filter;

typedef enum aa_dtype {
  AA_U8 = 0,  /* input only: the uint8 -> float cast the reference's caller does (test.py:55,67) is fused */
  AA_F32 = 1,
  AA_F64 = 2,
  AA_F16 = 3, /* output only, through aa_resize_forward_ex */
  AA_BF16 = 4 /* output only, through aa_resize_forward_ex */
} aa_dtype;

/* execution-path selector for aa_resize_forward (flags argument) */
#define AA_FLAG_AUTO 0u
#define AA_FLAG_FORCE_GENERAL 1u /* gather-form tile kernel: H pass then V pass, no FMA contraction:
                                    bit-identical to the reference for f32/f64                      */
#define AA_FLAG_FORCE_STREAM 2u  /* streaming fused kernel (fails with AA_ERR_UNSUPPORTED if the
                                    shape/layout is not eligible)                                   */
#define AA_FLAG_STREAM_TMA 4u    /* streaming kernel: stage input rows with cp.async.bulk (TMA)     */
#define AA_FLAG_STREAM_LDG 8u    /* streaming kernel: plain vectorised global loads, single role    */
#define AA_FLAG_VMMA 64u         /* uint8 input: vertical pass on the tensor cores (tcgen05 kind::i8 + TMA, aa_vmma.cu);
                                    fails with AA_ERR_UNSUPPORTED if not eligible.  AUTO picks it for uint8 inputs
                                    downsampled >= 2x vertically                                      */
/* NaN/Inf in float inputs.  The reference touches the taps j < xsize of a window and nothing else
 * (aa_interpolation_impl.h:73-85): an output is non-finite iff one of ITS taps is.  The fast kernels also multiply a few
 * zero-weight neighbours (unrolled tap loops, accumulators not yet open), so they check what they store; a CTA that stored
 * a non-finite value lists its region and a second, tiny kernel behind every fast float launch re-evaluates the listed
 * regions tap-exactly (csrc/aa_redo.cu).  With every path -- AUTO included -- the set of non-finite outputs is therefore
 * the reference's; finite images pay an empty launch (a few microseconds), uint8 inputs nothing. */
#define AA_FLAG_STRICT_NONFINITE 128u /* float inputs: the gather kernel that touches in-window taps only, i.e. the same
                                    non-finite placement as AUTO and, in addition, finite values bit-identical to the
                                    reference (same arithmetic as AA_FLAG_FORCE_GENERAL, at its speed)              */
#define AA_FLAG_ASSUME_FINITE 256u /* the caller guarantees finite float data (e.g. converted uint8 images): skip the
                                    drain launch -- one kernel per call.  If the data is not finite after all, a NaN/Inf
                                    can also reach outputs whose window ends within K-1 taps of it; none is ever lost */
#define AA_FLAG_ROUND_NEAREST 32u /* uint8 output: round to nearest (PIL) instead of truncating (.byte()) */

/* A 4-D tensor view [n, c, h, w] with ELEMENT strides, resident on CUDA device `device`.
 * Supported layouts: channels_first (stride_w == 1) and channels_last (stride_c == 1,
 * stride_w == c), both with dense rows; stride_n is free (batch slices are fine). */
typedef struct aa_tensor_desc {
  void* data;
  int32_t dtype;  /* aa_dtype */
  int32_t device; /* CUDA ordinal */
  int64_t n, c, h, w;
  int64_t stride_n, stride_c, stride_h, stride_w;
} aa_tensor_desc;

/* Per-axis tables in the reference's own representation (for bit-exactness checks). */
typedef struct aa_tables_desc {
  int64_t* xmin;     /* [out]       device, first input index of each output's window  (:254; the
                                     reference stores xmin*stride_bytes :258, we store xmin)        */
  int64_t* xsize;    /* [out]       device, window length                               (:255-257,:259) */
  void* weights;     /* [out * K]   device, float (AA_F32) or double (AA_F64), normalised, zero padded
                                     to K                                               (:262-278) */
  int32_t interp_size; /* K, written by the call = (int)ceilf(support)*2+1              (:210) */
} aa_tables_desc;

/* ---- queries (host only, no device needed) ------------------------------------------------ */

int aa_abi_version(void);
const char* aa_last_error(void);

/* K for one axis; replaces the `int& in_out_interp_size` result of
 * HelperInterpBase::_compute_indices_weights_aa, aa_interpolation_impl.h:194-213.
 * dtype selects the scalar_t the table arithmetic runs in (AA_U8 computes as AA_F32). */
int aa_interp_size(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype,
                   int32_t* interp_size_out);

/* The integer window tables of one axis computed ON THE HOST with the same IEEE operations as the table kernel
 * (what the library's launch planning uses instead of reading the device tables back).  xmin/xsize: [out_size] host
 * arrays; scale_factor <= 0 means "not given".  Same reference lines as aa_build_tables (:253-257); bit-identical to
 * it and to the oracle (tests/test_capi_cpu.py, tests/test_tables_gpu.py). */
int aa_host_tables(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype, double scale_factor,
                   int64_t* xmin, int64_t* xsize);

/* ---- tables -------------------------------------------------------------------------------- */

/* Builds one axis' tables with the sm_100a table kernel and copies them, in the reference's
 * representation, into caller-provided DEVICE buffers.  Replaces
 * HelperInterp{Linear,Cubic,Nearest}::compute_indices_weights, aa_interpolation_impl.h:302-328,
 * :337-363, :379-405 (+ :194-281).  Integer tables and weights are bit-exact. */
int aa_build_tables(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype,
                    int device, aa_tables_desc* dst, void* cuda_stream);
/* same with a caller-provided scale factor for the axis (see aa_scales below; <= 0: not given) */
int aa_build_tables_sf(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype, double scale_factor,
                       int device, aa_tables_desc* dst, void* cuda_stream);

/* Pre-populates the table cache for a forward and/or backward call (so that the real calls never
 * synchronise, e.g. under CUDA-graph capture). */
int aa_warm_tables(int64_t in_h, int64_t in_w, int64_t out_h, int64_t out_w, int filter,
                   int align_corners, int dtype, int device, void* cuda_stream);

/* Drops every cached table on every device (frees device memory). */
int aa_clear_table_cache(void);

/* Health query for asynchronous failures that cannot surface through a return code: the persistent
 * tensor-core kernel bounds every mbarrier wait and records a watchdog code instead of hanging the GPU.
 * Call after synchronising the stream (one 4-byte D2H copy); AA_ERR_CUDA + message when a watchdog fired since
 * the last call.  No reference counterpart (the reference is synchronous CPU code). */
int aa_check_device(int device);

/* Tuning aid for the tensor-core kernel (no reference counterpart): with AA_VMMA_PROF=1 in the environment every
 * mbarrier wait adds the cycles it spent to a per-device counter (summed over the waiting warps):
 *   [1] producer: weight-matrix slot free   [2] producer: stage free        [3] MMA: weights landed
 *   [4] MMA: accumulator buffer released    [5] MMA: tile landed (TMA)      [6] epilogue: accumulators ready
 *   [8] epilogue: barrier before the horizontal pass  [9] horizontal pass  [10] barrier after it
 *   [12] producer warp lifetime  [13] MMA warp lifetime  [14] epilogue warps' lifetimes (sum of 8)
 * Synchronise the stream first.  counters16: 16 x uint64 on the host. */
int aa_debug_counters(int device, uint64_t* counters16, int reset);

/* ---- the hot path --------------------------------------------------------------------------- */

/* out[n,c,oy,ox] = sum_y sum_x Wh[oy,y] * Ww[ox,x] * in[n,c,y,x]   (horizontal then vertical in the
 * general path, as the reference; see DESIGN.md for the streaming path's order).
 * Replaces ti_upsample_{bilinear,bicubic,nearest}2d_cpu, aa_interpolation_impl.h:731-807, i.e.
 * the body of linear_forward / cubic_forward / nearest_forward, for already-allocated outputs.
 * in->dtype: AA_U8 | AA_F32 | AA_F64; out->dtype: AA_F32 (for u8/f32 inputs) or AA_F64 (f64), or
 * AA_U8 (u8/f32 inputs) for the fused epilogue: clamp to [0,255] then truncate like the reference's caller
 * (torch.clamp + .byte(), test.py:71-75), or round to nearest with AA_FLAG_ROUND_NEAREST.
 * n, c must match; in and out must be in the same memory format.  n == 0 is a no-op. */
int aa_resize_forward(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter,
                      int align_corners, uint32_t flags, void* cuda_stream);

/* Decode-adjacent fused epilogue (the step after this path in an input pipeline; not in the reference:
 * there the caller would run `.permute()`, `(x/255 - mean)/std` and `.half()` as separate passes after
 * proto_downsample, test.py:52-75).  Same as aa_resize_forward, plus, fused into the output stores:
 *   - per-channel affine  v*scale[c] + bias[c]   (normalize != 0; c < 4),
 *   - out->dtype AA_F16 / AA_BF16 / AA_F32 / AA_U8,
 *   - a channels_first (planar) `out` for a channels_last `in` (HWC uint8 from a JPEG decoder -> CHW). */
typedef struct aa_epilogue {
  int32_t normalize;
  float scale[4];
  float bias[4];
} aa_epilogue;
int aa_resize_forward_ex(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners,
                         uint32_t flags, const aa_epilogue* epilogue, void* cuda_stream);

/* Caller-provided scale factors: the `scale_factors` argument of ti_upsample_*2d_cpu
 * (aa_interpolation_impl.h:735,740-742: get_scale_value -> area_pixel_compute_scale).  A value > 0 replaces the
 * table scale in/out of that axis by 1/scale_factor (torch's interpolate(scale_factor=s, recompute_scale_factor=False));
 * <= 0 or a null pointer means "not given" (what the reference's shim always passes, extension_interpolate.cpp:12).
 * Ignored when align_corners is set, exactly like area_pixel_compute_scale. */
typedef struct aa_scales {
  double scale_h;
  double scale_w;
} aa_scales;
int aa_resize_forward_sf(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners,
                         const aa_scales* scales, uint32_t flags, void* cuda_stream);
int aa_resize_backward_sf(const aa_tensor_desc* grad_out, const aa_tensor_desc* grad_in, int filter, int align_corners,
                          const aa_scales* scales, uint32_t flags, void* cuda_stream);

/* Variable-size inputs -> one fixed-size batch (the decode-adjacent caller: N decoded images of different sizes, one
 * (oH, oW) training resolution; the reference takes one [N,C,H,W] tensor per call, test.py:52-58, so such a caller would
 * loop).  Image i ([c, h_i, w_i], dtype and pixel layout common to all) is resized into out[i].  Images are grouped by
 * size class (h, w, strides); inside a class, runs of images that sit at a constant pointer distance and go to consecutive
 * output slots (slices of one staging buffer, the usual case for a decoder writing into a pool) take ONE launch per run;
 * isolated images take one launch each.  Every launch after the first of a class is a table-cache and plan-cache hit
 * (no allocation, no synchronisation).  aa_epilogue may be NULL (plain float32 / uint8 output as aa_resize_forward). */
typedef struct aa_image_desc {
  void* data;        /* device pointer to image i */
  int64_t h, w;      /* its size */
  int64_t stride_h;  /* elements between rows */
  int64_t stride_c;  /* elements between channel planes (channels_first); ignored for channels_last (stride_c == 1) */
} aa_image_desc;
int aa_resize_forward_ragged(const aa_image_desc* images, int32_t count, int32_t dtype, int64_t channels, int32_t channels_last,
                             const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                             const aa_epilogue* epilogue, void* cuda_stream, int32_t* launches_out);

/* Batched resized crops: the training-time RandomResizedCrop + RandomHorizontalFlip of an input pipeline, a box per image
 * resized to one common (oH, oW) in a single launch (torchvision's resized_crop(img, top, left, height, width, size,
 * antialias=True); not in the reference).  out[i] is the aa_resize_forward_ex result for the view
 * image_i[top:top+height, left:left+width] (same out dtypes and epilogue, table scale height/oH and width/oW or the
 * align_corners form), bit for bit the AA_FLAG_FORCE_GENERAL arithmetic; with hflip != 0 output column ox is stored at
 * oW-1-ox (channels keep their order).  The same image may appear several times in `images` (multi-crop).
 *   - input u8 or f32, planar (stride_c) or HWC (channels_last != 0), any stride_h; out [count, channels, oH, oW] f32, u8,
 *     f16 or bf16, channels_first or channels_last (channels_last only for an HWC input); epilogue may be NULL;
 *   - the weights are computed inside the kernel (no table cache, no allocation, no copy, no synchronisation: capturable
 *     in a CUDA graph); the crop descriptors travel in the kernel parameters, 512 crops per launch, so a call issues
 *     ceil(count / 512) launches (*launches_out);
 *   - only in-window taps inside the boxes are read: NaN/Inf placement is exact with one launch, float input included;
 *   - AA_ERR_INVALID (message names the crop index) for a box outside its image (top < 0, left < 0, height < 1, width < 1,
 *     top+height > h, left+width > w), a wrong `out` shape or a null pointer; AA_ERR_UNSUPPORTED for f64 input, the
 *     path-forcing flags (FORCE_STREAM, STREAM_TMA, STREAM_LDG, VMMA, FORCE_GENERAL) and a window longer than 65 taps
 *     (interp_size 2*ceil(support)+1 > 65: box/bicubic/bilinear downscales by more than 64x / 16x / 32x along an axis).
 *     ASSUME_FINITE and STRICT_NONFINITE change nothing.  Every check happens before the first launch.
 *   - count == 0 is a no-op. */
typedef struct aa_crop {
  int64_t top, left, height, width; /* the box in pixels of its image, torchvision's resized_crop order */
  int32_t hflip;                    /* != 0: flip the resized result horizontally */
} aa_crop;
int aa_resize_crops(const aa_image_desc* images, const aa_crop* crops, int32_t count, int32_t dtype, int64_t channels,
                    int32_t channels_last, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                    const aa_epilogue* epilogue, void* cuda_stream, int32_t* launches_out);

/* Batched resize-then-crop: the evaluation transforms of an input pipeline, Resize(size) followed by CenterCrop, FiveCrop or
 * TenCrop, with a resized size per crop and the crop taken after the resize (torchvision's crop(resize(img, ...), ...);
 * not in the reference).  out[i] is the (oH, oW) window at (crop_top, crop_left) of
 *     R_i = aa_resize_forward_ex(image_i[top:top+height, left:left+width] -> (resized_h, resized_w))
 * bit for bit the AA_FLAG_FORCE_GENERAL arithmetic (table scales height/resized_h and width/resized_w, or the align_corners
 * form; output index crop_top + oy of R_i has the window the table kernel builds for that index), flipped as `flip` says:
 * bit 0 stores column ox at oW-1-ox, bit 1 stores row oy at oH-1-oy; channels keep their order.  That is
 * hflip(crop(resize(img))), what TenCrop computes after Resize.  Only the window's outputs are computed.
 *   - inputs, out dtypes and layouts, epilogue, flags, launches (ceil(count / 512)), graph capturability and the reads
 *     staying inside the box are those of aa_resize_crops.  aa_resize_crops(c) is aa_resize_crops_ex with
 *     resized = (oH, oW), crop_top = crop_left = 0 and flip = (hflip != 0), bit for bit;
 *   - AA_ERR_INVALID (message names the crop index) for everything aa_resize_crops refuses with it, and for resized_h or
 *     resized_w < 1, a window outside the resized image (crop_top < 0, crop_left < 0, crop_top + oH > resized_h,
 *     crop_left + oW > resized_w: no zero padding) and flip bits other than 0 and 1; AA_ERR_UNSUPPORTED for everything
 *     aa_resize_crops refuses with it (the 65-tap bound applies to box -> resized) and resized_h or resized_w >= 2^31.
 *     Every check happens before the first launch;
 *   - count == 0 is a no-op. */
typedef struct aa_crop_ex {
  int64_t top, left, height, width; /* box in the image that is resized (the whole image for Resize + CenterCrop)   */
  int64_t resized_h, resized_w;     /* the size that box is resized to (torchvision Resize's output size)            */
  int64_t crop_top, crop_left;      /* origin, in the resized image, of the (oH, oW) window stored in out[i]          */
  int32_t flip;                     /* bit 0: flip the stored window horizontally, bit 1: vertically                  */
} aa_crop_ex;
int aa_resize_crops_ex(const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype, int64_t channels,
                       int32_t channels_last, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                       const aa_epilogue* epilogue, void* cuda_stream, int32_t* launches_out);

/* Padded resize-then-crop: aa_resize_crops_ex whose windows may reach past the resized image.  out[i] is the (oH, oW) window
 * at (crop_top, crop_left) of P_i, flipped as `flip` says, where P_i is R_i of aa_resize_crops_ex extended in every direction
 * by a constant.  What it reproduces:
 *   - torchvision v2 center_crop of a crop larger than the image (pad with 0, then crop): AA_FILL_INPUT with 0;
 *   - letterboxing (resize with the aspect ratio kept, centred on a constant border such as 114): AA_FILL_INPUT;
 *   - pad-to-batch (resize, place at the top left of a common canvas, pad with zeros after normalisation, as torchvision
 *     detection's batch_images): AA_FILL_OUTPUT with 0;
 *   - RandomCrop(size, padding=p, fill=v) + horizontal flip: pad(img, p, v), crop, hflip: AA_FILL_INPUT with the box filter,
 *     resized size = image size (one tap of weight 1) and a window origin in [-p, p].
 * Outputs inside R_i are bit-identical to aa_resize_crops_ex.  Outputs outside R_i are bit-identical to aa_resize_forward_ex
 * of a [1, C, 1, 1] float32 tensor holding value[c], resized to 1x1 with the same out dtype and flags, and with the same
 * epilogue (AA_FILL_INPUT: value is a pixel of the input, e.g. torchvision's pad fill before Normalize / ToDtype) or with
 * none (AA_FILL_OUTPUT: value is stored as it is, converted to out->dtype only: f16/bf16 round to nearest, u8 clamps, then
 * truncates or rounds as AA_FLAG_ROUND_NEAREST says).
 *   - fill == NULL or mode AA_FILL_NONE: exactly aa_resize_crops_ex (same refusals, same launches);
 *   - with a fill, a window may overhang any edge of R_i or lie wholly outside it (all fill).  Tiles of the output with no
 *     output inside R_i store the fill and read nothing; launches, graph capturability and the reads staying inside the box
 *     are those of aa_resize_crops_ex;
 *   - AA_ERR_INVALID for an unknown mode; AA_ERR_UNSUPPORTED with a fill for channels > 4 and (message names the crop index)
 *     for a crop_top, crop_top + oH, crop_left or crop_left + oW outside int32.  Every other check is that of
 *     aa_resize_crops_ex, the window check excepted; every check happens before the first launch. */
#define AA_FILL_NONE 0   /* windows must lie inside the resized image: exactly aa_resize_crops_ex */
#define AA_FILL_INPUT 1  /* value[c] is a pixel value of the input: it goes through the epilogue like a resized value */
#define AA_FILL_OUTPUT 2 /* value[c] is stored as it is, only converted to out->dtype (zeros after normalisation) */
typedef struct aa_fill {
  int32_t mode;
  float value[4]; /* per channel; channels <= 4 whenever mode != AA_FILL_NONE */
} aa_fill;
int aa_resize_crops_pad(const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype, int64_t channels,
                        int32_t channels_last, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                        const aa_epilogue* epilogue, const aa_fill* fill, void* cuda_stream, int32_t* launches_out);

/* grad_in = Wh^T * grad_out * Ww : the true adjoint of aa_resize_forward, gather form, no atomics,
 * no zero-fill pass.  Replaces ti_upsample_bilinear2d_backward_cpu,
 * aa_interpolation_backward_impl.h:185-219 (linear_backward), whose body is the NON-antialiased
 * adjoint (SURVEY section 0.2); also provides the cubic/box backward the reference stubs out
 * (test.py:111-116). */
int aa_resize_backward(const aa_tensor_desc* grad_out, const aa_tensor_desc* grad_in, int filter,
                       int align_corners, uint32_t flags, void* cuda_stream);

/* The reference's exported linear_backward arithmetic (non-AA 2-tap bilinear adjoint,
 * aa_interpolation_backward_impl.h:80-108), gather form.  Kept only so `linear_backward(...,
 * antialias semantics of the reference)` can be reproduced bit-compatibly when asked. */
int aa_resize_backward_nonaa_bilinear(const aa_tensor_desc* grad_out, const aa_tensor_desc* grad_in,
                                      int align_corners, void* cuda_stream);

/* ---- host-buffer convenience (what a non-torch host binds; used by bench.py's e2e) ---------- */

/* Same as aa_resize_forward but `in`/`out` describe HOST buffers (device field = target CUDA
 * ordinal).  The batch is cut into chunks that are copied H2D, resized and copied back D2H on
 * rotating streams so copies overlap compute; returns after the last byte of `out` is written.
 * Pinned host memory is recommended (pageable works, slower). */
int aa_resize_forward_host(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter,
                           int align_corners, uint32_t flags);

/* One process, several GPUs (SURVEY 7.1 step 6 / 8(e)): the batch is split by image into contiguous shards of
 * ceil(n / n_devices), every device gets its own stream set, staging buffers and table-cache entries, all devices are
 * enqueued before any is waited for, and the call returns after the last byte of `out` is written.  No collective: the
 * shards are independent.  `devices` = CUDA ordinals (NULL / n_devices <= 0: every visible device); in->device is ignored.
 * What a non-torch host binds to use the 8 B200s of a box from one thread; bit-identical to the single-device entry. */
int aa_resize_forward_host_multi(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners,
                                 uint32_t flags, const int32_t* devices, int32_t n_devices);

/* Number of this library's kernel launches issued by the calling thread since the last reset
 * (bench.py reports it as gpu_launches). */
int64_t aa_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* AA_RESIZE_H_ */
