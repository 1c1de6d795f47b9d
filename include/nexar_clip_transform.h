/*
 * nexar_clip_transform.h — C ABI of the B200 clip-transform library
 * (libnexar_clip_b200.so).
 *
 * One call turns a batch of decoded uint8 dashcam clips into the normalised
 * model-input tensor: temporal gather -> antialiased letterbox (or short-side
 * resize + crop) -> horizontal flip -> VideoAugmentation chain -> mean/std
 * normalise -> [B,C,T,cs,cs] (or any strided layout), fp32 or bf16.
 *
 * It replaces, for this path only, what the reference does on the CPU in
 *   nexar_video_aug.py:809-821  VideoTransform.forward        (driver, /255 rule)
 *   nexar_video_aug.py:705-739  letterbox_resize               (+ tv F.resize antialias)
 *   nexar_video_aug.py:746-755  horizontal_flip
 *   nexar_video_aug.py:200-315  VideoAugmentation per-frame chain
 *   nexar_video_aug.py:794-799  normalize_tensor
 *   nexar_video_aug.py:407-424,464-482  resize_tensor / crop (dead-code variant)
 *   nexar_videos.py:416-451     frame gather, THWC->CTHW permute, transform call
 * The random decisions (nexar_video_aug.py:97-182, :748; nexar_videos.py:410)
 * stay on the host, drawn from Python's `random` in the reference's order, and
 * arrive here as one NexarClipParams per clip.
 *
 * Conventions: plain pointers and sizes, no exceptions, no allocation inside
 * nexar_clip_transform (the caller owns src, dst, params and workspace; only
 * nexar_plan_create allocates, a few KB of device tables), asynchronous on the
 * given CUDA stream.  Every function returns NEXAR_OK or a negative code;
 * nexar_last_error() gives a thread-local message.
 */
#ifndef NEXAR_CLIP_TRANSFORM_H
#define NEXAR_CLIP_TRANSFORM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NEXAR_ABI_VERSION 1

enum {
  NEXAR_OK = 0,
  NEXAR_ERR_INVALID = -1,     /* bad argument (the reference raises ValueError/TypeError) */
  NEXAR_ERR_CUDA = -2,        /* a CUDA runtime call failed */
  NEXAR_ERR_WORKSPACE = -3,   /* workspace too small / missing */
  NEXAR_ERR_UNSUPPORTED = -4
};

/* Source frames.  U8 / F32: packed RGB, HWC.  NV12: what a hardware decoder emits (replaces the CPU decode + RGB
 * conversion of decord.VideoReader / cv2, nexar_videos.py:360,422): a Y plane [H][src_row_stride] followed by the
 * interleaved chroma plane [H/2][src_row_stride] (U0 V0 U1 V1 ...), 1.5 bytes per pixel; converted on the device to
 * RGB bytes with the BT.601 limited-range integer formula (C = Y-16, D = U-128, E = V-128; R = clip((298C+409E+128)>>8),
 * G = clip((298C-100D-208E+128)>>8), B = clip((298C+516D+128)>>8); nearest-neighbour chroma), then identical to U8.
 * frame_offsets then point at the Y planes; the workspace grows by one RGB copy of the batch.
 * nexar_plan_create(g, NEXAR_SRC_NV12, ...) is nexar_plan_create_yuv(g, {NV12, BT601, LIMITED, 0}, ...); the other
 * 4:2:0 variants (I420, BT.709, full range, padded luma height) are described by NexarYuvFormat below. */
enum { NEXAR_SRC_U8 = 0, NEXAR_SRC_F32 = 1, NEXAR_SRC_NV12 = 2 };
enum { NEXAR_DST_F32 = 0, NEXAR_DST_BF16 = 1 };

/* NexarClipParams.flags */
enum {
  NEXAR_FLIP = 1u << 0,        /* nexar_video_aug.py:748 */
  NEXAR_AUG = 1u << 1,         /* VideoAugmentation active and not skipped (:112) */
  NEXAR_AFFINE = 1u << 2,      /* :130-136 */
  NEXAR_GRAYSCALE = 1u << 3,   /* :139 */
  NEXAR_NOISE = 1u << 4,       /* :140 */
  NEXAR_BLUR = 1u << 5,        /* :141 */
  NEXAR_POSTERIZE = 1u << 6,   /* :174 */
  NEXAR_SOLARIZE = 1u << 7,    /* :173 */
  NEXAR_INVERT = 1u << 8,      /* :172 */
  NEXAR_CUTOUT = 1u << 9       /* :144 */
};

#define NEXAR_MAX_CUTOUT 8
#define NEXAR_MAX_BLUR_TAPS 33

/* Where the antialiased-resize output lands on the cs x cs canvas. */
typedef struct NexarGeometry {
  int32_t src_h, src_w;        /* decoded frame size */
  int32_t canvas;              /* crop_size */
  int32_t resize_h, resize_w;  /* size of the resize output (new_h, new_w) */
  int32_t off_y, off_x;        /* canvas(y,x) = resized(y-off_y, x-off_x); letterbox: the pads; crop: -top,-left */
} NexarGeometry;

/* One per clip; every float already rounded the way torch rounds the Python
 * double (float32 of the float64 value). */
typedef struct NexarClipParams {
  uint32_t flags;
  int32_t crop_dy, crop_dx;    /* added to off_y/off_x: per-clip random crop (nexar_video_aug.py:472-473) */
  float brightness;            /* ratio of tv _blend */
  float contrast, contrast_q;  /* ratio and float32(1.0 - ratio) */
  float saturation, saturation_q;
  float hue;
  float grid[6];               /* theta^T / [0.5w, 0.5h] of tv _gen_affine_grid: x' = gx(x,y) = x*grid[0]+y*grid[1]+grid[2]; y' likewise [3..5] */
  float solarize_threshold;
  int32_t posterize_bits;
  float noise_level;
  uint32_t noise_seed[2];
  int32_t blur_ksize;          /* int(sigma*4)*2+1 */
  float blur_taps[NEXAR_MAX_BLUR_TAPS]; /* tv _get_gaussian_kernel1d */
  int32_t n_cutout;
  int32_t cutout[NEXAR_MAX_CUTOUT][4]; /* top, left, height, width */
} NexarClipParams;

typedef struct NexarPlan NexarPlan;   /* geometry + device tap tables */

typedef struct NexarTransformArgs {
  uint32_t struct_size;         /* sizeof(NexarTransformArgs), for ABI checking */
  int32_t n_clips, frames_per_clip;
  const void* src;              /* device: base of the decoded frames */
  const int64_t* frame_offsets; /* device [n_clips*frames_per_clip]: BYTE offset of each output frame's
                                   source frame from src (temporal sampling = gather; repeats allowed) */
  int64_t src_row_stride;       /* bytes between source rows */
  const NexarClipParams* params;/* device [n_clips] */
  uint32_t any_flags;           /* host hint: bitwise OR of params[i].flags; stages no clip needs are not launched */
  void* dst;                    /* device */
  int32_t dst_dtype;            /* NEXAR_DST_* */
  int32_t normalize;            /* 0: leave values in [0,1] */
  int64_t dst_stride[5];        /* ELEMENT strides for (clip, channel, frame, y, x) */
  float mean[3], std[3];
  void* workspace;              /* device, >= nexar_workspace_bytes(...) */
  size_t workspace_bytes;
  void* stream;                 /* cudaStream_t */
} NexarTransformArgs;

int nexar_abi_version(void);
size_t nexar_sizeof_clip_params(void);     /* for binding checks */
size_t nexar_sizeof_transform_args(void);
const char* nexar_last_error(void);

/* nexar_video_aug.py:713-719 (float64 truncation, floor-div pads) */
int nexar_letterbox_geometry(int32_t src_h, int32_t src_w, int32_t crop_size, NexarGeometry* out);
/* nexar_video_aug.py:411-415 then the centre crop of :468-469 */
int nexar_resize_crop_geometry(int32_t src_h, int32_t src_w, int32_t size, int32_t crop_size, NexarGeometry* out);
/* ATen _upsample_bilinear2d_aa tap table for one axis (host).  start/count: [out_size];
 * weights: [out_size*kmax_capacity] row-major.  *kmax receives the table width used. */
int nexar_aa_taps(int32_t in_size, int32_t out_size, int32_t* start, int32_t* count, float* weights,
                  int32_t kmax_capacity, int32_t* kmax);

int nexar_plan_create(const NexarGeometry* geom, int32_t src_dtype, NexarPlan** out);

/* YUV 4:2:0 decoder surfaces (nearest-neighbour chroma, one chroma sample per 2 x 2 pixels).
 *
 * Addressing, with pitch = NexarTransformArgs.src_row_stride and L = luma_rows (0 means src_h; L >= src_h, even):
 *   Y plane at frame_offsets[i]:                        L rows of pitch bytes; the visible src_h x src_w picture is its
 *                                                       top-left corner (rows src_h..L-1 and bytes src_w..pitch-1 are
 *                                                       never read)
 *   NV12: UV plane at frame_offsets[i] + L*pitch:       L/2 rows of pitch bytes, U0 V0 U1 V1 ...
 *   I420: U plane at frame_offsets[i] + L*pitch:        L/2 rows of pitch/2 bytes (pitch must be even),
 *         V plane at frame_offsets[i] + L*pitch*5/4:    L/2 rows of pitch/2 bytes
 * so every surface is an [L*3/2][pitch] byte block.  A 1080p NVDEC surface, for example, has L = 1088.
 *
 * Conversion, the classic 8-bit integer form with every coefficient round(256 * c) of the standard's float value:
 *   C = Y - Yo, D = U - 128, E = V - 128
 *   R = clip((Ys C + Rv E + 128) >> 8), G = clip((Ys C - Gu D - Gv E + 128) >> 8), B = clip((Ys C + Bu D + 128) >> 8)
 *                    Yo  Ys   Rv   Gu  Gv   Bu
 *   BT.601 limited   16  298  409  100 208  516     (NEXAR_SRC_NV12)
 *   BT.601 full       0  256  359   88 183  454
 *   BT.709 limited   16  298  459   55 136  541
 *   BT.709 full       0  256  403   48 120  475
 * into the packed RGB copy in the workspace; from there it is the NEXAR_SRC_U8 path bit for bit.
 *
 * The conversion reads 16 luma pixels per thread with 16-byte loads when src, pitch and src_w are multiples of 16;
 * that path also needs every frame_offsets[i] to be a multiple of 16 (not checked: the offsets live on the device).
 * Any other even size, pitch or alignment takes a byte-wise kernel. */
enum { NEXAR_YUV_NV12 = 0, NEXAR_YUV_I420 = 1 };
enum { NEXAR_YUV_BT601 = 0, NEXAR_YUV_BT709 = 1 };
enum { NEXAR_YUV_LIMITED = 0, NEXAR_YUV_FULL = 1 };

typedef struct NexarYuvFormat {
  uint32_t struct_size;         /* sizeof(NexarYuvFormat), for ABI checking */
  int32_t layout;               /* NEXAR_YUV_NV12 / NEXAR_YUV_I420 */
  int32_t matrix;               /* NEXAR_YUV_BT601 / NEXAR_YUV_BT709 */
  int32_t range;                /* NEXAR_YUV_LIMITED / NEXAR_YUV_FULL */
  int32_t luma_rows;            /* luma rows of the surface (0: src_h) */
} NexarYuvFormat;

/* A plan for YUV 4:2:0 surfaces.  geom->src_h / src_w are the visible picture (both even). */
int nexar_plan_create_yuv(const NexarGeometry* geom, const NexarYuvFormat* fmt, NexarPlan** out);

/* A plan for YUV 4:2:0 surfaces of 16-bit little-endian samples (10-, 12- or 16-bit decoder output).
 * fmt->layout NEXAR_YUV_NV12 is semi-planar (P010 / P012 / P016: interleaved U V words), NEXAR_YUV_I420 planar
 * (libavcodec's yuv420p10le).  sample_shift aligns each sample to the top of a 16-bit word: 0 for MSB-aligned samples
 * (P010 / P012 / P016), 6 for LSB-aligned 10-bit samples (yuv420p10le), 4 for LSB-aligned 12-bit samples; any other
 * value is NEXAR_ERR_INVALID.
 *
 * Addressing is the 8-bit addressing above in bytes with 2-byte samples: pitch = src_row_stride is in bytes and must be
 * even with 2*src_w <= pitch; the chroma starts at L*pitch (NV12: L/2 rows of pitch bytes, U0 V0 U1 V1 ... words;
 * I420: U plane of L/2 rows of pitch/2 bytes, then the V plane at L*pitch*5/4).
 *
 * Conversion: every sample is read as the word w = (sample << sample_shift) & 0xFFFF, and with the coefficients of the
 * table above, unchanged,
 *   C = w_Y - (Yo << 8), D = w_U - 32768, E = w_V - 32768
 *   R = clip((Ys C + Rv E + 32768) >> 16), G = clip((Ys C - Gu D - Gv E + 32768) >> 16), B = clip((Ys C + Bu D + 32768) >> 16)
 * to RGB bytes, then the NEXAR_SRC_U8 path.  A word x << 8 converts exactly as the 8-bit code x does
 * ((256 x + 32768) >> 16 == (x + 128) >> 8), so P010 words made from an NV12 surface give its result bit for bit; and
 * (64 X + 32768) >> 16 == (X + 512) >> 10, so 10-bit content is rounded once from its full precision.  A 10-bit code is
 * read as 4 x an 8-bit code, the limited-range convention of BT.709 / BT.2100 (for full range it differs from the
 * code / 1023 scaling by 0.25 %).
 *
 * The conversion reads 16 luma pixels of two rows per thread with 16-byte loads when src and every frame_offsets[i]
 * are multiples of 16 (the offsets are not checked), src_w % 16 == 0 and the pitch keeps the chroma rows 16-byte
 * aligned (pitch % 16 == 0 for NV12, pitch % 32 == 0 for I420); any other even size, pitch or alignment takes a
 * byte-wise kernel. */
int nexar_plan_create_yuv16(const NexarGeometry* geom, const NexarYuvFormat* fmt, int32_t sample_shift, NexarPlan** out);
/* The integer coefficients {Yo, Ys, Rv, Gu, Gv, Bu} the conversion uses for (matrix, range), for binding checks. */
int nexar_yuv_coefficients(int32_t matrix, int32_t range, int32_t out[6]);
size_t nexar_sizeof_yuv_format(void);

void nexar_plan_destroy(NexarPlan* plan);
int nexar_plan_geometry(const NexarPlan* plan, NexarGeometry* out);

/* Bytes of scratch nexar_clip_transform needs for this batch shape (covers the
 * worst case: every clip augmented and blurred). */
size_t nexar_workspace_bytes(const NexarPlan* plan, int32_t n_clips, int32_t frames_per_clip);
/* Exact requirement for a batch whose NexarTransformArgs.any_flags is known (no augmentation: a few KB). */
size_t nexar_workspace_bytes_for(const NexarPlan* plan, int32_t n_clips, int32_t frames_per_clip, uint32_t any_flags);

/* The hot path.  Enqueues the kernels on args->stream and returns.  Limits: n_clips * frames_per_clip <= 65535 per
 * call (split larger batches), and, for augmented batches, one frame of the destination must span < 2^31 elements
 * (2 * |dst_stride[1]| + (canvas - 1) * (|dst_stride[3]| + |dst_stride[4]|)); both return NEXAR_ERR_UNSUPPORTED. */
int nexar_clip_transform(const NexarPlan* plan, const NexarTransformArgs* args);

/* Materialised sliding windows for inference (extends the single centred window of nexar_inference.py:211-231 to the
 * stride-s windows of BASELINE config 4).  `frames` holds the per-frame result of one video as [n_frames][3] planes of
 * plane_bytes each (layout BTCHW of nexar_clip_transform); dst receives [n_windows][3][window] planes with
 * dst[k][c][t] = frames[min(k * stride + t, n_frames - 1)][c] (the last frame repeats past the end, nexar_videos.py:429-433). */
int nexar_gather_windows(const void* frames, int64_t n_frames, int64_t plane_bytes, int32_t window, int32_t stride,
                         int64_t n_windows, void* dst, void* stream);

/* Number of kernel launches the last nexar_clip_transform call on this thread enqueued. */
int nexar_last_launch_count(void);

/* Optional timing of the dominant (resize) kernel: after nexar_profile_begin(n) the next n calls record a
 * CUDA event pair around that kernel on the call's stream; nexar_profile_end synchronises those events,
 * writes up to `cap` per-call durations in ms and returns how many it wrote.  Used by bench.py. */
int nexar_profile_begin(int32_t max_calls);
int nexar_profile_end(float* ms_out, int32_t cap);

/* Tuning knobs for experiments, per calling thread (the library keeps no process-global mutable state; the profile
 * events above are per thread too).  Resize kernel: 0 = auto (the fixed-point fast kernel when the geometry allows it,
 * followed by the colour and geometry kernels for augmented clips, the colour kernel being a programmatic dependent launch
 * that overlaps the resize kernel's last wave), 1 = force the general fp32 kernels, 2 = as 0 without that overlap.
 * 4 selected a fused thread-block-cluster kernel (resize + colour + geometry in one launch); it was measured slower and
 * removed, and 4 now returns NEXAR_ERR_UNSUPPORTED.  Any other value is NEXAR_ERR_INVALID.  A refused value leaves the
 * setting unchanged.  Bands: the number of
 * row bands each frame is split into by the fast kernel (0 = auto). */
int nexar_set_resize_kernel(int32_t variant);
int nexar_set_fast_bands(int32_t bands);
/* Geometry (affine gather) kernel: 0 = auto (the kernel specialised for the 720p -> 224 / -> 320 letterboxes writing a
 * planar row-contiguous tensor when the call has that shape), 1 = always the general kernel. */
int nexar_set_geometry_kernel(int32_t variant);
/* Experiment: process an augmented batch in chunks of `clips` whole clips (resize, colour and geometry kernels of one
 * chunk back to back, for L2 locality of the intermediate); 0 = the whole batch at once (default: measured faster on
 * B200 at every batch size tried).  The result does not depend on it. */
int nexar_set_chunk_clips(int32_t clips);

#ifdef __cplusplus
}
#endif
#endif /* NEXAR_CLIP_TRANSFORM_H */
