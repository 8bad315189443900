/* include/b200dsp.h — C-ABI of libb200dsp: the B200-native raw-frame DSP hot path.
 *
 * This is the drop-in boundary.  Every entry point is what a GStreamer element's
 * vmethod would call in place of the reference's CPU library call; the reference
 * interface each one replaces is cited (paths under /root/reference/subprojects/):
 *
 *   b200_vcs_*   replace  gst_video_converter_new / _frame / _free
 *                         gst-plugins-base/gst-libs/gst/video/video-converter.c:2421, :2782, :2618
 *                called from GstVideoFilterClass::set_info / ::transform_frame
 *                         gst-plugins-base/gst/videoconvertscale/gstvideoconvertscale.c:906, :1981
 *                device-memory calling convention follows gst_cuda_converter_convert_frame
 *                         gst-plugins-bad/gst-libs/gst/cuda/gstcudaconverter.cpp:1911
 *   b200_comp_*  replace  the BlendFunction / FillCheckerFunction / FillColorFunction table
 *                         gst-plugins-base/gst/compositor/blend.h:50-79
 *                called from GstVideoAggregatorClass::aggregate_frames
 *                         gst-plugins-base/gst/compositor/compositor.c:1739
 *   b200_ars_*   replace  gst_audio_resampler_new / _get_out_frames / _resample / _reset / _free
 *                         gst-plugins-base/gst-libs/gst/audio/audio-resampler.c:1344, :1648, :1750, :1458, :1616
 *                called from GstBaseTransformClass::transform
 *                         gst-plugins-base/gst/audioresample/gstaudioresample.c:885, :743
 *
 * Conventions: plain C, POD descriptors, raw pointers + sizes, an opaque
 * `void *cuda_stream` (a cudaStream_t / CUstream; NULL = legacy default stream).
 * No GLib, GStreamer or torch type crosses this boundary.  All calls return a
 * b200_status; 0 is success.  Device pointers must belong to the device the handle
 * was created on.  Launch-only calls are asynchronous on `cuda_stream` exactly like
 * gst_cuda_converter_convert_frame(): the caller owns synchronisation
 * (gst-plugins-bad/sys/nvcodec/gstcudaconvertscale.c:1541-1579).
 *
 * Enum values are GStreamer's own so an element can pass GstVideoInfo fields
 * through without translation.
 */
#ifndef B200DSP_H
#define B200DSP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200DSP_VERSION_MAJOR 0
#define B200DSP_VERSION_MINOR 1

typedef enum {
  B200_OK = 0,
  B200_ERR_INVALID_ARG = -1,     /* -> set_info FALSE / GST_FLOW_NOT_NEGOTIATED */
  B200_ERR_UNSUPPORTED = -2,     /* format / mode not implemented -> caps not accepted */
  B200_ERR_NO_DEVICE = -3,       /* no CUDA device / driver: product never falls back to CPU */
  B200_ERR_CUDA = -4,            /* a CUDA call failed -> GST_FLOW_ERROR */
  B200_ERR_NOMEM = -5,
  B200_ERR_STATE = -6
} b200_status;

const char *b200_strerror (int status);
/* last CUDA error string recorded on this thread (for GST_ELEMENT_ERROR text) */
const char *b200_last_cuda_error (void);
int b200_version (void);
/* number of CUDA devices visible, or a negative b200_status */
int b200_device_count (void);

/* pinned host staging memory (what a GstCudaBufferPool-style pool hands upstream
 * so H2D/D2H can be asynchronous; gst-plugins-bad/gst-libs/gst/cuda/gstcudamemory.cpp:446-522) */
int b200_host_alloc (size_t size, void **ptr);            /* near the calling thread's current device */
int b200_host_free (void *ptr);
/* the same, placed on the NUMA node `device` hangs off (mbind before first touch, then cudaHostRegister): with one
 * pipeline per GPU on a multi-socket host the staging buffers must not cross the socket interconnect.
 * b200_device_numa_node: that node from sysfs, -1 if unknown. */
int b200_host_alloc_near (int device, size_t size, void **ptr);
int b200_device_numa_node (int device);

/* ------------------------------------------------------------------ video types */
/* GstVideoFormat values (gst-libs/gst/video/video-format.h:195-) */
typedef enum {
  B200_VIDEO_FORMAT_I420 = 2, B200_VIDEO_FORMAT_YV12 = 3,
  B200_VIDEO_FORMAT_YUY2 = 4, B200_VIDEO_FORMAT_UYVY = 5, B200_VIDEO_FORMAT_Y42B = 18, B200_VIDEO_FORMAT_YVYU = 19,
  B200_VIDEO_FORMAT_Y444 = 20,   /* 4:2:2 / 4:4:4 inputs (capture formats) -> packed RGB: opt-in, see DESIGN.md */
  B200_VIDEO_FORMAT_RGBx = 7, B200_VIDEO_FORMAT_BGRx = 8, B200_VIDEO_FORMAT_xRGB = 9,
  B200_VIDEO_FORMAT_xBGR = 10, B200_VIDEO_FORMAT_RGBA = 11, B200_VIDEO_FORMAT_BGRA = 12,
  B200_VIDEO_FORMAT_ARGB = 13, B200_VIDEO_FORMAT_ABGR = 14,
  B200_VIDEO_FORMAT_NV12 = 23, B200_VIDEO_FORMAT_NV21 = 24,
  /* compositor formats only (blend.c PLANAR_YUV_BLEND at 10 / 12 / 16 bits, little endian; Y444 and Y42B above are
   * compositor formats too) */
  B200_VIDEO_FORMAT_I420_10LE = 43, B200_VIDEO_FORMAT_I422_10LE = 45, B200_VIDEO_FORMAT_Y444_10LE = 47,
  B200_VIDEO_FORMAT_I420_12LE = 73, B200_VIDEO_FORMAT_I422_12LE = 75, B200_VIDEO_FORMAT_Y444_12LE = 77,
  B200_VIDEO_FORMAT_Y444_16LE = 88
} b200_video_format;

/* GstVideoScaleMethod of the element (gst/videoconvertscale/gstvideoconvertscale.h:59-71) */
typedef enum {
  B200_SCALE_NEAREST = 0, B200_SCALE_BILINEAR, B200_SCALE_4TAP, B200_SCALE_LANCZOS,
  B200_SCALE_BILINEAR2, B200_SCALE_SINC, B200_SCALE_HERMITE, B200_SCALE_SPLINE,
  B200_SCALE_CATROM, B200_SCALE_MITCHELL
} b200_scale_method;

/* GstVideoColorMatrix / GstVideoColorRange / GstVideoChromaSite (video-color.h:40-83, video-chroma.h:43-52) */
enum { B200_COLOR_MATRIX_UNKNOWN = 0, B200_COLOR_MATRIX_RGB = 1, B200_COLOR_MATRIX_FCC = 2,
  B200_COLOR_MATRIX_BT709 = 3, B200_COLOR_MATRIX_BT601 = 4, B200_COLOR_MATRIX_SMPTE240M = 5,
  B200_COLOR_MATRIX_BT2020 = 6 };
enum { B200_COLOR_RANGE_UNKNOWN = 0, B200_COLOR_RANGE_0_255 = 1, B200_COLOR_RANGE_16_235 = 2 };
enum { B200_CHROMA_SITE_UNKNOWN = 0, B200_CHROMA_SITE_NONE = 1, B200_CHROMA_SITE_H_COSITED = 2,
  B200_CHROMA_SITE_V_COSITED = 4, B200_CHROMA_SITE_ALT_LINE = 8 };

#define B200_VIDEO_MAX_PLANES 4

/* The subset of GstVideoInfo the arithmetic depends on (gst-libs/gst/video/video-info.h:399-438).
 * stride/offset are per PLANE, in bytes, offset relative to the frame base pointer —
 * arbitrary values are honoured (GstCudaMemory uses a common pitch for all planes,
 * gst-plugins-bad/gst-libs/gst/cuda/gstcudamemory.cpp:194-345). */
typedef struct {
  int32_t format;                /* b200_video_format */
  int32_t width, height;
  int32_t stride[B200_VIDEO_MAX_PLANES];
  uint64_t offset[B200_VIDEO_MAX_PLANES];
  int32_t color_matrix;          /* 0 = default by height, like gst_video_info_set_format */
  int32_t color_range;           /* 0 = default */
  int32_t chroma_site;           /* 0 = default by height, like gst_video_info_from_caps */
} b200_video_info;

/* fill default system-memory layout + caps-default colorimetry for (format, w, h);
 * replaces gst_video_info_set_format (video-info.c:292) for the supported formats */
int b200_video_info_set_format (b200_video_info * info, int format, int width, int height);
/* total bytes of one frame with this layout (GstVideoInfo.size) */
size_t b200_video_info_size (const b200_video_info * info);

/* the videoconvertscale properties that reach the converter
 * (gstvideoconvertscale.c:130-144 defaults, :991-1087 option mapping) */
typedef struct {
  int32_t method;                /* b200_scale_method; element default BILINEAR */
  double envelope;               /* 2.0 */
  double sharpness;              /* 1.0 */
  double sharpen;                /* 0.0 */
  /* GST_VIDEO_CONVERTER_OPT_DEST_X/Y/WIDTH/HEIGHT as the element sets them for add-borders
   * (gstvideoconvertscale.c:926-952, :1068-1072): the input is scaled into this rectangle of the output frame and
   * the rest is filled with border_argb.  dest_width == 0 or dest_height == 0: the whole frame, no border.
   * For 4:2:0 outputs dest_x / dest_y are rounded down to even (video-converter.c:2335-2336). */
  int32_t dest_x, dest_y, dest_width, dest_height;
  uint32_t border_argb;          /* GST_VIDEO_CONVERTER_OPT_BORDER_ARGB, default 0xff000000 */
  int32_t fill_border;           /* GST_VIDEO_CONVERTER_OPT_FILL_BORDER, default 1 */
  int32_t reserved[2];
} b200_vcs_config;
void b200_vcs_config_init (b200_vcs_config * cfg);

typedef struct b200_vcs b200_vcs;

/* Build the per-caps plan (tap tables, matrix, chroma pairing, tiling) and upload it.
 * Format pairs (anything else: B200_ERR_UNSUPPORTED):
 *   NV12 / NV21 / I420 / YV12      -> the eight 4-byte RGB orders, or NV12 / NV21 / I420 / YV12
 *   the eight 4-byte RGB orders    -> the eight 4-byte RGB orders, or NV12 / NV21 / I420 / YV12
 *   YUY2 / UYVY / YVYU             -> the eight 4-byte RGB orders, or NV12 / NV21 / I420 / YV12
 *   Y42B / Y444                    -> the eight 4-byte RGB orders, or NV12 / NV21 / I420 / YV12
 * A YUV -> YUV pair must name the same colour matrix on both sides (what the element's caps fixation produces).
 * device >= 0: CUDA device ordinal (the element's cuda-device-id property,
 * gst-plugins-bad/sys/nvcodec/gstcudabasetransform.c:89-90).
 * device == -1: host-side plan only (no CUDA calls; convert() then fails with
 * B200_ERR_NO_DEVICE) — used by caps negotiation dry-runs and CPU-only tests. */
int b200_vcs_create (const b200_video_info * in, const b200_video_info * out,
    const b200_vcs_config * cfg, int device, b200_vcs ** handle);
void b200_vcs_destroy (b200_vcs * h);

/* one frame, device memory, asynchronous on cuda_stream. in_frame/out_frame are the
 * frame BASE device pointers; planes live at base + info.offset[i].
 * A handle serves one stream at a time (the element's streaming thread): kernel_variant 5 keeps per-handle
 * scratch images between its two launches. */
int b200_vcs_convert (b200_vcs * h, const void *in_frame, void *out_frame, void *cuda_stream);
/* n independent frames (same caps) in one launch: what a batching element / multi-stream
 * mux feeds; n <= B200_VCS_MAX_BATCH.  Slot i reads in_frames[i] and writes out_frames[i] only.
 *
 * Frame placement (b200_vcs_convert and _batch alike):
 *   - packed RGB outputs are written in 32-bit words: the frame base, info.offset[0] and info.stride[0] must be
 *     multiples of 4.  b200_vcs_create refuses such an offset or stride, convert such a base, with
 *     B200_ERR_INVALID_ARG before anything is written.
 *   - packed RGB inputs: the same rule (refused the same way) wherever the conversion has a YUV output.
 *   - any other base, offset and stride is accepted and gives the same bytes.  The fast kernels need more
 *     (the exact-2:1 kernels 8-byte aligned YUV planes, the plane and 4:2:0 packing kernels 4- or 8-byte
 *     aligned frames); a batch in which any frame falls short runs a kernel that reads and writes bytes.
 *     Device allocations (cudaMalloc, the torch caching allocator) are 256-byte aligned and always take the
 *     fast kernels. */
#define B200_VCS_MAX_BATCH 64
int b200_vcs_convert_batch (b200_vcs * h, int n, const void *const *in_frames,
    void *const *out_frames, void *cuda_stream);
/* system-memory peers: host frames in, host frames out.  H2D / kernel / D2H are
 * pipelined over internal device frame slots on side streams; returns when all n
 * outputs are complete in host memory.  Host buffers should come from
 * b200_host_alloc (pinned) for the copies to overlap. */
int b200_vcs_convert_host (b200_vcs * h, int n, const void *const *in_host,
    void *const *out_host);
/* diagnostic: the host<->device copies of b200_vcs_convert_host alone (both directions in flight, no kernel; the
 * outputs receive whatever the device slots hold).  Timed by the caller it is the link's ceiling for the same call. */
int b200_vcs_copy_probe (b200_vcs * h, int n, const void *const *in_host, void *const *out_host);

/* plan introspection (tests, debugging, gst-inspect style dumps) */
typedef struct {
  int32_t h_taps, v_taps;        /* 0 = no scaling in that direction */
  int32_t h_first;               /* 1: horizontal pass before vertical */
  int32_t matrix_first;          /* 1: matrix before scaling (net upscale) */
  int32_t p[5];                  /* AYUV->ARGB mulhi parameters p1..p5 */
  int32_t tile_w, tile_h;        /* generic kernel output tile */
  int32_t smem_bytes;
  int32_t kernel_variant;        /* 0 = generic tiled, 1 = lanczos 2:1 specialised, 2 = light (copy / 2-tap axes), 3 = n-tap any ratio, 4 = YUV plane scaling,
                                  * 5 = chain + chroma down-sampling (4:2:0 -> the other 4:2:0 family; 2 launches),
                                  * 6 = lanczos 2:1 with mma.sync FIRs (cross-check only: set_kernel_variant; measured slower),
                                  * 7 = lanczos 2:1 with both FIR passes as tcgen05.mma.kind::i8 banded products, accumulators in TMEM
                                  *     (bit-exact; set_kernel_variant(7) or B200_L2_TC=1 - not the default, see DESIGN.md) */
  int32_t n_launches_per_convert;
} b200_vcs_plan_info;
int b200_vcs_get_plan_info (const b200_vcs * h, b200_vcs_plan_info * info);
/* copy out the integer tap tables: dir 0 = horizontal, 1 = vertical.
 * offsets[out_size], taps[out_size * n_taps] (int16) */
int b200_vcs_get_taps (const b200_vcs * h, int dir, uint32_t * offsets, int16_t * taps,
    size_t offsets_len, size_t taps_len);
/* the x256 integer colour matrix of the plan (prepare_matrix, video-converter.c:1324-1370), row-major 4x4: YUV -> RGB
 * for RGB outputs, RGB -> YUV for a packed RGB input; all zero for plans without a matrix stage */
int b200_vcs_get_matrix (const b200_vcs * h, int32_t im[16]);
/* per input line chroma pairing mode (0 own row, 1 first of pair, 2 second of pair) */
int b200_vcs_get_chroma_plan (const b200_vcs * h, uint8_t * mode, size_t len);
/* force a kernel variant (0 generic, 1-3 the fast kernels, 6 the tensor-path 2:1 kernel, each if eligible); for A/B tests */
int b200_vcs_set_kernel_variant (b200_vcs * h, int variant);
/* name of the __global__ function b200_vcs_convert launches for this handle (what a profiler's launch list shows) */
const char *b200_vcs_kernel_name (const b200_vcs * h);

/* ------------------------------------------------------------------ compositor */
typedef enum { B200_COMP_BG_CHECKER = 0, B200_COMP_BG_BLACK = 1, B200_COMP_BG_WHITE = 2,
  B200_COMP_BG_TRANSPARENT = 3 } b200_comp_background;      /* compositor.c:742 */
typedef enum { B200_COMP_OP_SOURCE = 0, B200_COMP_OP_OVER = 1, B200_COMP_OP_ADD = 2 } b200_comp_operator;

/* one sink pad's prepared frame + its pad properties (compositor.c:190-196) */
typedef struct {
  const void *data;              /* device pointer to the pad's packed 4x8-bit frame */
  int32_t width, height, stride;
  int32_t xpos, ypos;
  double alpha;                  /* pad alpha 0.0..1.0 */
  int32_t op;                    /* b200_comp_operator */
  int32_t reserved;
} b200_comp_pad;

typedef struct b200_comp b200_comp;
#define B200_COMP_MAX_PADS 64
/* out_format: a packed 8-bit RGB format with alpha (RGBA/BGRA/ARGB/ABGR; b200_comp_blend) or a 4:2:0 YUV format
 * (I420/YV12/NV12/NV21; b200_comp_blend_yuv) */
int b200_comp_create (int out_format, int width, int height, int device, b200_comp ** handle);
void b200_comp_destroy (b200_comp * h);
/* background fill + every pad in z-order in ONE pass over the destination.
 * pads[] is in sink-pad (z) order, lowest first.  Pads with alpha 0 are skipped and
 * fully obscured pads give the same bytes as the reference's culling (compositor.c:519-601). */
int b200_comp_blend (b200_comp * h, void *dst, int32_t dst_stride, int background,
    const b200_comp_pad * pads, int n_pads, void *cuda_stream);

/* System-memory peers (what GstVideoAggregator hands a compositor without cudaupload in front): pads[].data are HOST
 * pointers (pinned by b200_host_alloc for the copies to be asynchronous), dst_host receives the frame.
 * _submit queues upload -> blend -> download on the handle's own three streams over a ring of 3 device slots and
 * returns at once; _wait (h, k) returns when all but the k most recent submissions are complete in host memory
 * (k = 1: push frame n-1 downstream while frame n is in flight - no per-buffer device synchronisation);
 * b200_comp_blend_host = _submit + _wait (h, 0).  Host buffers of a submission must stay untouched until it completed. */
int b200_comp_blend_host_submit (b200_comp * h, void *dst_host, int32_t dst_stride, int background,
    const b200_comp_pad * pads, int n_pads);
int b200_comp_blend_host_wait (b200_comp * h, int keep_in_flight);
int b200_comp_blend_host (b200_comp * h, void *dst_host, int32_t dst_stride, int background,
    const b200_comp_pad * pads, int n_pads);

/* 4:2:0 output (I420, YV12, NV12, NV21 given to b200_comp_create): blend.c PLANAR_YUV_BLEND / NV_YUV_BLEND.
 * Every pad frame has the OUTPUT's format (the aggregator converts pads that differ, see INTEGRATION.md);
 * plane strides / offsets of the destination and of every pad come from their b200_video_info. */
typedef struct {
  const void *data;              /* device pointer to the pad's frame */
  b200_video_info info;          /* format (== output format), width, height, plane layout */
  int32_t xpos, ypos;
  double alpha;
  int32_t op;                    /* b200_comp_operator: SOURCE copies, OVER and ADD blend with the pad alpha */
  int32_t reserved;
} b200_comp_pad_yuv;
/* dst_info->color_range picks the black / white background levels (16..235 unless B200_COLOR_RANGE_0_255) */
int b200_comp_blend_yuv (b200_comp * h, void *dst, const b200_video_info * dst_info, int background,
    const b200_comp_pad_yuv * pads, int n_pads, void *cuda_stream);
/* system-memory peers of the YUV compositor: pad frames and the destination are HOST buffers laid out as their
 * b200_video_info says (b200_video_info_size bytes each); same device ring, streams and _wait as b200_comp_blend_host_submit
 * (gstcudamemorycopy.c's role folded into the element).  The destination's stride padding is preserved. */
int b200_comp_blend_yuv_host_submit (b200_comp * h, void *dst_host, const b200_video_info * dst_info, int background,
    const b200_comp_pad_yuv * pads, int n_pads);
int b200_comp_blend_yuv_host (b200_comp * h, void *dst_host, const b200_video_info * dst_info, int background,
    const b200_comp_pad_yuv * pads, int n_pads);

/* ------------------------------------------------------------------ audio resampler */
typedef struct b200_ars b200_ars;
/* GstAudioFormat values (gst-libs/gst/audio/audio-format.h:97-140) of the sample formats audioresample hands to
 * its resampler unconverted (audio-converter.c:700-727), native (little) endian */
enum { B200_AUDIO_FORMAT_S16LE = 4, B200_AUDIO_FORMAT_S32LE = 12, B200_AUDIO_FORMAT_F32LE = 28,
  B200_AUDIO_FORMAT_F64LE = 30 };
typedef struct {
  int32_t in_rate, out_rate, channels;
  int32_t quality;               /* 0..10, element default 4 (gstaudioresample.c:68) */
  int32_t format;                /* B200_AUDIO_FORMAT_*; 0 = F32LE */
  /* the element's resample-method / sinc-filter-mode / sinc-filter-interpolation properties (gstaudioresample.c:160-186).
   * 0 = the element default in each; other values are the reference's enum value + 1 so that a zeroed config is the
   * default configuration: */
  int32_t resample_method;       /* 0 or B200_ARS_METHOD_KAISER; any B200_ARS_METHOD_* */
  int32_t sinc_filter_mode;      /* 0 or B200_ARS_FILTER_MODE_AUTO; _INTERPOLATED; _FULL */
  int32_t sinc_filter_interpolation;     /* 0 or B200_ARS_FILTER_INTERPOLATION_CUBIC; _NONE; _LINEAR */
  int32_t reserved[4];
} b200_ars_config;
enum { B200_ARS_METHOD_NEAREST = 1, B200_ARS_METHOD_LINEAR = 2, B200_ARS_METHOD_CUBIC = 3,
  B200_ARS_METHOD_BLACKMAN_NUTTALL = 4, B200_ARS_METHOD_KAISER = 5 };
enum { B200_ARS_FILTER_MODE_INTERPOLATED = 1, B200_ARS_FILTER_MODE_FULL = 2, B200_ARS_FILTER_MODE_AUTO = 3 };
enum { B200_ARS_FILTER_INTERPOLATION_NONE = 1, B200_ARS_FILTER_INTERPOLATION_LINEAR = 2,
  B200_ARS_FILTER_INTERPOLATION_CUBIC = 3 };

int b200_ars_create (const b200_ars_config * cfg, int device, b200_ars ** handle);
void b200_ars_destroy (b200_ars * h);
/* discard history (flush / discont), gst_audio_resampler_reset */
int b200_ars_reset (b200_ars * h);
/* rate change on a live stream (gst_audio_resampler_update as audioresample drives it, audio-resampler.c:1503): the filter
 * is re-designed for the new rates, the phase is rescaled, the history follows the tap count - no samples are lost and no
 * reset happens.  A rate <= 0 keeps the current one.  Synchronises the device (rate changes are rare events). */
int b200_ars_update (b200_ars * h, int in_rate, int out_rate);
/* frames the next process() call will produce for in_frames of input */
size_t b200_ars_get_out_frames (b200_ars * h, size_t in_frames);
size_t b200_ars_get_in_frames (b200_ars * h, size_t out_frames);
size_t b200_ars_get_max_latency (b200_ars * h);
/* Interleaved device buffers of the configured sample format.  in == NULL feeds silence (drain).
 * Consumes all in_frames, writes b200_ars_get_out_frames() frames, asynchronous on cuda_stream. */
int b200_ars_process (b200_ars * h, const void *in, size_t in_frames, void *out,
    size_t out_capacity_frames, size_t * out_frames, void *cuda_stream);
/* System-memory peers (an audioresample between system-memory elements): in_host / out_host are HOST buffers (pinned by
 * b200_host_alloc for the copies to be asynchronous).  _submit queues upload -> resample -> download on the handle's own
 * three streams over a ring of 3 device slots, returns the frame count at once (it only depends on the stream position);
 * _wait (h, k) returns when all but the k most recent submissions are complete in host memory (k = 1: push buffer n-1
 * while buffer n is in flight); b200_ars_process_host = _submit + _wait (h, 0).  Do not mix with b200_ars_process on
 * another stream without synchronising: the history lives on the handle. */
int b200_ars_process_host_submit (b200_ars * h, const void *in_host, size_t in_frames, void *out_host,
    size_t out_capacity_frames, size_t * out_frames);
int b200_ars_process_host_wait (b200_ars * h, int keep_in_flight);
int b200_ars_process_host (b200_ars * h, const void *in_host, size_t in_frames, void *out_host,
    size_t out_capacity_frames, size_t * out_frames);
typedef struct { int32_t n_taps, n_phases, in_step, out_step, filter_mode, oversample; } b200_ars_plan_info;
int b200_ars_get_plan_info (const b200_ars * h, b200_ars_plan_info * info);
int b200_ars_get_phase_taps (const b200_ars * h, int phase, float *taps, size_t len);

#ifdef __cplusplus
}
#endif
#endif /* B200DSP_H */
