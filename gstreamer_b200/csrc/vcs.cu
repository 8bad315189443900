// gstreamer_b200/csrc/vcs.cu — b200_vcs_* entry points (product code).
//
// Replaces gst_video_converter_new/_frame/_free for the element's transform_frame()
// (gst-plugins-base/gst/videoconvertscale/gstvideoconvertscale.c:1981-2005); device
// calling convention after gst_cuda_converter_convert_frame
// (gst-plugins-bad/gst-libs/gst/cuda/gstcudaconverter.cpp:1911).
#include "common.h"
#include "vcs_plan.h"
#include "vcs_device.h"
#include "vcs_kernels.cuh"
#include "vcs_lanczos2.cuh"
#include "vcs_lanczos2_v2.cuh"
#include "vcs_l2mma.cuh"
#ifndef B200_CUDA_EMU
#include "vcs_l2tc.cuh"          // tcgen05 / TMEM: no host emulation
#endif
#include "vcs_light.cuh"
#include "vcs_ntap.cuh"
#include "vcs_planes.cuh"
#include "vcs_down420.cuh"
#include "vcs_rgb420.cuh"
#include "vcs_yuy2_420.cuh"

#include <string.h>
#include <new>
#include <vector>

using namespace b200;

struct b200_vcs {
  VcsPlan plan;
  int device = -1;
  VcsDev dev;                     // kernel parameter block (device pointers inside)
  int variant = 0;
  // device tables
  uint32_t *d_hoff = nullptr, *d_voff = nullptr;
  int16_t *d_hcoef = nullptr, *d_vcoef = nullptr, *d_hsum = nullptr, *d_vsum = nullptr;
  uint8_t *d_cmode = nullptr;
  // host<->device pipeline for system-memory peers
  static const int kSlots = 4, kChunk = 4;
  uint8_t *slot_in[kSlots] = {nullptr}, *slot_out[kSlots] = {nullptr};
  cudaStream_t s_h2d = nullptr, s_run = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_in[kSlots] = {nullptr}, ev_run[kSlots] = {nullptr}, ev_out[kSlots] = {nullptr};
  bool pipeline_ready = false;
  int slot_frames = 0;            // frames each slot holds (one kernel launch per slot-full)
  Lanczos2Tables l2_tables;
  Lanczos2State l2;
  Lanczos2V2Tables l2v2_tables;      // second form of the headline kernel (vcs_lanczos2_v2.cuh) where the plan allows it
  Lanczos2V2State l2v2;
  NtapState ntap;
  L2mmaTables mma_tables;         // experimental tensor-path variant of the 2:1 kernel (variant 6, opt-in)
  L2mmaState mma;
#ifndef B200_CUDA_EMU
  L2tcTables tc_tables;           // tcgen05 formulation of the 2:1 kernel (variant 7)
  L2tcState tc;
#endif
  PlanesState planes;
  // 4:2:0 -> other 4:2:0 family: scaled A,Y,U,V scratch images between the two launches
  Down420Dev down;
  BorderDev border;               // destination rectangle: what to fill around it
  uint8_t *d_scratch = nullptr;
  int scratch_frames = 0;
  size_t scratch_frame_bytes = 0;
  // packed RGB -> 4:2:0 at an unchanged or shrinking size: [word-wide scaler on 4-byte pixels ->] matrix + down-sample + pack
  Rgb420Dev rgb420;
  Rgb2AyuvDev rgb2ayuv;           // the frame grows: the matrix runs first, on its own
  Yuy2AyuvDev yuy2ayuv;           // packed 4:2:2 input: unpack + horizontal chroma up-sampling, on its own
  bool rgb420_ok = false, rgb420_scaled = false;
  int rgb420_pre = 0;             // 0: none, 1: vcs_rgb2ayuv_kernel, 2: vcs_yuy2_ayuv_kernel
  PlaneFastState rgb420_scaler;
  Yuy2Dev yuy2;                   // YUY2 / UYVY -> I420 / YV12 at an unchanged size (plan.yuy2_420)
  size_t in_bytes = 0, out_bytes = 0;
};

namespace {

size_t frame_bytes (const b200_video_info & i)
{
  return b200_video_info_size (&i);
}

int upload_axis (const AxisPlan & a, uint32_t **off, int16_t **coef, int16_t **sum, AxisDev * d)
{
  int st;
  if ((st = upload (off, a.offset.data (), a.offset.size ())) != B200_OK) return st;
  if ((st = upload (coef, a.coef.data (), a.coef.size ())) != B200_OK) return st;
  if ((st = upload (sum, a.sum.data (), a.sum.size ())) != B200_OK) return st;
  d->offset = *off; d->coef = *coef; d->sum = *sum;
  d->mode = a.mode; d->n_taps = a.n_taps; d->coef_per_out = a.coef_per_out; d->span = a.span;
  d->out_size = a.out_size; d->in_size = a.in_size;
  return B200_OK;
}

int launch_convert (b200_vcs * h, int n, const VcsBatch & batch, cudaStream_t stream);

// the exact-2:1 kernels load luma and semi-planar chroma as 64-bit words (the plan holds plane offsets and strides to
// multiples of 8); a batch with any frame off an 8-byte boundary runs the generic kernel, whose YUV input path reads bytes
bool in_dword_aligned (const VcsBatch & batch, int n)
{
  for (int i = 0; i < n; i++) if (((uintptr_t) batch.in[i]) & 7) return false;
  return true;
}

// packed RGB -> 4:2:0 with every scaler in front of the matrix (the frame does not grow) and no destination rectangle:
// vcs_rgb420.cuh.  Leaves rgb420_ok false (the generic chain runs) for what the fast kernels decline.
int prepare_rgb420 (b200_vcs * h)
{
  const VcsPlan & p = h->plan;
  h->rgb420_ok = false;
  const bool packed422 = p.in_422_444 && p.ystep == 2;            // YUY2 / UYVY / YVYU
  if (!(p.rgb_in || packed422) || !p.yuv_out || p.yuy2_420 || getenv ("B200_RGB420_GENERIC")) return B200_OK;
  Rgb420Dev & r = h->rgb420;
  memset (&r, 0, sizeof (r));
  if (p.rgb_in) {
    const int pos_r = p.in_sel & 0xf, pos_g = (p.in_sel >> 4) & 0xf, pos_b = (p.in_sel >> 8) & 0xf;
    for (int i = 0; i < 3; i++) {
      if (!rgb420_split_row (p.m_rgb2yuv[i], pos_r, pos_g, pos_b, &r.ca[i], &r.cb[i])) return B200_OK;
      r.off[i] = p.m_rgb2yuv[i][3];
    }
  } else if ((p.in.stride[0] & 3) || (p.in.offset[0] & 3)) return B200_OK;      // pixel pairs are read as words
  const Down420Dev & q = h->down;
  r.ow = q.ow; r.oh = q.oh; r.hmode = q.hmode; r.vavg = q.vavg;
  r.stride_y = q.stride_y; r.stride_u = q.stride_u; r.stride_v = q.stride_v; r.cstep = q.cstep;
  r.off_y = q.off_y; r.off_u = q.off_u; r.off_v = q.off_v;
  const unsigned long long cbase = q.cstep == 2 ? std::min (q.off_u, q.off_v) : (q.off_u | q.off_v);
  r.wvec = ((q.stride_y | q.stride_u | q.stride_v) & 3) == 0 && ((q.off_y | cbase) & 3) == 0;
  h->rgb420_scaled = p.h.scaling || p.v.scaling;
  // a kernel of its own in front of the scalers: the RGB -> YUV matrix when the frame grows (chain_scale puts the
  // scalers behind it), unpack + horizontal chroma up-sampling for packed 4:2:2
  h->rgb420_pre = packed422 ? 2 : (p.matrix_first && h->rgb420_scaled) ? 1 : 0;
  int in_stride = p.in.stride[0];
  unsigned long long in_off = p.in.offset[0];
  if (h->rgb420_pre) {
    const int dstride = (p.in.width * 4 + 15) & ~15;
    if (h->rgb420_pre == 1) {
      Rgb2AyuvDev & m = h->rgb2ayuv;
      memset (&m, 0, sizeof (m));
      m.w = p.in.width; m.h = p.in.height; m.sstride = p.in.stride[0]; m.soff = p.in.offset[0]; m.dstride = dstride;
      for (int i = 0; i < 3; i++) { m.ca[i] = r.ca[i]; m.cb[i] = r.cb[i]; m.off[i] = r.off[i]; }
    } else {
      Yuy2AyuvDev & m = h->yuy2ayuv;
      memset (&m, 0, sizeof (m));
      m.w = p.in.width; m.h = p.in.height; m.sstride = p.in.stride[0]; m.soff = p.in.offset[0]; m.dstride = dstride;
      // byte positions inside a pixel-pair word, from the plan's sample offsets (YUY2: Y0 U Y1 V; UYVY: U Y0 V Y1; YVYU: Y0 V Y1 U)
      m.ypos = (int) (p.in_off_y - p.in.offset[0]); m.upos = (int) (p.in_off_u - p.in.offset[0]); m.vpos = (int) (p.in_off_v - p.in.offset[0]);
      m.cosited = p.h_cosited ? 1 : 0;
    }
    in_stride = dstride; in_off = 0;
  }
  if (!h->rgb420_scaled) {
    r.sstride = in_stride; r.soff = in_off;
    r.svec = (r.sstride & 15) == 0 && (r.soff & 15) == 0;
  } else {
    PlanePlan pl;
    pl.src_plane = 0; pl.iw = p.in.width; pl.ih = p.in.height; pl.ow = p.out.width; pl.oh = p.out.height;
    pl.ne = 4; pl.swz = 0; pl.mode = PM_SCALE;
    pl.have_h = p.h.scaling; pl.have_v = p.v.scaling; pl.h_first = p.h_first;
    pl.h = p.h; pl.v = p.v;
    const int sstride = (p.out.width * 4 + 15) & ~15;
    std::vector<int32_t> hp, vp;
    if (!plan_plane_fast (pl, in_stride, in_off, sstride, 0, &h->rgb420_scaler, &hp, &vp)) return B200_OK;
    const int st = prepare_plane_fast (pl, hp, vp, &h->rgb420_scaler);
    if (st != B200_OK) return st;
    r.sstride = sstride; r.soff = 0; r.svec = 1;
  }
  h->rgb420_ok = true;
  return B200_OK;
}

int launch (b200_vcs * h, int n, const VcsBatch & batch, cudaStream_t stream)
{
  const VcsPlan & p = h->plan;
  // every kernel that writes packed RGB stores whole 32-bit pixels: refuse a frame off a 4-byte boundary before
  // anything (the border fill included) touches it.  The plan builder already holds the plane offset and stride to it.
  if (p.frame_out.format >= B200_VIDEO_FORMAT_RGBx && p.frame_out.format <= B200_VIDEO_FORMAT_ABGR)
    for (int i = 0; i < n; i++) if (((uintptr_t) batch.out[i]) & 3) return B200_ERR_INVALID_ARG;
  if (p.has_dest && p.fill_border) {
    // border and rectangle are disjoint byte sets: the fill simply goes first on the same stream
    BorderBatch b;
    int wmax = 0, hmax = 0;
    for (int i = 0; i < n; i++) b.out[i] = batch.out[i];
    for (int i = 0; i < h->border.n_planes; i++) {
      wmax = max (wmax, h->border.pl[i].pw); hmax = max (hmax, h->border.pl[i].ph);
    }
    dim3 grid ((wmax + 255) / 256, hmax, h->border.n_planes * n);
    vcs_border_kernel <<<grid, 256, 0, stream>>> (h->border, b);
    B200_CUDA_TRY (cudaGetLastError ());
  }
  return launch_convert (h, n, batch, stream);
}

int launch_convert (b200_vcs * h, int n, const VcsBatch & batch, cudaStream_t stream)
{
  const VcsPlan & p = h->plan;
  if (p.planes_mode) {
    bool aligned = true;                                            // the word-wide halve / copy path needs 8-byte aligned frames
    for (int i = 0; i < n; i++) aligned = aligned && ((((uintptr_t) batch.in[i]) | ((uintptr_t) batch.out[i])) & 7) == 0;
    return launch_planes (h->planes, batch, n, stream, aligned);
  }
  if (h->variant == 6 && h->mma.ready) {
    bool aligned = true;                                            // 64-bit plane loads
    for (int i = 0; i < n; i++) aligned = aligned && (((uintptr_t) batch.in[i]) & 7) == 0 && (((uintptr_t) batch.out[i]) & 3) == 0;
    if (aligned) return launch_l2mma (h->dev, h->mma, batch, n, stream);
  }
#ifndef B200_CUDA_EMU
  if (h->variant == 7 && h->tc.ready) {
    bool aligned = true;                                            // 16-byte cp.async of the luma rows
    for (int i = 0; i < n; i++) aligned = aligned && (((uintptr_t) batch.in[i]) & 15) == 0 && (((uintptr_t) batch.out[i]) & 3) == 0;
    if (aligned) return launch_l2tc (h->dev, h->tc, batch, n, stream);
    if (p.lanczos2_ok && !p.planar && in_dword_aligned (batch, n)) return launch_lanczos2 (h->dev, h->l2, batch, n, stream);
  }
#endif
  if (h->variant == 1 && p.lanczos2_ok && !p.yuv_out && in_dword_aligned (batch, n)) {
    if (h->l2v2.ready && h->l2.x4) return launch_lanczos2_v2 (h->dev, h->l2, h->l2v2, batch, n, stream);
    if (!p.planar) return launch_lanczos2 (h->dev, h->l2, batch, n, stream);
  }
  if (h->variant == 2 && p.light_ok && !p.yuv_out) {
    // 32-bit plane loads: the frame itself must be word aligned (device allocations always are)
    bool aligned = true;
    for (int i = 0; i < n; i++) aligned = aligned && (((uintptr_t) batch.in[i]) & 3) == 0;
    if (aligned) return launch_light (h->dev, p, batch, n, stream);
  }
  if (h->variant == 3 && p.ntap_ok && !p.yuv_out) {
    bool aligned = true;
    for (int i = 0; i < n; i++) aligned = aligned && (((uintptr_t) batch.in[i]) & 3) == 0;
    if (aligned) return launch_ntap (h->dev, p, h->ntap, batch, n, stream);
  }
  dim3 grid ((p.out.width + p.tile_w - 1) / p.tile_w, (p.out.height + p.tile_h - 1) / p.tile_h, n);
  if (p.rgb_in)                                                    // packed pixels are read with 32-bit loads
    for (int i = 0; i < n; i++) if (((uintptr_t) batch.in[i]) & 3) return B200_ERR_INVALID_ARG;
  if (p.yuy2_420) {
    Yuy2Dev y = h->yuy2;
    Yuy2Batch b;
    for (int i = 0; i < n; i++) {
      b.src[i] = batch.in[i]; b.out[i] = batch.out[i];
      const uintptr_t a = (uintptr_t) batch.in[i];
      if ((a & 15) && y.svec > 1) y.svec = 1;
      if (a & 3) y.svec = 0;
      if (((uintptr_t) batch.out[i]) & 3) y.wvec = 0;
    }
    return launch_yuy2_420 (y, b, n, stream);
  }
  bool pairs_aligned = true;                                        // vcs_yuy2_ayuv_kernel reads pixel pairs as words
  if (h->rgb420_pre == 2)
    for (int i = 0; i < n; i++) pairs_aligned = pairs_aligned && (((uintptr_t) batch.in[i]) & 3) == 0;
  if (p.yuv_out && h->rgb420_ok && pairs_aligned) {
    Rgb420Dev r = h->rgb420;
    Rgb420Batch fin;
    for (int i = 0; i < n; i++) {
      fin.out[i] = batch.out[i];
      if (((uintptr_t) batch.out[i]) & 3) r.wvec = 0;
    }
    const int pre = h->rgb420_pre;
    const int pre_stride = pre == 1 ? h->rgb2ayuv.dstride : pre == 2 ? h->yuy2ayuv.dstride : 0;
    const size_t pre_bytes = (size_t) pre_stride * p.in.height;
    const size_t scaled_bytes = h->rgb420_scaled ? (size_t) r.sstride * p.out.height : 0;
    const size_t frame = pre_bytes + scaled_bytes;
    if (frame && (n > h->scratch_frames || frame != h->scratch_frame_bytes)) {
      B200_CUDA_TRY (cudaFree (h->d_scratch));                      // synchronises with launches still reading it
      h->d_scratch = nullptr; h->scratch_frames = 0;
      B200_CUDA_TRY (cudaMalloc ((void **) &h->d_scratch, frame * n));
      h->scratch_frames = n; h->scratch_frame_bytes = frame;
    }
    VcsBatch mid;                                                   // the scaler's view: in = the pre kernel's image or the frame
    for (int i = 0; i < n; i++) mid.in[i] = batch.in[i];
    if (pre) {
      Rgb420Batch pre_b;
      for (int i = 0; i < n; i++) { pre_b.src[i] = batch.in[i]; pre_b.out[i] = h->d_scratch + frame * i + scaled_bytes; mid.in[i] = pre_b.out[i]; }
      const int s0 = pre == 1 ? launch_rgb2ayuv (h->rgb2ayuv, pre_b, n, stream) : launch_yuy2_ayuv (h->yuy2ayuv, pre_b, n, stream);
      if (s0 != B200_OK) return s0;
    }
    if (h->rgb420_scaled) {
      for (int i = 0; i < n; i++) { mid.out[i] = h->d_scratch + frame * i; fin.src[i] = mid.out[i]; }
      const int s1 = launch_plane_fast (h->rgb420_scaler, mid, n, stream);
      if (s1 != B200_OK) return s1;
    } else {
      for (int i = 0; i < n; i++) {
        fin.src[i] = mid.in[i];
        if (((uintptr_t) mid.in[i]) & 15) r.svec = 0;
      }
    }
    return launch_rgb420 (r, fin, n, stream, pre == 0);
  }
  if (p.yuv_out) {
    // launch 1 writes the scaled pixels of every frame to its scratch image, launch 2 down-samples and packs
    const size_t frame = (size_t) h->down.stride_s * (p.out.height + (p.extra_row ? 1 : 0));
    if (n > h->scratch_frames || frame != h->scratch_frame_bytes) {
      B200_CUDA_TRY (cudaFree (h->d_scratch));                      // synchronises with launches still reading it
      h->d_scratch = nullptr; h->scratch_frames = 0;
      B200_CUDA_TRY (cudaMalloc ((void **) &h->d_scratch, frame * n));
      h->scratch_frames = n; h->scratch_frame_bytes = frame;
    }
    VcsBatch mid;
    Down420Batch fin;
    for (int i = 0; i < n; i++) {
      mid.in[i] = batch.in[i]; mid.out[i] = h->d_scratch + frame * i;
      fin.scratch[i] = mid.out[i]; fin.out[i] = batch.out[i];
    }
    // the chain up to the scaled pixels: the light / n-tap kernels (matrix stage off) where the plan allows, else the generic one
    bool word_aligned = true;
    for (int i = 0; i < n; i++) word_aligned = word_aligned && (((uintptr_t) batch.in[i]) & 3) == 0;
    static const bool slow_chain = getenv ("B200_CROSS_GENERIC") != nullptr;     // A/B knob
    if (!slow_chain && in_dword_aligned (batch, n) && h->variant == 1 && p.lanczos2_ok && h->l2v2.ready && h->l2.x4) {
      const int s = launch_lanczos2_v2 (h->dev, h->l2, h->l2v2, mid, n, stream);      // exact 2:1, 8 taps: the headline kernel without its matrix
      if (s != B200_OK) return s;
    } else if (!slow_chain && word_aligned && h->variant == 2 && p.light_ok) {
      const int s = launch_light (h->dev, p, mid, n, stream);
      if (s != B200_OK) return s;
    } else if (!slow_chain && word_aligned && h->variant == 3 && p.ntap_ok && h->ntap.ready) {
      const int s = launch_ntap (h->dev, p, h->ntap, mid, n, stream);
      if (s != B200_OK) return s;
    } else {
      vcs_generic_kernel <<<grid, 256, p.smem_bytes, stream>>> (h->dev, mid);
      B200_CUDA_TRY (cudaGetLastError ());
    }
    if (p.extra_row) {
      // scratch row `oh`: the chain over a one-line view of the frame (its last line, chroma row unfiltered vertically)
      VcsDev x = h->dev;
      x.off_y += (unsigned long long) (p.in.height - 1) * x.stride_y;
      x.off_u += (unsigned long long) ((p.in.height - 1) >> 1) * x.stride_u;
      x.off_v += (unsigned long long) ((p.in.height - 1) >> 1) * x.stride_v;
      x.ih = 1; x.oh = 1; x.v.in_size = x.v.out_size = 1;
      x.off_out = (unsigned long long) p.out.height * x.stride_out;
      dim3 gx (grid.x, 1, n);
      vcs_generic_kernel <<<gx, 256, p.smem_bytes, stream>>> (x, mid);
      B200_CUDA_TRY (cudaGetLastError ());
    }
    const int cw = (p.out.width + 1) / 2, chh = (p.out.height + 1) / 2;
    dim3 blk (32, 8), g2 ((cw + 31) / 32, (chh + 7) / 8, n);
    vcs_down420_kernel <<<g2, blk, 0, stream>>> (h->down, fin);
    B200_CUDA_TRY (cudaGetLastError ());
    return B200_OK;
  }
  vcs_generic_kernel <<<grid, 256, p.smem_bytes, stream>>> (h->dev, batch);
  B200_CUDA_TRY (cudaGetLastError ());
  return B200_OK;
}

int ensure_pipeline (b200_vcs * h, int chunk)
{
  if (h->pipeline_ready && chunk <= h->slot_frames) return B200_OK;
  h->in_bytes = frame_bytes (h->plan.in);
  h->out_bytes = frame_bytes (h->plan.frame_out);
  if (!h->pipeline_ready) {
    B200_CUDA_TRY (cudaStreamCreateWithFlags (&h->s_h2d, cudaStreamNonBlocking));
    B200_CUDA_TRY (cudaStreamCreateWithFlags (&h->s_run, cudaStreamNonBlocking));
    B200_CUDA_TRY (cudaStreamCreateWithFlags (&h->s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < b200_vcs::kSlots; i++) {
      B200_CUDA_TRY (cudaEventCreateWithFlags (&h->ev_in[i], cudaEventDisableTiming));
      B200_CUDA_TRY (cudaEventCreateWithFlags (&h->ev_run[i], cudaEventDisableTiming));
      B200_CUDA_TRY (cudaEventCreateWithFlags (&h->ev_out[i], cudaEventDisableTiming));
    }
    h->pipeline_ready = true;
  }
  // (re)size the slots: each holds `chunk` frames, so that one kernel launch and one event triple serve a whole chunk
  for (int i = 0; i < b200_vcs::kSlots; i++) {
    B200_CUDA_TRY (cudaFree (h->slot_in[i])); h->slot_in[i] = nullptr;       // cudaFree waits for work still using it
    B200_CUDA_TRY (cudaFree (h->slot_out[i])); h->slot_out[i] = nullptr;
  }
  h->slot_frames = 0;
  for (int i = 0; i < b200_vcs::kSlots; i++) {
    B200_CUDA_TRY (cudaMalloc ((void **) &h->slot_in[i], h->in_bytes * chunk));
    B200_CUDA_TRY (cudaMalloc ((void **) &h->slot_out[i], h->out_bytes * chunk));
  }
  h->slot_frames = chunk;
  return B200_OK;
}

}  // namespace

extern "C" {

void b200_vcs_config_init (b200_vcs_config * cfg)
{
  if (!cfg) return;
  memset (cfg, 0, sizeof (*cfg));
  cfg->method = B200_SCALE_BILINEAR;    // DEFAULT_PROP_METHOD, gstvideoconvertscale.c:130
  cfg->envelope = 2.0; cfg->sharpness = 1.0; cfg->sharpen = 0.0;
  cfg->border_argb = 0xff000000u; cfg->fill_border = 1;   // DEFAULT_OPT_FILL_BORDER / _BORDER_ARGB, video-converter.c:778, :782
}

int b200_video_info_set_format (b200_video_info * info, int format, int width, int height)
{
  if (!info || width < 1 || height < 1) return B200_ERR_INVALID_ARG;
  memset (info, 0, sizeof (*info));
  info->format = format; info->width = width; info->height = height;
  switch (format) {
    case B200_VIDEO_FORMAT_NV12: case B200_VIDEO_FORMAT_NV21:
      // video-info.c:1053-1063
      info->stride[0] = (width + 3) & ~3; info->stride[1] = info->stride[0];
      info->offset[0] = 0; info->offset[1] = (uint64_t) info->stride[0] * ((height + 1) & ~1);
      info->color_matrix = height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
      info->color_range = B200_COLOR_RANGE_16_235;
      info->chroma_site = height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
      return B200_OK;
    case B200_VIDEO_FORMAT_I420: case B200_VIDEO_FORMAT_YV12:
      // video-info.c:997-1009 (YV12: same layout, the format description swaps planes 1 and 2)
      info->stride[0] = (width + 3) & ~3;
      info->stride[1] = info->stride[2] = ((((width + 1) & ~1) / 2) + 3) & ~3;
      info->offset[0] = 0; info->offset[1] = (uint64_t) info->stride[0] * ((height + 1) & ~1);
      info->offset[2] = info->offset[1] + (uint64_t) info->stride[1] * (((height + 1) & ~1) / 2);
      info->color_matrix = height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
      info->color_range = B200_COLOR_RANGE_16_235;
      info->chroma_site = height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
      return B200_OK;
    case B200_VIDEO_FORMAT_YUY2: case B200_VIDEO_FORMAT_UYVY: case B200_VIDEO_FORMAT_YVYU:
    case B200_VIDEO_FORMAT_Y42B: case B200_VIDEO_FORMAT_Y444:
      if (format == B200_VIDEO_FORMAT_Y42B) {                      // video-info.c:1020-1029
        info->stride[0] = (width + 3) & ~3;
        info->stride[1] = info->stride[2] = ((width + 7) & ~7) / 2;
        info->offset[1] = (uint64_t) info->stride[0] * height;
        info->offset[2] = info->offset[1] + (uint64_t) info->stride[1] * height;
      } else if (format == B200_VIDEO_FORMAT_Y444) {               // :1030-1041
        info->stride[0] = info->stride[1] = info->stride[2] = (width + 3) & ~3;
        info->offset[1] = (uint64_t) info->stride[0] * height;
        info->offset[2] = info->offset[1] * 2;
      } else info->stride[0] = (width * 2 + 3) & ~3;               // :882-889
      info->color_matrix = height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
      info->color_range = B200_COLOR_RANGE_16_235;
      info->chroma_site = height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
      return B200_OK;
    case B200_VIDEO_FORMAT_RGBx: case B200_VIDEO_FORMAT_BGRx: case B200_VIDEO_FORMAT_xRGB:
    case B200_VIDEO_FORMAT_xBGR: case B200_VIDEO_FORMAT_RGBA: case B200_VIDEO_FORMAT_BGRA:
    case B200_VIDEO_FORMAT_ARGB: case B200_VIDEO_FORMAT_ABGR:
      info->stride[0] = width * 4;      // video-info.c:890-894
      info->color_matrix = B200_COLOR_MATRIX_RGB; info->color_range = B200_COLOR_RANGE_0_255;
      return B200_OK;
    case B200_VIDEO_FORMAT_I420_10LE: case B200_VIDEO_FORMAT_I420_12LE:       // video-info.c:1142-1156
    case B200_VIDEO_FORMAT_I422_10LE: case B200_VIDEO_FORMAT_I422_12LE: {     // :1157-1169
      const bool is420 = format == B200_VIDEO_FORMAT_I420_10LE || format == B200_VIDEO_FORMAT_I420_12LE;
      const int hh = (height + 1) & ~1;
      info->stride[0] = (width * 2 + 3) & ~3;
      info->stride[1] = info->stride[2] = (width + 3) & ~3;
      info->offset[1] = (uint64_t) info->stride[0] * hh;
      info->offset[2] = info->offset[1] + (uint64_t) info->stride[1] * (is420 ? hh / 2 : hh);
      info->color_matrix = height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
      info->color_range = B200_COLOR_RANGE_16_235;
      info->chroma_site = height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
      return B200_OK;
    }
    case B200_VIDEO_FORMAT_Y444_10LE: case B200_VIDEO_FORMAT_Y444_12LE: case B200_VIDEO_FORMAT_Y444_16LE:   // :1170-1188
      info->stride[0] = info->stride[1] = info->stride[2] = (width * 2 + 3) & ~3;
      info->offset[1] = (uint64_t) info->stride[0] * height;
      info->offset[2] = info->offset[1] * 2;
      info->color_matrix = height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
      info->color_range = B200_COLOR_RANGE_16_235;
      info->chroma_site = height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
      return B200_OK;
    default:
      return B200_ERR_UNSUPPORTED;
  }
}

size_t b200_video_info_size (const b200_video_info * info)
{
  if (!info) return 0;
  switch (info->format) {
    case B200_VIDEO_FORMAT_NV12: case B200_VIDEO_FORMAT_NV21:
      return (size_t) info->offset[1] + (size_t) info->stride[1] * (((info->height + 1) & ~1) / 2);
    case B200_VIDEO_FORMAT_I420: case B200_VIDEO_FORMAT_YV12: {
      const size_t ch = (size_t) (((info->height + 1) & ~1) / 2);
      const size_t e1 = (size_t) info->offset[1] + (size_t) info->stride[1] * ch;
      const size_t e2 = (size_t) info->offset[2] + (size_t) info->stride[2] * ch;
      return e1 > e2 ? e1 : e2;
    }
    case B200_VIDEO_FORMAT_Y42B: case B200_VIDEO_FORMAT_Y444:
    case B200_VIDEO_FORMAT_Y444_10LE: case B200_VIDEO_FORMAT_Y444_12LE: case B200_VIDEO_FORMAT_Y444_16LE:
      return (size_t) info->offset[2] + (size_t) info->stride[2] * info->height;
    case B200_VIDEO_FORMAT_I420_10LE: case B200_VIDEO_FORMAT_I420_12LE:
      return (size_t) info->offset[2] + (size_t) info->stride[2] * (((info->height + 1) & ~1) / 2);
    case B200_VIDEO_FORMAT_I422_10LE: case B200_VIDEO_FORMAT_I422_12LE:
      return (size_t) info->offset[2] + (size_t) info->stride[2] * ((info->height + 1) & ~1);
    default:
      return (size_t) info->offset[0] + (size_t) info->stride[0] * info->height;
  }
}

int b200_vcs_create (const b200_video_info * in, const b200_video_info * out,
    const b200_vcs_config * cfg, int device, b200_vcs ** handle)
{
  if (!handle) return B200_ERR_INVALID_ARG;
  *handle = nullptr;
  b200_vcs_config defcfg;
  if (!cfg) { b200_vcs_config_init (&defcfg); cfg = &defcfg; }
  b200_vcs *h = new (std::nothrow) b200_vcs ();
  if (!h) return B200_ERR_NOMEM;
  int st = build_vcs_plan (in, out, cfg, &h->plan);
  if (st != B200_OK) { delete h; return st; }
  if (h->plan.has_dest) {
    // per-plane rectangles: chroma planes use GST_VIDEO_FORMAT_INFO_SCALE_WIDTH / _HEIGHT (round up), :7209-7221
    const VcsPlan & q = h->plan;
    const b200_video_info & f = q.frame_out;
    BorderDev & b = h->border;
    memset (&b, 0, sizeof (b));
    const bool rgb = f.format >= B200_VIDEO_FORMAT_RGBx && f.format <= B200_VIDEO_FORMAT_ABGR;
    const bool planar = f.format == B200_VIDEO_FORMAT_I420 || f.format == B200_VIDEO_FORMAT_YV12;
    if (rgb) {
      b.n_planes = 1;
      b.pl[0] = BorderPlane {f.offset[0], f.stride[0], f.width, f.height, 4, q.dest[0], q.dest[1], q.dest[2], q.dest[3],
        (unsigned) q.border_px[0] | ((unsigned) q.border_px[1] << 8) | ((unsigned) q.border_px[2] << 16) | ((unsigned) q.border_px[3] << 24)};
    } else {
      const int cx = (q.dest[0] + 1) / 2, cy = (q.dest[1] + 1) / 2, cw = (q.dest[2] + 1) / 2, chh = (q.dest[3] + 1) / 2;
      const int CW = (f.width + 1) / 2, CH = (f.height + 1) / 2;
      b.pl[0] = BorderPlane {f.offset[0], f.stride[0], f.width, f.height, 1, q.dest[0], q.dest[1], q.dest[2], q.dest[3], (unsigned) q.border_yuv[0]};
      if (planar) {
        const int pu = f.format == B200_VIDEO_FORMAT_YV12 ? 2 : 1, pv = 3 - pu;
        b.n_planes = 3;
        b.pl[1] = BorderPlane {f.offset[pu], f.stride[pu], CW, CH, 1, cx, cy, cw, chh, (unsigned) q.border_yuv[1]};
        b.pl[2] = BorderPlane {f.offset[pv], f.stride[pv], CW, CH, 1, cx, cy, cw, chh, (unsigned) q.border_yuv[2]};
      } else {
        const unsigned u = (unsigned) q.border_yuv[1], v = (unsigned) q.border_yuv[2];
        b.n_planes = 2;
        b.pl[1] = BorderPlane {f.offset[1], f.stride[1], CW, CH, 2, cx, cy, cw, chh, f.format == B200_VIDEO_FORMAT_NV21 ? (v | (u << 8)) : (u | (v << 8))};
      }
    }
  }
  if (h->plan.planes_mode) {                                       // YUV -> same YUV family: plane scaling
    h->device = device;
    h->variant = 4;
    h->in_bytes = frame_bytes (h->plan.in); h->out_bytes = frame_bytes (h->plan.frame_out);
    if (device >= 0) {
      int ndev = b200_device_count ();
      if (ndev <= 0) { delete h; return ndev < 0 ? ndev : B200_ERR_NO_DEVICE; }
      if (device >= ndev) { delete h; return B200_ERR_INVALID_ARG; }
      DeviceGuard g (device);
      if (!g.ok) { delete h; return B200_ERR_CUDA; }
      if ((st = prepare_planes (h->plan, &h->planes)) != B200_OK) { b200_vcs_destroy (h); return st; }
    }
    *handle = h;
    return B200_OK;
  }
  if (h->plan.yuv_out && !h->plan.rgb_in && !h->plan.in_422_444 && !h->plan.has_dest) {
    // the chain's first launch may be the second form of the exact-2:1 kernel with its matrix stage off
    h->l2_tables = build_lanczos2_tables (h->plan);
    h->l2v2_tables = build_lanczos2_v2_tables (h->plan, h->l2_tables);
    h->plan.lanczos2_ok = h->l2_tables.ok && h->l2v2_tables.ok && !getenv ("B200_L2_V1") && !getenv ("B200_L2_X4") && !getenv ("B200_CROSS_GENERIC");
  }
  if (!h->plan.yuv_out && !h->plan.in_422_444) {
    h->l2_tables = build_lanczos2_tables (h->plan);
    h->l2v2_tables = build_lanczos2_v2_tables (h->plan, h->l2_tables);
    // planar (I420 / YV12) input exists in the second form of the kernel only
    h->plan.lanczos2_ok = h->l2_tables.ok && (!h->plan.planar || (h->l2v2_tables.ok && !getenv ("B200_L2_V1") && !getenv ("B200_L2_X4")));
    h->mma_tables = build_l2mma_tables (h->plan);
#ifndef B200_CUDA_EMU
    h->tc_tables = build_l2tc_tables (h->plan, h->l2_tables);
#endif
  }
  const VcsPlan & p = h->plan;
  h->device = device;
  // the kernel this plan will run (also reported for host-only handles: caps negotiation dry-runs, CPU tests)
  h->variant = h->plan.lanczos2_ok ? 1 : (h->plan.light_ok ? 2 : (h->plan.ntap_ok ? 3 : 0));
  if (device >= 0) {
    int ndev = b200_device_count ();
    if (ndev <= 0) { delete h; return ndev < 0 ? ndev : B200_ERR_NO_DEVICE; }
    if (device >= ndev) { delete h; return B200_ERR_INVALID_ARG; }
    DeviceGuard g (device);
    if (!g.ok) { delete h; return B200_ERR_CUDA; }
    VcsDev & d = h->dev;
    memset (&d, 0, sizeof (d));
    d.iw = p.in.width; d.ih = p.in.height; d.ow = p.out.width; d.oh = p.out.height;
    d.stride_y = p.in.stride[0]; d.stride_c = p.in.stride[1]; d.stride_out = p.out.stride[0];
    d.off_y = p.in.offset[0]; d.off_c = p.in.offset[1]; d.off_out = p.out.offset[0];
    d.u_index = p.u_index; d.h_cosited = p.h_cosited; d.v_pairs = p.v_pairs;
    d.planar = p.planar ? 1 : 0; d.chroma_nearest = p.chroma_nearest ? 1 : 0;
    if (p.planar) {
      d.off_u = p.in.offset[p.plane_u]; d.off_v = p.in.offset[p.plane_v];
      d.stride_u = p.in.stride[p.plane_u]; d.stride_v = p.in.stride[p.plane_v];
    } else {                                                      // interleaved pairs: both components walk the same rows
      d.off_u = p.in.offset[1] + p.u_index; d.off_v = p.in.offset[1] + (p.u_index ^ 1);
      d.stride_u = d.stride_v = p.in.stride[1];
    }
    d.cstep = p.planar ? 1 : 2;
    d.ystep = 1; d.chshift = 1; d.cvshift = 1;
    if (p.in_422_444) {                                           // capture formats: explicit sample geometry
      d.off_y = p.in_off_y; d.off_u = p.in_off_u; d.off_v = p.in_off_v;
      d.stride_u = p.in_stride_u; d.stride_v = p.in_stride_v; d.cstep = p.cstep_in;
      d.ystep = p.ystep; d.chshift = p.chshift; d.cvshift = p.cvshift;
    }
    d.h_first = p.h_first; d.matrix_first = p.matrix_first;
    d.yuv_out = p.yuv_out ? 1 : 0;
    d.rgb_in = p.rgb_in ? 1 : 0; d.in_sel = p.in_sel;
    for (int i = 0; i < 3; i++) for (int j = 0; j < 4; j++) d.m[i][j] = p.m_rgb2yuv[i][j];
    if (p.yuv_out) {                                              // the chain's output is the scratch image
      d.stride_out = p.out.width * 4; d.off_out = 0;
      Down420Dev & q = h->down;
      memset (&q, 0, sizeof (q));
      q.ow = p.out.width; q.oh = p.out.height; q.stride_s = d.stride_out;
      q.hmode = p.down_h; q.vavg = p.down_v ? 1 : 0; q.extra_row = p.extra_row ? 1 : 0;
      q.stride_y = p.out.stride[0]; q.off_y = p.out.offset[0];
      q.stride_u = p.out.stride[p.out_plane_u]; q.stride_v = p.out.stride[p.out_plane_v];
      q.cstep = p.out_cstep;
      q.off_u = p.out.offset[p.out_plane_u] + (p.out_cstep == 2 ? p.out_u_index : 0);
      q.off_v = p.out.offset[p.out_plane_v] + (p.out_cstep == 2 ? (p.out_u_index ^ 1) : 0);
      if ((st = prepare_rgb420 (h)) != B200_OK) { b200_vcs_destroy (h); return st; }
      if (p.yuy2_420) {
        Yuy2Dev & y = h->yuy2;
        memset (&y, 0, sizeof (y));
        const bool uyvy = p.in.format == B200_VIDEO_FORMAT_UYVY;
        y.w = p.in.width; y.h = p.in.height; y.sstride = p.in.stride[0]; y.soff = p.in.offset[0];
        y.sel_y = uyvy ? 0x7531 : 0x6420; y.sel_c = uyvy ? 0x6420 : 0x7531;
        y.svec = ((y.sstride | y.soff) & 15) == 0 ? 2 : (((y.sstride | y.soff) & 3) == 0 ? 1 : 0);
        y.stride_y = q.stride_y; y.stride_u = q.stride_u; y.stride_v = q.stride_v;
        y.off_y = q.off_y; y.off_u = q.off_u; y.off_v = q.off_v;
        y.wvec = ((q.stride_y | q.stride_u | q.stride_v) & 3) == 0 && ((q.off_y | q.off_u | q.off_v) & 3) == 0;
      }
    }
    d.p1 = p.p[0]; d.p2 = p.p[1]; d.p3 = p.p[2]; d.p4 = p.p[3]; d.p5 = p.p[4];
    d.sel = p.byte_sel[0] | (p.byte_sel[1] << 4) | (p.byte_sel[2] << 8) | (p.byte_sel[3] << 12);
    d.tile_w = p.tile_w; d.tile_h = p.tile_h; d.max_rows = p.max_rows; d.cols_pitch = p.cols_pitch;
    d.max_crows = p.max_crows;
    if ((st = upload_axis (p.h, &h->d_hoff, &h->d_hcoef, &h->d_hsum, &d.h)) != B200_OK ||
        (st = upload_axis (p.v, &h->d_voff, &h->d_vcoef, &h->d_vsum, &d.v)) != B200_OK ||
        (st = upload (&h->d_cmode, p.chroma_mode.data (), p.chroma_mode.size ())) != B200_OK) {
      b200_vcs_destroy (h);
      return st;
    }
    d.chroma_mode = h->d_cmode;
    if ((st = allow_max_dyn_smem (vcs_generic_kernel)) != B200_OK) { b200_vcs_destroy (h); return st; }
    if (h->mma_tables.ok) {
      st = prepare_l2mma (h->mma_tables, &h->mma);
      if (st != B200_OK) { b200_vcs_destroy (h); return st; }
    }
    if (p.lanczos2_ok) {
      st = prepare_lanczos2 (h->l2_tables, h->dev, &h->l2);
      if (st != B200_OK) { b200_vcs_destroy (h); return st; }
      h->variant = 1;
      if (h->l2v2_tables.ok && !getenv ("B200_L2_V1")) {            // tuning knob: B200_L2_V1 keeps the first form
        if ((st = prepare_lanczos2_v2 (h->l2v2_tables, &h->l2v2)) != B200_OK) { b200_vcs_destroy (h); return st; }
      }
#ifndef B200_CUDA_EMU
      if ((st = prepare_l2tc (h->tc_tables, &h->tc)) != B200_OK) { b200_vcs_destroy (h); return st; }
      { const char *e = getenv ("B200_L2_TC"); if (e && e[0] == '1' && h->tc.ready) h->variant = 7; }   // tuning knob
#endif
    } else if (p.light_ok) {
      if ((st = allow_max_dyn_smem (light_kernel_for (p))) != B200_OK) { b200_vcs_destroy (h); return st; }
      h->variant = 2;
    } else if (p.ntap_ok) {
      st = prepare_ntap (p, &h->ntap);
      if (st != B200_OK) { b200_vcs_destroy (h); return st; }
      h->variant = 3;
    }
  }
  // variant 6 (mma.sync formulation of the 2:1 kernel) measured 12.7 us/frame against 8.4 for the SIMT kernel
  // (profiles/r02_first_bench_l2mma.json): kept selectable through b200_vcs_set_kernel_variant for cross-checks only
  *handle = h;
  return B200_OK;
}

void b200_vcs_destroy (b200_vcs * h)
{
  if (!h) return;
  if (h->device >= 0) {
    DeviceGuard g (h->device);
    cudaFree (h->d_hoff); cudaFree (h->d_voff); cudaFree (h->d_hcoef); cudaFree (h->d_vcoef);
    cudaFree (h->d_hsum); cudaFree (h->d_vsum); cudaFree (h->d_cmode);
    cudaFree (h->l2.d_htab); cudaFree (h->l2.d_vtab); cudaFree (h->ntap.d_h); cudaFree (h->ntap.d_v);
    cudaFree (h->l2.d_htab4); cudaFree (h->l2.d_vtab4); cudaFree (h->l2.d_v4); cudaFree (h->l2v2.d_vkind);
    cudaFree (h->mma.d_bh); cudaFree (h->mma.d_bv); cudaFree (h->mma.d_h4); cudaFree (h->mma.d_v4);
#ifndef B200_CUDA_EMU
    cudaFree (h->tc.d_band); cudaFree (h->tc.d_vband); cudaFree (h->tc.d_hx4); cudaFree (h->tc.d_vx4);
#endif
    free_planes (&h->planes);
    free_plane_fast (&h->rgb420_scaler);
    cudaFree (h->d_scratch);
    for (int i = 0; i < b200_vcs::kSlots; i++) {
      cudaFree (h->slot_in[i]); cudaFree (h->slot_out[i]);
      if (h->ev_in[i]) cudaEventDestroy (h->ev_in[i]);
      if (h->ev_run[i]) cudaEventDestroy (h->ev_run[i]);
      if (h->ev_out[i]) cudaEventDestroy (h->ev_out[i]);
    }
    if (h->s_h2d) cudaStreamDestroy (h->s_h2d);
    if (h->s_run) cudaStreamDestroy (h->s_run);
    if (h->s_d2h) cudaStreamDestroy (h->s_d2h);
  }
  delete h;
}

int b200_vcs_convert_batch (b200_vcs * h, int n, const void *const *in_frames,
    void *const *out_frames, void *cuda_stream)
{
  if (!h || !in_frames || !out_frames || n < 1 || n > B200_VCS_MAX_BATCH) return B200_ERR_INVALID_ARG;
  if (h->device < 0) return B200_ERR_NO_DEVICE;
  DeviceGuard g (h->device);
  if (!g.ok) return B200_ERR_CUDA;
  VcsBatch b;
  for (int i = 0; i < n; i++) {
    if (!in_frames[i] || !out_frames[i]) return B200_ERR_INVALID_ARG;
    b.in[i] = (const uint8_t *) in_frames[i];
    b.out[i] = (uint8_t *) out_frames[i];
  }
  return launch (h, n, b, (cudaStream_t) cuda_stream);
}

int b200_vcs_convert (b200_vcs * h, const void *in_frame, void *out_frame, void *cuda_stream)
{
  return b200_vcs_convert_batch (h, 1, &in_frame, &out_frame, cuda_stream);
}

int b200_vcs_convert_host (b200_vcs * h, int n, const void *const *in_host, void *const *out_host)
{
  if (!h || !in_host || !out_host || n < 1) return B200_ERR_INVALID_ARG;
  if (h->device < 0) return B200_ERR_NO_DEVICE;
  for (int i = 0; i < n; i++) if (!in_host[i] || !out_host[i]) return B200_ERR_INVALID_ARG;
  DeviceGuard g (h->device);
  if (!g.ok) return B200_ERR_CUDA;
  // Three-stage software pipeline over kSlots device slots of `chunk` frames: the upload of chunk c+1 and the download
  // of chunk c-1 overlap the kernel of chunk c (the copy engines run beside the SMs).  One kernel launch and one event
  // triple per chunk, not per frame; with few frames the chunk shrinks so that all three stages still overlap.
  const int K = b200_vcs::kSlots;
  // measured: 16 frames in chunks of 4 lose 14 % to pipeline fill / drain against single frames
  const int chunk = n >= 16 * b200_vcs::kChunk ? b200_vcs::kChunk : (n >= 32 ? 2 : 1);
  int st = ensure_pipeline (h, chunk);
  if (st != B200_OK) return st;
  int c = 0;
  for (int i0 = 0; i0 < n; i0 += chunk, c++) {
    const int s = c % K, m = min (chunk, n - i0);
    if (c >= K) {
      B200_CUDA_TRY (cudaStreamWaitEvent (h->s_h2d, h->ev_run[s], 0));   // input slot consumed
      B200_CUDA_TRY (cudaStreamWaitEvent (h->s_run, h->ev_out[s], 0));   // output slot drained
    }
    VcsBatch b;
    for (int j = 0; j < m; j++) {
      b.in[j] = h->slot_in[s] + (size_t) j * h->in_bytes; b.out[j] = h->slot_out[s] + (size_t) j * h->out_bytes;
      B200_CUDA_TRY (cudaMemcpyAsync ((void *) b.in[j], in_host[i0 + j], h->in_bytes, cudaMemcpyHostToDevice, h->s_h2d));
    }
    B200_CUDA_TRY (cudaEventRecord (h->ev_in[s], h->s_h2d));
    B200_CUDA_TRY (cudaStreamWaitEvent (h->s_run, h->ev_in[s], 0));
    if ((st = launch (h, m, b, h->s_run)) != B200_OK) return st;
    B200_CUDA_TRY (cudaEventRecord (h->ev_run[s], h->s_run));
    B200_CUDA_TRY (cudaStreamWaitEvent (h->s_d2h, h->ev_run[s], 0));
    for (int j = 0; j < m; j++)
      B200_CUDA_TRY (cudaMemcpyAsync (out_host[i0 + j], b.out[j], h->out_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
    B200_CUDA_TRY (cudaEventRecord (h->ev_out[s], h->s_d2h));
  }
  B200_CUDA_TRY (cudaStreamSynchronize (h->s_d2h));
  return B200_OK;
}

int b200_vcs_copy_probe (b200_vcs * h, int n, const void *const *in_host, void *const *out_host)
{
  // the copies of b200_vcs_convert_host without the kernels: H2D of every input on one stream, D2H of every output
  // (whatever the slots hold) on another, both directions in flight together - the link's ceiling for this call
  if (!h || !in_host || !out_host || n < 1) return B200_ERR_INVALID_ARG;
  if (h->device < 0) return B200_ERR_NO_DEVICE;
  DeviceGuard g (h->device);
  if (!g.ok) return B200_ERR_CUDA;
  int st = ensure_pipeline (h, max (h->slot_frames, 1));
  if (st != B200_OK) return st;
  const int K = b200_vcs::kSlots, chunk = h->slot_frames;
  for (int i = 0; i < n; i++) {
    const int s = (i / chunk) % K, j = i % chunk;
    if (!in_host[i] || !out_host[i]) return B200_ERR_INVALID_ARG;
    B200_CUDA_TRY (cudaMemcpyAsync (h->slot_in[s] + (size_t) j * h->in_bytes, in_host[i], h->in_bytes, cudaMemcpyHostToDevice, h->s_h2d));
    B200_CUDA_TRY (cudaMemcpyAsync (out_host[i], h->slot_out[s] + (size_t) j * h->out_bytes, h->out_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
  }
  B200_CUDA_TRY (cudaStreamSynchronize (h->s_h2d));
  B200_CUDA_TRY (cudaStreamSynchronize (h->s_d2h));
  return B200_OK;
}

int b200_vcs_get_plan_info (const b200_vcs * h, b200_vcs_plan_info * info)
{
  if (!h || !info) return B200_ERR_INVALID_ARG;
  const VcsPlan & p = h->plan;
  memset (info, 0, sizeof (*info));
  info->h_taps = p.h.scaling ? p.h.n_taps : 0;
  info->v_taps = p.v.scaling ? p.v.n_taps : 0;
  info->h_first = p.h_first; info->matrix_first = p.matrix_first;
  for (int i = 0; i < 5; i++) info->p[i] = p.p[i];
  info->tile_w = p.tile_w; info->tile_h = p.tile_h; info->smem_bytes = p.smem_bytes;
  info->kernel_variant = p.yuv_out ? 5 : p.planes_mode ? 4 : h->variant == 7 ? 7 : (h->variant == 6 && h->mma.ready) ? 6 : (h->variant == 1 && p.lanczos2_ok) ? 1 : (h->variant == 2 && p.light_ok) ? 2 : (h->variant == 3 && p.ntap_ok) ? 3 : 0;
  info->n_launches_per_convert = (p.yuy2_420 ? 1 : h->rgb420_ok ? (1 + (h->rgb420_pre ? 1 : 0) + (h->rgb420_scaled ? 1 : 0)) : p.yuv_out ? (p.extra_row ? 3 : 2) : 1) + (p.has_dest && p.fill_border ? 1 : 0);
  return B200_OK;
}

int b200_vcs_get_taps (const b200_vcs * h, int dir, uint32_t * offsets, int16_t * taps,
    size_t offsets_len, size_t taps_len)
{
  if (!h || (dir != 0 && dir != 1)) return B200_ERR_INVALID_ARG;
  const AxisPlan & a = dir == 0 ? h->plan.h : h->plan.v;
  if (offsets) {
    if (offsets_len < a.offset.size ()) return B200_ERR_INVALID_ARG;
    memcpy (offsets, a.offset.data (), a.offset.size () * sizeof (uint32_t));
  }
  if (taps) {
    if (taps_len < a.coef.size ()) return B200_ERR_INVALID_ARG;
    memcpy (taps, a.coef.data (), a.coef.size () * sizeof (int16_t));
  }
  return (int) a.coef_per_out;
}

int b200_vcs_get_matrix (const b200_vcs * h, int32_t im[16])
{
  if (!h || !im) return B200_ERR_INVALID_ARG;
  const VcsPlan & p = h->plan;
  const bool has = !p.planes_mode && (!p.yuv_out || p.rgb_in);
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) im[4 * i + j] = has ? p.im[i][j] : 0;
  return B200_OK;
}

int b200_vcs_get_chroma_plan (const b200_vcs * h, uint8_t * mode, size_t len)
{
  if (!h || !mode || len < h->plan.chroma_mode.size ()) return B200_ERR_INVALID_ARG;
  memcpy (mode, h->plan.chroma_mode.data (), h->plan.chroma_mode.size ());
  return B200_OK;
}

int b200_vcs_set_kernel_variant (b200_vcs * h, int variant)
{
  if (!h || variant < 0 || (variant > 3 && variant != 6 && variant != 7)) return B200_ERR_INVALID_ARG;
  if (h->plan.planes_mode || h->plan.yuv_out) return B200_ERR_UNSUPPORTED;   // one kernel only
  if (variant == 6 && !h->mma.ready) return B200_ERR_UNSUPPORTED;
#ifndef B200_CUDA_EMU
  if (variant == 7 && !h->tc.ready) return B200_ERR_UNSUPPORTED;
#else
  if (variant == 7) return B200_ERR_UNSUPPORTED;
#endif
  if (variant == 3 && !(h->plan.ntap_ok && h->ntap.ready)) return B200_ERR_UNSUPPORTED;
  if (variant == 1 && !h->plan.lanczos2_ok) return B200_ERR_UNSUPPORTED;
  if (variant == 2 && !h->plan.light_ok) return B200_ERR_UNSUPPORTED;
  h->variant = variant;
  return B200_OK;
}

const char *b200_vcs_kernel_name (const b200_vcs * h)
{
  if (!h) return "";
  const VcsPlan & p = h->plan;
  if (p.planes_mode) {
    for (int i = 0; i < p.n_planes; i++) if (h->planes.fast[i].ok) return h->planes.fast[i].vfirst ? "vcs_planes_fast_vfirst_kernel" : "vcs_planes_fast_kernel";
    return "vcs_planes_kernel";
  }
  if (p.yuy2_420) return "vcs_yuy2_420_kernel";
  if (h->rgb420_ok) return h->rgb420_pre == 2 ? "vcs_yuy2_ayuv_kernel" : "vcs_rgb420_kernel";
  if (h->variant == 6 && h->mma.ready) return "vcs_l2mma_kernel";
#ifndef B200_CUDA_EMU
  if (h->variant == 7 && h->tc.ready) return "vcs_l2tc_kernel";
#endif
  if ((h->variant == 1 || h->variant == 7) && p.lanczos2_ok) return (h->l2v2.ready && h->l2.x4) ? "vcs_lanczos2_v2_kernel" : "vcs_lanczos2_kernel";
  if (h->variant == 2 && p.light_ok) return "vcs_light_kernel";
  if (h->variant == 3 && p.ntap_ok) return "vcs_ntap_kernel";
  return "vcs_generic_kernel";
}

}  // extern "C"
