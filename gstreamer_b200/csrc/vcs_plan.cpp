// gstreamer_b200/csrc/vcs_plan.cpp — host-side plan builder for convert+scale (product code).
//
// Follows the *numbers* of the reference's setup exactly (they decide every output
// byte) while producing flat tables for the fused CUDA kernels:
//   tap positions/weights      gst-libs/gst/video/video-resampler.c:204-288, :343-429
//   integer taps + DC bisection gst-libs/gst/video/video-scaler.c:338-449
//   2-tap specials             video-scaler.c:254-257, :609-618 (h, 16.16 stepping), :846-879 (v, 8-bit tap)
//   stage order                video-converter.c:1685-1718 (chain_scale), :2509-2539
//   colour matrix              video-converter.c:1324-1442 (+ :899-1040 algebra), video-color.c:204-252, :423-459
//   chroma pairing             video-converter.c:571-617, :2991-3021; video-chroma.c:959-1036
//   element option mapping     gst/videoconvertscale/gstvideoconvertscale.c:991-1087
#include "vcs_plan.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>

namespace b200 {

namespace {

enum Kernel1D { K_NEAREST, K_LINEAR, K_CUBIC, K_SINC, K_LANCZOS };

struct FilterSpec {
  Kernel1D kind = K_LINEAR;
  int max_taps = 128;            // GST_VIDEO_RESAMPLER_OPT_MAX_TAPS
  double cubic_b = 1.0 / 3.0, cubic_c = 1.0 / 3.0;
  double envelope = 2.0, sharpness = 1.0, sharpen = 0.0;
};

// gstvideoconvertscale.c:991-1050: element "method" -> resampler method + extra options
FilterSpec filter_from_method (const b200_vcs_config & cfg)
{
  FilterSpec f;
  f.envelope = cfg.envelope;
  f.sharpness = cfg.sharpness;
  f.sharpen = cfg.sharpen;
  switch (cfg.method) {
    case B200_SCALE_NEAREST:   f.kind = K_NEAREST; break;
    case B200_SCALE_BILINEAR:  f.kind = K_LINEAR; f.max_taps = 2; break;
    case B200_SCALE_4TAP:      f.kind = K_SINC; f.max_taps = 4; break;
    case B200_SCALE_LANCZOS:   f.kind = K_LANCZOS; break;
    case B200_SCALE_BILINEAR2: f.kind = K_LINEAR; break;
    case B200_SCALE_SINC:      f.kind = K_SINC; break;
    case B200_SCALE_HERMITE:   f.kind = K_CUBIC; f.cubic_b = 0.0; f.cubic_c = 0.0; break;
    case B200_SCALE_SPLINE:    f.kind = K_CUBIC; f.cubic_b = 1.0; f.cubic_c = 0.0; break;
    case B200_SCALE_CATROM:    f.kind = K_CUBIC; f.cubic_b = 0.0; f.cubic_c = 0.5; break;
    case B200_SCALE_MITCHELL:
    default:                   f.kind = K_CUBIC; break;
  }
  return f;
}

inline double sinc_pi (double x) { return x == 0 ? 1.0 : sin (M_PI * x) / (M_PI * x); }
inline double window (double x) { return (x <= -1 || x >= 1) ? 0.0 : sinc_pi (x); }

struct Weigher {
  Kernel1D kind;
  double fx, ex, b, c, sharpen;
  double operator() (double dist) const      // dist = x - (xi + l), signed
  {
    switch (kind) {
      case K_NEAREST: return 1.0;
      case K_LINEAR: { double a = fabs (dist) * fx; return a < 1.0 ? 1.0 - a : 0.0; }
      case K_CUBIC: {
        double a = fabs (dist) * fx, a2 = a * a, a3 = a2 * a;
        if (a <= 1.0)
          return ((12.0 - 9.0 * b - 6.0 * c) * a3 + (-18.0 + 12.0 * b + 6.0 * c) * a2 + (6.0 - 2.0 * b)) / 6.0;
        if (a <= 2.0)
          return ((-b - 6.0 * c) * a3 + (6.0 * b + 30.0 * c) * a2 + (-12.0 * b - 48.0 * c) * a + (8.0 * b + 24.0 * c)) / 6.0;
        return 0.0;
      }
      case K_SINC: return sinc_pi (dist * fx);
      case K_LANCZOS:
      default: return (sinc_pi (dist * fx) - sharpen) * window (dist * ex);
    }
  }
};

struct RealTaps {
  int n = 0;
  std::vector<uint32_t> first;
  std::vector<double> w;         // out_size * n
};

// video-resampler.c:343-429 (tap count) + :204-288 (positions, normalisation, edge folding)
RealTaps real_taps (const FilterSpec & f, int in_size, int out_size)
{
  RealTaps r;
  Weigher wf;
  wf.kind = f.kind; wf.b = f.cubic_b; wf.c = f.cubic_c; wf.sharpen = f.sharpen;
  double ratio = in_size / (double) out_size;
  wf.fx = (ratio > 1.0 ? 1.0 / ratio : 1.0) * f.sharpness;
  double env = f.envelope;
  int n = 0;
  if (f.kind == K_NEAREST) n = 1;
  else if (f.kind == K_LINEAR) env = 1.0;
  else if (f.kind == K_CUBIC) env = 2.0;
  if (n == 0) {
    double dx = ceil (2.0 * env / wf.fx);
    n = (int) std::min<double> (std::max<double> (dx, 0), f.max_taps);
  }
  wf.fx = 2.0 * env / n;
  wf.ex = 2.0 / n;
  n = std::min (n, in_size);
  r.n = n;
  r.first.resize (out_size);
  r.w.assign ((size_t) out_size * n, 0.0);
  const int centre = (n - 1) / 2;
  const double half = n == 1 ? 0.0 : 0.5;
  for (int j = 0; j < out_size; j++) {
    double pos = ((0.5 + (double) j - 0.0) / out_size) * (double) in_size - half;
    pos = std::min<double> (std::max<double> (pos, 0), in_size - 1);
    int xi = (int) floor (pos - centre);
    double *t = &r.w[(size_t) j * n];
    double total = 0;
    for (int l = 0; l < n; l++) { t[l] = wf (pos - (xi + l)); total += t[l]; }
    for (int l = 0; l < n; l++) t[l] /= total;
    int first = xi;
    if (xi < 0) {                       // fold taps hanging over the left edge
      int sh = -xi, l;
      for (l = 0; l < sh; l++) t[sh] += t[l];
      for (l = 0; l < n - sh; l++) t[l] = t[sh + l];
      for (; l < n; l++) t[l] = 0;
      first += sh;
    }
    if (xi > in_size - n) {             // ... and over the right edge
      int sh = xi - (in_size - n), l;
      for (l = 0; l < sh; l++) t[n - sh - 1] += t[n - sh + l];
      for (l = 0; l < n - sh; l++) t[n - 1 - l] = t[n - 1 - sh - l];
      for (l = 0; l < sh; l++) t[l] = 0;
      first -= sh;
    }
    r.first[j] = (uint32_t) first;
  }
  return r;
}

// video-scaler.c:338-388: floor(bias + w * 2^prec) with the bias bisected until the
// taps sum to 2^prec; the last attempt is kept when no bias achieves it.
void integer_taps (const double *w, int16_t * q, int n, int prec)
{
  const double mul = (double) (1 << prec);
  const int target = 1 << prec;
  double lo = 0.0, hi = 1.0, bias = 0.5;
  for (int it = 0; it < 64; it++) {
    int sum = 0;
    for (int j = 0; j < n; j++) { q[j] = (int16_t) floor (bias + w[j] * mul); sum += q[j]; }
    if (sum == target || lo == hi) break;
    if (sum < target) { if (bias > lo) lo = bias; bias += (hi - lo) / 2; }
    else { if (bias < hi) hi = bias; bias -= (hi - lo) / 2; }
  }
}

void identity_axis (AxisPlan * a, int size)
{
  a->in_size = a->out_size = size;
  a->mode = PASS_COPY; a->n_taps = 1; a->coef_per_out = 0; a->span = 1; a->scaling = false;
  a->offset.resize (size);
  for (int i = 0; i < size; i++) a->offset[i] = (uint32_t) i;
  a->coef.clear (); a->sum.clear ();
}

void scaled_axis (AxisPlan * a, const FilterSpec & f, int in_size, int out_size, bool horizontal,
    bool two_tap_stepping = true)
{
  RealTaps r = real_taps (f, in_size, out_size);
  a->in_size = in_size; a->out_size = out_size; a->scaling = true;
  a->n_taps = r.n; a->span = r.n;
  if (r.n == 1) {                       // video_scale_h_near_u32 / video_scale_v_near_u8
    a->mode = PASS_COPY; a->coef_per_out = 0; a->offset = r.first;
  } else if (r.n == 2 && horizontal && two_tap_stepping) {  // video_scale_h_2tap_4u8 / _1u8: edge-aligned 16.16 stepping
    a->mode = PASS_2TAP; a->coef_per_out = 1;
    a->offset.resize (out_size); a->coef.resize (out_size);
    int inc = out_size == 1 ? 0 : (int) ((((int64_t) in_size - 1) << 16) / (out_size - 1)) - 1;
    for (int i = 0; i < out_size; i++) {
      int tmp = i * inc;                // int arithmetic like ldreslinl
      a->offset[i] = (uint32_t) (tmp >> 16);
      a->coef[i] = (int16_t) ((tmp >> 8) & 0xff);
    }
  } else if (r.n == 2 && !horizontal) { // video_scale_v_2tap_u8: centre-aligned, 8-bit second tap
    a->mode = PASS_2TAP; a->coef_per_out = 1;
    a->offset = r.first; a->coef.resize (out_size);
    for (int i = 0; i < out_size; i++) {
      int16_t q[2];
      integer_taps (&r.w[(size_t) i * 2], q, 2, 8);
      a->coef[i] = q[1];
    }
  } else {                              // n-tap FIR at 6-bit precision (SCALE_U8_LQ)
    a->mode = PASS_NTAP; a->coef_per_out = r.n;
    a->offset = r.first; a->coef.resize ((size_t) out_size * r.n); a->sum.resize (out_size);
    for (int i = 0; i < out_size; i++) {
      int16_t *q = &a->coef[(size_t) i * r.n];
      integer_taps (&r.w[(size_t) i * r.n], q, r.n, 6);
      int s = 0;
      for (int k = 0; k < r.n; k++) s += q[k];
      a->sum[i] = (int16_t) s;
    }
  }
}

struct Mat4 {
  double m[4][4];
  static Mat4 identity () { Mat4 r; for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) r.m[i][j] = i == j; return r; }
};
// left-multiply: dst = a * b, accumulating k = 0..3 in order (rounding must match)
Mat4 mul (const Mat4 & a, const Mat4 & b)
{
  Mat4 r;
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) {
      double x = 0;
      for (int k = 0; k < 4; k++) x += a.m[i][k] * b.m[k][j];
      r.m[i][j] = x;
    }
  return r;
}
Mat4 diag (double a, double b, double c) { Mat4 r = Mat4::identity (); r.m[0][0] = a; r.m[1][1] = b; r.m[2][2] = c; return r; }
Mat4 shift (double a, double b, double c) { Mat4 r = Mat4::identity (); r.m[0][3] = a; r.m[1][3] = b; r.m[2][3] = c; return r; }

int colour_matrix (VcsPlan * p)
{
  int off[3], scl[3];
  if (p->in.color_range == B200_COLOR_RANGE_16_235) { off[0] = 16; scl[0] = 219; off[1] = off[2] = 128; scl[1] = scl[2] = 224; }
  else { off[0] = 0; scl[0] = 255; off[1] = off[2] = 128; scl[1] = scl[2] = 255; }
  double kr, kb;
  switch (p->in.color_matrix) {
    case B200_COLOR_MATRIX_FCC: kr = 0.30; kb = 0.11; break;
    case B200_COLOR_MATRIX_BT709: kr = 0.2126; kb = 0.0722; break;
    case B200_COLOR_MATRIX_BT601: kr = 0.2990; kb = 0.1140; break;
    case B200_COLOR_MATRIX_SMPTE240M: kr = 0.212; kb = 0.087; break;
    case B200_COLOR_MATRIX_BT2020: kr = 0.2627; kb = 0.0593; break;
    default: return B200_ERR_INVALID_ARG;   // YUV input needs a YUV matrix (video-info.c:187-209)
  }
  double kg = 1.0 - kr - kb;
  Mat4 m = Mat4::identity ();
  m = mul (shift (-off[0], -off[1], -off[2]), m);
  m = mul (diag (1 / ((float) scl[0]), 1 / ((float) scl[1]), 1 / ((float) scl[2])), m);
  Mat4 k = Mat4::identity ();
  k.m[0][0] = 1.; k.m[0][1] = 0.; k.m[0][2] = 2 * (1 - kr);
  k.m[1][0] = 1.; k.m[1][1] = -2 * kb * (1 - kb) / kg; k.m[1][2] = -2 * kr * (1 - kr) / kg;
  k.m[2][0] = 1.; k.m[2][1] = 2 * (1 - kb); k.m[2][2] = 0.;
  m = mul (k, m);
  m = mul (diag ((float) 255, (float) 255, (float) 255), m);     // ARGB out, full range
  m = mul (shift (0, 0, 0), m);
  m = mul (diag (256.0f, 256.0f, 256.0f), m);                    // SCALE_F
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) p->im[i][j] = (int) rint (m.m[i][j]);
  // the reference only takes its fused AYUV->ARGB routine for matrices of this shape
  if (p->im[0][0] != p->im[1][0] || p->im[1][0] != p->im[2][0] || p->im[0][1] != 0 || p->im[2][2] != 0)
    return B200_ERR_UNSUPPORTED;
  p->p[0] = p->im[0][0]; p->p[1] = p->im[0][2]; p->p[2] = p->im[2][1]; p->p[3] = p->im[1][1]; p->p[4] = p->im[1][2];
  return B200_OK;
}

// packed RGB in, YUV out: chain_convert (video-converter.c:1720-1868): identity -> compute_matrix_to_RGB (:1373-1404;
// for an RGB unpack format only the range normalisation) -> compute_matrix_to_YUV (:1406-1442): RGB_to_YCbCr (:1037-1066)
// of the OUTPUT matrix, output range scale + offset -> prepare_matrix (:1324-1370): x256, rint.  Only matrices the
// reference routes to video_converter_matrix8_table (is_no_clip_matrix :1262-1300) are accepted.
int colour_matrix_rgb2yuv (VcsPlan * p)
{
  double kr, kb;
  switch (p->out.color_matrix) {
    case B200_COLOR_MATRIX_FCC: kr = 0.30; kb = 0.11; break;
    case B200_COLOR_MATRIX_BT709: kr = 0.2126; kb = 0.0722; break;
    case B200_COLOR_MATRIX_BT601: kr = 0.2990; kb = 0.1140; break;
    case B200_COLOR_MATRIX_SMPTE240M: kr = 0.212; kb = 0.087; break;
    case B200_COLOR_MATRIX_BT2020: kr = 0.2627; kb = 0.0593; break;
    default: return B200_ERR_INVALID_ARG;
  }
  const double kg = 1.0 - kr - kb;
  Mat4 m = Mat4::identity ();
  if (p->in.color_range == B200_COLOR_RANGE_16_235) {
    m = mul (shift (-16, -16, -16), m);
    m = mul (diag (1 / ((float) 219), 1 / ((float) 219), 1 / ((float) 219)), m);
  } else {
    m = mul (shift (0, 0, 0), m);
    m = mul (diag (1 / ((float) 255), 1 / ((float) 255), 1 / ((float) 255)), m);
  }
  Mat4 k = Mat4::identity ();
  k.m[0][0] = kr; k.m[0][1] = kg; k.m[0][2] = kb;
  double x = 1 / (2 * (1 - kb));
  k.m[1][0] = -x * kr; k.m[1][1] = -x * kg; k.m[1][2] = x * (1 - kb);
  x = 1 / (2 * (1 - kr));
  k.m[2][0] = x * (1 - kr); k.m[2][1] = -x * kg; k.m[2][2] = -x * kb;
  m = mul (k, m);
  if (p->out.color_range == B200_COLOR_RANGE_16_235) {
    m = mul (diag ((float) 219, (float) 224, (float) 224), m);
    m = mul (shift (16, 128, 128), m);
  } else {
    m = mul (diag ((float) 255, (float) 255, (float) 255), m);
    m = mul (shift (0, 128, 128), m);
  }
  m = mul (diag (256.0f, 256.0f, 256.0f), m);
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) p->im[i][j] = (int) rint (m.m[i][j]);
  for (int t = 0; t < 8; t++)
    for (int i = 0; i < 3; i++) {
      const int r = (t & 4) ? 255 : 0, g = (t & 2) ? 255 : 0, b = (t & 1) ? 255 : 0;
      const int v = (p->im[i][0] * r + p->im[i][1] * g + p->im[i][2] * b + p->im[i][3]) >> 8;
      if (v < 0 || v > 255) return B200_ERR_UNSUPPORTED;       // the reference would run video_orc_matrix8: not built
    }
  for (int i = 0; i < 3; i++) for (int j = 0; j < 4; j++) p->m_rgb2yuv[i][j] = p->im[i][j];
  return B200_OK;
}

// Which lines reach the chroma upsampler and how they pair up (see DESIGN.md "chroma plan").
void chroma_pairing (VcsPlan * p)
{
  const int ih = p->in.height;
  std::vector<uint8_t> wanted (ih, p->v.scaling ? 0 : 1);
  if (p->v.scaling)
    for (int r = 0; r < p->v.out_size; r++)
      for (int k = 0; k < p->v.span; k++) wanted[p->v.offset[r] + k] = 1;
  p->chroma_mode.assign (ih, 0);
  int open_pair = -2;
  for (int y = 1; y < ih; y++) {        // line 0 always rides the clamped pair (-1,0)
    if (!wanted[y]) continue;
    if (open_pair == y - 1) p->chroma_mode[y] = 2;
    else { p->chroma_mode[y] = 1; open_pair = y; }
  }
}

void tile_geometry (VcsPlan * p)
{
  const int ow = p->out.width, oh = p->out.height;
  int tw = ow >= 64 ? 64 : (ow >= 32 ? 32 : 16), th = 16;
  const int budget = 200 * 1024;
  for (;;) {
    int max_rows = 0, max_cols = 0;
    for (int y0 = 0; y0 < oh; y0 += th) {
      int y1 = std::min (y0 + th, oh) - 1;
      max_rows = std::max (max_rows, (int) (p->v.offset[y1] + p->v.span - p->v.offset[y0]));
    }
    for (int x0 = 0; x0 < ow; x0 += tw) {
      int x1 = std::min (x0 + tw, ow) - 1;
      max_cols = std::max (max_cols, (int) (p->h.offset[x1] + p->h.span - p->h.offset[x0]));
    }
    int pitch = (max_cols + 3) & ~3;
    int crows = p->cvshift ? max_rows / 2 + 3 : max_rows + 1;    // chroma rows staged per tile
    size_t planes = (size_t) 3 * max_rows * pitch;
    size_t hup = (size_t) 2 * crows * pitch;
    size_t mid = p->h_first ? (size_t) 3 * max_rows * tw : (size_t) 3 * th * pitch;
    size_t coefs = ((size_t) tw * std::max (p->h.coef_per_out, 1) + (size_t) th * std::max (p->v.coef_per_out, 1)) * 2 + 64;
    size_t total = planes + hup + mid + coefs + 64;
    if (total <= (size_t) budget || (tw == 1 && th == 1)) {
      p->tile_w = tw; p->tile_h = th; p->max_rows = max_rows; p->max_cols = max_cols;
      p->cols_pitch = pitch; p->max_crows = crows; p->smem_bytes = (int) total;
      return;
    }
    // shrink the dimension that contributes most
    if (max_rows >= max_cols && th > 1) th = std::max (1, th / 2);
    else if (tw > 1) tw = std::max (1, tw / 2);
    else th = std::max (1, th / 2);
  }
}

// Geometry of the light kernel (vcs_light.cuh): packed 4-byte pixels in shared memory, input
// columns taken from a 4-aligned start, 128 output columns per tile.
// the fast kernels read luma rows with 32-bit loads and chroma with 32-bit (interleaved) or 16-bit
// (planar) loads, and keep row offsets in 32 bits
bool fast_layout_ok (const VcsPlan * p)
{
  const int iw = p->in.width;
  if ((p->in.stride[0] & 3) || (p->in.offset[0] & 3) || p->in.stride[0] < ((iw + 3) & ~3)) return false;
  if ((int64_t) p->in.stride[0] * p->in.height >= (1ll << 31)) return false;
  if (p->planar) {
    if (p->in.stride[1] != p->in.stride[2]) return false;
    for (int k = 1; k <= 2; k++) {
      if ((p->in.stride[k] & 1) || (p->in.offset[k] & 1) || p->in.stride[k] < ((((iw + 1) / 2) + 1) & ~1)) return false;
      if ((int64_t) p->in.stride[k] * p->in.height >= (1ll << 31)) return false;
    }
    return true;
  }
  if ((p->in.stride[1] & 3) || (p->in.offset[1] & 3) || p->in.stride[1] < ((iw + 3) & ~3)) return false;
  return (int64_t) p->in.stride[1] * p->in.height < (1ll << 31);
}

// fast stage A of the light and n-tap kernels (vcs_unpack_fast_cs): NV12 / NV21, real chroma filtering, every line's
// chroma_mode the standard one (all lines pulled in order), 64-bit loads possible (8-byte aligned rows; a last item may
// read up to 7 bytes past the width: inside the row's stride)
void std_pairs_check (VcsPlan * p)
{
  bool std_pairs = !p->chroma_nearest && p->v_pairs && !p->in_422_444 && !p->rgb_in && !p->planes_mode &&
      !(p->in.stride[0] & 7) && !(p->in.offset[0] & 7) && p->in.stride[0] >= ((p->in.width + 7) & ~7) && !(p->in.height & 1) &&
      (int) p->chroma_mode.size () >= p->in.height;
  if (p->planar)                                  // I420 / YV12: 32-bit loads of 4 samples + the next one from each chroma plane
    for (int k = 1; k <= 2; k++)
      std_pairs = std_pairs && !(p->in.stride[k] & 3) && !(p->in.offset[k] & 3) && p->in.stride[k] >= ((((p->in.width + 7) & ~7) >> 1));
  else
    std_pairs = std_pairs && !(p->in.stride[1] & 7) && !(p->in.offset[1] & 7) && p->in.stride[1] >= ((p->in.width + 7) & ~7);
  for (int y = 0; std_pairs && y < p->in.height; y++)
    if (p->chroma_mode[y] != (y == 0 ? 0 : ((y & 1) ? 1 : 2))) std_pairs = false;
  p->light_std_pairs = std_pairs;
}

void light_geometry (VcsPlan * p)
{
  p->light_ok = false;
  if (!(p->h.mode == PASS_COPY || p->h.mode == PASS_2TAP) || !(p->v.mode == PASS_COPY || p->v.mode == PASS_2TAP))
    return;
  if (!fast_layout_ok (p)) return;
  // the packed 16-bit-lane lerps need fractions in [0,255] (h) and weights in [0,256] (v)
  if (p->h.mode == PASS_2TAP) for (int16_t c : p->h.coef) if (c < 0 || c > 255) return;
  if (p->v.mode == PASS_2TAP) for (int16_t c : p->v.coef) if (c < 0 || c > 256) return;
  const int ow = p->out.width, oh = p->out.height, tw = 128;
  const char *env_th = getenv ("B200_LIGHT_TH");              // tuning aid
  static const int heights[] = {32, 16, 8, 4, 2, 1};              // 32 rows measured best on C1 (4.77 us vs 5.67 at 16)
  for (int hi = 0; hi < 6; hi++) {
    const int th = (env_th && hi == 0) ? atoi (env_th) : heights[hi];
    int max_rows = 0, max_cols = 0;
    for (int y0 = 0; y0 < oh; y0 += th) {
      int y1 = std::min (y0 + th, oh) - 1;
      max_rows = std::max (max_rows, (int) (p->v.offset[y1] + p->v.span - p->v.offset[y0]));
    }
    for (int x0 = 0; x0 < ow; x0 += tw) {
      int x1 = std::min (x0 + tw, ow) - 1;
      int c0 = (int) p->h.offset[x0] & ~3, c1 = ((int) (p->h.offset[x1] + p->h.span) + 3) & ~3;
      max_cols = std::max (max_cols, c1 - c0);
    }
    const int cp = max_cols + 4;                                  // +4 words: rows start on distinct banks
    const size_t t_words = p->h_first ? 0 : (size_t) th * cp;     // horizontal first: the two passes are fused, no intermediate tile
    const size_t total = ((size_t) max_rows * cp + t_words + 4 * (size_t) max_rows + 4 + th) * 4;   // S, T, work list, v table
    if (total <= (env_th ? 200 : 96) * 1024) {
      p->light_ok = true; p->light_tw = tw; p->light_th = th; p->light_rows = max_rows; p->light_cp = cp;
      p->light_smem = (int) total;

      return;
    }
  }
}

// 4 signed 8-bit taps per word, zero padded to a whole number of words; false when a tap does not
// fit or the 16-bit accumulator of the reference could wrap (the kernel accumulates in 32 bits)
bool pack_taps_s8 (const AxisPlan & a, int *ntw, std::vector<int32_t> * out)
{
  *ntw = 0; out->clear ();
  if (a.mode != PASS_NTAP) return true;
  const int n = a.n_taps, w = (n + 3) / 4;
  out->assign ((size_t) a.out_size * w, 0);
  for (int j = 0; j < a.out_size; j++) {
    int mag = 0;
    for (int k = 0; k < n; k++) {
      const int t = a.coef[(size_t) j * n + k];
      if (t < -128 || t > 127) return false;
      mag += abs (t);
      (*out)[(size_t) j * w + k / 4] |= (int32_t) ((uint32_t) (uint8_t) (int8_t) t << (8 * (k & 3)));
    }
    if (255 * mag + 32 > 32767) return false;
  }
  *ntw = w;
  return true;
}

// Geometry of the n-tap kernel (vcs_ntap.cuh)
void ntap_geometry (VcsPlan * p)
{
  p->ntap_ok = false;
  const bool hn = p->h.mode == PASS_NTAP, vn = p->v.mode == PASS_NTAP;
  if (!(hn || vn) || p->h.mode == PASS_2TAP || p->v.mode == PASS_2TAP) return;
  if (!fast_layout_ok (p)) return;
  if (!pack_taps_s8 (p->h, &p->ntw_h, &p->h_packed) || !pack_taps_s8 (p->v, &p->ntw_v, &p->v_packed)) return;
  p->ntap_alpha_opaque = true;
  if (hn) for (int16_t s : p->h.sum) if (s < 64 || s > 128) p->ntap_alpha_opaque = false;
  if (vn) for (int16_t s : p->v.sum) if (s < 64 || s > 128) p->ntap_alpha_opaque = false;
  const int ow = p->out.width, oh = p->out.height;
  // tile shape: the one that stages the fewest input pixels per output pixel (filter halos shrink
  // with the tile) among those whose shared memory lets at least two CTAs share an SM
  static const int shapes[][2] = {{128, 32}, {128, 16}, {64, 32}, {128, 8}, {64, 16}, {32, 32}, {64, 8}, {32, 16},
                                  {64, 4}, {32, 8}, {32, 4}, {32, 2}, {32, 1}};
  double best = 0;
  const char *env_shape = getenv ("B200_NTAP_SHAPE");             // tuning aid: "tw,th"
  int etw = 0, eth = 0;
  if (env_shape && sscanf (env_shape, "%d,%d", &etw, &eth) != 2) etw = eth = 0;
  for (auto & sh : shapes) {
    const int tw = sh[0], th = sh[1];
    if (etw && (tw != etw || th != eth)) continue;
    if (th > 16 && oh < 2 * th) continue;
    int max_rows = 0, max_cols = 0;
    for (int y0 = 0; y0 < oh; y0 += th) {
      int y1 = std::min (y0 + th, oh) - 1;
      max_rows = std::max (max_rows, (int) (p->v.offset[y1] + p->v.span - p->v.offset[y0]));
    }
    for (int x0 = 0; x0 < ow; x0 += tw) {
      int x1 = std::min (x0 + tw, ow) - 1;
      int c0 = (int) p->h.offset[x0] & ~3, c1 = ((int) (p->h.offset[x1] + p->h.span) + 3) & ~3;
      max_cols = std::max (max_cols, c1 - c0);
    }
    // rows: whole groups of 4; pitch (word columns per line): the zero-padded horizontal taps may
    // read up to ntw_h + 1 words past the window start; the h-scaled tile keeps 1 + ntw_v groups of
    // slack for the zero-padded vertical taps
    const int rows = ((max_rows + 3) & ~3), ngr = rows / 4, groups = ngr + 1 + p->ntw_v;
    const int pitch = max_cols / 4 + 2 + p->ntw_h;
    const size_t s_words = ((size_t) ngr * 3 * pitch + 2) * 4;
    const size_t t_words = (size_t) groups * tw * 4;
    const size_t tap_words = (size_t) tw * std::max (p->ntw_h, 1) + (size_t) th * std::max (p->ntw_v, 1) + th;
    size_t total = (s_words + t_words + tap_words + 4 * (size_t) rows + 12) * 4;
    if (!p->h_first) {
      // vertical first: plain planes S[3][rows][pitch], v-scaled rows T[3][th][pitch], 16-bit v taps one per word
      total = ((size_t) 3 * rows * pitch + 4 + (size_t) 3 * th * pitch + 4 + (size_t) tw * std::max (p->ntw_h, 1) +
          (size_t) th * std::max (p->v.n_taps, 1) + th + 4 * (size_t) rows + 12) * 4;
    }
    if (total > 100 * 1024) continue;
    // staged input pixels + h-scaled pixels per output pixel; small tiles pay extra per-tile overhead
    const double cost = ((double) rows * max_cols + (double) rows * tw) / ((double) std::min (tw, ow) * std::min (th, oh))
        + 64.0 / th + 256.0 / tw;
    if (!p->ntap_ok || cost < best) {
      best = cost;
      p->ntap_ok = true; p->ntap_tw = tw; p->ntap_th = th; p->ntap_rows = rows; p->ntap_pitch = pitch;
      p->ntap_smem = (int) total;
    }
  }
}

// Walk every tile the fast kernels will run and check each shared-memory index range against the
// geometry chosen above; a violation (none is known) downgrades the plan to the generic kernel instead
// of risking an out-of-bounds access.  tests/test_host_plan.py sweeps random sizes over this.
void validate_fast_geometry (VcsPlan * p)
{
  const int ow = p->out.width, oh = p->out.height;
  auto tile_ok = [&] (int tw, int th, int rows_cap, int words_cap, int ntw_h, int extra_words) {
    for (int y0 = 0; y0 < oh; y0 += th) {
      const int y1 = std::min (y0 + th, oh) - 1;
      const int R = (int) (p->v.offset[y1] + p->v.span - p->v.offset[y0]);
      if (R > rows_cap || R < 1) return false;
      for (int y = y0; y <= y1; y++) {                            // every output row's window inside the staged rows
        const int rb = (int) p->v.offset[y] - (int) p->v.offset[y0];
        if (rb < 0 || rb + p->v.span > R) return false;
      }
    }
    for (int x0 = 0; x0 < ow; x0 += tw) {
      const int x1 = std::min (x0 + tw, ow) - 1;
      const int cxa = (int) p->h.offset[x0] & ~3, cx1 = (int) (p->h.offset[x1] + p->h.span);
      const int ng = (cx1 - cxa + 3) >> 2;
      if (ng + extra_words > words_cap) return false;
      for (int x = x0; x <= x1; x++) {
        const int base = (int) p->h.offset[x] - cxa;
        if (base < 0 || base + p->h.span > cx1 - cxa) return false;
        if ((base >> 2) + ntw_h + 1 > words_cap) return false;    // funnel-shift FIR reads words wi .. wi + ntw_h
      }
    }
    return true;
  };
  if (p->light_ok && !tile_ok (p->light_tw, p->light_th, p->light_rows, p->light_cp / 4, 0, 0)) p->light_ok = false;
  if (p->ntap_ok) {
    bool ok = tile_ok (p->ntap_tw, p->ntap_th, p->ntap_rows, p->ntap_pitch, p->ntw_h, 0);
    if (ok && p->h_first) {                                       // vertical FIR over 4-line groups: g0 + ntw_v < groups
      const int groups = p->ntap_rows / 4 + 1 + p->ntw_v;
      for (int y0 = 0; y0 < oh && ok; y0 += p->ntap_th)
        for (int y = y0; y < std::min (y0 + p->ntap_th, oh); y++) {
          const int rb = (int) p->v.offset[y] - (int) p->v.offset[y0];
          if ((rb >> 2) + p->ntw_v >= groups) { ok = false; break; }
        }
    }
    if (!ok) p->ntap_ok = false;
  }
}

// setup_scale (video-converter.c:8092-8245) for planar in/out (4:2:0 same family; Y42B / Y444 -> I420 / YV12): what each output plane does
int build_planes (VcsPlan * p, const FilterSpec & f)
{
  const bool semi = p->out.format == B200_VIDEO_FORMAT_NV12 || p->out.format == B200_VIDEO_FORMAT_NV21;
  const int iw = p->in.width, ih = p->in.height, ow = p->out.width, oh = p->out.height;
  p->planes_mode = true;
  p->n_planes = semi ? 2 : 3;
  for (int i = 0; i < p->n_planes; i++) {
    PlanePlan & q = p->planes[i];
    q = PlanePlan ();
    // exactly one side YV12: U and V planes swap (the source plane is the one holding the same component)
    q.src_plane = (!semi && i > 0 && (p->in.format == B200_VIDEO_FORMAT_YV12) != (p->out.format == B200_VIDEO_FORMAT_YV12)) ? 3 - i : i;
    // chroma plane size of the input: 4:2:0 halves both directions, Y42B the width only, Y444 neither
    const int in_wsub = p->in.format == B200_VIDEO_FORMAT_Y444 ? 0 : 1;
    const int in_hsub = (p->in.format == B200_VIDEO_FORMAT_Y444 || p->in.format == B200_VIDEO_FORMAT_Y42B) ? 0 : 1;
    q.iw = i ? (iw + in_wsub) >> in_wsub : iw; q.ih = i ? (ih + in_hsub) >> in_hsub : ih;
    q.ow = i ? (ow + 1) / 2 : ow; q.oh = i ? (oh + 1) / 2 : oh;
    q.ne = (semi && i == 1) ? 2 : 1;
    if (p->in.stride[q.src_plane] < q.iw * q.ne || p->out.stride[i] < q.ow * q.ne) return B200_ERR_INVALID_ARG;
    FilterSpec fs = f;
    if (i > 0 && fs.kind != K_NEAREST) fs.kind = K_LINEAR;         // chroma resampler (cr_method), :7981-7986
    const bool same_w = q.iw == q.ow, same_h = q.ih == q.oh;
    if (same_w && same_h) { q.mode = PM_COPY; continue; }
    if (q.ne == 1 && fs.kind == K_LINEAR) {                        // convert_plane_{v,h,hv}_halve
      if (same_w && q.ih == 2 * q.oh) { q.mode = PM_HALVE_V; continue; }
      if (same_h && q.iw == 2 * q.ow) { q.mode = PM_HALVE_H; continue; }
      if (q.iw == 2 * q.ow && q.ih == 2 * q.oh) { q.mode = PM_HALVE_HV; continue; }
    }
    if (q.ne == 1 && fs.kind == K_NEAREST) {                       // convert_plane_{v,h,hv}_double
      if ((same_w && 2 * q.ih == q.oh) || (same_h && 2 * q.iw == q.ow) || (2 * q.iw == q.ow && 2 * q.ih == q.oh)) {
        q.mode = PM_DOUBLE; continue;
      }
    }
    q.mode = PM_SCALE;
    q.have_h = !same_w; q.have_v = !same_h;
    // get_functions (video-scaler.c:1283-1420): only the single-byte plane has the stepping 2-tap h scaler
    if (q.have_h) scaled_axis (&q.h, fs, q.iw, q.ow, true, q.ne == 1); else identity_axis (&q.h, q.iw);
    if (q.have_v) scaled_axis (&q.v, fs, q.ih, q.oh, false); else identity_axis (&q.v, q.ih);
    // gst_video_scaler_2d (:1542-1545): horizontal first when width * v.offset[last] <= width * height
    q.h_first = !(q.have_h && q.have_v) || (int64_t) q.v.offset[q.oh - 1] <= (int64_t) q.oh;
  }
  return B200_OK;
}

}  // namespace

// packed RGB -> 4:2:0 (the encoder-feeding direction): no table row in the reference, its generic chain: unpack to
// ARGB, the scalers that shrink, the RGB -> YUV table matrix, the scalers that grow, chroma down-sampling (RGB has no
// sub-sampling, so only the down side exists and it exists at every size: video-converter.c:2850-2895), 4:2:0 pack.
// Generic kernel + vcs_down420_kernel.  Written without device access: opt-in until it has run green on a GPU.
// packed RGB -> the same packed RGB format at another size (a compositor's scaled RGBA pads): the reference's one-plane
// convert_scale_planes rows (video-converter.c:8879-8896): 4-byte pixels through gst_video_scaler_2d with the element's
// method, the stepping 2-tap horizontal scaler (video_scale_h_2tap_4u8), every byte - alpha or padding included - a
// channel.  vcs_planes_kernel with ne = 4.
// memory byte index of the A (or padding), R, G, B component of a packed 4-byte format
static void rgb_component_bytes (int format, int pos[4])
{
  switch (format) {
    case B200_VIDEO_FORMAT_BGRA: case B200_VIDEO_FORMAT_BGRx: pos[0] = 3; pos[1] = 2; pos[2] = 1; pos[3] = 0; break;
    case B200_VIDEO_FORMAT_RGBA: case B200_VIDEO_FORMAT_RGBx: pos[0] = 3; pos[1] = 0; pos[2] = 1; pos[3] = 2; break;
    case B200_VIDEO_FORMAT_ABGR: case B200_VIDEO_FORMAT_xBGR: pos[0] = 0; pos[1] = 3; pos[2] = 2; pos[3] = 1; break;
    default: pos[0] = 0; pos[1] = 1; pos[2] = 2; pos[3] = 3; break;          // ARGB / xRGB
  }
}

static int build_rgb_same_plan (VcsPlan * p)
{
  const b200_video_info *in = &p->in, *out = &p->out;
  const int iw = in->width, ih = in->height, ow = out->width, oh = out->height;
  if (in->stride[0] < iw * 4 || out->stride[0] < ow * 4) return B200_ERR_INVALID_ARG;
  const FilterSpec f = filter_from_method (p->cfg);
  p->planes_mode = true;
  p->n_planes = 1;
  PlanePlan & q = p->planes[0];
  q = PlanePlan ();
  q.src_plane = 0; q.iw = iw; q.ih = ih; q.ow = ow; q.oh = oh; q.ne = 4;
  // another byte order (BGRA -> RGBA ...) has no table row: the reference's chain runs - byte-shuffle unpack, the same
  // 4-byte-pixel scalers, byte-shuffle pack, no matrix and (alpha value 1.0) no alpha stage - so it differs from the
  // same-format rows only in the pass order rule (chain_scale :1697-1714 instead of gst_video_scaler_2d :1542-1545)
  // and in where each byte lands; a format's padding byte travels as alpha, like in the reference's unpack
  const bool cross = in->format != out->format;
  if (cross) {
    int pi[4], po[4];
    rgb_component_bytes (in->format, pi);
    rgb_component_bytes (out->format, po);
    unsigned swz = 0;
    for (int comp = 0; comp < 4; comp++) swz |= (unsigned) pi[comp] << (4 * po[comp]);
    q.swz = swz == 0x3210u ? 0u : swz;
  }
  if (iw == ow && ih == oh) { q.mode = PM_COPY; return B200_OK; }
  q.mode = PM_SCALE;
  q.have_h = iw != ow; q.have_v = ih != oh;
  if (q.have_h) scaled_axis (&q.h, f, iw, ow, true, true); else identity_axis (&q.h, iw);
  if (q.have_v) scaled_axis (&q.v, f, ih, oh, false); else identity_axis (&q.v, ih);
  if (cross) q.h_first = (int64_t) ow * ih <= (int64_t) iw * oh;
  else q.h_first = !(q.have_h && q.have_v) || (int64_t) q.v.offset[oh - 1] <= (int64_t) oh;
  return B200_OK;
}

static int build_rgb_in_plan (VcsPlan * p)
{
  const b200_video_info *in = &p->in, *out = &p->out;
  if (out->format >= B200_VIDEO_FORMAT_RGBx && out->format <= B200_VIDEO_FORMAT_ABGR) return build_rgb_same_plan (p);
  const bool out_pl = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12;
  const bool out_semi = out->format == B200_VIDEO_FORMAT_NV12 || out->format == B200_VIDEO_FORMAT_NV21;
  if (!out_pl && !out_semi) return B200_ERR_UNSUPPORTED;
  if (in->stride[0] < in->width * 4 || (in->stride[0] & 3) || (in->offset[0] & 3)) return B200_ERR_INVALID_ARG;
  const int ocw = (out->width + 1) / 2;
  if (out->stride[0] < out->width) return B200_ERR_INVALID_ARG;
  if (out_pl) {
    if (out->stride[1] < ocw || out->stride[2] < ocw) return B200_ERR_INVALID_ARG;
    p->out_plane_u = out->format == B200_VIDEO_FORMAT_YV12 ? 2 : 1;
    p->out_plane_v = 3 - p->out_plane_u;
    p->out_cstep = 1; p->out_u_index = 0;
  } else {
    if (out->stride[1] < 2 * ocw) return B200_ERR_INVALID_ARG;
    p->out_plane_u = p->out_plane_v = 1;
    p->out_cstep = 2; p->out_u_index = out->format == B200_VIDEO_FORMAT_NV21 ? 1 : 0;
  }
  // caps defaults of the output size where the caller left them open (the fixation forwards only primaries and
  // transfer across an RGB/YUV change, gstvideoconvertscale.c:1394-1408)
  if (p->in.color_range == 0) p->in.color_range = B200_COLOR_RANGE_0_255;
  if (p->out.color_matrix == 0) p->out.color_matrix = out->height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
  if (p->out.color_range == 0) p->out.color_range = B200_COLOR_RANGE_16_235;
  if (p->out.chroma_site == 0) p->out.chroma_site = out->height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
  int st = colour_matrix_rgb2yuv (p);
  if (st != B200_OK) return st;
  p->rgb_in = p->yuv_out = true;
  switch (in->format) {                 // source byte of R, G, B, A (nibbles 0..3)
    case B200_VIDEO_FORMAT_BGRA: case B200_VIDEO_FORMAT_BGRx: p->in_sel = 0x3012; break;
    case B200_VIDEO_FORMAT_RGBA: case B200_VIDEO_FORMAT_RGBx: p->in_sel = 0x3210; break;
    case B200_VIDEO_FORMAT_ABGR: case B200_VIDEO_FORMAT_xBGR: p->in_sel = 0x0123; break;
    default: p->in_sel = 0x0321; break;                            // ARGB / xRGB
  }
  { uint8_t s[4] = {0, 1, 2, 3}; memcpy (p->byte_sel, s, 4); }
  p->planar = false; p->u_index = 0; p->h_cosited = false; p->v_pairs = false; p->chroma_nearest = false;
  FilterSpec f = filter_from_method (p->cfg);
  const int iw = in->width, ih = in->height, ow = out->width, oh = out->height;
  if (iw != ow) scaled_axis (&p->h, f, iw, ow, true); else identity_axis (&p->h, iw);
  if (ih != oh) scaled_axis (&p->v, f, ih, oh, false); else identity_axis (&p->v, ih);
  p->matrix_first = !((int64_t) ow * oh <= (int64_t) iw * ih);     // chain_scale: shrink before the matrix, grow after
  p->h_first = (int64_t) ow * ih <= (int64_t) iw * oh;
  p->chroma_mode.assign (ih, 0);
  p->down_h = (p->out.chroma_site & B200_CHROMA_SITE_H_COSITED) ? 2 : 1;
  p->down_v = (p->out.chroma_site & B200_CHROMA_SITE_V_COSITED) == 0;
  p->extra_row = false;                 // the line past an odd frame is the last line itself (no chroma up-sampler)
  tile_geometry (p);
  p->light_ok = p->ntap_ok = p->lanczos2_ok = false;
  return B200_OK;
}

static int build_inner_plan (const b200_video_info * in, const b200_video_info * out,
    const b200_vcs_config * cfg, VcsPlan * p, bool resample_forced);

// border pixel of setup_borderline (video-converter.c:2189-2258): packed RGB outputs take border_argb's bytes in the
// format's order; YUV outputs convert it with the un-scaled (no x256) rint'ed RGB -> YCbCr matrix of the OUTPUT
// colorimetry and hand-added 16 / 128 / 128 offsets
static int border_colour (VcsPlan * p, const b200_video_info & fo, uint32_t argb_word)
{
  const int a = argb_word >> 24, r = (argb_word >> 16) & 0xff, g = (argb_word >> 8) & 0xff, b = argb_word & 0xff;
  const bool rgb = fo.format >= B200_VIDEO_FORMAT_RGBx && fo.format <= B200_VIDEO_FORMAT_ABGR;
  if (rgb) {
    const uint8_t comp[4] = {(uint8_t) a, (uint8_t) r, (uint8_t) g, (uint8_t) b};
    uint8_t sel[4];
    switch (fo.format) {
      case B200_VIDEO_FORMAT_BGRA: case B200_VIDEO_FORMAT_BGRx: { uint8_t s_[4] = {3, 2, 1, 0}; memcpy (sel, s_, 4); break; }
      case B200_VIDEO_FORMAT_RGBA: case B200_VIDEO_FORMAT_RGBx: { uint8_t s_[4] = {1, 2, 3, 0}; memcpy (sel, s_, 4); break; }
      case B200_VIDEO_FORMAT_ABGR: case B200_VIDEO_FORMAT_xBGR: { uint8_t s_[4] = {0, 3, 2, 1}; memcpy (sel, s_, 4); break; }
      default: { uint8_t s_[4] = {0, 1, 2, 3}; memcpy (sel, s_, 4); break; }
    }
    for (int i = 0; i < 4; i++) p->border_px[i] = comp[sel[i]];
    return B200_OK;
  }
  // the plan's `out` carries the resolved output colorimetry (the input's for 4:2:0 -> 4:2:0, the caps defaults of
  // the frame for packed RGB input)
  int matrix = p->out.color_matrix ? p->out.color_matrix : p->in.color_matrix;
  int range = p->out.color_range ? p->out.color_range : p->in.color_range;
  double kr, kb;
  switch (matrix) {
    case B200_COLOR_MATRIX_FCC: kr = 0.30; kb = 0.11; break;
    case B200_COLOR_MATRIX_BT709: kr = 0.2126; kb = 0.0722; break;
    case B200_COLOR_MATRIX_BT601: kr = 0.2990; kb = 0.1140; break;
    case B200_COLOR_MATRIX_SMPTE240M: kr = 0.212; kb = 0.087; break;
    case B200_COLOR_MATRIX_BT2020: kr = 0.2627; kb = 0.0593; break;
    default: return B200_ERR_INVALID_ARG;
  }
  const double kg = 1.0 - kr - kb;
  Mat4 k = Mat4::identity ();
  k.m[0][0] = kr; k.m[0][1] = kg; k.m[0][2] = kb;
  double x = 1 / (2 * (1 - kb));
  k.m[1][0] = -x * kr; k.m[1][1] = -x * kg; k.m[1][2] = x * (1 - kb);
  x = 1 / (2 * (1 - kr));
  k.m[2][0] = x * (1 - kr); k.m[2][1] = -x * kg; k.m[2][2] = -x * kb;
  Mat4 m = mul (k, Mat4::identity ());
  if (range == B200_COLOR_RANGE_16_235) { m = mul (diag ((float) 219, (float) 224, (float) 224), m); m = mul (shift (16, 128, 128), m); }
  else { m = mul (diag ((float) 255, (float) 255, (float) 255), m); m = mul (shift (0, 128, 128), m); }
  int im[3][3];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) im[i][j] = (int) rint (m.m[i][j]);
  const int yy = 16 + ((r * im[0][0] + g * im[0][1] + b * im[0][2]) >> 8);
  const int uu = 128 + ((r * im[1][0] + g * im[1][1] + b * im[1][2]) >> 8);
  const int vv = 128 + ((r * im[2][0] + g * im[2][1] + b * im[2][2]) >> 8);
  p->border_yuv[0] = std::min (std::max (yy, 0), 255);
  p->border_yuv[1] = std::min (std::max (uu, 0), 255);
  p->border_yuv[2] = std::min (std::max (vv, 0), 255);
  return B200_OK;
}

int build_vcs_plan (const b200_video_info * in, const b200_video_info * out,
    const b200_vcs_config * cfg, VcsPlan * p)
{
  if (!in || !out || !cfg || !p) return B200_ERR_INVALID_ARG;
  // packed RGB is written in 32-bit words: the plane and each of its lines must start on a 4-byte boundary
  // (b200_vcs_convert_batch holds the frame base to the same)
  if (out->format >= B200_VIDEO_FORMAT_RGBx && out->format <= B200_VIDEO_FORMAT_ABGR && ((out->stride[0] & 3) || (out->offset[0] & 3)))
    return B200_ERR_INVALID_ARG;
  if (cfg->dest_width == 0 || cfg->dest_height == 0 ||
      (cfg->dest_x == 0 && cfg->dest_y == 0 && cfg->dest_width == out->width && cfg->dest_height == out->height)) {
    int st = build_inner_plan (in, out, cfg, p, false);
    if (st == B200_OK) p->frame_out = p->out;
    return st;
  }
  // GST_VIDEO_CONVERTER_OPT_DEST_* (video-converter.c:2333-2362): the chain scales into the rectangle; for sub-sampled
  // outputs its origin is rounded down to the chroma grid; it is clipped to the frame
  if (out->width < 1 || out->height < 1 || out->width > 32767 || out->height > 32767) return B200_ERR_INVALID_ARG;
  const bool yuv = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12 ||
      out->format == B200_VIDEO_FORMAT_NV12 || out->format == B200_VIDEO_FORMAT_NV21;
  const bool planar = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12;
  int dx = cfg->dest_x, dy = cfg->dest_y, dw = cfg->dest_width, dh = cfg->dest_height;
  if (yuv) { dx &= ~1; dy &= ~1; }
  if (dx < 0 || dy < 0 || dw < 0 || dh < 0) return B200_ERR_INVALID_ARG;
  if (dw > out->width - dx) dw = out->width - dx;
  if (dh > out->height - dy) dh = out->height - dy;
  if (dw < 1 || dh < 1) return B200_ERR_INVALID_ARG;               // an empty rectangle: degenerate in the reference too
  b200_video_info inner = *out;
  inner.width = dw; inner.height = dh;
  if (!yuv) inner.offset[0] += (uint64_t) dy * out->stride[0] + (uint64_t) dx * 4;
  else {
    inner.offset[0] += (uint64_t) dy * out->stride[0] + (uint64_t) dx;
    if (planar) {
      inner.offset[1] += (uint64_t) (dy / 2) * out->stride[1] + (uint64_t) (dx / 2);
      inner.offset[2] += (uint64_t) (dy / 2) * out->stride[2] + (uint64_t) (dx / 2);
    } else inner.offset[1] += (uint64_t) (dy / 2) * out->stride[1] + (uint64_t) dx;
  }
  // colorimetry defaults belong to the whole frame, not to the rectangle
  const bool in_rgb = in->format >= B200_VIDEO_FORMAT_RGBx && in->format <= B200_VIDEO_FORMAT_ABGR;
  if (yuv && in_rgb) {
    if (inner.color_matrix == 0) inner.color_matrix = out->height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
    if (inner.color_range == 0) inner.color_range = B200_COLOR_RANGE_16_235;
    if (inner.chroma_site == 0) inner.chroma_site = out->height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
  }
  const bool in_422p = in->format == B200_VIDEO_FORMAT_YUY2 || in->format == B200_VIDEO_FORMAT_UYVY || in->format == B200_VIDEO_FORMAT_YVYU;
  if (yuv && in_422p && inner.chroma_site == 0)
    inner.chroma_site = out->height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
  // video_converter_compute_resample (:2850-2895) compares the input with the whole output frame
  const bool forced = in->width != out->width || in->height != out->height;
  int st = build_inner_plan (in, &inner, cfg, p, forced);
  if (st != B200_OK) return st;
  p->has_dest = true;
  p->frame_out = *out;
  p->dest[0] = dx; p->dest[1] = dy; p->dest[2] = dw; p->dest[3] = dh;
  p->fill_border = cfg->fill_border != 0;
  return border_colour (p, *out, cfg->border_argb);
}

static int build_inner_plan (const b200_video_info * in, const b200_video_info * out,
    const b200_vcs_config * cfg, VcsPlan * p, bool resample_forced)
{
  if (!in || !out || !cfg || !p) return B200_ERR_INVALID_ARG;
  if (in->width < 1 || in->height < 1 || out->width < 1 || out->height < 1 ||
      in->width > 32767 || in->height > 32767 || out->width > 32767 || out->height > 32767)
    return B200_ERR_INVALID_ARG;        // caps range [1,32767], gstvideoconvertscale.c:168-169
  const bool in_rgb = in->format >= B200_VIDEO_FORMAT_RGBx && in->format <= B200_VIDEO_FORMAT_ABGR;
  const bool in_422 = in->format == B200_VIDEO_FORMAT_YUY2 || in->format == B200_VIDEO_FORMAT_UYVY ||
      in->format == B200_VIDEO_FORMAT_YVYU || in->format == B200_VIDEO_FORMAT_Y42B || in->format == B200_VIDEO_FORMAT_Y444;
  if (in->format != B200_VIDEO_FORMAT_NV12 && in->format != B200_VIDEO_FORMAT_NV21 &&
      in->format != B200_VIDEO_FORMAT_I420 && in->format != B200_VIDEO_FORMAT_YV12 && !in_rgb && !in_422)
    return B200_ERR_UNSUPPORTED;
  p->in = *in; p->out = *out; p->cfg = *cfg;
  if (in_rgb) return build_rgb_in_plan (p);
  if (in_422) {
    // capture formats: unpack_YUY2 / _UYVY / _YVYU / _Y42B / _Y444 (video-format.c:155-274, :1009-1104), horizontal chroma
    // up-sampling only (4:2:2: v_factor 0 selects video_chroma_none, video-chroma.c:989-994; 4:4:4: no resampler at all),
    // then the usual chain to packed RGB.  Generic kernel (device-verified: tests/test_vcs_rgbin_gpu.py).
    // Packed 4:2:2 (YUY2 / UYVY / YVYU) also converts to 4:2:0 (capture -> encoder): the chain closed by chroma
    // down-sampling, or the table rows YUY2 / UYVY -> I420 / YV12 at an unchanged size (yuy2_420 below).  Planar
    // 4:2:2 / 4:4:4 -> planar 4:2:0 are plane-scaling table rows, -> semi-planar 4:2:0 the chain again.
    const bool out_rgb = out->format >= B200_VIDEO_FORMAT_RGBx && out->format <= B200_VIDEO_FORMAT_ABGR;
    const bool out_420 = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12 ||
        out->format == B200_VIDEO_FORMAT_NV12 || out->format == B200_VIDEO_FORMAT_NV21;
    const bool in_packed = in->format == B200_VIDEO_FORMAT_YUY2 || in->format == B200_VIDEO_FORMAT_UYVY || in->format == B200_VIDEO_FORMAT_YVYU;
    const bool out_pl420 = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12;
    if (!in_packed && out_pl420) {
      // planar 4:2:2 / 4:4:4 -> planar 4:2:0: plane-scaling table rows like I420 -> I420 (video-converter.c:8607-8628; the
      // same colour matrix on both sides, :8989 - what the element's fixation produces): no chain, no chroma siting
      if (p->in.color_matrix == 0) p->in.color_matrix = in->height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
      if (p->out.color_matrix != 0 && p->out.color_matrix != p->in.color_matrix) return B200_ERR_UNSUPPORTED;
      if (in->stride[0] < in->width || out->stride[0] < out->width) return B200_ERR_INVALID_ARG;
      return build_planes (p, filter_from_method (*cfg));
    }
    // (planar 4:2:2 / 4:4:4 -> NV12 / NV21 has no table row: the chain, like the packed inputs)
    if (!out_rgb && !out_420) return B200_ERR_UNSUPPORTED;
    const int w = in->width;
    p->in_422_444 = true;
    p->cvshift = 0;
    p->chshift = in->format == B200_VIDEO_FORMAT_Y444 ? 0 : 1;
    switch (in->format) {
      case B200_VIDEO_FORMAT_YUY2: case B200_VIDEO_FORMAT_YVYU: case B200_VIDEO_FORMAT_UYVY: {
        if (in->stride[0] < 4 * ((w + 1) / 2)) return B200_ERR_INVALID_ARG;
        const int yo = in->format == B200_VIDEO_FORMAT_UYVY ? 1 : 0;
        const int uo = in->format == B200_VIDEO_FORMAT_YUY2 ? 1 : (in->format == B200_VIDEO_FORMAT_YVYU ? 3 : 0);
        const int vo = in->format == B200_VIDEO_FORMAT_YUY2 ? 3 : (in->format == B200_VIDEO_FORMAT_YVYU ? 1 : 2);
        p->ystep = 2; p->cstep_in = 4;
        p->in_off_y = in->offset[0] + yo; p->in_off_u = in->offset[0] + uo; p->in_off_v = in->offset[0] + vo;
        p->in_stride_u = p->in_stride_v = in->stride[0];
        break;
      }
      default: {
        const int cw = p->chshift ? (w + 1) / 2 : w;
        if (in->stride[0] < w || in->stride[1] < cw || in->stride[2] < cw) return B200_ERR_INVALID_ARG;
        p->ystep = 1; p->cstep_in = 1;
        p->in_off_y = in->offset[0]; p->in_off_u = in->offset[1]; p->in_off_v = in->offset[2];
        p->in_stride_u = in->stride[1]; p->in_stride_v = in->stride[2];
        break;
      }
    }
  }
  // caps defaults (video-info.c:165-185, :211-225)
  if (p->in.color_matrix == 0) p->in.color_matrix = in->height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
  if (p->in.color_range == 0) p->in.color_range = B200_COLOR_RANGE_16_235;
  if (p->in.chroma_site == 0) p->in.chroma_site = in->height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE;
  {
    const bool in_pl = in->format == B200_VIDEO_FORMAT_I420 || in->format == B200_VIDEO_FORMAT_YV12;
    const bool out_pl = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12;
    const bool out_semi = out->format == B200_VIDEO_FORMAT_NV12 || out->format == B200_VIDEO_FORMAT_NV21;
    if (out_pl || out_semi) {
      // the reference has plane-scaling fast paths for NV12->NV12, NV21->NV21, I420/YV12 -> I420/YV12
      // (video-converter.c:8722-8760); the other 4:2:0 pairs run the chain with chroma down-sampling
      if (!((in_pl && out_pl) || (out_semi && in->format == out->format))) {
        // the remaining 4:2:0 pairs have no table row: the generic chain, closed by chain_downsample
        // (video-converter.c:2018-2032) and the 4:2:0 pack functions
        p->yuv_out = true;
      } else {
        if (in->stride[0] < in->width || out->stride[0] < out->width) return B200_ERR_INVALID_ARG;
        if (p->in.color_matrix == 0) p->in.color_matrix = in->height > 576 ? B200_COLOR_MATRIX_BT709 : B200_COLOR_MATRIX_BT601;
        return build_planes (p, filter_from_method (*cfg));
      }
    }
  }
  if (p->yuv_out) {
    const bool out_pl = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12;
    const int ocw = (out->width + 1) / 2;
    // chain_convert (video-converter.c:1720-1868) compares the two colour matrices only (not the range): equal ->
    // no matrix stage.  A differing one would run video_orc_matrix8, whose SIMD program and C backup disagree
    // (video-orc.orc:2079-2133 vs video-converter.c:1136-1176): refused.  The element's caps fixation carries the
    // input colorimetry over to a YUV output (gstvideoconvertscale.c:1335-1427), so equal is the negotiated case.
    if (p->out.color_matrix != 0 && p->out.color_matrix != p->in.color_matrix) return B200_ERR_UNSUPPORTED;
    // a changing sub-sampling (4:2:2 in) does not carry the input's chroma-site over (gstvideoconvertscale.c:1411-1424):
    // the output keeps the default of its size
    if (p->out.chroma_site == 0)
      p->out.chroma_site = !p->in_422_444 ? p->in.chroma_site : (out->height > 576 ? B200_CHROMA_SITE_H_COSITED : B200_CHROMA_SITE_NONE);
    if (out->stride[0] < out->width) return B200_ERR_INVALID_ARG;
    if (out_pl) {
      if (out->stride[1] < ocw || out->stride[2] < ocw) return B200_ERR_INVALID_ARG;
      p->out_plane_u = out->format == B200_VIDEO_FORMAT_YV12 ? 2 : 1;
      p->out_plane_v = 3 - p->out_plane_u;
      p->out_cstep = 1; p->out_u_index = 0;
    } else {
      if (out->stride[1] < 2 * ocw) return B200_ERR_INVALID_ARG;
      p->out_plane_u = p->out_plane_v = 1;
      p->out_cstep = 2; p->out_u_index = out->format == B200_VIDEO_FORMAT_NV21 ? 1 : 0;
    }
    { uint8_t s[4] = {0, 1, 2, 3}; memcpy (p->byte_sel, s, 4); }   // scratch pixels stay A,Y,U,V
  } else
  switch (out->format) {                // (A,R,G,B) component placed at each output byte
    case B200_VIDEO_FORMAT_BGRA: case B200_VIDEO_FORMAT_BGRx: { uint8_t s[4] = {3, 2, 1, 0}; memcpy (p->byte_sel, s, 4); break; }
    case B200_VIDEO_FORMAT_RGBA: case B200_VIDEO_FORMAT_RGBx: { uint8_t s[4] = {1, 2, 3, 0}; memcpy (p->byte_sel, s, 4); break; }
    case B200_VIDEO_FORMAT_ABGR: case B200_VIDEO_FORMAT_xBGR: { uint8_t s[4] = {0, 3, 2, 1}; memcpy (p->byte_sel, s, 4); break; }
    case B200_VIDEO_FORMAT_ARGB: case B200_VIDEO_FORMAT_xRGB: { uint8_t s[4] = {0, 1, 2, 3}; memcpy (p->byte_sel, s, 4); break; }
    default: return B200_ERR_UNSUPPORTED;
  }
  p->planar = in->format == B200_VIDEO_FORMAT_I420 || in->format == B200_VIDEO_FORMAT_YV12;
  const int min_out_stride = p->yuv_out ? out->width : out->width * 4;
  if (p->in_422_444) {
    if (out->stride[0] < min_out_stride) return B200_ERR_INVALID_ARG;
  } else if (p->planar) {
    const int cw = (in->width + 1) / 2;
    if (in->stride[0] < in->width || in->stride[1] < cw || in->stride[2] < cw || out->stride[0] < min_out_stride)
      return B200_ERR_INVALID_ARG;
    p->plane_u = in->format == B200_VIDEO_FORMAT_YV12 ? 2 : 1;   // YV12 keeps V in plane 1
    p->plane_v = 3 - p->plane_u;
  } else if (in->stride[0] < in->width || in->stride[1] < ((in->width + 1) & ~1) || out->stride[0] < min_out_stride)
    return B200_ERR_INVALID_ARG;
  p->u_index = in->format == B200_VIDEO_FORMAT_NV21 ? 1 : 0;
  p->h_cosited = (p->in.chroma_site & B200_CHROMA_SITE_H_COSITED) != 0;
  p->v_pairs = (p->in.chroma_site & B200_CHROMA_SITE_V_COSITED) == 0 && !p->in_422_444;   // line pairs: 4:2:0 only

  if (!p->yuv_out) {
    int st = colour_matrix (p);
    if (st != B200_OK) return st;
  }

  FilterSpec f = filter_from_method (*cfg);
  const int iw = in->width, ih = in->height, ow = out->width, oh = out->height;
  if (iw != ow) scaled_axis (&p->h, f, iw, ow, true); else identity_axis (&p->h, iw);
  if (ih != oh) scaled_axis (&p->v, f, ih, oh, false); else identity_axis (&p->v, ih);
  // chain_scale: shrink before the matrix, grow after it; horizontal first unless the
  // vertical pass leaves fewer pixels for the second pass
  const int64_t s0 = (int64_t) iw * ih, s3 = (int64_t) ow * oh;
  p->matrix_first = !p->yuv_out && !(s3 <= s0);
  p->h_first = (int64_t) ow * ih <= (int64_t) iw * oh;
  chroma_pairing (p);
  // unchanged size, planar 4:2:0 in, packed RGB out: the reference never builds the chain, its fast path
  // (convert_I420_BGRA / _ARGB / _pack_ARGB, video-converter.c:6772-6988, table :8766-8800) feeds each
  // chroma sample to its 2x2 pixels unfiltered
  p->chroma_nearest = !p->yuv_out && p->planar && iw == ow && ih == oh;
  if (p->chroma_nearest) {
    p->v_pairs = false;
    std::fill (p->chroma_mode.begin (), p->chroma_mode.end (), 0);
  }
  if (p->yuv_out && p->in_422_444) {
    const bool out_pl = out->format == B200_VIDEO_FORMAT_I420 || out->format == B200_VIDEO_FORMAT_YV12;
    // table rows YUY2 / UYVY -> I420 / YV12 (video-converter.c:8493-8507; a border rectangle disables them, :8993)
    p->yuy2_420 = (in->format == B200_VIDEO_FORMAT_YUY2 || in->format == B200_VIDEO_FORMAT_UYVY) && out_pl &&
        iw == ow && ih == oh && !resample_forced;
    if (p->yuy2_420 && out->stride[0] < 2 * ((ow + 1) / 2)) return B200_ERR_INVALID_ARG;   // whole pairs of luma per line
  }
  if (p->yuv_out) {
    // video_converter_compute_resample (video-converter.c:2850-2895): chroma resamplers exist on BOTH sides as soon
    // as the size or the site differs (the sub-sampling is 4:2:0 on both), on neither otherwise
    const bool resample = iw != ow || ih != oh || p->out.chroma_site != p->in.chroma_site || resample_forced || p->in_422_444;
    if (!resample) {
      p->chroma_nearest = true; p->v_pairs = false;
      std::fill (p->chroma_mode.begin (), p->chroma_mode.end (), 0);
      p->down_h = 0; p->down_v = false;
    } else {
      p->down_h = (p->out.chroma_site & B200_CHROMA_SITE_H_COSITED) ? 2 : 1;
      p->down_v = (p->out.chroma_site & B200_CHROMA_SITE_V_COSITED) == 0;
      // odd height and no vertical scaler: the down-sampler's second line of the last pair is line `oh`.  A vertical
      // scaler would clamp that request to its last line (video-converter.c:3070-3080: the pair averages a line
      // with itself); without one it reaches do_unpack_lines' clamp (:2973) through a fresh up-sampler pair
      // (oh, oh+1), i.e. the LAST SOURCE LINE WITH ITS CHROMA ROW NOT VERTICALLY FILTERED, pushed through the
      // horizontal stages.  The device code rebuilds that line as row `oh` of the scratch image by running the chain
      // on a one-line view of the frame (line ih-1 with chroma row (ih-1)>>1: a 1-line frame has no vertical filter).
      p->extra_row = (oh & 1) && ih == oh && p->down_v && p->v_pairs && p->chroma_mode[ih - 1] != 0;
    }
    tile_geometry (p);
    p->light_ok = p->ntap_ok = p->lanczos2_ok = false;
    if (!p->rgb_in && !p->in_422_444 && !p->has_dest) {
      // 4:2:0 in: the first launch (the chain up to the scaled A,Y,U,V pixels) may run the light / n-tap kernels with their
      // matrix stage switched off (VcsDev::yuv_out) instead of the generic kernel
      std_pairs_check (p);
      light_geometry (p);
      ntap_geometry (p);
      validate_fast_geometry (p);
    }
    return B200_OK;
  }
  if (p->in_422_444) {
    std::fill (p->chroma_mode.begin (), p->chroma_mode.end (), 0);
    tile_geometry (p);
    p->light_ok = p->ntap_ok = p->lanczos2_ok = false;
    return B200_OK;
  }
  tile_geometry (p);
  std_pairs_check (p);
  light_geometry (p);
  ntap_geometry (p);
  validate_fast_geometry (p);

  // the specialised kernel covers exactly the headline shape class: even 2:1 in both
  // directions with the 8-tap lanczos the reference derives for it
  p->lanczos2_ok = false;
  return B200_OK;
}

}  // namespace b200
