"""Kernel logic without a GPU: the product's own kernel sources (vcs_generic_kernel, vcs_planes_kernel,
vcs_down420_kernel, vcs_border_kernel) and glue (vcs.cu), compiled for the host against a stand-in CUDA runtime
(tests/cudaemu: blocks run one after another, threads of a block are real threads, __syncthreads is a barrier), driven
through the same C-ABI and compared with the oracle.  TEST INFRASTRUCTURE — the product never loads this library and has
no CPU fallback; the `-m gpu` tests remain the parity tests proper.  What it buys: indexing and integer arithmetic of the
kernels that use neither PTX nor warp shuffles are checked on every CPU run, including the paths written after the
round's device budget was spent (packed RGB input, RGB -> RGB, destination rectangle + borders)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from oracle import bindings as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "cudaemu"))

pytestmark = pytest.mark.timeout(600)           # emulated barriers: a logic error must fail, not hang the CPU suite

RGB = ["BGRA", "RGBA", "ARGB", "ABGR", "BGRx", "RGBx", "xRGB", "xBGR"]
YUV = ["NV12", "NV21", "I420", "YV12"]
YUV_422_444 = ["YUY2", "UYVY", "YVYU", "Y42B", "Y444"]


@pytest.fixture(scope="module")
def emu():
    import build_emu
    from gstreamer_b200 import _lib
    lib = C.CDLL(build_emu.build())
    for name, (res, args) in _lib._SIGS.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    return lib


def frame_for(fmt, iw, ih, seed):
    if fmt in YUV_422_444:
        d = ob.vcs_desc(iw, ih, iw, ih, 1, in_fmt=ob.FMT[fmt], out_fmt=12)
        return np.random.default_rng(seed).integers(0, 256, ob.vcs_sizes(d)[0], dtype=np.uint8)
    if fmt in RGB:
        return np.random.default_rng(seed).integers(0, 256, iw * ih * 4, dtype=np.uint8)
    return ob.i420_random_frame(iw, ih, seed) if fmt in ("I420", "YV12") else ob.nv12_random_frame(iw, ih, seed)


def run(emu, fi, fo, size, method, frame, colorimetry=None, dest=None, border=0xff000000, site=None, out_site=None, force_generic=True):
    """one conversion through the emulated C-ABI; returns the output frame (filled with 0x5A beforehand)"""
    from gstreamer_b200 import _lib
    iw, ih, W, H = size
    ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
    assert emu.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih) == 0
    assert emu.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], W, H) == 0
    if site is not None:
        ii.chroma_site = site
    if fi in YUV and fo in YUV:                      # what the element's caps fixation does
        oi.color_matrix, oi.color_range, oi.chroma_site = ii.color_matrix, ii.color_range, ii.chroma_site
    if fi in YUV_422_444 and fo in YUV:              # ... across a sub-sampling change: the site stays the output's own
        oi.color_matrix, oi.color_range = ii.color_matrix, ii.color_range
    if out_site is not None:
        oi.chroma_site = out_site
    if colorimetry:
        oi.color_matrix, oi.color_range, oi.chroma_site = colorimetry
    cfg = _lib.VcsConfigC()
    emu.b200_vcs_config_init(C.byref(cfg))
    cfg.method = method
    if dest:
        cfg.dest_x, cfg.dest_y, cfg.dest_width, cfg.dest_height = dest
        cfg.border_argb = border
    h = C.c_void_p()
    st = emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h))
    assert st == 0, (st, fi, fo, size)
    try:
        if force_generic:
            emu.b200_vcs_set_kernel_variant(h, 0)    # the fast kernels (PTX, shuffles) are not emulated
        out = np.full(emu.b200_video_info_size(C.byref(oi)), 0x5A, dtype=np.uint8)
        src = np.ascontiguousarray(frame)
        assert emu.b200_vcs_convert(h, src.ctypes.data, out.ctypes.data, None) == 0
    finally:
        emu.b200_vcs_destroy(h)
    return out


def expected(fi, fo, size, method, frame, colorimetry=None, dest=None, border=0xff000000, site=None, out_site=None):
    iw, ih, W, H = size
    d = ob.vcs_desc(iw, ih, W, H, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site)
    if out_site is not None:
        d.out_chroma_site = out_site
    if colorimetry:
        d.out_matrix, d.out_range, d.out_chroma_site = colorimetry
    if dest:
        return ob.oracle_vcs_convert_dest(d, frame, dest, border, fill=0x5A)
    want = np.full(ob.vcs_sizes(d)[1], 0x5A, dtype=np.uint8)
    assert ob.oracle().oracle_vcs_convert(C.byref(d), np.ascontiguousarray(frame).ctypes.data, want.ctypes.data) == 0
    return want


def check(got, want, tag):
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{tag}: {len(bad)} of {got.size} bytes differ, first at {bad[:5].ravel().tolist()}"


SMALL = [(64, 48, 32, 24), (40, 30, 64, 48), (33, 17, 20, 31), (57, 35, 29, 35), (50, 21, 50, 21), (100, 60, 150, 30), (7, 5, 3, 9)]


# ---- 1. the emulator itself, on paths the device has already confirmed bit-exact ------------------------------------
@pytest.mark.parametrize("size", SMALL, ids=lambda s: "%dx%d-%dx%d" % s)
def test_emulator_agrees_on_device_verified_paths(emu, size):
    """generic kernel (4:2:0 -> packed RGB), plane kernel (same family) and chain + chroma down-sampling (other family)
    are bit-exact on a B200 (tests/test_vcs_gpu.py, _planes_gpu, _cross_gpu); the emulated build must say the same"""
    iw, ih = size[:2]
    for fi, fo, method in [("NV12", "BGRA", 3), ("I420", "RGBA", 1), ("NV21", "xRGB", 0), ("NV12", "NV12", 1), ("I420", "YV12", 9),
                           ("NV12", "I420", 3), ("YV12", "NV21", 1), ("I420", "NV12", 0)]:
        frame = frame_for(fi, iw, ih, 3)
        for site in (1, 2):
            got = run(emu, fi, fo, size, method, frame, site=site)
            check(got, expected(fi, fo, size, method, frame, site=site), f"{fi}->{fo} m{method} site{site}")


# ---- 2. the remaining converter paths (device-verified since: tests/test_vcs_rgbin_gpu.py) ------------------------------------
@pytest.mark.parametrize("size", SMALL, ids=lambda s: "%dx%d-%dx%d" % s)
def test_rgb_to_420(emu, size, monkeypatch):
    iw, ih = size[:2]
    for k, (fi, fo) in enumerate([("BGRA", "NV12"), ("RGBA", "I420"), ("ARGB", "NV21"), ("ABGR", "YV12"), ("xRGB", "NV12"), ("BGRx", "I420")]):
        frame = frame_for(fi, iw, ih, 4)
        method = [1, 3, 0, 9, 4, 5][k]
        check(run(emu, fi, fo, size, method, frame), expected(fi, fo, size, method, frame), f"{fi}->{fo} m{method}")
    frame = frame_for("BGRA", iw, ih, 5)
    for col in [(3, 2, 2), (4, 1, 1), (6, 2, 6), (2, 1, 4), (5, 2, 1)]:
        check(run(emu, "BGRA", "NV12", size, 3, frame, colorimetry=col), expected("BGRA", "NV12", size, 3, frame, colorimetry=col),
              f"colorimetry {col}")


@pytest.mark.parametrize("size", SMALL, ids=lambda s: "%dx%d-%dx%d" % s)
def test_422_444_inputs(emu, size, monkeypatch):
    """YUY2 / UYVY / YVYU / Y42B / Y444 -> packed RGB through the generic kernel (luma pitch 2 in the packed formats,
    per-line chroma rows, horizontal-only or no chroma up-sampling)"""
    iw, ih = size[:2]
    for k, fi in enumerate(YUV_422_444):
        frame = frame_for(fi, iw, ih, 10 + k)
        method = [1, 3, 0, 9, 4][k]
        fo = RGB[k]
        for site in (1, 2):
            check(run(emu, fi, fo, size, method, frame, site=site), expected(fi, fo, size, method, frame, site=site),
                  f"{fi}->{fo} m{method} site{site}")


@pytest.mark.parametrize("size", SMALL + [(64, 48, 64, 24), (64, 48, 32, 48)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_rgb_to_rgb(emu, size, monkeypatch):
    iw, ih = size[:2]
    for k, (fi, fo) in enumerate([("BGRA", "BGRA"), ("RGBA", "RGBA"), ("xBGR", "xBGR"), ("BGRA", "RGBA"), ("ARGB", "BGRx"),
                                  ("RGBx", "ABGR"), ("xRGB", "BGRA")]):
        frame = frame_for(fi, iw, ih, 6)
        for method in [[1, 3], [0], [4], [9, 1], [3], [5], [1]][k]:
            check(run(emu, fi, fo, size, method, frame, force_generic=False), expected(fi, fo, size, method, frame), f"{fi}->{fo} m{method}")


@pytest.mark.parametrize("pair", [("NV12", "BGRA"), ("I420", "RGBA"), ("NV12", "NV12"), ("I420", "YV12"), ("NV12", "I420"),
                                  ("YV12", "NV21"), ("BGRA", "NV12"), ("RGBA", "RGBA"), ("BGRA", "ARGB")], ids=lambda p: "%s-%s" % p)
def test_destination_rectangle_and_borders(emu, pair, monkeypatch):
    fi, fo = pair
    rng = np.random.default_rng(9)
    for t in range(6):
        iw, ih, W, H = (int(v) for v in rng.integers(2, 64, 4))
        if t % 2:
            dest = ob.vcs_borders(iw, ih, W, H)
        else:
            dw, dh = int(rng.integers(1, W + 1)), int(rng.integers(1, H + 1))
            dest = (int(rng.integers(0, W - dw + 1)), int(rng.integers(0, H - dh + 1)), dw, dh)
        if dest[2] < 1 or dest[3] < 1:
            continue
        border = [0xff000000, 0x80ff4020, 0xff10c0f0][t % 3]
        method = [1, 3, 0, 9][t % 4]
        frame = frame_for(fi, iw, ih, t)
        size = (iw, ih, W, H)
        generic = not (fi in RGB and fo in RGB)
        got = run(emu, fi, fo, size, method, frame, dest=dest, border=border, force_generic=generic)
        check(got, expected(fi, fo, size, method, frame, dest=dest, border=border), f"{size} dest {dest} m{method}")


def test_odd_height_without_vertical_scaler(emu):
    """the third launch of the cross-family path (device-verified) — keeps the emulator honest about multi-launch glue"""
    for size in [(64, 49, 32, 49), (50, 21, 50, 21), (33, 5, 70, 5)]:
        frame = frame_for("NV12", size[0], size[1], 2)
        for site, out_site in ((1, 1), (2, 1), (1, 6)):
            if size[:2] == size[2:] and site == out_site:
                continue
            got = run(emu, "NV12", "I420", size, 3, frame, site=site, out_site=out_site)
            check(got, expected("NV12", "I420", size, 3, frame, site=site, out_site=out_site), f"{size} {site}->{out_site}")


@pytest.mark.parametrize("size", [(400, 300, 150, 100), (160, 90, 300, 200), (262, 146, 131, 73), (129, 67, 200, 67), (96, 200, 96, 75),
                                  (514, 130, 258, 66), (70, 40, 35, 20)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_planes_fast_kernel(emu, size, monkeypatch):
    """vcs_planes_fast_kernel (the word-wide plane scaler): 1- and 2-byte planes, every pass-mode pair (nearest, bilinear,
    n-tap in either direction), several tiles per plane, odd widths whose last word overhangs the line; and the byte-wise
    kernel (B200_PLANES_SLOW) must agree with the same oracle"""
    iw, ih = size[:2]
    for fi, fo in [("NV12", "NV12"), ("I420", "I420"), ("NV21", "NV21"), ("I420", "YV12")]:
        frame = frame_for(fi, iw, ih, 5)
        for method in (0, 1, 3, 9, 4):
            check(run(emu, fi, fo, size, method, frame), expected(fi, fo, size, method, frame), f"{fi}->{fo} m{method}")


# ---- 2b. the fast kernels (device-verified; here as a CPU regression net for future changes to them) -----------------------
@pytest.mark.parametrize("case", [
    # (in, out, size, method, expected kernel_variant)
    ("NV12", "BGRA", (128, 96, 64, 48), 3, 1), ("NV21", "RGBA", (144, 80, 72, 40), 9, 1),          # lanczos2 (exact 2:1, 8 taps)
    ("NV12", "BGRA", (96, 54, 64, 36), 1, 2), ("I420", "xRGB", (64, 48, 96, 72), 0, 2), ("NV12", "ARGB", (100, 60, 150, 30), 1, 2),
    ("YV12", "BGRA", (64, 48, 64, 48), 1, 2),                                                       # light (copy / 2-tap axes)
    ("NV12", "BGRA", (200, 120, 133, 80), 1, 2), ("NV21", "RGBA", (648, 360, 427, 240), 1, 2),      # light, fast stage A: several tiles,
    ("NV12", "xBGR", (136, 72, 200, 100), 1, 2), ("NV12", "BGRA", (264, 10, 100, 33), 0, 2),        # edges, up-scale, nearest
    ("NV21", "RGBA", (166, 256, 490, 272), 1, 2), ("NV12", "BGRA", (162, 20, 81, 10), 1, 2),        # width % 8 != 0: last odd pixel
    ("NV12", "BGRA", (96, 54, 64, 36), 3, 3), ("I420", "RGBA", (64, 48, 96, 72), 9, 3), ("NV21", "ABGR", (120, 66, 40, 22), 5, 3),
    ("NV12", "BGRA", (100, 60, 150, 30), 3, 3),                                                     # n-tap, both pass orders
    ("NV12", "BGRA", (648, 360, 427, 240), 3, 3), ("NV21", "RGBA", (166, 256, 100, 150), 3, 3),     # n-tap, fast stage A: several
    ("NV12", "xRGB", (200, 120, 300, 90), 9, 3), ("NV12", "BGRA", (264, 40, 100, 33), 5, 3),        # tiles, edges, odd widths, v-first
], ids=lambda c: "%s-%s-%dx%d-%dx%d-m%d-v%d" % (c[0], c[1], *c[2], c[3], c[4]))
def test_fast_kernels(emu, case):
    """vcs_lanczos2_kernel (warp shuffles), vcs_light_kernel (ballot work lists, 16-bit-lane lerps) and the n-tap kernels
    (funnel shifts + dp4a) from their own sources: PTX helpers take their plain-C branch (B200_CUDA_EMU), warp collectives
    are emulated lane by lane"""
    from gstreamer_b200 import _lib
    fi, fo, size, method, variant = case
    iw, ih, W, H = size
    frame = frame_for(fi, iw, ih, 8)
    ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
    emu.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih)
    emu.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], W, H)
    ii.chroma_site = 2
    cfg = _lib.VcsConfigC()
    emu.b200_vcs_config_init(C.byref(cfg))
    cfg.method = method
    h = C.c_void_p()
    assert emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h)) == 0
    try:
        info = _lib.VcsPlanInfoC()
        emu.b200_vcs_get_plan_info(h, C.byref(info))
        assert int(info.kernel_variant) == variant
        out = np.full(W * H * 4, 0x5A, dtype=np.uint8)
        assert emu.b200_vcs_convert(h, frame.ctypes.data, out.ctypes.data, None) == 0
    finally:
        emu.b200_vcs_destroy(h)
    check(out, expected(fi, fo, size, method, frame, site=2), str(case))


# ---- 3. the tensor-path variant of the 2:1 kernel (variant 6, opt-in) ----------------------------------------------------
@pytest.mark.parametrize("size", [(128, 96, 64, 48), (256, 48, 128, 24), (144, 80, 72, 40), (16, 16, 8, 8), (272, 112, 136, 56)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_l2mma_variant(emu, size):
    """vcs_l2mma_kernel: both FIR passes as u8 x s8 banded matrix products (mma.sync.m16n8k32, emulated from the PTX
    fragment layouts), staging, packing and the matrix epilogue — against the oracle for every 8-tap method, both
    semi-planar orders, frame borders on all four sides of every tile"""
    from gstreamer_b200 import _lib
    iw, ih, W, H = size
    for fi, fo, method in [("NV12", "BGRA", 3), ("NV21", "RGBA", 9), ("NV12", "xRGB", 5), ("NV12", "ABGR", 6), ("NV21", "BGRx", 8), ("NV12", "RGBx", 7)]:
        frame = frame_for(fi, iw, ih, 7)
        ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
        emu.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih)
        emu.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], W, H)
        ii.chroma_site = 2                          # h-cosited (the caps default above 576 lines)
        cfg = _lib.VcsConfigC()
        emu.b200_vcs_config_init(C.byref(cfg))
        cfg.method = method
        h = C.c_void_p()
        assert emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h)) == 0
        try:
            assert emu.b200_vcs_set_kernel_variant(h, 6) == 0, "not eligible"
            info = _lib.VcsPlanInfoC()
            emu.b200_vcs_get_plan_info(h, C.byref(info))
            assert int(info.kernel_variant) == 6
            out = np.full(W * H * 4, 0x5A, dtype=np.uint8)
            assert emu.b200_vcs_convert(h, frame.ctypes.data, out.ctypes.data, None) == 0
        finally:
            emu.b200_vcs_destroy(h)
        check(out, expected(fi, fo, size, method, frame, site=2), f"{fi}->{fo} m{method}")


@pytest.mark.parametrize("size", [(512, 144, 256, 72), (256, 240, 128, 120), (496, 128, 248, 64)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_lanczos2_x4_variant(emu, size, monkeypatch):
    """the SIMT 2:1 kernel with its taps times 4 (B200_L2_X4=1): interior tiles and row groups read the scaled tables and
    take the rounded, saturated output as byte 1 of a saturating 16-bit pack; tiles and row groups at a frame border keep
    the plain tables — sizes with interior tiles in both directions"""
    from gstreamer_b200 import _lib
    monkeypatch.setenv("B200_L2_X4", "1")
    iw, ih, W, H = size
    for fi, fo, method in [("NV12", "BGRA", 3), ("NV21", "RGBA", 9)]:
        frame = frame_for(fi, iw, ih, 12)
        ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
        emu.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih)
        emu.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], W, H)
        ii.chroma_site = 2
        cfg = _lib.VcsConfigC()
        emu.b200_vcs_config_init(C.byref(cfg))
        cfg.method = method
        h = C.c_void_p()
        assert emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h)) == 0
        try:
            info = _lib.VcsPlanInfoC()
            emu.b200_vcs_get_plan_info(h, C.byref(info))
            assert int(info.kernel_variant) == 1
            out = np.full(W * H * 4, 0x5A, dtype=np.uint8)
            assert emu.b200_vcs_convert(h, frame.ctypes.data, out.ctypes.data, None) == 0
        finally:
            emu.b200_vcs_destroy(h)
        check(out, expected(fi, fo, size, method, frame, site=2), f"{fi}->{fo} m{method}")


@pytest.mark.parametrize("size", [(512, 248, 256, 124), (752, 376, 376, 188)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_lanczos2_v2_interior_tiles(emu, size):
    """vcs_lanczos2_v2_kernel (the default for plans with uniform interior taps): sizes with tiles that touch no frame border
    in either direction, so the constant-tap H path on the shifted chroma grid, the prefetching item loop and all three row
    group kinds of the V phase run; byte orders with a compile-time selector (BGRA, RGBA) and with the run-time one"""
    from gstreamer_b200 import _lib
    iw, ih, W, H = size
    for fi, fo, method in [("NV12", "BGRA", 3), ("NV21", "RGBA", 9), ("NV12", "ARGB", 5), ("NV21", "xBGR", 3), ("I420", "BGRA", 3),
                           ("YV12", "RGBA", 7), ("I420", "ABGR", 9)]:     # planar input: the kernel's PLANAR instantiation
        frame = frame_for(fi, iw, ih, 21)
        ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
        emu.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih)
        emu.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], W, H)
        ii.chroma_site = 2
        cfg = _lib.VcsConfigC()
        emu.b200_vcs_config_init(C.byref(cfg))
        cfg.method = method
        h = C.c_void_p()
        assert emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h)) == 0
        try:
            info = _lib.VcsPlanInfoC()
            emu.b200_vcs_get_plan_info(h, C.byref(info))
            assert int(info.kernel_variant) == 1
            out = np.full(W * H * 4, 0x5A, dtype=np.uint8)
            assert emu.b200_vcs_convert(h, frame.ctypes.data, out.ctypes.data, None) == 0
        finally:
            emu.b200_vcs_destroy(h)
        check(out, expected(fi, fo, size, method, frame, site=2), f"{fi}->{fo} m{method}")


def test_lanczos2_v2_as_first_launch_of_the_cross_family_chain(emu):
    """exact 2:1 with 8 taps into the OTHER 4:2:0 family: launch 1 is vcs_lanczos2_v2_kernel<YUVOUT> ({255, Y, U, V} pixels, no
    matrix), launch 2 the chroma down-sampler - interior, border and clamped-row tiles, semi-planar and planar inputs"""
    size = (512, 248, 256, 124)
    for fi, fo, method in [("NV12", "I420", 3), ("I420", "NV12", 3), ("NV21", "YV12", 9), ("YV12", "NV21", 6), ("NV12", "NV21", 3)]:
        frame = frame_for(fi, size[0], size[1], 31)
        for site in (2, 3):                          # h-cosited sites: the kernel's chroma up-sampler
            got = run(emu, fi, fo, size, method, frame, site=site)
            check(got, expected(fi, fo, size, method, frame, site=site), f"{fi}->{fo} m{method} site{site}")


# ---- 4. compositor and audio resampler sources under the same emulation --------------------------------------------------
@pytest.mark.parametrize("fmt", ["RGBA", "BGRA", "ARGB", "ABGR"])
@pytest.mark.parametrize("background", [0, 1, 2, 3])
def test_compositor_kernel(emu, fmt, background):
    """comp_kernel (ballot-culled pad list, PRMT blend, reciprocal-multiply overlay) against the oracle"""
    from gstreamer_b200 import _lib
    W, H = 96, 64
    rng = np.random.default_rng(background * 7 + len(fmt))
    n = 5
    pads = (_lib.CompPadC * n)()
    opads = (ob.OraclePad * n)()
    keep = []
    for k in range(n):
        w, h = int(rng.integers(1, 70)), int(rng.integers(1, 50))
        src = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        keep.append(src)
        x, y = int(rng.integers(-30, W)), int(rng.integers(-20, H))
        a, op = float(rng.choice([1.0, 0.5, 0.25, 0.9])), int(rng.integers(0, 3))
        pads[k].data, pads[k].width, pads[k].height, pads[k].stride = src.ctypes.data, w, h, w * 4
        pads[k].xpos, pads[k].ypos, pads[k].alpha, pads[k].op = x, y, a, op
        opads[k].data, opads[k].width, opads[k].height, opads[k].stride = src.ctypes.data, w, h, w * 4
        opads[k].xpos, opads[k].ypos, opads[k].alpha, opads[k].op = x, y, a, op
    want = np.zeros((H, W, 4), dtype=np.uint8)
    ob.oracle().oracle_compositor(ob.FMT[fmt], want.ctypes.data, W, H, W * 4, background, opads, n)
    hc = C.c_void_p()
    assert emu.b200_comp_create(ob.FMT[fmt], W, H, 0, C.byref(hc)) == 0
    out = np.zeros((H, W, 4), dtype=np.uint8)
    try:
        assert emu.b200_comp_blend(hc, out.ctypes.data, W * 4, background, pads, n, None) == 0
    finally:
        emu.b200_comp_destroy(hc)
    check(out.ravel(), want.ravel(), f"{fmt} background {background}")


COMP_YUV_FORMATS = [2, 3, 23, 24, 20, 18, 43, 73, 45, 75, 47, 77, 88]
COMP_YUV_IDS = ["I420", "YV12", "NV12", "NV21", "Y444", "Y42B", "I420_10LE", "I420_12LE", "I422_10LE", "I422_12LE", "Y444_10LE", "Y444_12LE",
                "Y444_16LE"]


@pytest.mark.parametrize("fmt", COMP_YUV_FORMATS, ids=COMP_YUV_IDS)
def test_compositor_420_kernel(emu, fmt):
    """the planar / semi-planar YUV compositor (b200_comp_blend_yuv: per-plane blend, pad positions rounded up to the format's
    grid, round-up chroma rectangles; 8-bit and little-endian 10 / 12 / 16-bit samples) against the oracle: random layouts,
    both ranges, every background, one trial beyond a launch chunk of pads"""
    from gstreamer_b200 import _lib
    o = ob.oracle()
    rng = np.random.default_rng(fmt)
    for trial in range(8):
        W, H, bg, rg = int(rng.integers(1, 120)), int(rng.integers(1, 90)), int(rng.integers(0, 4)), int(rng.integers(0, 2))
        n = int(rng.integers(0, 6)) if trial % 4 else 30
        oi = _lib.VideoInfoC()
        assert emu.b200_video_info_set_format(C.byref(oi), fmt, W, H) == 0
        oi.color_range = 2 if rg else 1
        opads = (ob.OraclePad * max(n, 1))()
        pads = (_lib.CompPadYuvC * max(n, 1))()
        keep = []
        for i in range(n):
            w, h = int(rng.integers(1, 80)), int(rng.integers(1, 60))
            a = rng.integers(0, 256, o.oracle_compositor_yuv_size(fmt, w, h), dtype=np.uint8)
            keep.append(a)
            x, y = int(rng.integers(-40, W + 5)), int(rng.integers(-40, H + 5))
            al, op = float(rng.choice([0.0, 0.3, 0.5, 0.999, 1.0, 0.004])), int(rng.integers(0, 3))
            opads[i].data, opads[i].width, opads[i].height, opads[i].stride = a.ctypes.data, w, h, 0
            opads[i].xpos, opads[i].ypos, opads[i].alpha, opads[i].op = x, y, al, op
            assert emu.b200_video_info_set_format(C.byref(pads[i].info), fmt, w, h) == 0
            pads[i].data, pads[i].xpos, pads[i].ypos, pads[i].alpha, pads[i].op = a.ctypes.data, x, y, al, op
        sz = o.oracle_compositor_yuv_size(fmt, W, H)
        want = np.zeros(sz, dtype=np.uint8)
        assert o.oracle_compositor_yuv(fmt, want.ctypes.data, W, H, bg, rg, opads, n) == 0
        hc = C.c_void_p()
        assert emu.b200_comp_create(fmt, W, H, 0, C.byref(hc)) == 0
        out = np.zeros(sz, dtype=np.uint8)
        try:
            assert emu.b200_comp_blend_yuv(hc, out.ctypes.data, C.byref(oi), bg, pads, n, None) == 0
        finally:
            emu.b200_comp_destroy(hc)
        check(out, want, f"fmt {fmt} trial {trial} {W}x{H} bg {bg} range {rg} pads {n}")


@pytest.mark.parametrize("fmt", ["F32", "S16", "F64"])
def test_audio_nearest_decimation_skip_quirk(emu, fmt, monkeypatch):
    """the product's history after a skip (tests/test_oracle_vs_ref.py::test_audio_nearest_decimation_skip_quirk): part of what
    the reference keeps is what its buffer shift left in place, not the stream's tail"""
    from gstreamer_b200 import _lib
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o = ob.oracle()
    for (a, b, ch) in [(48000, 11025, 3), (96000, 8000, 1), (400, 3, 2)]:
        for seed in range(3):
            rng = np.random.default_rng(seed)
            ho = o.oracle_ars_new_opts(a, b, ch, 4, ofmt, 0, 2, 2)
            cfg = _lib.ArsConfigC()
            cfg.in_rate, cfg.out_rate, cfg.channels, cfg.quality, cfg.format, cfg.resample_method = a, b, ch, 4, gfmt, 1
            h = C.c_void_p()
            assert emu.b200_ars_create(C.byref(cfg), 0, C.byref(h)) == 0
            try:
                for n in [int(v) for v in rng.choice([1, 2, 7, 37, 100, 160, 480], 6)]:
                    x = ob.audio_test_signal(rng, n, ch, fmt)
                    cap = int(n * b / a) + 64
                    want = np.full((cap, ch), 7, dtype=dt)
                    got = want.copy()
                    nw = o.oracle_ars_process_any(ho, x.ctypes.data, n, want.ctypes.data, cap)
                    ng = C.c_size_t()
                    assert emu.b200_ars_process(h, x.ctypes.data, n, got.ctypes.data, cap, C.byref(ng), None) == 0
                    assert ng.value == nw and got.tobytes() == want.tobytes(), (a, b, ch, seed, n)
            finally:
                emu.b200_ars_destroy(h)
                o.oracle_ars_free(ho)


AUDIO_OPTS = [("kaiser", "auto", "cubic"), ("blackman-nuttall", "auto", "cubic"), ("kaiser", "full", "none"),
              ("kaiser", "interpolated", "cubic"), ("blackman-nuttall", "full", "none"), ("kaiser", "interpolated", "none"),
              ("kaiser", "full", "linear"), ("kaiser", "interpolated", "linear"), ("blackman-nuttall", "interpolated", "linear"),
              ("nearest", "auto", "cubic"), ("linear", "auto", "cubic"), ("cubic", "auto", "cubic")]


@pytest.mark.parametrize("fmt", ["F32", "S16", "S32", "F64"])
@pytest.mark.parametrize("opts", AUDIO_OPTS, ids=lambda o: "-".join(o))
def test_audio_kernels(emu, fmt, opts, monkeypatch):
    """the resampler kernels (tiled F32 / S16, direct S32 / F64, interpolated) with the default configuration and with the
    element's resample-method / sinc-filter-* properties, bit for bit against the oracle — the first end-to-end check of
    those option sets through the product's own kernel code"""
    from gstreamer_b200 import _lib
    from gstreamer_b200.audio import CudaAudioResample as A
    method, mode, interp = opts
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o = ob.oracle()
    M = {"nearest": 0, "linear": 1, "cubic": 2, "blackman-nuttall": 3, "kaiser": 4}
    MO = {"interpolated": 0, "full": 1, "auto": 2}
    I = {"none": 0, "linear": 1, "cubic": 2}
    rates = [(48000, 44100, 2, 4), (44100, 48000, 66, 2) if fmt in ("F32", "S16") else (96000, 44100, 1, 6)]
    if M[method] < 3:                                         # tap counts off the lane widths: 3, 12; and the 96k -> 44.1k pair
        rates += [(3, 2, 3, 5), (48000, 8000, 2, 1), (96000, 44100, 1, 6)]
    if opts == AUDIO_OPTS[0]:
        rates += [(44100, 44100, 3, 4)]                       # equal rates: gst_audio_resampler's nearest functions
        if fmt in ("F32", "S16"):
            rates += [(48000, 44100, 128, 4), (44100, 48000, 256, 2)]   # whole 128-channel blocks: the persistent pipelined kernels
    for (a, b, ch, q) in rates:
        ho = o.oracle_ars_new_opts(a, b, ch, q, ofmt, M[method], MO[mode], I[interp])
        cfg = _lib.ArsConfigC()
        cfg.in_rate, cfg.out_rate, cfg.channels, cfg.quality, cfg.format = a, b, ch, q, gfmt
        cfg.resample_method, cfg.sinc_filter_mode, cfg.sinc_filter_interpolation = A.METHODS[method], A.FILTER_MODES[mode], A.INTERPOLATIONS[interp]
        h = C.c_void_p()
        assert emu.b200_ars_create(C.byref(cfg), 0, C.byref(h)) == 0
        rng = np.random.default_rng(a + ch)
        try:
            for n in [300, 100, 1, None]:
                x = None
                if n is None:
                    n = emu.b200_ars_get_max_latency(h)
                else:
                    x = ob.audio_test_signal(rng, n, ch, fmt)
                cap = int(n * b / a) + 64
                want = np.zeros((cap, ch), dtype=dt)
                nw = o.oracle_ars_process_any(ho, x.ctypes.data if x is not None else None, n, want.ctypes.data, cap)
                got = np.full((cap, ch), 7, dtype=dt)
                ng = C.c_size_t()
                assert emu.b200_ars_process(h, x.ctypes.data if x is not None else None, n, got.ctypes.data, cap, C.byref(ng), None) == 0
                assert ng.value == nw and got[:nw].tobytes() == want[:nw].tobytes(), (a, b, ch, q, n)
                assert (got[nw:] == 7).all()
        finally:
            emu.b200_ars_destroy(h)
            o.oracle_ars_free(ho)


@pytest.mark.parametrize("fmt", ["F32", "S16"])
def test_audio_pipeline_many_tiles_per_cta(emu, monkeypatch, fmt):
    """ars_pipe_kernel's stage hand-over (full / empty barriers, two stages): B200_ARS_GRID=2 makes each persistent CTA walk
    a dozen tiles, with start-up zeros, a silent call (no input pointer) and a last partial tile"""
    from gstreamer_b200 import _lib
    monkeypatch.setenv("B200_ARS_GRID", "2")
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o = ob.oracle()
    for (a, b, ch, grid) in [(48000, 44100, 256, "2"), (44100, 48000, 128, "3"), (48000, 44100, 128, "1")]:
        monkeypatch.setenv("B200_ARS_GRID", grid)
        ho = o.oracle_ars_new_fmt(a, b, ch, 4, ofmt)
        cfg = _lib.ArsConfigC()
        cfg.in_rate, cfg.out_rate, cfg.channels, cfg.quality, cfg.format = a, b, ch, 4, gfmt
        h = C.c_void_p()
        assert emu.b200_ars_create(C.byref(cfg), 0, C.byref(h)) == 0
        rng = np.random.default_rng(ch + a)
        try:
            for n in [700, 333, None, 90]:
                x = None
                if n is None:
                    n = 200
                else:
                    x = ob.audio_test_signal(rng, n, ch, fmt)
                cap = int(n * b / a) + 64
                want = np.zeros((cap, ch), dtype=dt)
                nw = o.oracle_ars_process_any(ho, x.ctypes.data if x is not None else None, n, want.ctypes.data, cap)
                got = np.full((cap, ch), 7, dtype=dt)
                ng = C.c_size_t()
                assert emu.b200_ars_process(h, x.ctypes.data if x is not None else None, n, got.ctypes.data, cap, C.byref(ng), None) == 0
                assert ng.value == nw and got[:nw].tobytes() == want[:nw].tobytes(), (a, b, ch, n)
                assert (got[nw:] == 7).all()
        finally:
            emu.b200_ars_destroy(h)
            o.oracle_ars_free(ho)


# ---- 5. the randomised three-way runs (tools/emu_fuzz*.py) keep working: a few seconds of each -------------------------
@pytest.mark.parametrize("tool", ["emu_fuzz.py", "emu_fuzz_audio.py", "emu_fuzz_comp.py"])
def test_random_run_tools(emu, tool):
    """reference build (when present) vs oracle vs emulated kernels on random configurations; the long runs are recorded
    in profiles/r01_race_check.txt"""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "tools", tool), "6", "4"], capture_output=True, text=True, timeout=300)
    last = p.stdout.strip().splitlines()[-1] if p.stdout.strip() else ""
    assert p.returncode == 0 and (" 0 problems" in last or " 0 mismatches" in last), (p.stdout[-600:], p.stderr[-600:])


# ---- 7. variable rate: b200_ars_update on a live stream, emulated kernels vs the oracle ------------------------------------
@pytest.mark.parametrize("fmt", ["F32", "S16", "S32", "F64"])
def test_audio_rate_update(emu, fmt):
    """the product's gst_audio_resampler_update: rescaled phase, phase-error-limited divisor, re-designed filter, history
    moved by half the tap-count change - byte-identical with the oracle across every change"""
    from gstreamer_b200 import _lib
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o = ob.oracle()
    for ch, q, pairs in [(2, 4, [(48000, 44100), (48000, 96000), (48000, 32000), (44100, 48000)]),
                         (3, 6, [(48000, 44100), (48000, 44101), (48001, 44100), (8000, 7999)]),
                         (1, 0, [(96000, 8000), (96000, 44100), (32000, 48000)]),
                         (128, 4, [(48000, 44100), (47999, 44100), (48000, 44100)] if fmt == "F32" else [(48000, 44100), (48000, 44000)])]:
        a, b = pairs[0]
        ho = o.oracle_ars_new_fmt(a, b, ch, q, ofmt)
        cfg = _lib.ArsConfigC()
        cfg.in_rate, cfg.out_rate, cfg.channels, cfg.quality, cfg.format = a, b, ch, q, gfmt
        h = C.c_void_p()
        assert emu.b200_ars_create(C.byref(cfg), 0, C.byref(h)) == 0
        rng = np.random.default_rng(a + ch)
        try:
            for k, (a, b) in enumerate(pairs):
                if k:
                    assert o.oracle_ars_update(ho, a, b) == 0
                    assert emu.b200_ars_update(h, a, b) == 0
                for n in [int(v) for v in rng.choice([1, 7, 160, 481], 3)]:
                    x = ob.audio_test_signal(rng, n, ch, fmt)
                    cap = int(o.oracle_ars_get_out_frames(ho, n)) + 64
                    want = np.zeros((cap, ch), dtype=dt)
                    got = want.copy()
                    nw = o.oracle_ars_process_any(ho, x.ctypes.data, n, want.ctypes.data, cap)
                    ng = C.c_size_t()
                    assert emu.b200_ars_get_out_frames(h, n) == nw
                    assert emu.b200_ars_process(h, x.ctypes.data, n, got.ctypes.data, cap, C.byref(ng), None) == 0
                    assert ng.value == nw and got[:nw].tobytes() == want[:nw].tobytes(), (ch, k, a, b, n)
        finally:
            emu.b200_ars_destroy(h)
            o.oracle_ars_free(ho)


@pytest.mark.parametrize("size", [(400, 300, 150, 100), (160, 90, 300, 200), (262, 146, 131, 73), (129, 67, 200, 67), (96, 200, 96, 75),
                                  (70, 40, 35, 20)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_planes_fast_kernel_packed_rgb(emu, size):
    """the word-wide plane scaler on 4-byte pixels (packed RGB -> packed RGB of the same or another byte order): stage A
    de-interleaves 4 pixels into one word per component, the store re-packs (and re-orders) them"""
    iw, ih = size[:2]
    for k, (fi, fo) in enumerate([("BGRA", "BGRA"), ("RGBA", "BGRA"), ("xRGB", "RGBA"), ("ARGB", "ABGR")]):
        frame = frame_for(fi, iw, ih, 11 + k)
        for method in [(1, 3), (0, 9), (4, 1), (3,)][k]:
            check(run(emu, fi, fo, size, method, frame, force_generic=False), expected(fi, fo, size, method, frame), f"{fi}->{fo} m{method}")


@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (1, 1, 1, 1), (2, 2, 2, 2), (7, 5, 7, 5), (16, 2, 16, 2),
                                  (400, 300, 150, 100), (262, 146, 131, 73), (129, 67, 100, 67), (96, 200, 96, 75), (100, 60, 150, 30),
                                  (70, 40, 35, 20), (41, 23, 17, 9),
                                  (40, 30, 64, 48), (33, 17, 50, 31), (129, 67, 200, 67), (48, 37, 48, 100),
                                  (60, 100, 150, 60)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_rgb_to_420_fast_kernels(emu, size, monkeypatch):
    """vcs_rgb420_kernel (matrix + chroma down-sampling + pack; alone at an unchanged size, behind the word-wide scaler on
    4-byte pixels where the frame shrinks, behind vcs_rgb2ayuv_kernel + that scaler where it grows): every input byte order, both output layouts, co-sited and centred chroma
    sites, full and video range; the generic chain (B200_RGB420_GENERIC) must agree with the same oracle"""
    from gstreamer_b200 import _lib
    iw, ih, W, H = size
    ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
    emu.b200_video_info_set_format(C.byref(ii), ob.FMT["BGRA"], iw, ih)
    emu.b200_video_info_set_format(C.byref(oi), ob.FMT["NV12"], W, H)
    cfg = _lib.VcsConfigC()
    emu.b200_vcs_config_init(C.byref(cfg))
    cfg.method = 1
    h = C.c_void_p()
    assert emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h)) == 0
    emu.b200_vcs_kernel_name.restype = C.c_char_p
    name = emu.b200_vcs_kernel_name(h).decode()
    emu.b200_vcs_destroy(h)
    assert name == "vcs_rgb420_kernel" or min(W, H) < 8, name
    for k, (fi, fo) in enumerate([("BGRA", "NV12"), ("RGBA", "I420"), ("ARGB", "NV21"), ("ABGR", "YV12"), ("xRGB", "NV12"), ("BGRx", "I420")]):
        frame = frame_for(fi, iw, ih, 40 + k)
        for method in [(1, 3), (3,), (0, 9), (4,), (1,), (5,)][k]:
            check(run(emu, fi, fo, size, method, frame), expected(fi, fo, size, method, frame), f"{fi}->{fo} m{method}")
    frame = frame_for("BGRA", iw, ih, 5)
    cols = [(3, 2, 2), (4, 1, 1), (6, 2, 6), (2, 1, 4), (5, 2, 1), (3, 1, 3)]               # (matrix, range, chroma site)
    for col in (cols if W * H < 12000 else cols[(iw + ih) % 3::3]):                         # two of them on the larger frames
        check(run(emu, "BGRA", "NV12", size, 1, frame, colorimetry=col), expected("BGRA", "NV12", size, 1, frame, colorimetry=col),
              f"colorimetry {col}")
    monkeypatch.setenv("B200_RGB420_GENERIC", "1")
    check(run(emu, "BGRA", "NV12", size, 1, frame), expected("BGRA", "NV12", size, 1, frame), "generic chain")


@pytest.mark.parametrize("case", [((100, 60), (160, 120), (31, 17, 100, 60)), ((200, 120), (320, 240), (40, 20, 100, 60)),
                                  ((100, 60), (161, 101), (11, 3, 139, 90)), ((160, 90), (160, 200), (0, 55, 160, 90)),
                                  ((64, 64), (200, 100), (51, 1, 97, 99))], ids=lambda c: "%dx%d-in-%dx%d-%d" % (c[0] + c[1] + c[2][:1]))
def test_rgb_to_420_fast_kernels_destination_rectangle(emu, case):
    """the same kernels writing into a destination rectangle of the output frame (odd origins and sizes included: the plan
    shifts the plane origins, the kernels fall back from word stores to byte stores where the rectangle is unaligned)"""
    (iw, ih), (W, H), dest = case
    pairs = [("BGRA", "NV12"), ("RGBA", "I420"), ("xRGB", "NV21"), ("ABGR", "YV12")]
    for k in ((0, 1) if (dest[0] & 1) else (2, 3)):            # two of the four pairs per case keep the CPU suite short
        fi, fo = pairs[k]
        frame = frame_for(fi, iw, ih, 70 + k)
        method = [1, 3, 0, 9][k]
        size = (iw, ih, W, H)
        got = run(emu, fi, fo, size, method, frame, dest=dest, border=0xff204080)
        check(got, expected(fi, fo, size, method, frame, dest=dest, border=0xff204080), f"{fi}->{fo} m{method} dest {dest}")


@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (1, 1, 1, 1), (2, 3, 2, 3), (130, 34, 130, 34),
                                  (64, 48, 32, 24), (40, 30, 64, 48), (33, 17, 20, 31), (100, 60, 150, 30), (57, 35, 29, 35)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_packed_422_to_420(emu, size):
    """capture -> encoder: YUY2 / UYVY -> I420 / YV12 at an unchanged size is the table row (vcs_yuy2_420_kernel: luma copy in
    whole pairs, avgub of the line pair's chroma); every other pair or size runs the chain with the output size's default
    chroma site: vcs_yuy2_ayuv_kernel (unpack + horizontal chroma up-sampling), the word-wide scaler on the A,Y,U,V pixels,
    vcs_rgb420_kernel<MATRIX = false> (down-sample + pack) - and the generic kernels (B200_RGB420_GENERIC) must agree"""
    import os
    iw, ih, W, H = size
    for k, (fi, fo) in enumerate([("YUY2", "I420"), ("UYVY", "YV12"), ("UYVY", "I420"), ("YVYU", "I420"), ("YUY2", "NV12"),
                                  ("UYVY", "NV21"), ("YVYU", "YV12")]):
        frame = frame_for(fi, iw, ih, 90 + k)
        for method in [(1, 3), (0,), (9,), (4,), (1, 5), (3,), (1,)][k]:
            for site in ((1, 2) if k < 4 else (1 + (method & 1),)):
                want = expected(fi, fo, size, method, frame, site=site)
                check(run(emu, fi, fo, size, method, frame, site=site), want, f"{fi}->{fo} m{method} site{site}")
                if k in (3, 4):
                    os.environ["B200_RGB420_GENERIC"] = "1"
                    try:
                        check(run(emu, fi, fo, size, method, frame, site=site), want, f"generic {fi}->{fo} m{method} site{site}")
                    finally:
                        del os.environ["B200_RGB420_GENERIC"]


def test_packed_422_to_420_unaligned_frame(emu):
    """a frame that does not start on a 4-byte boundary: the table-row kernel falls back to byte loads, the chain to the
    generic kernels (vcs_yuy2_ayuv_kernel reads pixel pairs as words)"""
    for fi, fo, size in [("YUY2", "I420", (50, 22, 50, 22)), ("UYVY", "NV12", (50, 22, 50, 22)), ("YUY2", "NV21", (64, 48, 32, 24))]:
        frame = frame_for(fi, size[0], size[1], 3)
        want = expected(fi, fo, size, 1, frame, site=1)
        for shift in (1, 2):
            buf = np.zeros(frame.size + 8, dtype=np.uint8)
            off = (-buf.ctypes.data) % 4 + shift
            view = buf[off:off + frame.size]
            view[:] = frame
            assert view.ctypes.data % 4 == shift
            check(run(emu, fi, fo, size, 1, view, site=1), want, f"{fi}->{fo} shift {shift}")


@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (2, 3, 2, 3), (64, 48, 32, 24), (40, 30, 64, 48),
                                  (33, 17, 20, 31), (100, 60, 150, 30), (64, 48, 64, 24), (64, 48, 128, 96), (262, 146, 131, 73)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_planar_422_444_to_420(emu, size):
    """Y42B / Y444 -> I420 / YV12: the reference's plane-scaling rows - every output plane from the plane holding the same
    component, chroma planes with their own geometry (4:2:2 -> 4:2:0 at an unchanged size is the line-pair average of
    convert_plane_v_halve, 4:4:4 -> 4:2:0 the 2 x 2 one); plane kernels unchanged, only their geometry is new"""
    for k, (fi, fo) in enumerate([("Y42B", "I420"), ("Y444", "YV12"), ("Y42B", "YV12"), ("Y444", "I420")]):
        frame = frame_for(fi, size[0], size[1], 120 + k)
        for method in [(1, 3), (0, 9), (4,), (1, 5)][k]:
            check(run(emu, fi, fo, size, method, frame, force_generic=False), expected(fi, fo, size, method, frame), f"{fi}->{fo} m{method}")


@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (2, 3, 2, 3), (64, 48, 32, 24), (40, 30, 64, 48),
                                  (33, 17, 20, 31), (100, 60, 150, 30), (57, 35, 29, 35)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_planar_422_444_to_semi_planar_420(emu, size):
    """Y42B / Y444 -> NV12 / NV21: no table row, the chain (generic kernel with the planar 4:2:2 / 4:4:4 input stage, matrix
    off, then vcs_down420_kernel); 4:4:4 has no up-sampler at all - the odd-height corner reads the last line as unpacked"""
    for k, (fi, fo) in enumerate([("Y42B", "NV12"), ("Y444", "NV21"), ("Y444", "NV12"), ("Y42B", "NV21")]):
        frame = frame_for(fi, size[0], size[1], 140 + k)
        for method in [(1, 3), (0, 9), (1,), (4,)][k]:
            for site in (1, 2):
                check(run(emu, fi, fo, size, method, frame, site=site), expected(fi, fo, size, method, frame, site=site),
                      f"{fi}->{fo} m{method} site{site}")


# ---- 8. batches: every slot reads its own frame, one handle serves batches of changing sizes -----------------------------
# (in, out, size, method, kernel variant forced or None, input chroma site, output chroma site, destination rectangle)
BATCH_ROUTES = {
    "generic": ("NV12", "BGRA", (40, 30, 24, 18), 3, 0, 2, None, None),
    "lanczos2-v2": ("NV12", "BGRA", (256, 64, 128, 32), 3, None, 2, None, None),
    "lanczos2-v2-planar": ("I420", "RGBA", (256, 64, 128, 32), 3, None, 2, None, None),
    "light": ("NV12", "BGRA", (96, 54, 64, 36), 1, None, 2, None, None),
    "ntap": ("NV12", "BGRA", (96, 54, 64, 36), 3, None, 2, None, None),
    "l2mma": ("NV12", "BGRA", (128, 48, 64, 24), 3, 6, 2, None, None),
    "planes-fast": ("I420", "YV12", (70, 40, 35, 20), 3, None, None, None, None),
    "chain-lanczos2-v2": ("NV12", "I420", (256, 64, 128, 32), 3, None, 2, None, None),
    "chain-extra-row": ("NV12", "I420", (40, 29, 24, 29), 1, None, 1, 1, None),
    "rgb420": ("BGRA", "NV12", (40, 30, 40, 30), 1, None, None, None, None),
    "rgb420-scaled": ("RGBA", "I420", (48, 36, 24, 18), 3, None, None, None, None),
    "rgb420-pre1": ("BGRA", "NV12", (24, 18, 40, 30), 1, None, None, None, None),
    "rgb420-pre2": ("UYVY", "I420", (48, 36, 24, 18), 1, None, None, 1, None),
    "yuy2-420": ("YUY2", "I420", (40, 30, 40, 30), 1, None, 1, None, None),
    "borders-rgb": ("NV12", "BGRA", (40, 30, 40, 40), 1, None, 1, None, (0, 5, 40, 30)),
    "borders-420": ("NV12", "I420", (40, 30, 40, 40), 1, None, 1, 1, (0, 4, 40, 30)),
}


@pytest.mark.parametrize("route", list(BATCH_ROUTES))
def test_batches_of_distinct_frames(emu, route, monkeypatch):
    """n = 3 distinct frames in one b200_vcs_convert_batch, then n = 2, 5, 1, 5 on the same handle (the chain's and the
    rgb420 pre-pass's scratch images grow, stay, shrink and grow back); every slot against the oracle of its own frame,
    outputs 256 bytes apart with the gaps checked"""
    from gstreamer_b200 import _lib
    fi, fo, size, method, force, site, out_site, dest = BATCH_ROUTES[route]
    iw, ih, W, H = size
    ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
    assert emu.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih) == 0
    assert emu.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], W, H) == 0
    if site is not None:
        ii.chroma_site = site
    if fi in YUV and fo in YUV:
        oi.color_matrix, oi.color_range, oi.chroma_site = ii.color_matrix, ii.color_range, ii.chroma_site
    if fi in YUV_422_444 and fo in YUV:
        oi.color_matrix, oi.color_range = ii.color_matrix, ii.color_range
    if out_site is not None:
        oi.chroma_site = out_site
    cfg = _lib.VcsConfigC()
    emu.b200_vcs_config_init(C.byref(cfg))
    cfg.method = method
    if dest:
        cfg.dest_x, cfg.dest_y, cfg.dest_width, cfg.dest_height = dest
    h = C.c_void_p()
    assert emu.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(h)) == 0
    try:
        if force is not None:
            assert emu.b200_vcs_set_kernel_variant(h, force) == 0
        osz = emu.b200_video_info_size(C.byref(oi))
        pitch = (osz + 256 + 255) & ~255
        seed = 0
        for n in (3, 2, 5, 1, 5):
            frames = [frame_for(fi, iw, ih, 200 + seed + k) for k in range(n)]
            seed += n
            buf = np.full(pitch * n + 256, 0x5A, dtype=np.uint8)
            base = (-buf.ctypes.data) % 256
            ins = (C.c_void_p * n)(*[f.ctypes.data for f in frames])
            outs = (C.c_void_p * n)(*[buf.ctypes.data + base + k * pitch for k in range(n)])
            assert emu.b200_vcs_convert_batch(h, n, ins, outs, None) == 0
            for k, f in enumerate(frames):
                got = buf[base + k * pitch: base + k * pitch + osz]
                want = expected(fi, fo, size, method, f, dest=dest, border=0xff000000, site=site, out_site=out_site) if dest else \
                    expected(fi, fo, size, method, f, site=site, out_site=out_site,
                             colorimetry=(oi.color_matrix, oi.color_range, oi.chroma_site) if fi in RGB and fo in YUV else None)
                check(got, want, f"{route} n={n} slot {k}")
                assert (buf[base + k * pitch + osz: base + (k + 1) * pitch] == 0x5A).all(), f"{route} n={n}: slot {k} wrote past its frame"
    finally:
        emu.b200_vcs_destroy(h)
