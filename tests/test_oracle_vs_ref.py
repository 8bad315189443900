"""Pins the oracle (oracle/*.c, our restatement) against the reference's own sources compiled in
place (oracle/_ref/libgstref.so).

Every result of the reference build a test compares with is stored in tests/golden/ref_pins.npz,
reduced by key() to one 64-bit number (integers as themselves, arrays by a digest of their bytes),
so the comparison runs on any machine.  Where the reference sources are present, rebuild the
library and re-record the file with

    make -C oracle ref && B200_RECORD_REF_PINS=1 python -m pytest -p no:xdist tests/test_oracle_vs_ref.py

which runs the same comparisons against the live reference build while it records."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from oracle import bindings as ob

PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pins.npz")
RECORD = os.environ.get("B200_RECORD_REF_PINS") == "1"
_MASK = (1 << 64) - 1


def key(v):
    """one 64-bit number for a result: an integer stands for itself; an array, a list or a tuple of parts for the first
    8 bytes of the BLAKE2b digest of their shapes and bytes"""
    if isinstance(v, (bool, int, np.integer)):
        return int(v) & _MASK
    h = hashlib.blake2b(digest_size=8)
    for part in (v if isinstance(v, tuple) else (v,)):
        a = np.ascontiguousarray(part)
        h.update(repr(a.shape).encode())
        h.update(a.tobytes())
    return int.from_bytes(h.digest(), "little")


def _load():
    if RECORD:
        return {}, {}
    z = np.load(PINS)
    vals, store, at = z["vals"], {}, 0
    for name, n in zip(z["names"].tolist(), z["counts"].tolist()):
        store[name] = [int(v) for v in vals[at:at + n]]
        at += n
    arrays = {name: z[f"a{i}"] for i, name in enumerate(z["array_names"].tolist())}
    return store, arrays


_STORE, _ARRAYS = _load()


@pytest.fixture(scope="module", autouse=True)
def _write_pins():
    yield
    if RECORD:
        names = sorted(_STORE)
        anames = sorted(_ARRAYS)
        np.savez_compressed(PINS, names=np.array(names), counts=np.array([len(_STORE[n]) for n in names], dtype=np.int64),
                            vals=np.array([v for n in names for v in _STORE[n]], dtype=np.uint64),
                            array_names=np.array(anames, dtype=str), **{f"a{i}": _ARRAYS[n] for i, n in enumerate(anames)})


class Pins:
    """the reference's results in the order one test asks for them: fn() runs against the reference build while recording,
    everywhere else the stored value is read back (a test without stored values fails)"""

    def __init__(self, name):
        self.name, self.k = name, 0

    def __call__(self, fn):
        k, self.k = self.k, self.k + 1
        if RECORD:
            _STORE.setdefault(self.name, []).append(key(fn()))
        return _STORE[self.name][k]

    def array(self, fn):
        """the whole array, for the tests that look inside the reference's output"""
        k, self.k = self.k, self.k + 1
        name = f"{self.name}#{k}"
        if RECORD:
            _ARRAYS[name] = np.ascontiguousarray(fn())
        return _ARRAYS[name]


@pytest.fixture
def pin(request):
    return Pins(request.node.name)


def live():
    """the reference build itself, only while recording"""
    return ob.ref() if RECORD else None


def ref_convert(pin, frame, *args, out_size=None, **kw):
    """key of the reference converter's output for one frame (ob.RefVcs arguments)"""
    def run():
        r = ob.RefVcs(*args, **kw)
        try:
            return r.convert(frame, None if out_size is None else np.zeros(out_size, dtype=np.uint8))
        finally:
            r.close()
    return pin(run)


def _info(fn, h):
    v = [C.c_int() for _ in range(6)]
    fn(h, *[C.byref(t) for t in v])
    return [t.value for t in v]


# the reference element test's size matrix (tests/check/elements/videoscale.c:451-492) and more
SIZES = [(640, 480, 320, 240), (320, 240, 640, 480), (641, 481, 111, 30), (111, 30, 641, 481),
         (641, 481, 30, 111), (30, 111, 641, 481), (1, 1, 1, 1), (2, 2, 1, 1), (1, 1, 2, 2), (16, 16, 16, 16),
         (100, 100, 50, 150), (3, 5, 7, 2), (17, 33, 64, 7), (640, 480, 641, 481), (1920, 1080, 1280, 720)]


def _vfirst(iw, ih, ow, oh):
    return ih != oh and (iw == ow or ow * ih > iw * oh)


@pytest.mark.parametrize("size", SIZES, ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("method", range(10))
def test_video_matches_reference(size, method, pin):
    iw, ih, ow, oh = size
    frame = ob.nv12_random_frame(iw, ih, seed=iw + 3 * oh + method)
    want = ref_convert(pin, frame, iw, ih, ow, oh, method)
    got = key(ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, method), frame))
    if _vfirst(iw, ih, ow, oh) and got != want:
        pytest.xfail("reference ring aliasing (vertical-first chain); see test_vertical_first_two_step")
    assert got == want


@pytest.mark.parametrize("size", [(100, 100, 150, 50), (641, 481, 640, 480), (720, 480, 640, 360), (17, 33, 64, 7), (40, 90, 40, 31),
                          (64, 64, 64, 32)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("method", [3, 4, 5, 6, 9])
def test_vertical_first_two_step(size, method, pin):
    """On vertical-first chains the reference's unpack ring is one line short and a tap reads a
    recycled line.  Its INTENDED arithmetic is pinned by composing two reference runs that
    cannot alias: NV12 -> AYUV at the same size (chroma up-sampling only), then AYUV -> BGRA with
    scaling (identity unpack, no temp-line ring in front of the vertical scaler)."""
    iw, ih, ow, oh = size
    assert _vfirst(iw, ih, ow, oh)
    d = ob.vcs_desc(iw, ih, ow, oh, method)
    frame = ob.nv12_random_frame(iw, ih, seed=7)

    def two_step():
        r1 = ob.RefVcs(iw, ih, iw, ih, method, out_fmt=ob.FMT["AYUV"], matrix=d.in_matrix, rng=d.in_range,
                       site=d.in_chroma_site, out_matrix=d.in_matrix, out_rng=d.in_range, out_site=0)
        ayuv = r1.convert(frame)
        r1.close()
        r2 = ob.RefVcs(iw, ih, ow, oh, method, in_fmt=ob.FMT["AYUV"], matrix=d.in_matrix, rng=d.in_range, site=0)
        out = r2.convert(ayuv)
        r2.close()
        return out
    want = pin(two_step)
    got = ob.oracle_vcs_convert(d, frame)
    assert key(got) == want


@pytest.mark.parametrize("in_fmt", ["NV12", "NV21"])
@pytest.mark.parametrize("out_fmt", ["RGBx", "BGRx", "xRGB", "xBGR", "RGBA", "BGRA", "ARGB", "ABGR"])
def test_video_formats(in_fmt, out_fmt, pin):
    iw, ih, ow, oh = 98, 66, 45, 37
    frame = ob.nv12_random_frame(iw, ih, 5)
    want = ref_convert(pin, frame, iw, ih, ow, oh, 3, in_fmt=ob.FMT[in_fmt], out_fmt=ob.FMT[out_fmt])
    got = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, 3, in_fmt=ob.FMT[in_fmt], out_fmt=ob.FMT[out_fmt]), frame)
    assert key(got) == want


PLANAR_SIZES = [(640, 480, 320, 240), (320, 240, 640, 480), (641, 481, 111, 30), (64, 48, 64, 48), (65, 49, 65, 49),
                (1, 1, 1, 1), (2, 2, 2, 2), (3, 5, 7, 2), (17, 33, 64, 7), (1920, 1080, 1280, 720), (30, 111, 641, 481)]


@pytest.mark.parametrize("size", PLANAR_SIZES, ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("method", [0, 1, 3, 9])
@pytest.mark.parametrize("in_fmt", ["I420", "YV12"])
def test_planar_420_matches_reference(in_fmt, size, method, pin):
    """I420 / YV12: unpack_I420 in front of the same chain; at unchanged size the reference takes its
    convert_I420_BGRA family fast path (nearest chroma), video-converter.c:8766-8800"""
    iw, ih, ow, oh = size
    frame = ob.i420_random_frame(iw, ih, seed=iw + oh + method)
    want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[in_fmt])
    got = key(ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[in_fmt]), frame))
    if _vfirst(iw, ih, ow, oh) and got != want:
        pytest.xfail("reference ring aliasing (vertical-first chain)")
    assert got == want


@pytest.mark.parametrize("in_fmt", ["I420", "YV12"])
@pytest.mark.parametrize("out_fmt", ["RGBx", "BGRx", "xRGB", "xBGR", "RGBA", "BGRA", "ARGB", "ABGR"])
@pytest.mark.parametrize("size", [(98, 66, 45, 37), (98, 66, 98, 66)], ids=["scaled", "same-size"])
@pytest.mark.parametrize("matrix,rng,site", [(3, 2, 2), (4, 1, 1), (6, 2, 6), (2, 1, 4)])
def test_planar_420_formats_and_colorimetry(in_fmt, out_fmt, size, matrix, rng, site, pin):
    iw, ih, ow, oh = size
    frame = ob.i420_random_frame(iw, ih, 5)
    kw = dict(in_fmt=ob.FMT[in_fmt], out_fmt=ob.FMT[out_fmt], site=site, matrix=matrix, rng=rng)
    want = ref_convert(pin, frame, iw, ih, ow, oh, 3, **kw)
    got = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, 3, **kw), frame)
    assert key(got) == want


@pytest.mark.parametrize("site", [1, 2, 4, 6])
@pytest.mark.parametrize("matrix,rng", [(3, 2), (4, 2), (4, 1), (6, 2), (2, 1), (5, 2)])
def test_video_colorimetry_and_siting(site, matrix, rng, pin):
    iw, ih, ow, oh = 130, 74, 65, 37
    frame = ob.nv12_random_frame(iw, ih, site + matrix)
    want = ref_convert(pin, frame, iw, ih, ow, oh, 3, site=site, matrix=matrix, rng=rng)
    got = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, 3, site=site, matrix=matrix, rng=rng), frame)
    assert key(got) == want


@pytest.mark.parametrize("size", [(64, 48, 40, 30), (64, 48, 100, 70), (64, 48, 64, 48), (130, 74, 65, 37)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("in_fmt", ["NV12", "I420"])
def test_default_converter_is_mitchell(size, in_fmt, pin):
    """a GstVideoAggregatorConvertPad builds its converter with NO options (gstvideoaggregator.c:508-513):
    cubic b = c = 1/3, exactly what the element's method=mitchell sets"""
    iw, ih, ow, oh = size
    frame = ob.i420_random_frame(iw, ih, 3) if in_fmt == "I420" else ob.nv12_random_frame(iw, ih, 3)
    a = ref_convert(pin, frame, iw, ih, ow, oh, -1, in_fmt=ob.FMT[in_fmt])
    b = ref_convert(pin, frame, iw, ih, ow, oh, 9, in_fmt=ob.FMT[in_fmt])
    assert a == b
    if not _vfirst(iw, ih, ow, oh):
        assert key(ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, 9, in_fmt=ob.FMT[in_fmt]), frame)) == a


def test_reference_threads_equal_single_thread(pin):
    """the reference's own invariant (tests/check/libs/video.c:3189-3260) holds for our build of it
    on the headline shape: n-threads=4 output == n-threads=1 output (and == the oracle's)"""
    iw, ih, ow, oh = 1920, 1080, 960, 540
    frame = ob.nv12_random_frame(iw, ih, 1)
    a = pin(lambda: ob.RefVcs(iw, ih, ow, oh, 3, n_threads=1).convert(frame))
    b = pin(lambda: ob.RefVcs(iw, ih, ow, oh, 3, n_threads=4).convert(frame))
    assert a == b
    assert key(ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, 3), frame)) == a


def test_compositor_matches_reference(pin):
    rng = np.random.default_rng(7)
    o = ob.oracle()
    for trial in range(150):
        W, H = int(rng.integers(1, 90)), int(rng.integers(1, 70))
        fmt, bg = int(rng.choice([11, 12, 13, 14])), int(rng.integers(0, 4))
        n = int(rng.integers(0, 6))
        pads = (ob.OraclePad * max(n, 1))()
        keep = []
        for i in range(n):
            w, h = int(rng.integers(1, 60)), int(rng.integers(1, 50))
            a = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
            keep.append(a)
            pads[i].data, pads[i].width, pads[i].height, pads[i].stride = a.ctypes.data, w, h, w * 4
            pads[i].xpos, pads[i].ypos = int(rng.integers(-30, W + 5)), int(rng.integers(-30, H + 5))
            pads[i].alpha, pads[i].op = float(rng.choice([0.0, 0.3, 0.5, 0.999, 1.0, 0.004])), int(rng.integers(0, 3))
        d1 = np.full((H, W, 4), 0x77, dtype=np.uint8)
        d2 = d1.copy()
        want = pin(lambda: (live().ref_compositor(fmt, d1.ctypes.data, W, H, W * 4, bg, pads, n), d1)[1])
        o.oracle_compositor(fmt, d2.ctypes.data, W, H, W * 4, bg, pads, n)
        assert key(d2) == want, f"trial {trial}"


@pytest.mark.parametrize("cfg", [(48000, 44100, 2, 4), (44100, 48000, 3, 4), (8000, 16000, 1, 4), (48000, 24000, 2, 4),
                                 (12345, 54321, 2, 4), (101, 99, 1, 4), (44100, 8000, 2, 10), (48000, 96000, 2, 0),
                                 (96000, 8000, 1, 7), (22050, 48000, 2, 9), (48000, 44100, 256, 4),
                                 # interpolated filter mode (phase table would exceed 1 MiB)
                                 (44100, 48001, 2, 4), (48000, 44101, 1, 6), (96000, 8001, 2, 3), (7999, 48000, 3, 10)],
                         ids=lambda c: "%d-%d-%dch-q%d" % c)
def test_audio_matches_reference(cfg, pin):
    a, b, ch, q = cfg
    o, r = ob.oracle(), live()
    ho, hr = o.oracle_ars_new(a, b, ch, q), (r.ref_ars_new(a, b, ch, q) if r else None)
    io = _info(o.oracle_ars_info, ho)
    assert key(io) == pin(lambda: _info(r.ref_ars_info, hr))
    if io[4] == 1:
        for ph in sorted({0, 1, io[1] // 2, io[1] - 1}):
            t1 = np.zeros(io[0], dtype=np.float32)
            t2 = t1.copy()
            o.oracle_ars_phase_taps(ho, ph, t1.ctypes.data)
            assert key(t1) == pin(lambda: (r.ref_ars_phase_taps(hr, ph, t2.ctypes.data), t2)[1])
    rng = np.random.default_rng(a + b)
    for n in [480, 480, 100, 1, 2000, None]:
        x = None
        if n is None:
            n = io[0] // 2        # drain: push silence like the element (gstaudioresample.c:590-662)
        else:
            x = rng.standard_normal((n, ch)).astype(np.float32)
        cap = int(n * b / a) + 64
        o1 = np.zeros((cap, ch), dtype=np.float32)
        o2 = o1.copy()
        n1 = o.oracle_ars_process(ho, x.ctypes.data if x is not None else None, n, o1.ctypes.data, cap)

        def ref_process():
            n2 = r.ref_ars_process(hr, x.ctypes.data if x is not None else None, n, o2.ctypes.data, cap)
            return n2, o2[:n2]
        assert key((n1, o1[:n1])) == pin(ref_process), n
    o.oracle_ars_free(ho)
    if r:
        r.ref_ars_free(hr)


@pytest.mark.parametrize("cfg", [(48000, 44100, 2, 4), (44100, 48000, 3, 4), (8000, 16000, 1, 4), (48000, 24000, 2, 4),
                                 (101, 99, 1, 4), (44100, 8000, 2, 10), (48000, 96000, 2, 0), (96000, 8000, 1, 7),
                                 (12345, 54321, 2, 4), (44100, 48001, 2, 4), (48000, 44101, 1, 6), (96000, 8001, 2, 3),
                                 (7999, 48000, 3, 10), (48000, 44100, 64, 4)],
                         ids=lambda c: "%d-%d-%dch-q%d" % c)
@pytest.mark.parametrize("fmt", ["S16", "S32", "F64"])
def test_audio_sample_formats_match_reference(fmt, cfg, pin):
    """S16 / S32 / F64: integer tap quantisation, integer cubic coefficients, the SSE2 / SSE4.1 inner products
    (audio-resampler-x86-sse2.c, -sse41.c) in FULL and interpolated filter modes — byte-identical output"""
    a, b, ch, q = cfg
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o, r = ob.oracle(), live()
    ho, hr = o.oracle_ars_new_fmt(a, b, ch, q, ofmt), (r.ref_ars_new_fmt(a, b, ch, q, gfmt) if r else None)
    io = _info(o.oracle_ars_info, ho)
    assert key(io) == pin(lambda: _info(r.ref_ars_info, hr))
    rng = np.random.default_rng(a + b)
    for n in [480, 480, 100, 1, 2000, None]:
        x = None
        if n is None:
            n = io[0] // 2
        else:
            x = ob.audio_test_signal(rng, n, ch, fmt)
        cap = int(n * b / a) + 64
        o1 = np.zeros((cap, ch), dtype=dt)
        o2 = o1.copy()
        n1 = o.oracle_ars_process_any(ho, x.ctypes.data if x is not None else None, n, o1.ctypes.data, cap)

        def ref_process():
            n2 = r.ref_ars_process(hr, x.ctypes.data if x is not None else None, n, o2.ctypes.data, cap)
            return n2, o2[:n2]
        assert key((n1, o1[:n1])) == pin(ref_process), n
    o.oracle_ars_free(ho)
    if r:
        r.ref_ars_free(hr)


def test_compositor_420_matches_reference(pin):
    """I420 / YV12 / NV12 / NV21 output: blend.c PLANAR_YUV_BLEND / NV_YUV_BLEND rectangle arithmetic,
    compositor_orc_blend_u8, the four backgrounds — random layouts, byte-identical frames"""
    o = ob.oracle()
    rng = np.random.default_rng(11)
    for trial in range(200):
        fmt = int(rng.choice([2, 3, 23, 24]))
        W, H, bg, rg = int(rng.integers(1, 90)), int(rng.integers(1, 70)), int(rng.integers(0, 4)), int(rng.integers(0, 2))
        n = int(rng.integers(0, 5))
        pads = (ob.OraclePad * max(n, 1))()
        keep = []
        for i in range(n):
            w, h = int(rng.integers(1, 60)), int(rng.integers(1, 50))
            a = rng.integers(0, 256, o.oracle_compositor_yuv_size(fmt, w, h), dtype=np.uint8)
            keep.append(a)
            pads[i].data, pads[i].width, pads[i].height, pads[i].stride = a.ctypes.data, w, h, 0
            pads[i].xpos, pads[i].ypos = int(rng.integers(-30, W + 5)), int(rng.integers(-30, H + 5))
            pads[i].alpha, pads[i].op = float(rng.choice([0.0, 0.3, 0.5, 0.999, 1.0, 0.004])), int(rng.integers(0, 3))
        sz = o.oracle_compositor_yuv_size(fmt, W, H)
        d1 = np.zeros(sz, dtype=np.uint8)
        d2 = d1.copy()
        # (status, frame): the reference must return 0 too
        want = pin(lambda: (live().ref_compositor_yuv(fmt, d1.ctypes.data, W, H, bg, rg, pads, n), d1))
        assert o.oracle_compositor_yuv(fmt, d2.ctypes.data, W, H, bg, rg, pads, n) == 0
        assert key((0, d2)) == want, f"trial {trial}"


@pytest.mark.parametrize("fmt", [20, 18, 43, 73, 45, 75, 47, 77, 88], ids=["Y444", "Y42B", "I420_10LE", "I420_12LE", "I422_10LE", "I422_12LE",
                                                                         "Y444_10LE", "Y444_12LE", "Y444_16LE"])
def test_compositor_planar_444_422_and_high_depth_match_reference(fmt, pin):
    """the other PLANAR_YUV_BLEND instantiations (blend.c:596-646): Y444 / Y42B at 8 bits, the little-endian 10 / 12 / 16-bit
    I420 / I422 / Y444 families with compositor_orc_blend_u10 / _u12 / _u16 (32-bit wrapping arithmetic), their x / y
    rounding, chroma rectangles, checker / black / white / transparent backgrounds at the format's depth - random layouts
    with samples over the whole 16-bit range (the reference does not mask them either), byte-identical frames"""
    o = ob.oracle()
    rng = np.random.default_rng(100 + fmt)
    for trial in range(120):
        W, H, bg, rg = int(rng.integers(1, 90)), int(rng.integers(1, 70)), int(rng.integers(0, 4)), int(rng.integers(0, 2))
        n = int(rng.integers(0, 5))
        pads = (ob.OraclePad * max(n, 1))()
        keep = []
        for i in range(n):
            w, h = int(rng.integers(1, 60)), int(rng.integers(1, 50))
            a = rng.integers(0, 256, o.oracle_compositor_yuv_size(fmt, w, h), dtype=np.uint8)
            keep.append(a)
            pads[i].data, pads[i].width, pads[i].height, pads[i].stride = a.ctypes.data, w, h, 0
            pads[i].xpos, pads[i].ypos = int(rng.integers(-30, W + 5)), int(rng.integers(-30, H + 5))
            pads[i].alpha, pads[i].op = float(rng.choice([0.0, 0.3, 0.5, 0.999, 1.0, 0.004, 0.00002])), int(rng.integers(0, 3))
        sz = o.oracle_compositor_yuv_size(fmt, W, H)
        assert sz > 0
        d1 = np.full(sz, 0xA5, dtype=np.uint8)          # stride padding must stay untouched in both
        d2 = d1.copy()
        want = pin(lambda: (live().ref_compositor_yuv(fmt, d1.ctypes.data, W, H, bg, rg, pads, n), d1))
        assert o.oracle_compositor_yuv(fmt, d2.ctypes.data, W, H, bg, rg, pads, n) == 0
        assert key((0, d2)) == want, f"trial {trial}"


YUV_PAIRS = [("NV12", "NV12"), ("NV21", "NV21"), ("I420", "I420"), ("YV12", "YV12"), ("I420", "YV12"), ("YV12", "I420")]
YUV_SIZES = [(64, 48, 32, 24), (64, 48, 128, 96), (64, 48, 40, 30), (64, 48, 100, 70), (65, 49, 33, 25), (33, 17, 20, 9),
             (64, 48, 64, 24), (64, 48, 32, 48), (64, 48, 64, 96), (64, 48, 128, 48), (640, 480, 320, 240), (320, 240, 640, 480),
             (1920, 1080, 1280, 720), (100, 100, 50, 150), (3, 5, 7, 2), (2, 2, 1, 1), (1, 1, 2, 2), (16, 16, 16, 16)]


@pytest.mark.parametrize("size", YUV_SIZES, ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("pair", YUV_PAIRS, ids=lambda p: "%s-%s" % p)
def test_yuv_plane_scaling_matches_reference(pair, size, pin):
    """convert_scale_planes (video-converter.c:7757-7769, setup_scale :7958-8245, gst_video_scaler_2d
    video-scaler.c:1451-1640): per-plane scalers, linear chroma resampler, halve / double kernels, both 2-D
    pass orders, all ten element methods"""
    iw, ih, ow, oh = size
    fi, fo = ob.FMT[pair[0]], ob.FMT[pair[1]]
    frame = ob.i420_random_frame(iw, ih, 5) if pair[0] in ("I420", "YV12") else ob.nv12_random_frame(iw, ih, 5)
    for m in range(10):
        got = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, m, in_fmt=fi, out_fmt=fo), frame)
        want = ref_convert(pin, frame, iw, ih, ow, oh, m, in_fmt=fi, out_fmt=fo, out_size=got.size)
        assert key(got) == want, f"method {m}"


def _one_tap_vertical_repeat(iw, ih, ow, oh, method):
    """1-tap vertical pass (nearest, or a 1-line input) that repeats source lines, with the matrix after the scalers"""
    return (method == 0 or ih == 1) and oh > ih and ow * oh <= iw * ih


@pytest.mark.parametrize("size", [(64, 2, 16, 3), (64, 8, 16, 9), (202, 12, 40, 51), (128, 5, 40, 6)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_one_tap_vertical_repeat_defect_is_double_conversion(size, pin):
    """Second reference defect we do NOT reproduce: with a 1-tap vertical pass the reference hands the cached h-scaled
    line itself downstream, and the in-place AYUV->ARGB matrix then converts that cached line; every later output row
    that repeats the same source line is converted AGAIN (ARGB output, where pack is the identity).  Pinned here: each
    row where the reference differs is exactly matrix(our row) — i.e. our row is the reference's own single conversion."""
    iw, ih, ow, oh = size
    assert _one_tap_vertical_repeat(iw, ih, ow, oh, 0)
    frame = ob.nv12_random_frame(iw, ih, 1)
    d = ob.vcs_desc(iw, ih, ow, oh, 0, in_fmt=23, out_fmt=13)
    ours = ob.oracle_vcs_convert(d, frame).reshape(oh, ow, 4)

    def run():
        r = ob.RefVcs(iw, ih, ow, oh, 0, in_fmt=23, out_fmt=13)
        out = r.convert(frame)
        r.close()
        return out
    ref = pin.array(run).reshape(oh, ow, 4)
    p = (C.c_int * 5)()
    im = ((C.c_int * 4) * 4)()
    ob.oracle().oracle_vcs_matrix(C.byref(d), p, im)
    p = list(p)

    def splat(v):
        sb = (v - 128) & 0xff
        w = (sb << 8) | sb
        return w - 65536 if w >= 32768 else w

    def matrix(px):                      # video_orc_convert_AYUV_ARGB on one pixel held as (A, Y, U, V)
        a, y, u, v = (int(t) for t in px)
        wy = (splat(y) * p[0]) >> 16
        rr = wy + ((splat(v) * p[1]) >> 16)
        bb = wy + ((splat(u) * p[2]) >> 16)
        gg = wy + ((splat(u) * p[3]) >> 16) + ((splat(v) * p[4]) >> 16)
        cl = lambda t: max(-128, min(127, t)) + 128
        return [a, cl(rr), cl(gg), cl(bb)]

    bad_rows = [y for y in range(oh) if np.any(ours[y] != ref[y])]
    assert bad_rows, "the defect should show on this shape"
    for y in bad_rows:
        assert y > 0 and np.array_equal(np.array([matrix(px) for px in ours[y]], dtype=np.uint8), ref[y])
    # the first output row of every source line is converted once by both
    assert np.array_equal(ours[0], ref[0])


# ------------------------------------------------------------------- 4:2:0 -> the other 4:2:0 family (generic chain)
CROSS_PAIRS = [("NV12", "I420"), ("I420", "NV12"), ("NV12", "NV21"), ("NV21", "YV12"), ("YV12", "NV21"), ("I420", "NV21")]
CROSS_SIZES = [(64, 48, 32, 24), (64, 48, 96, 72), (33, 17, 20, 31), (50, 21, 50, 21), (57, 35, 29, 35), (40, 33, 57, 33),
               (320, 240, 213, 120), (17, 9, 64, 31), (2, 2, 1, 1), (1, 1, 5, 4)]


def _cross(pin, pair, size, method, site, out_site=None, seed=3):
    iw, ih, ow, oh = size
    fi, fo = ob.FMT[pair[0]], ob.FMT[pair[1]]
    frame = ob.i420_random_frame(iw, ih, seed) if pair[0] in ("I420", "YV12") else ob.nv12_random_frame(iw, ih, seed)
    d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=fi, out_fmt=fo, site=site)
    if out_site is not None:
        d.out_chroma_site = out_site
    got = ob.oracle_vcs_convert(d, frame)
    # the element's caps fixation carries colorimetry (and, for an unchanged sub-sampling, the chroma site) over from
    # the input caps (gstvideoconvertscale.c:1335-1427): same matrix on both sides -> no matrix stage in the chain
    want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=fi, out_fmt=fo, site=site, matrix=d.in_matrix,
                       out_matrix=d.in_matrix, out_site=site if out_site is None else out_site, out_size=got.size)
    return key(got), want


def _one_tap_vertical_inplace(ih, oh, method):
    """the chroma down-sampler filters IN PLACE the line the 1-tap vertical pass handed through, so a repeated source
    line is filtered once per repeat (same defect class as the in-place matrix above)"""
    return (method == 0 or ih == 1) and oh > ih


@pytest.mark.parametrize("pair", CROSS_PAIRS, ids=lambda p: "%s-%s" % p)
@pytest.mark.parametrize("size", CROSS_SIZES, ids=lambda s: "%dx%d-%dx%d" % s)
def test_cross_family_420_matches_reference(pair, size, pin):
    """unpack -> chroma up -> scalers -> chroma DOWN (video-converter.c:2018-2032, :3194-3222; video-chroma.c:398-442,
    :742-785) -> pack_planar_420 / pack_NV12 / pack_NV21, all ten element methods, both default chroma sites"""
    iw, ih, ow, oh = size
    for method in range(10):
        for site in (1, 2):
            got, want = _cross(pin, pair, size, method, site)
            if got != want:
                if _vfirst(iw, ih, ow, oh) or _one_tap_vertical_inplace(ih, oh, method):
                    continue            # the two reference defect classes; intended arithmetic pinned below
                assert False, f"method {method} site {site}"


@pytest.mark.parametrize("site,out_site", [(1, 2), (2, 1), (6, 2), (2, 4), (4, 6), (1, 6)])
@pytest.mark.parametrize("size", [(64, 48, 32, 24), (33, 17, 20, 31), (50, 21, 50, 21), (57, 35, 29, 35), (40, 33, 57, 33)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_cross_family_420_output_chroma_site(size, site, out_site, pin):
    """a different output site picks the other down filters (co-sited horizontal 3-1 / 1-2-1 / 1-3; the vertical
    co-sited one is the reference's unimplemented resampler) and turns on both resamplers even at the same size"""
    iw, ih, ow, oh = size
    for method in (1, 3, 9):
        got, want = _cross(pin, ("NV12", "I420"), size, method, site, out_site)
        if _vfirst(iw, ih, ow, oh) and got != want:
            continue
        assert got == want, f"method {method}"


@pytest.mark.parametrize("size", [(100, 100, 150, 50), (64, 66, 64, 31), (40, 90, 40, 31), (48, 68, 36, 12)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("method", [3, 4, 5, 9])
def test_cross_family_420_vertical_first_two_step(size, method, pin):
    """vertical-first chains: the intended arithmetic, pinned by two reference runs that cannot alias
    (NV12 -> AYUV at the same size, then AYUV -> I420 with scaling and chroma down-sampling).  Filters whose
    vertical windows skip source lines are left out: the first run would pair chroma rows in a different pull order."""
    iw, ih, ow, oh = size
    assert _vfirst(iw, ih, ow, oh)
    d = ob.vcs_desc(iw, ih, ow, oh, method, out_fmt=ob.FMT["I420"])
    frame = ob.nv12_random_frame(iw, ih, seed=11)
    got = ob.oracle_vcs_convert(d, frame)

    def two_step():
        r1 = ob.RefVcs(iw, ih, iw, ih, method, out_fmt=ob.FMT["AYUV"], matrix=d.in_matrix, rng=d.in_range,
                       site=d.in_chroma_site, out_matrix=d.in_matrix, out_rng=d.in_range, out_site=0)
        ayuv = r1.convert(frame)
        r1.close()
        r2 = ob.RefVcs(iw, ih, ow, oh, method, in_fmt=ob.FMT["AYUV"], out_fmt=ob.FMT["I420"], matrix=d.in_matrix,
                       rng=d.in_range, site=0, out_matrix=d.in_matrix, out_rng=d.in_range, out_site=d.in_chroma_site)
        out = r2.convert(ayuv, np.zeros(got.size, dtype=np.uint8))
        r2.close()
        return out
    assert key(got) == pin(two_step)


def test_cross_family_420_differing_matrix_is_refused():
    d = ob.vcs_desc(64, 48, 32, 24, 1, out_fmt=ob.FMT["I420"])
    d.out_matrix = 4 if d.in_matrix == 3 else 3
    with pytest.raises(RuntimeError):
        ob.oracle_vcs_convert(d, ob.nv12_random_frame(64, 48, 1))


# ------------------------------------------------------------------- packed RGB -> 4:2:0 (the encoder-feeding direction)
RGB_IN = ["BGRA", "RGBA", "ARGB", "ABGR", "BGRx", "RGBx", "xRGB", "xBGR"]


def _rgb_frame(iw, ih, seed):
    return np.random.default_rng(seed).integers(0, 256, iw * ih * 4, dtype=np.uint8)


@pytest.mark.parametrize("fi", RGB_IN)
@pytest.mark.parametrize("fo", ["I420", "YV12", "NV12", "NV21"])
@pytest.mark.parametrize("size", [(64, 48, 32, 24), (64, 48, 96, 72), (33, 17, 20, 31), (50, 21, 50, 21), (57, 35, 29, 35),
                                  (100, 100, 150, 50), (40, 90, 40, 31), (1, 1, 5, 4), (2, 3, 1, 1)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_rgb_to_420_matches_reference(fi, fo, size, pin):
    """unpack to ARGB -> scalers that shrink -> RGB->YUV matrix (video_converter_matrix8_table) -> scalers that grow ->
    chroma down-sampling -> 4:2:0 pack; output colorimetry = the caps defaults of the output size.  No chroma
    up-sampler in this chain, so vertical-first geometries are compared directly too."""
    iw, ih, ow, oh = size
    frame = _rgb_frame(iw, ih, 3)
    for method in range(10):
        got = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo]), frame)
        want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], out_size=got.size)
        if _one_tap_vertical_inplace(ih, oh, method) and key(got) != want:
            continue
        assert key(got) == want, f"method {method}"


@pytest.mark.parametrize("matrix", [2, 3, 4, 5, 6])
@pytest.mark.parametrize("rng", [1, 2])
@pytest.mark.parametrize("site", [1, 2, 4, 6])
def test_rgb_to_420_colorimetry(matrix, rng, site, pin):
    for (iw, ih, ow, oh) in [(64, 48, 40, 30), (40, 30, 64, 48), (33, 33, 33, 33)]:
        frame = _rgb_frame(iw, ih, 5)
        d = ob.vcs_desc(iw, ih, ow, oh, 3, in_fmt=ob.FMT["BGRA"], out_fmt=ob.FMT["NV12"])
        d.out_matrix, d.out_range, d.out_chroma_site = matrix, rng, site
        got = ob.oracle_vcs_convert(d, frame)
        want = ref_convert(pin, frame, iw, ih, ow, oh, 3, in_fmt=ob.FMT["BGRA"], out_fmt=ob.FMT["NV12"], out_matrix=matrix,
                           out_rng=rng, out_site=site, out_size=got.size)
        assert key(got) == want


def test_rgb_to_yuv_matrix_known_answers():
    """bt709 and bt601, full-range RGB -> 16-235: the x256 integer matrices the reference derives (rows Y, U, V)"""
    im = (C.c_int * 16)()
    d = ob.vcs_desc(1920, 1080, 1920, 1080, 1, in_fmt=ob.FMT["BGRA"], out_fmt=ob.FMT["NV12"])
    assert ob.oracle().oracle_vcs_matrix_rgb2yuv(C.byref(d), im) == 0
    assert list(im)[:12] == [47, 157, 16, 4096, -26, -87, 112, 32768, 112, -102, -10, 32768]
    d = ob.vcs_desc(640, 480, 640, 480, 1, in_fmt=ob.FMT["BGRA"], out_fmt=ob.FMT["NV12"])
    assert ob.oracle().oracle_vcs_matrix_rgb2yuv(C.byref(d), im) == 0
    assert list(im)[:12] == [66, 129, 25, 4096, -38, -74, 112, 32768, 112, -94, -18, 32768]


@pytest.mark.parametrize("fi", RGB_IN)
@pytest.mark.parametrize("fo", RGB_IN)
def test_rgb_to_rgb_matches_reference(fi, fo, pin):
    """same format: the one-plane convert_scale_planes rows (video-converter.c:8879-8896; 4-byte pixels through
    gst_video_scaler_2d, stepping 2-tap horizontal, every byte a channel) — the compositor's scaled RGBA pads; another
    byte order: the chain without matrix or alpha stage"""
    for (iw, ih, ow, oh) in [(64, 48, 32, 24), (40, 30, 64, 48), (33, 17, 20, 31), (100, 100, 150, 50), (40, 90, 40, 31),
                             (50, 21, 50, 21), (3, 5, 7, 2)]:
        frame = _rgb_frame(iw, ih, 4)
        for method in (0, 1, 3, 4, 9):
            got = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo]), frame)
            want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], out_size=got.size)
            assert key(got) == want, f"{iw}x{ih}->{ow}x{oh} method {method}"


# ------------------------------------------------------------------- destination rectangle + borders (add-borders)
def test_add_borders_geometry():
    """gst_video_convert_scale_set_info (gstvideoconvertscale.c:920-952), pixel aspect ratio 1/1 on both sides"""
    assert ob.vcs_borders(1920, 1080, 1280, 720) == (0, 0, 1280, 720)          # same display aspect ratio: none
    assert ob.vcs_borders(1920, 1080, 1280, 1024) == (0, 152, 1280, 720)       # bars above / below
    assert ob.vcs_borders(640, 480, 1920, 1080) == (240, 0, 1440, 1080)        # pillar box
    assert ob.vcs_borders(100, 100, 150, 50) == (50, 0, 50, 50)
    assert ob.vcs_borders(7, 3, 10, 10) == (0, 3, 10, 4)                       # 10*3/7 = 4 (floor), borders 6 -> y = 3


@pytest.mark.parametrize("pair", [("NV12", "BGRA"), ("I420", "RGBA"), ("NV12", "NV12"), ("I420", "YV12"), ("NV12", "I420"),
                                  ("YV12", "NV21"), ("BGRA", "NV12"), ("RGBA", "I420"), ("BGRA", "BGRA")],
                         ids=lambda p: "%s-%s" % p)
def test_destination_rectangle_and_borders_match_reference(pair, pin):
    """GST_VIDEO_CONVERTER_OPT_DEST_X/Y/WIDTH/HEIGHT as the element sets them for add-borders, and arbitrary rectangles;
    border colour: the default opaque black and two others (setup_borderline's RGB -> YUV of the border pixel)"""
    rnd = np.random.default_rng(17)
    fi, fo = pair
    rgb_in = fi in RGB_IN
    checked = 0
    for t in range(40):
        iw, ih, W, H = (int(v) for v in rnd.integers(2, 70, 4))
        method = int(rnd.choice([0, 1, 3, 4, 9]))
        if t % 2:
            dest = ob.vcs_borders(iw, ih, W, H)
        else:
            dw, dh = int(rnd.integers(1, W + 1)), int(rnd.integers(1, H + 1))
            dest = (int(rnd.integers(0, W - dw + 1)), int(rnd.integers(0, H - dh + 1)), dw, dh)
        border = [0xff000000, 0x80ff4020, 0xff10c0f0][t % 3]
        if dest[2] < 1 or dest[3] < 1:
            continue                # extreme aspect ratios leave an empty rectangle: degenerate in the reference too
        frame = _rgb_frame(iw, ih, t) if rgb_in else (ob.i420_random_frame(iw, ih, t) if fi in ("I420", "YV12") else ob.nv12_random_frame(iw, ih, t))
        d = ob.vcs_desc(iw, ih, W, H, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo])
        kw = {}
        if not rgb_in and fo not in RGB_IN:
            kw = dict(matrix=d.in_matrix, out_matrix=d.in_matrix, site=d.in_chroma_site, out_site=d.in_chroma_site)
        got = ob.oracle_vcs_convert_dest(d, frame, dest, border)
        want = ref_convert(pin, frame, iw, ih, W, H, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], dest=dest, border_argb=border,
                           out_size=got.size, **kw)
        if key(got) != want:
            dw, dh = dest[2], dest[3]
            if fo not in RGB_IN or fi not in RGB_IN:            # the two reference defect classes, on the rectangle's size
                if _vfirst(iw, ih, dw, dh) or (method == 0 or ih == 1) and dh > ih:
                    continue
            assert False, (iw, ih, W, H, dest, method)
        checked += 1
    assert checked >= 25


@pytest.mark.parametrize("fmt", ["F32", "S16", "S32", "F64"])
@pytest.mark.parametrize("method,mode,interp", [(3, 2, 2), (3, 1, 2), (3, 0, 2), (4, 1, 2), (4, 0, 2), (4, 1, 0), (3, 1, 0),
                                                (4, 2, 0), (4, 0, 0), (3, 2, 0),
                                                (4, 2, 1), (4, 1, 1), (4, 0, 1), (3, 1, 1), (3, 0, 1),
                                                (0, 2, 2), (1, 2, 2), (2, 2, 2), (1, 0, 1), (2, 1, 0)])
def test_audio_method_and_filter_mode_properties(fmt, method, mode, interp, pin):
    """resample-method kaiser / blackman-nuttall, sinc-filter-mode interpolated / full / auto, sinc-filter-interpolation
    cubic / linear (two table rows per phase, 11x the oversampling) / none (FULL mode then computes every phase's taps directly; an interpolated table falls back to cubic with an
    oversampling of 1) — byte-identical output for every sample format"""
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o, r = ob.oracle(), live()
    for (a, b, ch, q) in [(48000, 44100, 2, 4), (44100, 48000, 1, 6), (8000, 16000, 2, 2), (96000, 44100, 1, 8), (44100, 44099, 1, 3),
                          (3, 2, 1, 5), (48000, 8000, 2, 1), (44100, 44100, 2, 4)]:   # equal rates: the nearest functions
        ho = o.oracle_ars_new_opts(a, b, ch, q, ofmt, method, mode, interp)
        hr = r.ref_ars_new_opts(a, b, ch, q, gfmt, method, mode, interp) if r else None
        assert ho and pin(lambda: bool(hr))
        io = _info(o.oracle_ars_info, ho)
        assert key(io) == pin(lambda: _info(r.ref_ars_info, hr)), (a, b, q)
        rng = np.random.default_rng(a + b)
        for n in [480, 100, 1, 1500, None]:
            x = None
            if n is None:
                n = io[0] // 2
            else:
                x = ob.audio_test_signal(rng, n, ch, fmt)
            cap = int(n * b / a) + 64
            o1 = np.zeros((cap, ch), dtype=dt)
            o2 = o1.copy()
            n1 = o.oracle_ars_process_any(ho, x.ctypes.data if x is not None else None, n, o1.ctypes.data, cap)

            def ref_process():
                n2 = r.ref_ars_process(hr, x.ctypes.data if x is not None else None, n, o2.ctypes.data, cap)
                return n2, o2[:n2]
            assert key((n1, o1[:n1])) == pin(ref_process), (a, b, q, n)
        o.oracle_ars_free(ho)
        if r:
            r.ref_ars_free(hr)


@pytest.mark.parametrize("fmt", ["F32", "S16", "F64"])
def test_audio_nearest_decimation_skip_quirk(fmt, pin):
    """nearest method while decimating: the next window can start beyond the data, gst_audio_resampler_resample then sets
    `skip` (:1796-1803), adds it to samp_index on EVERY later call (:1762, never cleared), and after such a call shifts its
    buffers by the absolute final index while counting the rest from the start index - so the tail of what it keeps is
    whatever the shift left in place.  The oracle keeps the same buffers and reproduces all of it."""
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o, r = ob.oracle(), live()
    for (a, b, ch) in [(48000, 11025, 3), (48000, 8000, 2), (96000, 8000, 1), (400, 3, 2)]:
        for seed in range(4):
            rng = np.random.default_rng(seed)
            ho = o.oracle_ars_new_opts(a, b, ch, 4, ofmt, 0, 2, 2)
            hr = r.ref_ars_new_opts(a, b, ch, 4, gfmt, 0, 2, 2) if r else None
            for n in [int(v) for v in rng.choice([1, 2, 7, 37, 100, 160, 480], 6)]:
                x = ob.audio_test_signal(rng, n, ch, fmt)
                cap = int(n * b / a) + 64
                o1 = np.full((cap, ch), 7, dtype=dt)
                o2 = o1.copy()
                n1 = o.oracle_ars_process_any(ho, x.ctypes.data, n, o1.ctypes.data, cap)
                assert key((n1, o1)) == pin(lambda: (r.ref_ars_process(hr, x.ctypes.data, n, o2.ctypes.data, cap), o2)), \
                    (a, b, ch, seed, n)
            o.oracle_ars_free(ho)
            if r:
                r.ref_ars_free(hr)


# ------------------------------------------------------------------- 4:2:2 and 4:4:4 inputs (capture formats) -> packed RGB
@pytest.mark.parametrize("fi", ["YUY2", "UYVY", "YVYU", "Y42B", "Y444"])
@pytest.mark.parametrize("size", [(64, 48, 32, 24), (64, 48, 96, 72), (33, 17, 20, 31), (50, 21, 50, 21), (100, 100, 150, 50),
                                  (40, 90, 40, 31), (1, 1, 5, 4), (7, 3, 3, 9)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_422_444_inputs_match_reference(fi, size, pin):
    """unpack_YUY2 / _UYVY / _YVYU / _Y42B / _Y444, horizontal chroma up-sampling only for 4:2:2 (v_factor 0 selects
    video_chroma_none), none for 4:4:4; then the usual scalers, fast matrix and pack.  No line pairs here, so vertical-first
    geometries compare directly as well."""
    iw, ih, ow, oh = size
    for k, method in enumerate(range(10)):
        fo = RGB_IN[k % 8]
        for site, matrix, rng in ((2, 3, 2), (1, 4, 1)):
            d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site, matrix=matrix, rng=rng)
            frame = np.random.default_rng(method).integers(0, 256, ob.vcs_sizes(d)[0], dtype=np.uint8)
            got = ob.oracle_vcs_convert(d, frame)
            want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site, matrix=matrix,
                               rng=rng, out_size=got.size)
            if _one_tap_vertical_repeat(iw, ih, ow, oh, method) and key(got) != want:
                continue
            assert key(got) == want, f"{fo} method {method} site {site}"


# ---- variable rate: gst_audio_resampler_update on a live stream (audio-resampler.c:1503-1615) -------------------------------
RATE_WALKS = [
    # (channels, quality, [(in, out), ...]): every pair after the first arrives through update() with a fresh option bag
    (2, 4, [(48000, 44100), (48000, 48000 * 2), (48000, 32000), (44100, 48000)]),
    (1, 4, [(44100, 48000), (44100, 44100 * 3 // 2), (44100, 8000), (44100, 96000)]),      # tap count changes both ways
    (3, 6, [(48000, 44100), (48000, 44101), (48001, 44100), (8000, 7999)]),                # FULL <-> interpolated, odd rates
    (2, 0, [(96000, 8000), (96000, 44100), (32000, 48000)]),
    (2, 10, [(44100, 48000), (22050, 48000), (44100, 16000)]),
    (5, 4, [(48000, 44100), (47999, 44100), (48000, 44100), (48000, 44099)]),              # clock-drift sized steps
]


@pytest.mark.parametrize("fmt", ["F32", "S16", "S32", "F64"])
@pytest.mark.parametrize("walk", RATE_WALKS, ids=lambda w: "%dch-q%d-%s" % (w[0], w[1], "_".join("%d-%d" % p for p in w[2])))
def test_audio_rate_update_matches_reference(fmt, walk, pin):
    """The element's rate change (gst_audio_resample_update_state -> gst_audio_resampler_update with a fresh option bag):
    the phase is rescaled, the divisor of the rates follows the phase-error rule, the filter is re-designed and the
    history moves by half the tap-count change - byte-identical output with the reference build across every change,
    with the stream cut into uneven buffers around them"""
    ch, q, pairs = walk
    ofmt, gfmt, dt, _ = ob.AUDIO_FORMATS[fmt]
    o, r = ob.oracle(), live()
    a, b = pairs[0]
    ho, hr = o.oracle_ars_new_fmt(a, b, ch, q, ofmt), (r.ref_ars_new_fmt(a, b, ch, q, gfmt) if r else None)
    rng = np.random.default_rng(a * 7 + b + ch)
    try:
        for k, (a, b) in enumerate(pairs):
            if k:
                assert o.oracle_ars_update(ho, a, b) == 0
                assert pin(lambda: r.ref_ars_update(hr, a, b, q, 4, 2, 2)) == 0      # kaiser, filter-mode auto, cubic interpolation
                vo = _info(o.oracle_ars_info, ho)

                def ref_info():
                    vr = _info(r.ref_ars_info, hr)
                    if vr[4] == 0:          # interpolated mode: the reference leaves the FULL-mode phase count of before in place
                        vr[1] = 0
                    return vr
                if vo[4] == 0:
                    vo[1] = 0
                assert key(vo) == pin(ref_info), (a, b)
            for n in [int(v) for v in rng.choice([1, 7, 160, 481, 1000], 4)]:
                x = ob.audio_test_signal(rng, n, ch, fmt)
                cap = int(n * b / a) + 64
                o1 = np.zeros((cap, ch), dtype=dt)
                o2 = o1.copy()
                assert o.oracle_ars_get_out_frames(ho, n) == pin(lambda: r.ref_ars_get_out_frames(hr, n))
                n1 = o.oracle_ars_process_any(ho, x.ctypes.data, n, o1.ctypes.data, cap)

                def ref_process():
                    n2 = r.ref_ars_process(hr, x.ctypes.data, n, o2.ctypes.data, cap)
                    return n2, o2[:n2]
                assert key((n1, o1[:n1])) == pin(ref_process), (k, a, b, n)
    finally:
        o.oracle_ars_free(ho)
        if r:
            r.ref_ars_free(hr)


# ------------------------------------------------------------------- packed 4:2:2 (capture) -> 4:2:0 (encoder input)
@pytest.mark.parametrize("fi", ["YUY2", "UYVY", "YVYU"])
@pytest.mark.parametrize("fo", ["I420", "YV12", "NV12", "NV21"])
@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (1, 1, 1, 1), (2, 3, 2, 3), (64, 48, 32, 24),
                                  (64, 48, 96, 72), (33, 17, 20, 31), (100, 100, 150, 50), (40, 90, 40, 31), (57, 35, 29, 35),
                                  (7, 3, 3, 9)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_packed_422_to_420_matches_reference(fi, fo, size, pin):
    """YUY2 / UYVY -> I420 / YV12 at an unchanged size: the table rows convert_YUY2_I420 / convert_UYVY_I420 (luma copy,
    avgub of the line pair's chroma); every other pair or size: the chain - unpack, horizontal chroma up-sampling, scalers,
    chroma down-sampling with the OUTPUT size's default site (the fixation does not carry the site across a
    sub-sampling change), 4:2:0 pack"""
    iw, ih, ow, oh = size
    for method in range(10):
        for site in (1, 2):
            out_site = 2 if oh > 576 else 1
            d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site)
            d.out_chroma_site = out_site
            frame = np.random.default_rng(method + 10 * site).integers(0, 256, ob.vcs_sizes(d)[0], dtype=np.uint8)
            got = ob.oracle_vcs_convert(d, frame)
            want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site, matrix=d.in_matrix,
                               out_matrix=d.in_matrix, out_site=out_site, out_size=got.size)
            if key(got) != want:
                if _one_tap_vertical_inplace(ih, oh, method) or _one_tap_vertical_repeat(iw, ih, ow, oh, method):
                    continue
                assert False, f"method {method} site {site}: output differs from the reference's"


# ------------------------------------------------------------------- planar 4:2:2 / 4:4:4 -> planar 4:2:0 (plane-scaling table rows)
@pytest.mark.parametrize("fi", ["Y42B", "Y444"])
@pytest.mark.parametrize("fo", ["I420", "YV12"])
@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (1, 1, 1, 1), (2, 3, 2, 3), (64, 48, 32, 24),
                                  (64, 48, 96, 72), (33, 17, 20, 31), (100, 100, 150, 50), (40, 90, 40, 31), (7, 3, 3, 9),
                                  (64, 48, 64, 24), (64, 48, 128, 96), (64, 48, 32, 48)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_planar_422_444_to_420_matches_reference(fi, fo, size, pin):
    """convert_scale_planes rows Y42B / Y444 -> I420 / YV12 (video-converter.c:8607-8628): every output plane scaled from the
    plane holding the same component with the chroma resampler method, halving / doubling special cases included; all ten
    element methods, byte-identical (no defect class on this route: no chain, no in-place filters)"""
    iw, ih, ow, oh = size
    for method in range(10):
        d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=2)
        frame = np.random.default_rng(method).integers(0, 256, ob.vcs_sizes(d)[0], dtype=np.uint8)
        got = ob.oracle_vcs_convert(d, frame)
        want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=2, matrix=d.in_matrix,
                           out_matrix=d.in_matrix, out_site=1, out_size=got.size)
        assert key(got) == want, f"method {method}"


@pytest.mark.parametrize("fi", ["Y42B", "Y444"])
@pytest.mark.parametrize("fo", ["NV12", "NV21"])
@pytest.mark.parametrize("size", [(64, 48, 64, 48), (50, 21, 50, 21), (33, 17, 33, 17), (1, 1, 1, 1), (2, 3, 2, 3), (64, 48, 32, 24),
                                  (64, 48, 96, 72), (33, 17, 20, 31), (100, 100, 150, 50), (40, 90, 40, 31), (7, 3, 3, 9),
                                  (57, 35, 29, 35), (40, 33, 57, 33)], ids=lambda s: "%dx%d-%dx%d" % s)
def test_planar_422_444_to_semi_planar_420_matches_reference(fi, fo, size, pin):
    """Y42B / Y444 -> NV12 / NV21: no table row, the chain (4:2:2: horizontal up-sampler; 4:4:4: none - an odd height at an
    unchanged size then reads the last line as unpacked), chroma down-sampling with the output size's default site"""
    iw, ih, ow, oh = size
    for method in range(10):
        for site in (1, 2):
            d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site)
            d.out_chroma_site = 1
            frame = np.random.default_rng(method).integers(0, 256, ob.vcs_sizes(d)[0], dtype=np.uint8)
            got = ob.oracle_vcs_convert(d, frame)
            want = ref_convert(pin, frame, iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site, matrix=d.in_matrix,
                               out_matrix=d.in_matrix, out_site=1, out_size=got.size)
            if key(got) != want:
                assert _one_tap_vertical_inplace(ih, oh, method), f"method {method} site {site}"
