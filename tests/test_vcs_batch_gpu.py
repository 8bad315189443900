"""b200_vcs_convert_batch on the device: every slot of a batch reads its own frame and writes its own output, on every
convert route, and one handle serves batches of changing sizes (the 4:2:0 scratch images and the host pipeline's
device slots grow and shrink with them).

Each slot gets a distinct frame, so a kernel that read frames.in[0] (or any other slot's frame) for a slot fails.  Each
output is compared with the oracle, byte for byte, row padding and the bytes between frames included.  The frame
placement tests (tests/test_frame_placement.py) cover the same routes on the CPU at unaligned pointers; here only two
placements are checked, one of each outcome: a 2:1 input 4 bytes past an 8-byte boundary (converted by the fallback) and
a packed-RGB output 2 bytes past a word boundary (refused, nothing written)."""
import numpy as np
import pytest

from oracle import bindings as ob

pytestmark = pytest.mark.gpu

FILL = 0x5A
INVALID_ARG = -1

# id -> (in, out, (iw, ih, ow, oh), method, env, forced kernel variant or None, input chroma site, output chroma site,
#        destination rectangle or None, expected kernel name)
ROUTES = {
    "generic": ("NV12", "BGRA", (200, 120, 96, 64), 3, {}, 0, 2, None, None, "vcs_generic_kernel"),
    "generic-yuy2": ("YUY2", "ARGB", (120, 68, 96, 54), 1, {}, None, 1, None, None, "vcs_generic_kernel"),
    "v2-nv12": ("NV12", "BGRA", (512, 248, 256, 124), 3, {}, None, 2, None, None, "vcs_lanczos2_v2_kernel"),
    "v2-i420": ("I420", "RGBA", (512, 248, 256, 124), 3, {}, None, 2, None, None, "vcs_lanczos2_v2_kernel"),
    "v1-nv12": ("NV12", "BGRA", (256, 128, 128, 64), 3, {"B200_L2_V1": "1"}, None, 2, None, None, "vcs_lanczos2_kernel"),
    "light": ("NV12", "BGRA", (648, 360, 427, 240), 1, {}, None, 2, None, None, "vcs_light_kernel"),
    "ntap": ("NV12", "BGRA", (648, 360, 427, 240), 3, {}, None, 2, None, None, "vcs_ntap_kernel"),
    "l2mma": ("NV12", "BGRA", (272, 112, 136, 56), 3, {}, 6, 2, None, None, "vcs_l2mma_kernel"),
    "l2tc": ("NV12", "BGRA", (512, 240, 256, 120), 3, {}, 7, 2, None, None, "vcs_l2tc_kernel"),
    "planes-fast": ("I420", "I420", (400, 300, 150, 100), 3, {}, None, None, None, None, None),
    "chain-v2": ("NV12", "I420", (512, 248, 256, 124), 3, {}, None, 2, None, None, "vcs_lanczos2_v2_kernel"),
    "chain-extra-row": ("NV12", "I420", (64, 49, 32, 49), 1, {}, None, 1, 1, None, None),
    "rgb420": ("BGRA", "NV12", (64, 48, 64, 48), 1, {}, None, None, None, None, "vcs_rgb420_kernel"),
    "rgb420-scaled": ("RGBA", "I420", (400, 300, 150, 100), 3, {}, None, None, None, None, "vcs_rgb420_kernel"),
    "rgb420-pre1": ("BGRA", "NV12", (40, 30, 64, 48), 1, {}, None, None, None, None, "vcs_rgb420_kernel"),
    "rgb420-pre2": ("UYVY", "NV12", (64, 48, 32, 24), 1, {}, None, None, 1, None, "vcs_yuy2_ayuv_kernel"),
    "yuy2-420": ("YUY2", "I420", (130, 34, 130, 34), 1, {}, None, 1, None, None, "vcs_yuy2_420_kernel"),
    "border-rgb": ("NV12", "BGRA", (200, 120, 200, 160), 1, {}, None, 2, None, (0, 20, 200, 120), None),
    "border-420": ("NV12", "I420", (200, 120, 200, 160), 1, {}, None, 2, 2, (0, 20, 200, 120), None),
}


class Route:
    """one element on one route, with the oracle for any frame"""

    def __init__(self, name, monkeypatch):
        import gstreamer_b200 as g
        fi, fo, (iw, ih, ow, oh), method, env, force, site, out_site, dest, kernel = ROUTES[name]
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        self.fi, self.fo, self.size, self.method, self.site, self.dest = fi, fo, (iw, ih, ow, oh), method, site, dest
        ii, oi = g.VideoInfo(ob.FMT[fi], iw, ih), g.VideoInfo(ob.FMT[fo], ow, oh)
        if site is not None:
            ii.set_colorimetry(chroma_site=site)
        g.transfer_colorimetry_from_input(ii, oi)
        if out_site is not None:
            oi.set_colorimetry(chroma_site=out_site)
        self.el = g.CudaVideoConvertScale(add_borders=False, method=method, cuda_device_id=0)
        if dest:
            # the element's add-borders rectangle, given explicitly through the C-ABI configuration
            import ctypes as C
            from gstreamer_b200 import _lib
            cfg = _lib.VcsConfigC()
            g.lib.b200_vcs_config_init(C.byref(cfg))
            cfg.method = method
            cfg.dest_x, cfg.dest_y, cfg.dest_width, cfg.dest_height = dest
            h = C.c_void_p()
            _lib.check(g.lib.b200_vcs_create(C.byref(ii.c), C.byref(oi.c), C.byref(cfg), 0, C.byref(h)))
            self.el._h, self.el.in_info, self.el.out_info = h, ii, oi
        else:
            self.el.set_info(ii, oi)
        if force is not None:
            self.el.set_kernel_variant(force)
        if kernel:
            assert self.el.kernel_name() == kernel, (name, self.el.kernel_name())
        self.ii, self.oi = ii, oi
        d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site)
        d.out_matrix, d.out_range, d.out_chroma_site = oi.c.color_matrix, oi.c.color_range, oi.c.chroma_site
        self.desc = d
        self.in_size = ob.vcs_sizes(d)[0]
        self.cache = {}

    def frame(self, seed):
        return np.random.default_rng(1000 + seed).integers(0, 256, self.in_size, dtype=np.uint8)

    def want(self, seed):
        if seed not in self.cache:
            if self.dest:
                self.cache[seed] = ob.oracle_vcs_convert_dest(self.desc, self.frame(seed), self.dest, fill=FILL)
            else:
                w = np.full(ob.vcs_sizes(self.desc)[1], FILL, dtype=np.uint8)
                import ctypes as C
                assert ob.oracle().oracle_vcs_convert(C.byref(self.desc), self.frame(seed).ctypes.data, w.ctypes.data) == 0
                self.cache[seed] = w
        return self.cache[seed]

    def run_batch(self, seeds, stream=None):
        """one b200_vcs_convert_batch call over frames `seeds`, outputs 256-byte aligned one after another in one buffer
        (a slot that writes past its frame lands in the gap or its neighbour); returns the outputs"""
        import torch
        osz = self.oi.size
        pitch = (osz + 256 + 255) & ~255
        src = [torch.from_numpy(self.frame(s)).cuda() for s in seeds]
        out = torch.full((pitch * len(seeds),), FILL, dtype=torch.uint8, device="cuda")
        self.el.transform_frames(src, [out[k * pitch:k * pitch + osz] for k in range(len(seeds))], stream=stream)
        torch.cuda.synchronize()
        host = out.cpu().numpy()
        for k in range(len(seeds)):
            assert (host[k * pitch + osz:(k + 1) * pitch] == FILL).all(), f"slot {k} wrote past its frame"
        return [host[k * pitch:k * pitch + osz] for k in range(len(seeds))]

    def check(self, seeds, outs, tag):
        for k, (s, got) in enumerate(zip(seeds, outs)):
            want = self.want(s)
            bad = np.flatnonzero(got != want[:got.size])
            assert bad.size == 0, f"{tag}: slot {k} (frame {s}): {bad.size} bytes differ from the oracle, first at {bad[:6].tolist()}"


@pytest.mark.parametrize("n", [2, 7, 64])
@pytest.mark.parametrize("route", list(ROUTES))
def test_distinct_frames_per_slot(cuda_device, monkeypatch, route, n):
    r = Route(route, monkeypatch)
    seeds = list(range(n))
    r.check(seeds, r.run_batch(seeds), f"{route} n={n}")


@pytest.mark.parametrize("route", list(ROUTES))
def test_batch_sizes_on_one_handle(cuda_device, monkeypatch, route):
    """n = 2, 5, 1, 5 on one handle: scratch images grow, stay, shrink and grow back"""
    r = Route(route, monkeypatch)
    base = 0
    for n in (2, 5, 1, 5):
        seeds = list(range(base, base + n))
        r.check(seeds, r.run_batch(seeds), f"{route} n={n}")
        base += n


def test_batch_limit(cuda_device, monkeypatch):
    import torch
    import gstreamer_b200 as g
    r = Route("v2-nv12", monkeypatch)
    src = [torch.zeros(r.in_size, dtype=torch.uint8, device="cuda")] * 65
    dst = [torch.full((r.oi.size,), FILL, dtype=torch.uint8, device="cuda") for _ in range(65)]
    with pytest.raises(g.B200Error) as e:
        r.el.transform_frames(src, dst)
    assert e.value.status == INVALID_ARG
    torch.cuda.synchronize()
    assert all(bool((d == FILL).all()) for d in dst)


@pytest.mark.parametrize("route", ["v2-nv12", "chain-v2"])
def test_host_frames_cross_every_chunk_size(cuda_device, monkeypatch, route):
    """b200_vcs_convert_host on one handle with n = 9, 64, 33, 9: chunks of 1, 4, 2 and 1 frame, the device slots
    re-sized each time the chunk grows"""
    import gstreamer_b200 as g
    r = Route(route, monkeypatch)
    base = 0
    for n in (9, 64, 33, 9):
        seeds = list(range(base, base + n))
        ins = [g.PinnedBuffer(r.in_size) for _ in seeds]
        outs = [g.PinnedBuffer(r.oi.size) for _ in seeds]
        for b, s in zip(ins, seeds):
            b.array[:] = r.frame(s)
        for b in outs:
            b.array[:] = FILL
        r.el.transform_host_frames([b.array for b in ins], [b.array for b in outs])
        r.check(seeds, [b.array.copy() for b in outs], f"{route} host n={n}")
        for b in ins + outs:
            b.free()
        base += n


def test_bench_configuration(cuda_device):
    """what bench.py times: 4K NV12 -> 1080p BGRA lanczos, the element's default add-borders, 32 distinct frames in one
    call on a non-default stream.  Every output equals a single-frame run of its input; three of them (first, last and
    one between) equal the oracle's"""
    import torch
    import gstreamer_b200 as g
    iw, ih, ow, oh, n = 3840, 2160, 1920, 1080, 32
    el = g.CudaVideoConvertScale(method=g.VideoScaleMethod.LANCZOS, cuda_device_id=0)
    ii, oi = g.VideoInfo(g.VideoFormat.NV12, iw, ih), g.VideoInfo(g.VideoFormat.BGRA, ow, oh)
    el.set_info(ii, oi)
    assert el.kernel_name() == "vcs_lanczos2_v2_kernel"
    frames = [np.random.default_rng(7000 + k).integers(0, 256, ii.size, dtype=np.uint8) for k in range(n)]
    src = [torch.from_numpy(f).cuda() for f in frames]
    out = [torch.full((oi.size,), FILL, dtype=torch.uint8, device="cuda") for _ in range(n)]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        el.transform_frames(src, out, stream=s)
    s.synchronize()
    one = torch.full((oi.size,), FILL, dtype=torch.uint8, device="cuda")
    for k in range(n):
        one.fill_(FILL)
        el.transform_frame(src[k], one)
        torch.cuda.synchronize()
        assert torch.equal(out[k], one), f"slot {k} differs from the single-frame run of the same input"
    for k in (0, 13, n - 1):
        want = ob.oracle_vcs_convert(ob.vcs_desc(iw, ih, ow, oh, 3), frames[k])
        assert np.array_equal(out[k].cpu().numpy(), want), f"slot {k} differs from the oracle"


def test_placement_on_the_device(cuda_device, monkeypatch):
    """the two outcomes of the placement contract, once each on the device (the CPU sweep covers the rest): a 2:1 input
    4 bytes past an 8-byte boundary converts through the byte-reading fallback, a packed-RGB output 2 bytes past a word
    boundary is refused before anything is written"""
    import torch
    import gstreamer_b200 as g
    r = Route("v2-nv12", monkeypatch)
    buf = torch.zeros(r.in_size + 64, dtype=torch.uint8, device="cuda")
    src = buf[4:4 + r.in_size]
    assert src.data_ptr() % 8 == 4
    src.copy_(torch.from_numpy(r.frame(3)).cuda())
    out = torch.full((r.oi.size,), FILL, dtype=torch.uint8, device="cuda")
    r.el.transform_frame(src, out)
    torch.cuda.synchronize()
    r.check([3], [out.cpu().numpy()], "input at +4")
    for route in ("v2-nv12", "light"):
        r = Route(route, monkeypatch)
        obuf = torch.full((r.oi.size + 64,), FILL, dtype=torch.uint8, device="cuda")
        with pytest.raises(g.B200Error) as e:
            r.el.transform_frame(torch.from_numpy(r.frame(0)).cuda(), obuf[2:2 + r.oi.size])
        assert e.value.status == INVALID_ARG
        torch.cuda.synchronize()
        assert bool((obuf == FILL).all()), route
