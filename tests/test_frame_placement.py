"""Frame placement on every convert route, without a GPU: base pointers at every small offset from a 16-byte boundary,
plane offsets and strides set through the frame layout, and a batch that mixes placements.

b200_vcs_convert_batch promises, for any base pointer and layout, either the oracle's bytes or a clean refusal
(B200_ERR_INVALID_ARG) - never a device fault.  A kernel that loads a uint2 / uint4 or stores a 32-bit word through a
pointer that is not a multiple of its size faults on the device and ends the CUDA context.  The emulated build with
UBSan (tests/cudaemu, variant "ubsan": vector types at CUDA's alignments, every report fatal) turns each such
access into an abort with a "misaligned address" report, so this module finds them on the CPU.

Every case runs in its own process, so a sanitizer abort fails that case and leaves the pytest worker alone.  The
child process is this file run as a script; it prints one line per conversion and the parent checks them:
  * status 0: output equal to the oracle's, row padding and the bytes around the frame untouched; or
  * status B200_ERR_INVALID_ARG: the output buffer untouched (at create time for a layout the route cannot take);
and in either case no UBSan report at all."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "cudaemu"))

pytestmark = pytest.mark.timeout(900)

INVALID_ARG = -1
FILL = 0x5A
GUARD = 64                                   # bytes before and after the output frame that must keep the fill byte

RGB = ("BGRA", "RGBA", "ARGB", "ABGR", "BGRx", "RGBx", "xRGB", "xBGR")
YUV420 = ("NV12", "NV21", "I420", "YV12")
PACKED422 = ("YUY2", "UYVY", "YVYU")

IN_OFFS = (0, 1, 2, 4, 8)                    # input base mod 16
OUT_OFFS = (0, 1, 2, 4)                      # output base mod 16
# (input layout, output layout): "padded" keeps every alignment with wider strides and gaps between the planes,
# "word" makes plane offsets and strides multiples of 4 but not of 8, "odd" makes them odd
LAYOUTS = (("default", "default"), ("padded", "padded"), ("word", "default"), ("odd", "default"), ("default", "odd"),
           ("default", "word"))

# route id -> what it converts and what must run for the default layout at aligned pointers:
#   (in, out, (iw, ih, ow, oh), method, env, kernel variant forced with b200_vcs_set_kernel_variant or None,
#    input chroma site or None, output chroma site or None, destination rectangle or None,
#    expected kernel name, expected plan_info kernel_variant, expected launches per convert)
ROUTES = {
    "generic-nv12-bgra": ("NV12", "BGRA", (40, 30, 24, 18), 3, {}, 0, 2, None, None, "vcs_generic_kernel", 0, 1),
    "generic-i420-rgba": ("I420", "RGBA", (40, 30, 56, 42), 1, {}, 0, 1, None, None, "vcs_generic_kernel", 0, 1),
    "generic-yuy2-argb": ("YUY2", "ARGB", (40, 30, 24, 18), 1, {}, None, 1, None, None, "vcs_generic_kernel", 0, 1),
    "v2-nv12-bgra": ("NV12", "BGRA", (256, 64, 128, 32), 3, {}, None, 2, None, None, "vcs_lanczos2_v2_kernel", 1, 1),
    "v2-i420-bgra": ("I420", "BGRA", (256, 64, 128, 32), 3, {}, None, 2, None, None, "vcs_lanczos2_v2_kernel", 1, 1),
    "v1-nv12-rgba": ("NV12", "RGBA", (128, 48, 64, 24), 3, {"B200_L2_V1": "1"}, None, 2, None, None, "vcs_lanczos2_kernel", 1, 1),
    "light-nv12-bgra": ("NV12", "BGRA", (96, 54, 64, 36), 1, {}, None, 2, None, None, "vcs_light_kernel", 2, 1),
    "ntap-nv12-bgra": ("NV12", "BGRA", (96, 54, 64, 36), 3, {}, None, 2, None, None, "vcs_ntap_kernel", 3, 1),
    "l2mma-nv12-bgra": ("NV12", "BGRA", (128, 48, 64, 24), 3, {}, 6, 2, None, None, "vcs_l2mma_kernel", 6, 1),
    "planes-nv12-nv12": ("NV12", "NV12", (40, 30, 24, 18), 3, {"B200_PLANES_SLOW": "1"}, None, None, None, None, "vcs_planes_kernel", 4, 1),
    "planes-fast-i420-i420": ("I420", "I420", (70, 40, 35, 20), 3, {}, None, None, None, None, "vcs_planes_fast_vfirst_kernel", 4, 1),
    "planes-fast-bgra-rgba": ("BGRA", "RGBA", (70, 40, 35, 20), 1, {}, None, None, None, None, "vcs_planes_fast_kernel", 4, 1),
    "chain-v2-nv12-i420": ("NV12", "I420", (256, 64, 128, 32), 3, {}, None, 2, None, None, "vcs_lanczos2_v2_kernel", 5, 2),
    # B200_CROSS_GENERIC: the generic kernel ahead of the down-sampler (kernel_name still names the plan's light kernel)
    "chain-extra-row-nv12-i420": ("NV12", "I420", (40, 29, 24, 29), 1, {"B200_CROSS_GENERIC": "1"}, None, 1, 1, None, "vcs_light_kernel", 5, 3),
    "rgb420-bgra-nv12": ("BGRA", "NV12", (40, 30, 40, 30), 1, {}, None, None, None, None, "vcs_rgb420_kernel", 5, 1),
    "rgb420-scaled-rgba-i420": ("RGBA", "I420", (48, 36, 24, 18), 3, {}, None, None, None, None, "vcs_rgb420_kernel", 5, 2),
    "rgb420-pre1-bgra-nv12": ("BGRA", "NV12", (24, 18, 40, 30), 1, {}, None, None, None, None, "vcs_rgb420_kernel", 5, 3),
    "rgb420-pre2-yuy2-nv12": ("YUY2", "NV12", (40, 30, 40, 30), 1, {}, None, None, 1, None, "vcs_yuy2_ayuv_kernel", 5, 2),
    "rgb420-pre2-scaled-uyvy-i420": ("UYVY", "I420", (48, 36, 24, 18), 1, {}, None, None, 1, None, "vcs_yuy2_ayuv_kernel", 5, 3),
    "yuy2-420-yuy2-i420": ("YUY2", "I420", (40, 30, 40, 30), 1, {}, None, 1, None, None, "vcs_yuy2_420_kernel", 5, 1),
    "border-nv12-bgra": ("NV12", "BGRA", (40, 30, 40, 40), 1, {}, 0, 1, None, (0, 5, 40, 30), "vcs_generic_kernel", 0, 2),
    "border-nv12-i420": ("NV12", "I420", (40, 30, 40, 40), 1, {}, None, 1, 1, (0, 4, 40, 30), "vcs_light_kernel", 5, 3),
}


def plane_rows(fmt, h):
    if fmt in ("NV12", "NV21"):
        return [h, (h + 1) // 2]
    if fmt in ("I420", "YV12"):
        return [h, (h + 1) // 2, (h + 1) // 2]
    if fmt in ("Y42B", "Y444"):
        return [h, h, h]
    return [h]


def apply_layout(info, fmt, kind):
    """rewrites info's strides and plane offsets; returns the frame size in bytes"""
    rows = plane_rows(fmt, info.height)
    if kind == "default":
        return None
    pad, start, gap = {"padded": (16, 48, 32), "word": (4, 4, 4), "odd": (1, 3, 5)}[kind]
    off = start
    for p, r in enumerate(rows):
        info.stride[p] = info.stride[p] + pad * (p + 1)
        info.offset[p] = off
        off += info.stride[p] * r + gap
    return off


def load(lib_path):
    from gstreamer_b200 import _lib  # noqa: F401  (signatures only)
    from gstreamer_b200._lib import _SIGS
    lib = C.CDLL(lib_path)
    for name, (res, args) in _SIGS.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    return lib


def placed(size, mod, align=64):
    """a zero-filled uint8 view of `size` bytes whose address is `mod` past a multiple of 16, inside a larger buffer"""
    buf = np.zeros(size + align + 2 * GUARD, dtype=np.uint8)
    start = GUARD + (-(buf.ctypes.data + GUARD)) % align + mod
    return buf, start


class Case:
    """one route at one layout: infos, handle, oracle output"""

    def __init__(self, lib, route, layout):
        from gstreamer_b200 import _lib
        from oracle import bindings as ob
        fi, fo, (iw, ih, ow, oh), method, env, force, site, out_site, dest, *_ = ROUTES[route]
        self.lib, self.fi, self.fo = lib, fi, fo
        ii, oi = _lib.VideoInfoC(), _lib.VideoInfoC()
        assert lib.b200_video_info_set_format(C.byref(ii), ob.FMT[fi], iw, ih) == 0
        assert lib.b200_video_info_set_format(C.byref(oi), ob.FMT[fo], ow, oh) == 0
        if site is not None:
            ii.chroma_site = site
        if fi in YUV420 and fo in YUV420:                      # the element's caps fixation
            oi.color_matrix, oi.color_range, oi.chroma_site = ii.color_matrix, ii.color_range, ii.chroma_site
        if fi in PACKED422 and fo in YUV420:
            oi.color_matrix, oi.color_range = ii.color_matrix, ii.color_range
        if out_site is not None:
            oi.chroma_site = out_site
        in_end = apply_layout(ii, fi, layout[0])
        out_end = apply_layout(oi, fo, layout[1])
        self.in_size = in_end or lib.b200_video_info_size(C.byref(ii))
        self.out_size = out_end or lib.b200_video_info_size(C.byref(oi))
        cfg = _lib.VcsConfigC()
        lib.b200_vcs_config_init(C.byref(cfg))
        cfg.method = method
        if dest:
            cfg.dest_x, cfg.dest_y, cfg.dest_width, cfg.dest_height = dest
            cfg.border_argb = 0xff204080
        self.h = C.c_void_p()
        self.status = lib.b200_vcs_create(C.byref(ii), C.byref(oi), C.byref(cfg), 0, C.byref(self.h))
        if self.status != 0:
            return
        if force is not None:                                   # a forced kernel the layout rules out: the plan's own
            st = lib.b200_vcs_set_kernel_variant(self.h, force)
            assert st == 0 or layout != ("default", "default"), (route, st)
        lib.b200_vcs_kernel_name.restype = C.c_char_p
        self.name = lib.b200_vcs_kernel_name(self.h).decode()
        info = _lib.VcsPlanInfoC()
        lib.b200_vcs_get_plan_info(self.h, C.byref(info))
        self.variant, self.launches = int(info.kernel_variant), int(info.n_launches_per_convert)
        # the oracle on the same layout (its descriptor carries strides and offsets too)
        d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[fi], out_fmt=ob.FMT[fo], site=site)
        d.out_matrix, d.out_range, d.out_chroma_site = oi.color_matrix, oi.color_range, oi.chroma_site
        for p in range(4):
            d.in_stride[p], d.in_offset[p] = ii.stride[p], ii.offset[p]
            d.out_stride[p], d.out_offset[p] = oi.stride[p], oi.offset[p]
        self.frames = [np.random.default_rng(seed).integers(0, 256, self.in_size, dtype=np.uint8) for seed in (1, 2)]
        self.want = []
        for f in self.frames:
            w = np.full(max(self.out_size, ob.vcs_sizes(d)[1]), FILL, dtype=np.uint8)
            if dest:
                r = ob.oracle_vcs_convert_dest(d, f, dest, 0xff204080, fill=FILL)
                w[:r.size] = r
            else:
                assert ob.oracle().oracle_vcs_convert(C.byref(d), f.ctypes.data, w.ctypes.data) == 0
            self.want.append(w[:self.out_size])

    def run(self, in_offs, out_offs):
        """one batch: slot k reads frame k % 2 at in_offs[k] and writes at out_offs[k]; returns (status, problems)"""
        n = len(in_offs)
        ins, outs, keep = [], [], []
        for k in range(n):
            ib, i0 = placed(self.in_size, in_offs[k])
            ib[i0:i0 + self.in_size] = self.frames[k % 2]
            ob_, o0 = placed(self.out_size, out_offs[k])
            ob_[:] = FILL
            keep += [ib, ob_]
            ins.append(ib.ctypes.data + i0)
            outs.append((ob_, o0))
        pin = (C.c_void_p * n)(*ins)
        pout = (C.c_void_p * n)(*[b.ctypes.data + o for b, o in outs])
        st = self.lib.b200_vcs_convert_batch(self.h, n, pin, pout, None)
        problems = []
        for k, (b, o) in enumerate(outs):
            if st == 0:
                got = b[o:o + self.out_size]
                bad = np.flatnonzero(got != self.want[k % 2])
                if bad.size:
                    problems.append(f"slot {k}: {bad.size} of {got.size} bytes differ from the oracle, first at {bad[:4].tolist()}")
                if not ((b[:o] == FILL).all() and (b[o + self.out_size:] == FILL).all()):
                    problems.append(f"slot {k}: bytes outside the frame written")
            elif st == INVALID_ARG:
                if not (b == FILL).all():
                    problems.append(f"slot {k}: refused, but the output buffer was written")
            else:
                problems.append(f"status {st}")
        return st, problems

    def close(self):
        if self.status == 0:
            self.lib.b200_vcs_destroy(self.h)


def worker(spec):
    import build_emu
    route, in_off = spec["route"], spec["in_off"]
    lib = load(os.path.join(build_emu.out_dir("ubsan"), "libb200emu.so"))
    for layout in LAYOUTS:
        c = Case(lib, route, layout)
        if c.status != 0:
            print(json.dumps({"layout": layout, "create": c.status}), flush=True)
            continue
        offs = OUT_OFFS if layout == ("default", "default") else (0, 2)
        if layout != ("default", "default") and in_off not in (0, 4):
            c.close()
            continue
        for out_off in offs:
            st, problems = c.run([in_off], [out_off])
            print(json.dumps({"layout": layout, "in_off": in_off, "out_off": out_off, "name": c.name, "variant": c.variant,
                              "launches": c.launches, "status": st, "problems": problems}), flush=True)
        c.close()
    if spec.get("mixed"):
        # one aligned slot and one 4 bytes past an 8-byte boundary, both ways round: the whole batch takes the fallback
        c = Case(lib, route, ("default", "default"))
        for offs in ([0, 4], [4, 0], [0, 0, 12]):
            st, problems = c.run(offs, [0] * len(offs))
            print(json.dumps({"layout": "mixed", "in_offs": offs, "name": c.name, "status": st, "problems": problems}), flush=True)
        c.close()


@pytest.fixture(scope="module")
def ubsan_lib():
    import build_emu
    return build_emu.build(variant="ubsan")


def run_child(spec, env_extra):
    env = dict(os.environ, UBSAN_OPTIONS="print_stacktrace=1", PYTHONDONTWRITEBYTECODE="1", **env_extra)
    p = subprocess.run([sys.executable, os.path.abspath(__file__), json.dumps(spec)], capture_output=True, text=True,
                       env=env, timeout=800, cwd=ROOT)
    report = [ln for ln in p.stderr.splitlines() if "runtime error" in ln]
    assert p.returncode == 0 and not report, \
        f"{spec}: exit {p.returncode}, UBSan: {report[:3]}\nlast cases:\n{p.stdout[-1500:]}\nstderr:\n{p.stderr[-3000:]}"
    return [json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith("{")]


def check_lines(route, lines):
    name, variant, launches = ROUTES[route][-3:]
    for r in lines:
        if "create" in r:
            # a layout the plan cannot take is refused as an invalid argument, never accepted and then faulted on
            assert r["create"] == INVALID_ARG and r["layout"] != ["default", "default"], r
            continue
        assert not r["problems"], r
        assert r["status"] in (0, INVALID_ARG), r
        if r["layout"] == ["default", "default"] and r["in_off"] == 0 and r["out_off"] == 0:
            assert r["status"] == 0, r
            assert (r["name"], r["variant"], r["launches"]) == (name, variant, launches), \
                f"{route} ran {r['name']} (variant {r['variant']}, {r['launches']} launches), expected {name}"


@pytest.mark.parametrize("in_off", IN_OFFS)
@pytest.mark.parametrize("route", list(ROUTES))
def test_placement(ubsan_lib, route, in_off):
    lines = run_child({"route": route, "in_off": in_off}, ROUTES[route][4])
    assert lines, route
    check_lines(route, lines)


@pytest.mark.parametrize("route", ["v2-nv12-bgra", "v2-i420-bgra", "v1-nv12-rgba", "chain-v2-nv12-i420", "light-nv12-bgra"])
def test_mixed_batch_takes_the_fallback(ubsan_lib, route):
    """a batch is one launch: a single slot the fast kernel cannot read sends every slot to the fallback, and each slot
    still reads its own frame"""
    lines = run_child({"route": route, "in_off": 0, "mixed": True}, ROUTES[route][4])
    mixed = [r for r in lines if r["layout"] == "mixed"]
    assert len(mixed) == 3
    for r in mixed:
        assert r["status"] == 0 and not r["problems"], r


def test_packed_rgb_output_refuses_unaligned_pointers(ubsan_lib):
    """every kernel that writes packed RGB stores 32-bit words: a base pointer off a 4-byte boundary is refused before
    anything is written, on the fast routes and the generic one alike"""
    for route in ("v2-nv12-bgra", "light-nv12-bgra", "ntap-nv12-bgra", "generic-nv12-bgra", "border-nv12-bgra"):
        lines = run_child({"route": route, "in_off": 0}, ROUTES[route][4])
        for r in lines:
            if r.get("layout") == ["default", "default"]:
                assert r["status"] == (INVALID_ARG if r["out_off"] & 3 else 0), (route, r)


if __name__ == "__main__":
    worker(json.loads(sys.argv[1]))
