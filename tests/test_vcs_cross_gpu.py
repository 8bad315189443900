"""4:2:0 -> the other 4:2:0 family (NV12 <-> I420, NV12 <-> NV21, ...): the reference's generic chain closed by chroma
down-sampling and the 4:2:0 pack functions (video-converter.c:2018-2032, :3194-3222; video-chroma.c:398-442, :742-785).
Product: vcs_generic_kernel (no matrix stage) into scratch A,Y,U,V images, then vcs_down420_kernel.
"""
import numpy as np
import pytest

from oracle import bindings as ob

pytestmark = pytest.mark.gpu

PAIRS = [("NV12", "I420"), ("I420", "NV12"), ("NV12", "NV21"), ("NV21", "YV12"), ("YV12", "NV21"), ("I420", "NV21")]
SIZES = [(64, 48, 32, 24), (64, 48, 96, 72), (65, 49, 33, 26), (33, 17, 20, 31), (50, 21, 50, 21), (57, 35, 29, 35),
         (40, 34, 57, 34), (100, 100, 150, 50), (64, 66, 64, 30), (320, 240, 213, 120), (17, 9, 64, 31), (2, 2, 1, 1),
         (1, 1, 5, 4), (640, 480, 320, 240), (1920, 1080, 1280, 720), (1280, 720, 1920, 1080)]


def planes_equal(got, want, oi, ow, oh, semi, fill=0x5A):
    """compare the pixel bytes of every plane; row padding must keep the fill byte.  Returns a list of problems."""
    bad = []
    for p in range(2 if semi else 3):
        w = ow if p == 0 else ((ow + 1) // 2) * (2 if semi else 1)
        h = oh if p == 0 else (oh + 1) // 2
        st, off = oi.stride[p], oi.offset[p]
        g_pl = got[off: off + st * h].reshape(h, st)
        w_pl = want[off: off + st * h].reshape(h, st)
        d = np.argwhere(g_pl[:, :w] != w_pl[:, :w])
        if d.size:
            bad.append(f"plane {p}: {len(d)} bytes differ, first at {d[:4].tolist()}")
        if not (g_pl[:, w:] == fill).all():
            bad.append(f"plane {p}: row padding written")
    return bad


def convert(size, method, frame, pair, site, out_site, batch=1):
    import torch
    import gstreamer_b200 as g
    iw, ih, ow, oh = size
    el = g.CudaVideoConvertScale(add_borders=False, method=method, cuda_device_id=0)
    ii, oi = g.VideoInfo(ob.FMT[pair[0]], iw, ih), g.VideoInfo(ob.FMT[pair[1]], ow, oh)
    ii.set_colorimetry(chroma_site=site)
    oi.set_colorimetry(matrix=ii.c.color_matrix, chroma_site=out_site)      # what the element's caps fixation does
    el.set_info(ii, oi)
    info = el.plan_info()
    assert int(info.kernel_variant) == 5 and int(info.n_launches_per_convert) in (2, 3)
    src = [torch.from_numpy(frame).cuda() for _ in range(batch)]
    dst = [torch.full((oi.size,), 0x5A, dtype=torch.uint8, device="cuda") for _ in range(batch)]
    if batch == 1:
        el.transform_frame(src[0], dst[0])
    else:
        el.transform_frames(src, dst)
    torch.cuda.synchronize()
    return [d.cpu().numpy() for d in dst], oi


def expected(size, method, frame, pair, site, out_site):
    iw, ih, ow, oh = size
    d = ob.vcs_desc(iw, ih, ow, oh, method, in_fmt=ob.FMT[pair[0]], out_fmt=ob.FMT[pair[1]], site=site)
    d.out_chroma_site = out_site
    return ob.oracle_vcs_convert(d, frame)


def random_frame(pair, iw, ih, seed):
    return ob.i420_random_frame(iw, ih, seed) if pair[0] in ("I420", "YV12") else ob.nv12_random_frame(iw, ih, seed)


# large shapes (the CPU oracle needs seconds per frame there): NV12 -> I420, bilinear / lanczos only
CROSS_CASES = [(p, s, m) for p in PAIRS for s in SIZES for m in (0, 1, 3, 4, 9)
               if not (s[0] * s[1] > 500_000 and (p != ("NV12", "I420") or m not in (1, 3)))]


@pytest.mark.parametrize("pair,size,method", CROSS_CASES, ids=lambda v: "-".join(str(x) for x in v) if isinstance(v, tuple) else str(v))
def test_cross_family_matches_oracle(cuda_device, pair, size, method):
    iw, ih, ow, oh = size
    frame = random_frame(pair, iw, ih, 5)
    for site, out_site in ((2, 2), (1, 1), (2, 1), (6, 4)):
        want = expected(size, method, frame, pair, site, out_site)
        (got,), oi = convert(size, method, frame, pair, site, out_site)
        assert got.size == want.size
        bad = planes_equal(got, want, oi, ow, oh, pair[1] in ("NV12", "NV21"))
        assert not bad, f"site {site}->{out_site}: {bad}"


def test_cross_family_batch(cuda_device):
    """distinct frames in batches of 5, 2 and 5 on ONE handle: the second batch reuses the scratch images of the first,
    the third grows them back"""
    import torch
    import gstreamer_b200 as g
    size = (640, 360, 426, 240)
    pair = ("NV12", "I420")
    el = g.CudaVideoConvertScale(add_borders=False, method=3, cuda_device_id=0)
    ii, oi = g.VideoInfo(ob.FMT[pair[0]], 640, 360), g.VideoInfo(ob.FMT[pair[1]], 426, 240)
    ii.set_colorimetry(chroma_site=2)
    oi.set_colorimetry(matrix=ii.c.color_matrix, chroma_site=2)
    el.set_info(ii, oi)
    assert int(el.plan_info().kernel_variant) == 5
    seed = 9
    for batch in (5, 2, 5):
        frames = [random_frame(pair, 640, 360, seed + k) for k in range(batch)]
        seed += batch
        dst = [torch.full((oi.size,), 0x5A, dtype=torch.uint8, device="cuda") for _ in frames]
        el.transform_frames([torch.from_numpy(f).cuda() for f in frames], dst)
        torch.cuda.synchronize()
        for k, (f, d) in enumerate(zip(frames, dst)):
            bad = planes_equal(d.cpu().numpy(), expected(size, 3, f, pair, 2, 2), oi, 426, 240, False)
            assert not bad, f"batch of {batch}, slot {k}: {bad}"


def test_cross_family_refusals(cuda_device):
    import gstreamer_b200 as g
    el = g.CudaVideoConvertScale(add_borders=False, method=1)
    ii, oi = g.VideoInfo(23, 64, 48), g.VideoInfo(2, 32, 24)
    oi.set_colorimetry(matrix=3 if ii.c.color_matrix == 4 else 4)           # a matrix stage: not built
    with pytest.raises(g.B200Error):
        el.set_info(ii, oi)


@pytest.mark.parametrize("size", [(64, 49, 32, 49), (50, 21, 50, 21), (33, 5, 70, 5), (1920, 1081, 1280, 1081), (7, 3, 7, 3)],
                         ids=lambda s: "%dx%d-%dx%d" % s)
def test_cross_family_odd_height_without_vertical_scaler(cuda_device, size):
    """the down-sampler's last pair reads line `oh`; with no vertical scaler to clamp it the reference rebuilds it from
    the last source line with a vertically unfiltered chroma row — a third launch over a one-line view of the frame"""
    import gstreamer_b200 as g
    iw, ih, ow, oh = size
    pair = ("NV12", "I420")
    frame = random_frame(pair, iw, ih, 3)
    for method in (1, 3):
        for site, out_site in ((1, 1), (2, 2), (2, 1), (1, 6), (4, 1)):
            if (iw, ih) == (ow, oh) and site == out_site:
                continue
            want = expected(size, method, frame, pair, site, out_site)
            (got,), oi = convert(size, method, frame, pair, site, out_site)
            assert not planes_equal(got, want, oi, ow, oh, False), (method, site, out_site)
    el = g.CudaVideoConvertScale(add_borders=False, method=1)
    ii, oi = g.VideoInfo(23, 64, 49), g.VideoInfo(2, 32, 49)
    g.transfer_colorimetry_from_input(ii, oi)
    el.set_info(ii, oi)
    assert int(el.plan_info().n_launches_per_convert) == 3
