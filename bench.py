#!/usr/bin/env python
"""bench.py — headline benchmark of the convert+scale hot path (BASELINE.json configs[1]).

Workload (N=1): 3840x2160 NV12 -> 1920x1080 BGRA, method=lanczos (8-tap, 6-bit taps), bt709
16-235, chroma-site mpeg2.  One "step" = one batch of FRAMES_PER_STEP distinct frames drawn from
a ring whose working set (>= 1.3 GB) is far larger than the 126 MB L2, so no L2 flush is needed.

  value      whole-job Mpix/s (input pixels), frames resident in HBM, kernel launches only
  e2e        same metric through the C-ABI host call (pinned host buffers, H2D + kernel + D2H
             inside the timed region)
  roofline   algorithmic bytes (20 736 000 B/frame, SURVEY §8d) / CUDA-event kernel time vs the
             measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the reference's own converter (oracle/_ref, compiled from /root/reference
             sources) — or the oracle port if that library is absent — on the host cores

N>1: one process per GPU (torchrun), independent streams, no collective on the data path
(SURVEY §8e): "scaling": "weak".  `--impl reference` times the reference CPU path instead.

`--dump-outputs DIR` writes what the last timed step returned (rank 0's frames, see dump_outputs) so
that two builds run with the same arguments can be compared output for output: the input frames
are generated from fixed seeds.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IW, IH, OW, OH = 3840, 2160, 1920, 1080
METHOD = 3  # GST_VIDEO_SCALE_LANCZOS
ALG_BYTES_PER_FRAME = 12_441_600 + 8_294_400
IN_PIX_PER_FRAME = IW * IH
FRAMES_PER_STEP = 32
RING = 64
WORKLOAD = "3840x2160 NV12 -> 1920x1080 BGRA, lanczos (8-tap), videoconvertscale semantics"
METRIC = "4K NV12->BGRA+lanczos->1080p throughput"
REF_NOTE = ("oracle/_ref: the reference's own video-converter.c compiled here, ORC C backups (no liborc SIMD JIT), n-threads = all "
            "cores but the converter caps its task count at rows/200 (about 10 effective threads for 4K -> 1080p)")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        if self._run_nvml():
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    f = [x.strip() for x in line.split(",")]
                    if len(f) >= 9:
                        self.samples.append(f)
            except Exception:
                pass
            self._stop.wait(0.1)

    def _run_nvml(self):
        """NVML (the library nvidia-smi itself queries) polled every millisecond: the timed region is tens of ms"""
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis:
                ids = [v for v in vis.split(",") if v.strip()]
                if self.gpu < len(ids) and ids[self.gpu].strip().isdigit():
                    idx = int(ids[self.gpu])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            return False
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = get_reasons(h)
                self.samples.append([str(self.gpu), str(sm), str(mx), "", hex(r)] +
                                    ["Active" if r & bits[k] else "Not Active" for k in
                                     ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            except Exception:
                pass
            self._stop.wait(0.001)
        return True

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit())
        mx = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for name, v in zip(names, s[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def ncu_traffic(kernel, frames_per_launch):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/)"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) * frames_per_launch / t["frames_per_launch"]
    except Exception:
        return None


def cpu_baseline(seconds=10.0, threads=None):
    """time the reference's CPU converter on frames of the same workload"""
    import numpy as np
    from oracle import bindings as ob
    cores = threads or os.cpu_count() or 1
    frames = [ob.nv12_random_frame(IW, IH, s) for s in range(2)]
    if ob.have_ref():
        kind = "reference"
        conv = ob.RefVcs(IW, IH, OW, OH, METHOD, n_threads=cores)
        out = np.zeros(OW * OH * 4, dtype=np.uint8)
        run = lambda f: conv.convert(f, out)
        impl = REF_NOTE
    else:
        kind = "port"
        cores = 1
        d = ob.vcs_desc(IW, IH, OW, OH, METHOD)
        run = lambda f: ob.oracle_vcs_convert(d, f)
        impl = "oracle port (scalar C)"
    run(frames[0])  # warm (tap tables are built lazily on first use)
    n, t0 = 0, time.perf_counter()
    while True:
        run(frames[n % 2])
        n += 1
        dt = time.perf_counter() - t0
        if dt >= seconds and n >= 3:
            break
    return {"value": n * IN_PIX_PER_FRAME / dt / 1e6, "unit": "Mpix/s", "cores": cores, "kind": kind,
            "sample": f"{n} frames of the same workload in {dt:.1f} s, {impl}"}


DUMP_SAMPLE = 4 << 20      # sampled bytes of a step's whole output


def dump_outputs(path, frames):
    """frames: the FRAMES_PER_STEP BGRA frames one step wrote.  Saved as float32 (about 50 MB):
    bgra_last_frame.npy   the step's last frame, (OH, OW, 4)
    bgra_sample.npy       the bytes at np.unique(default_rng(0).integers(0, n, DUMP_SAMPLE)) of all n output bytes
                          of the step, frame after frame"""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    out = torch.stack(frames)
    np.save(os.path.join(path, "bgra_last_frame.npy"), out[-1].view(OH, OW, 4).cpu().numpy().astype(np.float32))
    idx = np.unique(np.random.default_rng(0).integers(0, out.numel(), DUMP_SAMPLE))
    sample = out.view(-1)[torch.from_numpy(idx).to(out.device)]
    np.save(os.path.join(path, "bgra_sample.npy"), sample.cpu().numpy().astype(np.float32))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import bindings as ob
    import numpy as np
    cores = os.cpu_count() or 1
    per_step = FRAMES_PER_STEP
    frames = [ob.nv12_random_frame(IW, IH, s) for s in range(4)]
    if ob.have_ref():
        kind = "reference"
        conv = ob.RefVcs(IW, IH, OW, OH, METHOD, n_threads=cores)
        out = np.zeros(OW * OH * 4, dtype=np.uint8)
        run = lambda f: conv.convert(f, out)
        note = REF_NOTE
    else:
        kind, cores = "port", 1
        d = ob.vcs_desc(IW, IH, OW, OH, METHOD)
        run = lambda f: ob.oracle_vcs_convert(d, f)
        note = "oracle port (scalar C, 1 thread)"
    for _ in range(min(args.warmup, 3)):
        for k in range(4):
            run(frames[k])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for k in range(per_step):
            run(frames[k % 4])
    dt = time.perf_counter() - t0
    val = args.steps * per_step * IN_PIX_PER_FRAME / dt / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val,
            "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step": per_step},
            "cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": cores, "kind": kind,
                             "sample": f"{args.steps} steps x {per_step} frames; {note}"},
            "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_extras(steps):
    """the other BASELINE configs on this GPU (kernel-resident, CUDA events): C1 element default, C4 both backgrounds, C5;
    and the YUV -> YUV scaling cases of bench_extra.py --only planes"""
    import bench_extra as bx
    bx.QUIET = True
    a = argparse.Namespace(steps=steps, seconds=20, background=0, no_cpu=True, variant=-1)
    out = {}

    def slim(d, key="us_per_frame"):
        r = d["roofline"]
        e = {"us": d.get(key), "alg_bytes": r.get("alg_bytes_per_launch"), "achieved_gbs": r["achieved"], "frac": r["frac"],
             "config": d["config"]}
        if "achieved_gflops" in r:
            e["achieved_gflops_non_fma"] = r["achieved_gflops"]
        return e
    try:
        d = bx.bench_c1(a)
        d["us_per_frame"] = d["us_per_frame"]
        e = slim(d); e["alg_bytes"] = d["roofline"]["alg_bytes_per_launch"] // 64; e["kernel_variant"] = d["kernel_variant"]
        out["c1"] = e
        a.background = 0
        out["c4_checker"] = slim(bx.bench_c4(a))
        a.background = 3
        out["c4_transparent"] = slim(bx.bench_c4(a))
        a.steps = max(3, steps // 4)
        d = bx.bench_c5(a)
        d["us_per_frame"] = d["ms_per_buffer"] * 1e3
        out["c5"] = slim(d)
        # the transcoding-ladder cases (not BASELINE configs): YUV -> YUV plane scaling and the cross-family chain
        a.steps = max(3, steps // 2)
        ladder, rgb = [], []
        for d in bx.bench_planes(a):
            e = slim(d); e["alg_bytes"] = d["roofline"]["alg_bytes_per_launch"] // 32; e["kernel_variant"] = d["kernel_variant"]
            (rgb if d["config"].startswith(("BGRA", "RGBA", "YUY2", "UYVY")) else ladder).append(e)
        out["yuv_ladder"] = ladder
        out["rgb_paths"] = rgb          # packed RGB -> packed RGB scaling, packed RGB / packed 4:2:2 -> 4:2:0 (compositor / capture -> encoder)
    except Exception as e:          # an extra must never take the headline line down
        out["error"] = repr(e)
    return out


def run_ours(args):
    import numpy as np
    import torch
    import gstreamer_b200 as g
    from oracle import bindings as ob  # input generator only (synthetic frames)

    from gstreamer_b200 import multi
    rank, world, local = multi.rank_info()
    numa = multi.bind_to_gpu_numa(local)          # before any staging memory exists
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist = multi.init("nccl", device=dev)

    el = g.CudaVideoConvertScale(method=METHOD, cuda_device_id=local)
    ii, oi = g.VideoInfo(g.VideoFormat.NV12, IW, IH), g.VideoInfo(g.VideoFormat.BGRA, OW, OH)
    el.set_info(ii, oi)
    pinfo = el.plan_info()
    from gstreamer_b200 import _lib as _b200lib
    kname = _b200lib.lib.b200_vcs_kernel_name(el._h).decode()

    # ring of distinct frames resident in HBM
    base = [torch.from_numpy(ob.nv12_random_frame(IW, IH, multi.stream_seed(rank, s))).to(dev) for s in range(4)]
    ring_in = []
    for k in range(RING):
        t = base[k % 4].clone()
        t[:: 4099] = (t[:: 4099].to(torch.int32) + k).to(torch.uint8)  # make every frame distinct
        ring_in.append(t)
    ring_out = [torch.empty(oi.size, dtype=torch.uint8, device=dev) for _ in range(RING)]
    stream = torch.cuda.Stream(device=dev)

    def step(i):
        o = (i % (RING // FRAMES_PER_STEP)) * FRAMES_PER_STEP
        el.transform_frames(ring_in[o:o + FRAMES_PER_STEP], ring_out[o:o + FRAMES_PER_STEP], stream)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    profiling = os.environ.get("B200_PROFILE") == "1"      # ncu --profile-from-start off
    if profiling:
        torch.cuda.cudart().cudaProfilerStart()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for i in range(args.steps):
            step(i)
        e1.record(stream)
    barrier()
    if profiling:
        torch.cuda.cudart().cudaProfilerStop()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        o = ((args.steps - 1) % (RING // FRAMES_PER_STEP)) * FRAMES_PER_STEP      # what step(args.steps - 1) wrote
        dump_outputs(args.dump_outputs, ring_out[o:o + FRAMES_PER_STEP])

    # ---- sustained: the same launches back to back for >= 2 s (an issue-bound kernel follows the SM clock, and the
    # clock under a seconds-long load is not the burst clock)
    sustained = None
    if not profiling and args.sustained_seconds > 0:
        n_sus = max(50, int(args.sustained_seconds * 1e3 / max(ms / args.steps, 1e-3)))
        barrier()
        s2 = ClockSampler(local)
        if rank == 0:
            s2.start()
        with torch.cuda.stream(stream):
            e0.record(stream)
            for i in range(n_sus):
                step(i)
            e1.record(stream)
        barrier()
        sus_ms = e0.elapsed_time(e1)
        c2 = s2.stop() if rank == 0 else None
        sus_ms, = multi.reduce_max(dist, [sus_ms], device=dev)
        sustained = {"launches": n_sus, "seconds": sus_ms * 1e-3,
                     "value": n_sus * FRAMES_PER_STEP * world * IN_PIX_PER_FRAME / (sus_ms * 1e-3) / 1e6, "unit": "Mpix/s",
                     "us_per_launch": sus_ms * 1e3 / n_sus, "clocks": c2}

    # ---- e2e: host frames through the C-ABI (pinned staging next to the GPU, copies inside the timed region)
    e2e_frames = 32
    hin = [g.PinnedBuffer(ii.size, device=local) for _ in range(e2e_frames)]
    hout = [g.PinnedBuffer(oi.size, device=local) for _ in range(e2e_frames)]
    for k, b in enumerate(hin):
        b.array[:] = ob.nv12_random_frame(IW, IH, 77 + k % 4)
        b.array[:: 4099] += k
    inp, outp = [b.ptr for b in hin], [b.ptr for b in hout]
    for _ in range(max(1, min(args.warmup, 3))):
        el.transform_host_frames(inp, outp)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        el.transform_host_frames(inp, outp)     # returns when every output is back in host memory
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    checksum = int(hout[0].array[:4096].sum())
    # the link's ceiling for the same call: the same copies on the same buffers without the kernels
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        el.copy_probe(inp, outp)
    torch.cuda.synchronize()
    probe_s = time.perf_counter() - t0

    ms, e2e_s, probe_s = multi.reduce_max(dist, [ms, e2e_s, probe_s], device=dev)    # slowest rank defines the job
    extras = run_extras(10) if (rank == 0 and world == 1 and not args.no_extras and not profiling) else None
    if rank == 0:
        frames = args.steps * FRAMES_PER_STEP * world
        value = frames * IN_PIX_PER_FRAME / (ms * 1e-3) / 1e6
        peak, peak_src = measured_peak()
        achieved = args.steps * FRAMES_PER_STEP * ALG_BYTES_PER_FRAME / (ms * 1e-3) / 1e9   # per GPU
        e2e_val = e2e_steps * e2e_frames * world * IN_PIX_PER_FRAME / e2e_s / 1e6
        ceil_val = e2e_steps * e2e_frames * world * IN_PIX_PER_FRAME / probe_s / 1e6
        traffic = ncu_traffic(kname, FRAMES_PER_STEP)
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s",
            "frames_per_s": frames / (ms * 1e-3),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step": FRAMES_PER_STEP, "ring_frames": RING,
                       "l2": "inputs larger than L2 (ring %.0f MB in + %.0f MB out)" %
                             (RING * ii.size / 1e6, RING * oi.size / 1e6),
                       "kernel_variant": int(pinfo.kernel_variant), "parallelism": f"streams{world}", "numa": numa},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_source": "dram__bytes_read+write of the committed ncu --set full capture (profiles/traffic.json), not measured in this run",
                         "peak_source": peak_src, "kernel": kname,
                         "alg_bytes_per_launch": FRAMES_PER_STEP * ALG_BYTES_PER_FRAME,
                         "us_per_launch": ms * 1e3 / args.steps},
            "sustained": sustained,
            "e2e": {"value": e2e_val, "unit": "Mpix/s", "h2d_bytes_per_step": e2e_frames * ii.size,
                    "d2h_bytes_per_step": e2e_frames * oi.size, "frames_per_step": e2e_frames,
                    "steps": e2e_steps, "checksum": checksum,
                    "copy_ceiling": {"value": ceil_val, "unit": "Mpix/s", "frac_of_ceiling": e2e_val / ceil_val,
                                     "what": "the same H2D || D2H copies on the same pinned buffers without the kernels (b200_vcs_copy_probe)"},
                    "staging": "b200_host_alloc_near: mbind to the GPU's NUMA node, then cudaHostRegister"},
            "gpu_launches": args.steps * pinfo.n_launches_per_convert,
            "clocks": clocks,
        }
        if extras is not None:
            line["extra"] = extras
        if world == 1 and not profiling and not args.no_extras:
            # the reference's GPU path for the same conversion: its CUDA converter kernel (texture-bilinear, float
            # matrix - different arithmetic, so a speed reference only), compiled from the reference's own source
            gb = ob.run_refcuda_bench()
            if gb is not None and "us_per_frame" in gb:
                gb.update({"value": gb["mpix_per_s_in"], "unit": "Mpix/s", "frac": gb["achieved_gbs"] / peak,
                           "note": "reference cudaconvertscale kernel, bilinear texture sampling: not bit-exact with videoconvertscale"})
            line["gpu_baseline"] = gb
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C1 / C4 / C5 block of the line")
    ap.add_argument("--sustained-seconds", type=float, default=2.5)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output frames to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
