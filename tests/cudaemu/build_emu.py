#!/usr/bin/env python
"""tests/cudaemu/build_emu.py — TEST INFRASTRUCTURE.

Builds tests/cudaemu/_build/libb200emu.so: the product's convert+scale glue (vcs.cu), its host plan builder, the video
kernels (all but vcs_l2tc_kernel), the compositor and the audio resampler compiled with g++ against the stand-in runtime
in emu/ (warp collectives emulated lane by lane, PTX helpers on their plain-C branch).  The sources are the product's own files,
patched textually only where CUDA syntax has no C++ spelling:
    kernel <<<grid, block, smem, stream>>> (args);   ->   b200emu::launch (grid, block, smem, [&] { kernel (args); });
    extern __shared__ ... smem[];                    ->   uint8_t *smem = b200emu::dyn_smem;
    __shared__ T x[N];                               ->   static T x[N];
The library exports the same b200_vcs_* C-ABI; "device pointers" are host pointers.  It exists so that kernel indexing
and integer arithmetic can be checked against the oracle without a GPU — it is never loaded by gstreamer_b200.

build("ubsan") makes a second library in _build_ubsan/ with -fsanitize=undefined and every report fatal: with the
vector types at CUDA's alignments (emu/cuda_runtime.h) a misaligned uint2 / uint4 access, which faults on the device,
aborts the process there.  Each variant has its own directory, lock and stamp, so the builds do not replace each
other's library under pytest-xdist."""
import hashlib
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "gstreamer_b200", "csrc")
OUT = os.path.join(HERE, "_build")
LIB = os.path.join(OUT, "libb200emu.so")
# g++ keeps going after an alignment report even with -fno-sanitize-recover=alignment; =all makes every report fatal
VARIANTS = {None: [], "ubsan": ["-fsanitize=undefined", "-fno-sanitize-recover=all"]}

LAUNCH = re.compile(r"(\b\w+(?:<[^<>;()]*>)?)\s*<<<(.+?)>>>\s*\(([^;]*)\);")


def split_top(s):
    """split on commas that are not inside <...> or (...)"""
    parts, depth, cur = [], 0, ""
    for ch in s:
        if ch in "<(":
            depth += 1
        elif ch in ">)":
            depth -= 1
        if ch == "," and depth == 0:
            parts.append(cur.strip())
            cur = ""
        else:
            cur += ch
    parts.append(cur.strip())
    return parts


def patch(text):
    def repl(m):
        name, cfg, args = m.group(1), m.group(2), m.group(3)
        parts = split_top(cfg)
        assert len(parts) == 4, cfg
        return f"b200emu::launch ({parts[0]}, {parts[1]}, {parts[2]}, [&] {{ {name} ({args}); }});"
    text, n = LAUNCH.subn(repl, text)
    text = re.sub(r"extern __shared__ __align__ \((?:16|128)\) (\w+) (\w+)\[\];", r"\1 *\2 = (\1 *) b200emu::dyn_smem;", text)
    text = re.sub(r"(^|\n)(\s*)__shared__ ", r"\1\2static ", text)
    return text, n


def sources():
    return [os.path.join(CSRC, f) for f in ("vcs.cu", "vcs_planes.cuh", "vcs_planes_fast.cuh", "vcs_kernels.cuh", "vcs_down420.cuh", "vcs_rgb420.cuh", "vcs_yuy2_420.cuh", "vcs_l2mma.cuh", "vcs_lanczos2.cuh", "vcs_lanczos2_v2.cuh", "vcs_light.cuh",
                                            "vcs_ntap.cuh", "common.cu", "comp.cu", "ars.cu", "besi0_coeffs.inc",
                                            "vcs_plan.cpp", "vcs_plan.h", "vcs_device.h", "common.h")] + \
        [os.path.join(HERE, "emu", f) for f in sorted(os.listdir(os.path.join(HERE, "emu")))] + [os.path.abspath(__file__)]


def digest(variant=None):
    h = hashlib.sha256()
    h.update((repr(variant) + "/").encode())
    h.update((os.environ.get("B200_EMU_TSAN", "") + "/" + os.environ.get("B200_EMU_DROP_SYNC", "") + "/" + os.environ.get("B200_EMU_ASAN", "") + "/" + os.environ.get("B200_EMU_UBSAN", "")).encode())
    for s in sources():
        h.update(open(s, "rb").read())
    return h.hexdigest()


def out_dir(variant=None):
    return OUT if variant is None else OUT + "_" + variant


def build(force=False, variant=None):
    """returns the path of the library; variant None (the plain build, sanitizers from B200_EMU_* variables) or 'ubsan'"""
    # one builder at a time (pytest-xdist workers all arrive here after a source change); the others wait and then find
    # the stamp up to date
    import fcntl
    if variant not in VARIANTS:
        raise ValueError(f"unknown emulator build variant {variant!r}")
    out = out_dir(variant)
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        return _build_locked(force, variant, out)


def _build_locked(force, variant, out):
    stamp = os.path.join(out, "stamp")
    lib = os.path.join(out, "libb200emu.so")
    d = digest(variant)
    if not force and os.path.exists(lib) and os.path.exists(stamp) and open(stamp).read() == d:
        return lib
    gen = os.path.join(out, "gen")
    os.makedirs(gen, exist_ok=True)
    launches = 0
    for src, dst in (("vcs.cu", "vcs_emu.cpp"), ("vcs_planes.cuh", "vcs_planes.cuh"), ("vcs_planes_fast.cuh", "vcs_planes_fast.cuh"), ("vcs_kernels.cuh", "vcs_kernels.cuh"),
                     ("vcs_down420.cuh", "vcs_down420.cuh"), ("vcs_rgb420.cuh", "vcs_rgb420.cuh"), ("vcs_yuy2_420.cuh", "vcs_yuy2_420.cuh"), ("vcs_l2mma.cuh", "vcs_l2mma.cuh"), ("vcs_lanczos2.cuh", "vcs_lanczos2.cuh"), ("vcs_lanczos2_v2.cuh", "vcs_lanczos2_v2.cuh"),
                     ("vcs_light.cuh", "vcs_light.cuh"), ("vcs_ntap.cuh", "vcs_ntap.cuh"), ("common.cu", "common_emu.cpp"),
                     ("comp.cu", "comp_emu.cpp"), ("ars.cu", "ars_emu.cpp")):
        text, n = patch(open(os.path.join(CSRC, src)).read())
        if os.environ.get("B200_EMU_DROP_SYNC") and src == "vcs_kernels.cuh":    # negative control for the race detector
            text = text.replace("__syncthreads ();", "", 1)
        launches += n
        open(os.path.join(gen, dst), "w").write(text)
    assert launches >= 18, f"expected the launch sites of vcs.cu and vcs_planes.cuh, patched {launches}"
    for f in os.listdir(os.path.join(HERE, "emu")):                # stand-in headers next to the generated sources
        if f.endswith((".h", ".cuh")):
            open(os.path.join(gen, f), "w").write(open(os.path.join(HERE, "emu", f)).read())
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-Wno-unknown-pragmas", "-DB200_CUDA_EMU=1",
           "-I", gen, "-I", CSRC, "-o", lib + ".tmp",
           os.path.join(gen, "vcs_emu.cpp"), os.path.join(gen, "common_emu.cpp"), os.path.join(gen, "comp_emu.cpp"),
           os.path.join(gen, "ars_emu.cpp"), os.path.join(CSRC, "vcs_plan.cpp"),
           os.path.join(HERE, "emu", "emu_runtime.cpp")]
    if os.environ.get("B200_EMU_ASAN"):              # out-of-bounds accesses of frames, tables and static shared arrays
        cmd[1:1] = ["-fsanitize=address", "-fno-omit-frame-pointer"]
    if os.environ.get("B200_EMU_UBSAN"):             # misaligned vector accesses (a fault on the device), shifts, overflows
        cmd[1:1] = ["-fsanitize=undefined"]
    cmd[1:1] = VARIANTS[variant]
    if os.environ.get("B200_EMU_TSAN"):              # race detector build: every shared-memory access of the kernels is checked
        cmd[1:1] = ["-fsanitize=thread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout[-4000:] + r.stderr[-8000:])
        raise RuntimeError("emulation build failed")
    os.replace(lib + ".tmp", lib)                     # never write into a library another process has mapped
    open(stamp, "w").write(d)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, variant="ubsan" if "--ubsan" in sys.argv else None))
