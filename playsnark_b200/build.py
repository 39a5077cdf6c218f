"""Builds libplaysnark_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

One object file per translation unit, compiled in parallel and only when one of the files it includes
(transitively) has changed; then one link.  Objects live in playsnark_b200/_build/ (not shipped)."""
from __future__ import annotations

import glob
import os
import re
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libplaysnark_b200.so")

CU_SOURCES = [os.path.join(CSRC, f) for f in ("capi.cu", "capi_poly.cu", "capi_multi.cu", "capi_verify.cu", "group_g1.cu", "group_g2.cu", "accum_g2.cu")
              if os.path.exists(os.path.join(CSRC, f))]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
    "-lineinfo", "-Xcompiler", "-fPIC",
]

_INC = re.compile(r'^\s*#\s*include\s+"([^"]+)"', re.M)


def _deps(path: str, seen=None):
    """the file and every project header it includes, transitively"""
    seen = set() if seen is None else seen
    path = os.path.normpath(path)
    if path in seen or not os.path.exists(path):
        return seen
    seen.add(path)
    with open(path) as f:
        for inc in _INC.findall(f.read()):
            _deps(os.path.join(os.path.dirname(path), inc), seen)
    return seen


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) +
                  [os.path.join(ROOT, "include", "playsnark_b200.h")])


def stale(target: str, sources) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_cuda(force: bool = False, verbose: bool = False, out: str = LIB, extra_flags=()) -> str:
    if not force and not extra_flags and not stale(out, _sources()):
        return out
    nvcc = os.environ.get("NVCC", "nvcc")
    obj_dir = OBJ if out == LIB else out + ".obj"
    os.makedirs(obj_dir, exist_ok=True)
    jobs = []
    for src in CU_SOURCES:
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        if force or extra_flags or stale(obj, _deps(src)):
            jobs.append((src, obj))
    threads = max(1, (os.cpu_count() or 2) // max(1, len(jobs)))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + \
              ["-split-compile", str(threads), "-c", "-o", obj, src]
        print("[playsnark_b200] " + " ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd, cwd=ROOT)

    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(obj_dir, os.path.basename(s)[:-3] + ".o") for s in CU_SOURCES]
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + objs
    print("[playsnark_b200] " + " ".join(cmd), file=sys.stderr)
    subprocess.check_call(cmd, cwd=ROOT)
    return out


def build_variant(name: str, flags, tus=("capi_poly.cu",)) -> str:
    """A/B builds for kernel tuning: the listed translation units recompiled with extra -D flags, linked with the
    standard objects of the others into playsnark_b200/variants/lib_<name>.so (loaded through
    PLAYSNARK_B200_LIB by the tools/ab_*.py scripts)."""
    build_cuda()
    nvcc = os.environ.get("NVCC", "nvcc")
    vdir = os.path.join(OBJ, "variants")
    os.makedirs(vdir, exist_ok=True)
    objs = []
    for src in CU_SOURCES:
        base = os.path.basename(src)
        if base in tus:
            obj = os.path.join(vdir, "%s_%s.o" % (base[:-3], name))
            if stale(obj, _deps(src)):
                cmd = [nvcc] + NVCC_FLAGS + list(flags) + ["-split-compile", "0", "-c", "-o", obj, src]
                print("[playsnark_b200] " + " ".join(cmd), file=sys.stderr)
                subprocess.check_call(cmd, cwd=ROOT)
        else:
            obj = os.path.join(OBJ, base[:-3] + ".o")
        objs.append(obj)
    os.makedirs(os.path.join(HERE, "variants"), exist_ok=True)
    out = os.path.join(HERE, "variants", "lib_%s.so" % name)     # outside _build/: shipped to the GPU box
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + objs, cwd=ROOT)
    return out


TEST_BUILD = os.path.join(ROOT, "tests", "_build")
DEVICE_HARNESS = os.path.join(ROOT, "tests", "device_arith.cu")
PAIRING_HARNESS = os.path.join(ROOT, "tests", "device_pairing.cu")


def can_write(dir_path: str) -> bool:
    """dir_path exists and is writable, or can be created"""
    while not os.path.isdir(dir_path):
        parent = os.path.dirname(dir_path)
        if parent == dir_path:
            return False
        dir_path = parent
    return os.access(dir_path, os.W_OK | os.X_OK)


def harness_path(out_dir: str = TEST_BUILD, source: str = DEVICE_HARNESS, host: bool = False) -> str:
    """where build_device_harness puts `source`: out_dir/lib<name>.so (lib<name>_host.so for the host build)"""
    name = os.path.basename(source).rsplit(".", 1)[0]
    return os.path.join(out_dir, "lib%s%s.so" % (name, "_host" if host else ""))


def build_device_harness(out_dir: str = TEST_BUILD, source: str = DEVICE_HARNESS, host: bool = False) -> str:
    """TEST-ONLY: a device harness of the GPU suite (tests/device_arith.cu for tests/test_gpu_arith.py,
    tests/device_pairing.cu for tests/test_gpu_pairing.py) as out_dir/lib<name>.so for sm_100a, rebuilt when it or a
    header it includes has changed.  host=True compiles the same file with g++ -DPS_HOST_EMU instead (kernels become
    serial loops, for the CPU suite) as lib<name>_host.so.  Written under a temporary name and renamed, so a reader
    never loads a partial file."""
    so = harness_path(out_dir, source, host)
    if not stale(so, _deps(source)):
        return so
    os.makedirs(out_dir, exist_ok=True)
    tmp = "%s.%d.tmp" % (so, os.getpid())
    if host:
        cmd = ["g++", "-O2", "-std=c++17", "-x", "c++", "-DPS_HOST_EMU", "-fPIC", "-shared", "-o", tmp, source]
    else:
        cmd = [os.environ.get("NVCC", "nvcc")] + NVCC_FLAGS + ["-split-compile", "0", "-shared", "-o", tmp, source]
    print("[playsnark_b200] " + " ".join(cmd), file=sys.stderr)
    try:
        subprocess.check_call(cmd, cwd=ROOT)
        os.replace(tmp, so)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    return so


def build_host_emulation(out_dir: str) -> str:
    """TEST-ONLY: the same sources with -DPS_HOST_EMU (kernel bodies driven by serial loops)."""
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libps_hostemu.so")
    if not stale(so, _sources()):
        return so
    jobs = []
    for src in CU_SOURCES:
        obj = os.path.join(out_dir, "emu_" + os.path.basename(src)[:-3] + ".o")
        if stale(obj, _deps(src)):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-DPS_HOST_EMU", "-fPIC", "-c", "-o", obj, src], cwd=ROOT)

    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(out_dir, "emu_" + os.path.basename(s)[:-3] + ".o") for s in CU_SOURCES]
    subprocess.check_call(["g++", "-shared", "-o", so] + objs + ["-lpthread"], cwd=ROOT)
    return so


if __name__ == "__main__":
    build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv)
