"""
TEST TOOLING: build the host-emulated SwiFTly library (tests/emu/libswiftly_emu.so).

The same kernel sources as the CUDA product (csrc/*.cu, *.cuh) are compiled with
plain g++ and -DSWIFTLY_EMU; CUDA threads run as fibres (emu_runtime.h).  Used
only by tests marked "not gpu" to check kernel index algebra without a GPU.
"""

import fcntl
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "ska_sdp_distributed_fourier_transform_b200", "csrc")
OUT = os.path.join(HERE, "libswiftly_emu.so")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def deps():
    return sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + sorted(
        glob.glob(os.path.join(CSRC, "*.h"))
    ) + [os.path.join(HERE, "emu_runtime.h"), os.path.join(ROOT, "include", "swiftly_b200.h")]


def up_to_date():
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(d) <= t for d in deps())


def build(force=False, opt="-O1"):
    if not force and up_to_date():
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    # Several test processes (the spawned ranks of tests/test_dist_gloo.py) may ask for the
    # library at once: one builds while the others wait, and the library appears under its
    # name only once it is completely linked.
    with open(os.path.join(objdir, "build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and up_to_date():
            return OUT
        procs = []
        objs = []
        for src in sources():
            obj = os.path.join(objdir, os.path.basename(src) + ".o")
            objs.append(obj)
            cmd = ["g++", "-std=c++17", opt, "-fPIC", "-x", "c++", "-DSWIFTLY_EMU", "-I", HERE,
                   "-I", os.path.join(ROOT, "include"), "-Wno-unknown-pragmas", "-c", src, "-o",
                   obj]
            procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE,
                                                stderr=subprocess.STDOUT)))
        for cmd, p in procs:
            out, _ = p.communicate()
            if p.returncode != 0:
                sys.stderr.write(out.decode())
                raise RuntimeError("emulator build failed: " + " ".join(cmd))
        tmp = os.path.join(objdir, os.path.basename(OUT) + ".tmp")
        subprocess.check_call(["g++", "-shared", "-o", tmp] + objs)
        os.replace(tmp, OUT)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
