"""Builds libinfernos_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libinfernos_b200.so")
SOURCES = ["tail.cu", "codec_kernels.cu", "conv_simt.cu", "conv_umma.cu", "conv_resblock.cu", "conv_resblock_t.cu", "sched.cu", "server.cu", "decoder.cu", "encoder.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "infernos_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, extra_flags=(), so_out: str = SO, tag: str = "") -> str:
    """extra_flags / out / tag: variant builds (e.g. -DB2_RBT_ZERO_INIT into libinfernos_b200_zeroinit.so; load with B2_SO_PATH)."""
    if not force and not extra_flags and not needs_build():
        return SO
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC, s.replace(".cu", tag + ".o"))
        cmd = [nvcc(), *FLAGS, *extra_flags, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas"); cmd.insert(2, "-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {s}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc(), "-shared", "-o", so_out, *objs])
    return so_out


if __name__ == "__main__":
    if "--variant" in sys.argv:          # python -m infernos_b200.build --variant zeroinit -DB2_RBT_ZERO_INIT
        i = sys.argv.index("--variant")
        name, flags = sys.argv[i + 1], [a for a in sys.argv[i + 2:] if a.startswith("-D")]
        print(build(force=True, extra_flags=flags, so_out=os.path.join(HERE, f"libinfernos_b200_{name}.so"), tag="_" + name))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
