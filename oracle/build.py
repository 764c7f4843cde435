"""Build recipe for the CPU oracle (test infrastructure, not product code).

Compiles oracle/wr_oracle.c + oracle/wr_oracle_blend.c -> oracle/_build/libwr_oracle.so with gcc.  `-ffp-contract=off`
is REQUIRED: the raster contract (DESIGN.md section 3) is a sequence of individually rounded
fp32 operations and a fused multiply-add would change coverage at snap boundaries.

There is no `oracle/_ref`: the reference (/root/reference) contains no native source for this
path -- its arithmetic lives in the un-vendored nvdiffrast dependency (requirements.txt:55),
so nothing of the reference can be compiled here (recorded in DESIGN.md section 6).
"""
from __future__ import annotations

import atexit
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRCS = [os.path.join(HERE, "wr_oracle.c"), os.path.join(HERE, "wr_oracle_blend.c")]
OUT_DIR = os.path.join(HERE, "_build")

# -O3 -march=native as BASELINE.md section 4 states for the CPU arm; -ffp-contract=off keeps every operation
# individually rounded whatever the target supports.  Because of -march=native the library is specific to the
# host it was built on: its name carries a hash of the host's CPU flags and it is (re)built on first use on a
# new host (gcc is part of the image; ~3 s).
CFLAGS = ["-O3", "-march=native", "-fPIC", "-shared", "-std=c11", "-fopenmp", "-ffp-contract=off",
          "-fno-fast-math", "-Wall", "-Wextra"]


def _host_tag() -> str:
    import hashlib
    flags = ""
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags") or line.startswith("model name"):
                    flags += line
                    if line.startswith("flags"):
                        break
    except OSError:
        pass
    return hashlib.sha1(flags.encode()).hexdigest()[:10]


LIB = os.path.join(OUT_DIR, f"libwr_oracle_{_host_tag()}.so")


def build(force: bool = False) -> str:
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= max(os.path.getmtime(p) for p in SRCS):
        return LIB
    lib = LIB
    if not os.access(OUT_DIR if os.path.isdir(OUT_DIR) else HERE, os.W_OK):
        # A read-only tree (bench.py may run from one) on a host without a build for its CPU: build into a directory
        # private to this process (mkdtemp: mode 0700, a fresh name), never reused and removed at exit.
        out = tempfile.mkdtemp(prefix="wr_oracle_")
        atexit.register(shutil.rmtree, out, True)
        lib = os.path.join(out, os.path.basename(LIB))
    os.makedirs(os.path.dirname(lib), exist_ok=True)
    tmp = lib + f".{os.getpid()}.tmp"   # several ranks may build at once: write aside, then rename atomically
    cmd = ["gcc", *CFLAGS, *SRCS, "-o", tmp, "-lm"]
    subprocess.run(cmd, check=True)
    os.replace(tmp, lib)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
