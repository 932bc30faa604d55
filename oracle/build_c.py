"""Builds oracle/_cbuild/libsipref*.so from oracle/c/ref_kernels.c (gcc + OpenMP).

TEST / MEASUREMENT INFRASTRUCTURE ONLY: the threaded CPU restatement timed by bench.py's cpu_baseline and
`--impl reference` legs.  Two builds: a portable one (no -march flag: built in one container, may run on another host)
and, when gcc is present on the machine that RUNS the baseline, one with -march=native (BASELINE.md §4) tagged with the
CPU model it was built for; `build()` returns the native one when it matches this host.  A run loads
`runtime_library()`, which never writes into the tree (it may be read-only then)."""
from __future__ import annotations

import atexit
import hashlib
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "c", "ref_kernels.c")
DEPS = [SRC, os.path.join(HERE, "c", "ref_kernels_body.inc"), os.path.join(HERE, "c", "ref_kernels.h")]
OUT = os.path.join(HERE, "_cbuild", "libsipref.so")
FLAGS = ["-O3", "-fopenmp", "-fPIC", "-shared", "-std=c11", "-Wall"]


def _cpu_tag() -> str:
    """Short hash of this host's CPU model and ISA flags: a -march=native build is only reused on the same CPU."""
    model, flags = "", ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and not model:
                model = line.split(":", 1)[1].strip()
            elif line.startswith("flags") and not flags:
                flags = line.split(":", 1)[1].strip()
            if model and flags:
                break
    except OSError:
        return "generic"
    return hashlib.sha1((model + "|" + flags).encode()).hexdigest()[:12]


def _stale(out: str) -> bool:
    return not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in DEPS)


def needs_build() -> bool:
    return _stale(OUT)


def build(force: bool = False, native: bool = True, out_dir: str | None = None) -> str:
    out_dir = out_dir or os.path.dirname(OUT)
    out = os.path.join(out_dir, os.path.basename(OUT))
    os.makedirs(out_dir, exist_ok=True)
    have_gcc = shutil.which("gcc") is not None
    if (force or _stale(out)) and have_gcc:
        subprocess.run(["gcc"] + FLAGS + ["-o", out, SRC, "-lm"], check=True)
    if native and have_gcc:
        out_n = os.path.join(out_dir, "libsipref_native_%s.so" % _cpu_tag())
        try:
            if force or _stale(out_n):
                subprocess.run(["gcc"] + FLAGS + ["-march=native", "-o", out_n, SRC, "-lm"], check=True)
            return out_n
        except (subprocess.CalledProcessError, OSError):
            pass
    if not os.path.exists(out):
        raise RuntimeError("libsipref.so is missing and gcc is not available")
    return out


_RUNTIME = {}


def runtime_library() -> str:
    """The library a run loads: the in-tree -march=native build when it is current for this host, else, with gcc, a
    build in a temporary directory removed at exit, else the in-tree portable build."""
    if "path" not in _RUNTIME:
        native = os.path.join(HERE, "_cbuild", "libsipref_native_%s.so" % _cpu_tag())
        if not _stale(native):
            _RUNTIME["path"] = native
        elif shutil.which("gcc") is not None:
            tmp = tempfile.mkdtemp(prefix="sipref-")
            atexit.register(shutil.rmtree, tmp, True)
            _RUNTIME["path"] = build(out_dir=tmp)
        elif os.path.exists(OUT):
            _RUNTIME["path"] = OUT
        else:
            raise RuntimeError("libsipref.so is missing and gcc is not available")
    return _RUNTIME["path"]


def is_native(path: str) -> bool:
    return "native" in os.path.basename(path)


if __name__ == "__main__":
    print(build(force=True))
