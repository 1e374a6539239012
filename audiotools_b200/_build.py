"""In-tree build of ``audiotools_b200/csrc/libb2a.so`` for sm_100a (nvcc cross-compiles
without a GPU).  The .so is git-ignored but travels to the GPU box with the snapshot."""
import glob
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(CSRC, "libb2a.so")
STAMP = os.path.join(CSRC, ".libb2a.stamp")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _digest(files):
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in sorted(files):
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Build (if stale) and return the path of libb2a.so.  Safe to call from several processes at once (the ranks of a
    torchrun launch, the two ranks of a gloo test): an exclusive file lock serialises the builders and the library is
    moved into place atomically, so a concurrent importer never sees a half-written file.  An up-to-date library is
    returned without writing anything, so a built tree may be read-only."""
    import fcntl

    if not force and _up_to_date(_digest(_deps())):
        return OUT
    with open(os.path.join(CSRC, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _deps():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu"))) + sorted(glob.glob(os.path.join(CSRC, "*.h"))) + sorted(
        glob.glob(os.path.join(CSRC, "*.cuh"))) + [os.path.join(os.path.dirname(HERE), "include", "b2a.h")]


def _up_to_date(dig: str) -> bool:
    """The library exists and the stamp written after it names the digest ``dig`` of the current sources."""
    return os.path.exists(OUT) and os.path.exists(STAMP) and open(STAMP).read() == dig


def _build_locked(force: bool, verbose: bool) -> str:
    deps = _deps()
    srcs = [d for d in deps if d.endswith(".cu")]
    dig = _digest(deps)
    if not force and _up_to_date(dig):
        return OUT
    nvcc = _nvcc()
    objs, procs = [], []
    for s in srcs:
        o = s[:-3] + ".o"
        cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out.decode()}")
    tmp = OUT + ".tmp.%d" % os.getpid()
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs
    subprocess.check_call(cmd)
    os.replace(tmp, OUT)
    with open(STAMP, "w") as f:
        f.write(dig)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
