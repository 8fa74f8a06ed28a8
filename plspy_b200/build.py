"""Builds plspy_b200/libplsb200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

    python -m plspy_b200.build            # incremental (skips if up to date)
    python -m plspy_b200.build --force

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libplsb200.so")
SOURCES = ["abi.cu", "gram.cu", "nspace.cu", "boot.cu", "boot_quad.cu", "boot_os.cu", "boot_tf32.cu", "gram_tf32.cu", "split.cu", "rb.cu", "rb_dmma.cu", "half_gram.cu", "percentile.cu", "host_rng.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr",
]


def _deps():
    d = [os.path.join(CSRC, s) for s in SOURCES]
    d += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    d.append(os.path.join(os.path.dirname(HERE), "include", "plsb200.h"))
    return d


STAMP = OUT + ".srchash"


def _source_hash():
    import hashlib
    h = hashlib.sha256()
    for f in sorted(_deps()):
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def up_to_date():
    """The library is current when the hash of all sources recorded at build time matches (file times are not
    reliable after the tree has been copied to another machine)."""
    if not (os.path.exists(OUT) and os.path.exists(STAMP)):
        return False
    return open(STAMP).read().strip() == _source_hash()


def _object_hash(src):
    """Hash of everything one object file depends on: its source, the shared headers and the flags."""
    import hashlib
    h = hashlib.sha256()
    deps = [os.path.join(CSRC, src)] + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
    deps.append(os.path.join(os.path.dirname(HERE), "include", "plsb200.h"))
    for f in deps:
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC, os.path.splitext(s)[0] + ".o")
        objs.append(o)
        ostamp, want = o + ".srchash", _object_hash(s)
        if not force and os.path.exists(o) and os.path.exists(ostamp) and open(ostamp).read().strip() == want:
            continue                                       # this object is current: only changed sources are recompiled
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas"); cmd.insert(2, "-v")
        procs.append((s, ostamp, want, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, ostamp, want, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode:
            sys.stderr.write(out)
        if pr.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
        with open(ostamp, "w") as f:
            f.write(want)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT, *objs, "-lcudart"])
    with open(STAMP, "w") as f:
        f.write(_source_hash())
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
