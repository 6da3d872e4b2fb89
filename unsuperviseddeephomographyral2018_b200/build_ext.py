"""Build libudh.so in-tree with nvcc for sm_100a (no torch in the link line: the library is a plain C ABI).

Concurrency: several ranks (torchrun) may import the package at once on a fresh clone.  The build runs under an exclusive
fcntl lock on `build/.lock`, compiles into `build/`, links to a temporary name and publishes the library with an atomic
rename — a concurrent importer either waits for the lock and then finds the library up to date, or loads the previous
complete file; it never sees a half-written one.
"""
import fcntl
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")

LIB = os.path.join(HERE, "libudh.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + [os.path.join(HERE, "..", "include", "udh.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    with open(os.path.join(bdir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():         # another process built it while we waited for the lock
                return LIB
            nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
            objs, procs = [], []
            for src in sources():
                obj = os.path.join(bdir, os.path.basename(src)[:-3] + ".o")
                objs.append(obj)
                cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
                procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
            ok = True
            for src, p in procs:
                out, _ = p.communicate()
                if p.returncode != 0 or verbose:
                    sys.stderr.write("== %s\n%s\n" % (os.path.basename(src), out))
                ok = ok and p.returncode == 0
            if not ok:
                raise RuntimeError("nvcc failed building %s" % os.path.basename(LIB))
            tmp = "%s.tmp.%d" % (LIB, os.getpid())
            subprocess.check_call([nvcc, "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
            os.replace(tmp, LIB)                        # atomic publish
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


PROBE_LIB = os.path.join(HERE, "libudh_probe.so")


def build_probes(force=False):
    """Hardware probes (csrc/probes/: TMA / tcgen05 descriptor conventions, CTA-pair MMAs, MMA issue rates) live in their OWN
    library, libudh_probe.so, declared in include/udh_probe.h — the product library carries no debug kernels.  Links against
    libudh.so for the shared error / launch-count helpers."""
    lib = build()
    srcs = sorted(glob.glob(os.path.join(CSRC, "probes", "*.cu")))
    if not force and os.path.exists(PROBE_LIB) and all(os.path.getmtime(s) < os.path.getmtime(PROBE_LIB) for s in srcs) \
            and os.path.getmtime(lib) < os.path.getmtime(PROBE_LIB):
        return PROBE_LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tmp = "%s.tmp.%d" % (PROBE_LIB, os.getpid())
    subprocess.check_call([nvcc] + NVCC_FLAGS + ["-shared", "-o", tmp] + srcs + ["-L" + HERE, "-l:libudh.so", "-Xlinker", "-rpath=$ORIGIN"])
    os.replace(tmp, PROBE_LIB)
    return PROBE_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
