"""Build libunimatch_sm100.so in-tree with nvcc for sm_100a (no JIT cache, the .so travels with the repo).

    python unimatch_b200/csrc/build.py [--force] [-v]     (or: from unimatch_b200.csrc.build import build; build())

Run the file by path: `python -m unimatch_b200.csrc.build` imports the package first, which loads the library that is
about to be replaced.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(os.path.dirname(HERE), "libunimatch_sm100.so")
SOURCES = ["um_api.cu", "um_attention_simt.cu", "um_attention_tc.cu", "um_attention_tc2.cu", "um_conv_tc.cu", "um_ffn_tc.cu", "um_local.cu", "um_local_tc.cu", "um_local_stencil.cu", "um_misc.cu", "um_norm.cu", "um_stem.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-I", os.path.join(ROOT, "include"), "-I", HERE]


def _nvcc():
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: libunimatch_sm100.so cannot be built")


def have_nvcc():
    try:
        _nvcc()
        return True
    except RuntimeError:
        return False


if os.environ.get("UM_ATTN_DEBUG_BUILD") == "1":      # diagnostics of the attention kernel (timeline, dump, timing experiments)
    FLAGS = FLAGS + ["-DUM_ATTN_DEBUG=1"]


def _stamp():
    h = hashlib.sha256()
    h.update(" ".join(FLAGS).replace(ROOT, "").encode())       # a moved checkout keeps its library
    for f in sorted(os.listdir(HERE)) + [os.path.join(ROOT, "include", "unimatch_sm100.h")]:
        p = f if os.path.isabs(f) else os.path.join(HERE, f)
        if p.endswith((".cu", ".cuh", ".h", "build.py")):
            h.update(open(p, "rb").read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Idempotent and safe under concurrent callers (torchrun ranks importing the package at the same time): the stamp
    check and the build run under an exclusive file lock, objects are compiled into a per-process directory and the
    finished library / stamp are moved into place atomically, so no process ever maps a half-written .so."""
    import fcntl
    import tempfile
    stamp_file = LIB + ".stamp"
    stamp = _stamp()

    def fresh():
        return os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp

    if not force and fresh():
        return LIB
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    with open(os.path.join(bdir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and fresh():              # another process built it while we waited for the lock
                return LIB
            nvcc = _nvcc()
            work = tempfile.mkdtemp(prefix="obj.%d." % os.getpid(), dir=bdir)
            try:
                objs, procs = [], []
                for src in SOURCES:
                    obj = os.path.join(work, src.replace(".cu", ".o"))
                    cmd = [nvcc] + FLAGS + ["-c", os.path.join(HERE, src), "-o", obj]
                    if verbose:
                        cmd.insert(1, "-Xptxas=-v")
                    procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
                    objs.append(obj)
                for src, p in procs:
                    out, _ = p.communicate()
                    if verbose or p.returncode:
                        sys.stderr.write(out)
                    if p.returncode:
                        raise RuntimeError("nvcc failed on %s" % src)
                tmp_lib = os.path.join(work, "libunimatch_sm100.so")
                r = subprocess.run([nvcc, "-shared", "-o", tmp_lib] + objs + ["-lcudart", "-lcuda"],
                                   stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                if r.returncode:
                    sys.stderr.write(r.stdout)
                    raise RuntimeError("link failed")
                tmp_stamp = os.path.join(work, "stamp")
                open(tmp_stamp, "w").write(stamp)
                os.replace(tmp_lib, LIB)
                os.replace(tmp_stamp, stamp_file)
            finally:
                shutil.rmtree(work, ignore_errors=True)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
