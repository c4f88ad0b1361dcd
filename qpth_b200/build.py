"""Build libqpth_b200.so in-tree with nvcc for sm_100a (`python -m qpth_b200.build`)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
import glob  # noqa: E402

DEPS = sorted(glob.glob(os.path.join(HERE, "csrc", "*"))) + [os.path.join(os.path.dirname(HERE), "include", "qpth_b200.h")]
OUT = os.path.join(HERE, "libqpth_b200.so")


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def up_to_date():
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(d) <= t for d in DEPS)


# (source, extra defines, object suffix): the 256-thread build of every kernel + the 192- and 512-thread builds of the
# product-form solve kernels (three QPs per SM; large orders)
UNITS = [("qp_kernels.cu", [], "main"),
         ("qp_alt.cu", ["-DQPB_NT=192", "-DQPB_ALT_CTAS=3"], "alt192"),
         ("qp_alt.cu", ["-DQPB_NT=512", "-DQPB_ALT_CTAS=1"], "alt512")]


def build(force=False, verbose=False, extra=(), out=None):
    """Compile the three translation units in parallel and link them into one shared library."""
    out = out or OUT
    if not force and out == OUT and up_to_date():
        return out
    import tempfile
    base = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
            "-Xcompiler", "-fPIC"] + list(extra)
    if verbose:
        base.insert(1, "-Xptxas=-v")
    # objects go to a private temporary directory: a fixed name under /tmp may belong to another user of the machine
    with tempfile.TemporaryDirectory(prefix="qpth_b200_obj_") as objdir:
        procs, objs = [], []
        for src, defs, tag in UNITS:
            obj = os.path.join(objdir, tag + ".o")
            cmd = base + defs + ["-c", "-o", obj, os.path.join(HERE, "csrc", src)]
            if verbose:
                print(" ".join(cmd))
            procs.append((cmd, subprocess.Popen(cmd)))
            objs.append(obj)
        for cmd, rc in [(cmd, pr.wait()) for cmd, pr in procs]:      # every compiler exits before the directory goes
            if rc != 0:
                raise subprocess.CalledProcessError(rc, cmd)
        subprocess.check_call([nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + objs)
    return out


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print("built", OUT)
