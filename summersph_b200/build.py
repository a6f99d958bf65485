"""In-tree build of the CUDA engine: nvcc -> summersph_b200/libsph_b200.so (sm_100a only)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libsph_b200.so")
SOURCES = ["sph_engine.cu"]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inl")))      # every header sph_engine.cu may include
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(HERE, "..", "include", "sph_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def nvcc_command(out, extra=()):
    """The nvcc command line that builds the engine into `out`; `extra`: more flags, e.g. ["-DSCREEN_AUDIT"] for a variant."""
    cmd = [nvcc_path()] + NVCC_FLAGS + list(extra) + ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    if os.path.exists("/usr/bin/g++"):
        cmd[1:1] = ["-ccbin", "/usr/bin/g++"]
    return cmd


def build_extension(force=False, verbose=False):
    """Compile the engine for sm_100a. Returns the path of the shared library."""
    if not force and not needs_build():
        return SO
    cmd = nvcc_command(SO)
    env = dict(os.environ)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    log = res.stdout + res.stderr
    with open(os.path.join(HERE, "csrc", "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed")
    if verbose:
        print(log)
    return SO


if __name__ == "__main__":
    print(build_extension(force=True, verbose="-v" in sys.argv))
