"""In-tree build of libparasail_b200.so: hand-written CUDA for sm_100a + the C-ABI host side."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libparasail_b200.so")
SOURCES = ["scan.cu", "pairs.cu", "pairs16.cu", "wave32.cu", "db.cu", "host_scan.cu", "ctx.cu", "db_io.cu", "matrix.cpp", "fn_name.cpp",
           "result.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "parasail_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, defines=(), out=None):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> parasail_rs_b200/libparasail_b200.so
    (`defines`/`out` build tuning variants next to it, e.g. defines=["SW16_UNROLL=1"])"""
    out = out or OUT
    if out == OUT and not force and not _stale():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    # one object per source, compiled side by side (the kernel translation units dominate), then one link
    objdir = os.path.join(HERE, "build", os.path.splitext(os.path.basename(out))[0])
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + [f"-D{d}" for d in defines] + ["-c", "-o", obj, os.path.join(CSRC, src)]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    for src, obj, r in results:
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"nvcc failed compiling {src}")
        if verbose:
            sys.stderr.write(r.stderr)
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + [o for _, o, _ in results],
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libparasail_b200.so")
    return out


def build_tools():
    """the DPX issue-rate microbenchmark (tools/dpx_bench)"""
    root = os.path.dirname(HERE)
    src, out = os.path.join(root, "tools", "dpx_bench.cu"), os.path.join(root, "tools", "dpx_bench")
    if os.path.exists(out) and os.path.getmtime(out) > os.path.getmtime(src):
        return out
    nvcc = os.environ.get("NVCC", "nvcc")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-o", out, src], check=True)
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_tools())
