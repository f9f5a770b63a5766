"""Builds libpermutect_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m permutect_b200.csrc.build [--force]
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["pmt_call.cu", "pmt_forward.cu", "pmt_backward.cu", "pmt_loader.cu", "pmt_tc.cu", "pmt_tc_bwd.cu", "pmt_cnn_tc.cu", "pmt_cnn_bwd.cu", "pmt_head_bwd.cu", "pmt_loss.cu", "pmt_optim.cu", "pmt_posterior.cu", "pmt_context_fit.cu"]
HEADERS = ["pmt_device.cuh", "pmt_tile.cuh", "pmt_cnn.cuh", "pmt_host.h", "pmt_tc_ptx.cuh", "pmt_tc.cuh", "pmt_cnn_tc.cuh", "pmt_call.h", os.path.join("..", "..", "include", "permutect_b200.h")]
OUTPUT = os.path.join(HERE, "libpermutect_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _fingerprint() -> str:
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for name in SOURCES + HEADERS:
        with open(os.path.join(HERE, name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compiles every translation unit for sm_100a (in parallel, objects under csrc/build/) and links the shared library."""
    from concurrent.futures import ThreadPoolExecutor
    stamp = OUTPUT + ".stamp"
    fp = _fingerprint()
    if not force and os.path.exists(OUTPUT) and os.path.exists(stamp) and open(stamp).read() == fp:
        return OUTPUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + compile_flags + ["-c", "-o", obj, os.path.join(HERE, src)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, " ".join(cmd), res

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    log = ""
    for src, obj, cmd, res in results:
        log += cmd + "\n" + res.stdout + res.stderr
    failed = [src for src, _, _, res in results if res.returncode != 0]
    if not failed:
        link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", OUTPUT] + [r[1] for r in results]
        res = subprocess.run(link, capture_output=True, text=True)
        log += " ".join(link) + "\n" + res.stdout + res.stderr
        if res.returncode != 0:
            failed = ["link"]
    with open(os.path.join(HERE, "build.log"), "w") as f:
        f.write(log)
    if failed:
        raise RuntimeError(f"nvcc failed ({', '.join(failed)}):\n" + log[-4000:])
    if verbose:
        print(log)
    with open(stamp, "w") as f:
        f.write(fp)
    return OUTPUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
