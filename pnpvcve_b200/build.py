"""In-tree build of libpnpvcve.so (sm_100a only) with nvcc; no torch headers involved."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpnpvcve.so")
SOURCES = ["pnp_api.cu", "pnp_conv_rows.cu", "pnp_ops.cu", "pnp_raster.cu", "pnp_metrics.cu", "pnp_png.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v"]


def _newest_source_mtime():
    m = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(force=False, verbose=False, lib=LIB):
    """Compile `lib` (default: the in-tree library) when it is missing or older than its sources.  Returns its path."""
    if not force and os.path.isfile(lib) and os.path.getmtime(lib) >= _newest_source_mtime():
        return lib
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = list(NVCC_FLAGS)
    if os.environ.get("PNP_DIAG", "0") != "0":     # diagnostics build for tools/ (what-if bits, clock traces)
        flags.append("-DPNP_DIAG")
    if os.environ.get("PNP_WARP_BLOCKS"):          # tile-width sweep of the warp kernel (tools/warp_bench.py)
        flags.append("-DPNP_WARP_BLOCKS=" + os.environ["PNP_WARP_BLOCKS"])
    if os.environ.get("PNP_STEP_RING_LOG2"):       # 3 = the 8-barrier step ring that could dead-lock (validation only)
        flags.append("-DPNP_STEP_RING_LOG2=" + os.environ["PNP_STEP_RING_LOG2"])
    if os.environ.get("PNP_SPIN_LIMIT"):           # stress runs: trap a stuck pipeline after fewer polls
        flags.append("-DPNP_SPIN_LIMIT=" + os.environ["PNP_SPIN_LIMIT"])
    cmd = [nvcc] + flags + ["-o", lib] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed building {lib}")
    return lib


if __name__ == "__main__":
    print(build(force=True, verbose=True))
