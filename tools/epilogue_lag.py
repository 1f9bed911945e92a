"""How far does the epilogue of the row-stacked conv trail its MMA issuer, with and without debug bit 2048 (the ~2 us
per-row epilogue delay of tests/test_gpu_kernels.py::test_conv_720p_survives_a_slow_epilogue)?  Builds a PNP_DIAG copy
of the library in a temporary directory and launches one 720p conv per (variant, delay) in a process of its own (the
library reads its debug knobs once).  From the clock64 stamps of CTA 0 (pnp_conv_rows.cu, PNP_TRACING) it prints, per
output row, the lag: the last step the issuer had begun when the epilogue took the row, minus the step that completes
the row.  Step s accumulates into output rows s-1, s and s+1, so at lag L the rows from the one the epilogue takes to
the newest hold L + 3 accumulators; the ring has 8 (plain conv) or 5 (with the partition 1x1 convs, par), so L = 5 and
L = 2 mean a full ring: the issuer is held back by the epilogue alone.

   python tools/epilogue_lag.py"""
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(kind):
    import torch
    dev = torch.device("cuda:0")
    trace = torch.zeros(4096, dtype=torch.int64, device=dev)
    os.environ["PNP_TRACE_PTR"] = str(trace.data_ptr())
    from pnpvcve_b200 import ops
    h, w = 720, 1280
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn((1, h, w, 64), generator=g, device=dev).to(torch.bfloat16)
    out = ops.new_feature(1, h, w, dev)
    war = ops.new_wpack_rowstack(dev, with_par=True)
    ops.pack_conv3x3_rowstack(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05, war)
    for j in range(3):
        ops.pack_rows(torch.randn((64, 64), generator=g, device=dev) * 0.1, war[9 * ops.CHUNK_BYTES:], 64 * j)
    par = (torch.rand((1, 3, h, w), generator=g, device=dev) > 0.6).float() / 255.0
    bias = torch.randn(64, generator=g, device=dev) * 0.1

    def launch():
        if kind == "par":
            ops.conv3x3(x, war, out=out, bias=bias, par=par, act=ops.PNP_ACT_RELU)
        else:
            ops.conv3x3(x, war, out=out, bias=bias)

    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    trace.zero_()
    launch()
    torch.cuda.synchronize()
    t = trace.cpu().tolist()
    starts = [t[s * 8] for s in range(64) if t[s * 8]]          # issuer: start of step s
    # epilogue: the moment it holds row `ord` (behind the delay and the step_done wait); CTA 0 owns one segment from
    # the top row, so row `ord` completes with step ord + 1
    took = [t[2816 + o * 4 + 1] for o in range(64)] if kind == "par" else [t[o * 8 + 3] for o in range(64)]
    lags = []
    for o, e in enumerate(took):
        if not e or o + 1 >= len(starts) - 1:                     # (the last row of the segment completes with it)
            break
        lags.append(sum(1 for s in starts if s <= e) - 1 - (o + 1))
    print(" ".join(str(v) for v in lags))


def main():
    if len(sys.argv) > 2 and sys.argv[1] == "--child":
        return child(sys.argv[2])
    from pnpvcve_b200 import build
    with tempfile.TemporaryDirectory() as tmp:
        lib = os.path.join(tmp, "libpnpvcve_diag.so")
        os.environ["PNP_DIAG"] = "1"
        build.build(force=True, lib=lib)
        for kind, ring in (("plain", 8), ("par", 5)):
            for bits in ("0", "2048"):
                env = dict(os.environ, PNP_LIB_PATH=lib, PNP_DEBUG_SKIP=bits)
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", kind], cwd=ROOT, env=env,
                                     capture_output=True, text=True, check=True)
                lags = [int(v) for v in res.stdout.split()]
                print(f"{kind:5s} (ring {ring} rows) debug bits {bits:>4s}: rows {len(lags)}, lag in steps max {max(lags)} "
                      f"median {sorted(lags)[len(lags) // 2]}; per row: {' '.join(map(str, lags))}")


if __name__ == "__main__":
    main()
