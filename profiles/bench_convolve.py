"""b2_convolve1d throughput on the tutorial-sized block: float32 (256, 1024, 1024) per GPU along axis -1 (time last,
the layout of tutorials/reflectivity.py) and along axis 0, nh in {5, 11, 21, 41, 81}, plus float64 at nh = 41.
1 GiB in + 1 GiB out (float32): far above the 126 MB L2, so every pass streams from HBM.

Same-run references: torch ``copy_`` of the same byte count (the HBM rate) and cuDNN through
torch.nn.functional.conv1d (axis -1) / conv2d with an (nh, 1) filter (axis 0) on the same data (the library
baseline).  Each output is checked against a float64 direct sum over a slice before timing.

    python profiles/bench_convolve.py [--iters 50] [--out profiles/r03_bench_convolve.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pylops_mpi_b200 as pm  # noqa: E402

DIMS = (256, 1024, 1024)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, plim, clk = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def reference_slice(x, h, offset, axis):
    """float64 direct sum y[i] = sum_k h[k] x[i + offset - k] over the first two outer slices (axis -1) / the
    first 4096 columns (axis 0)"""
    xs = (x[:2] if axis == -1 else x[:, :4, :1024]).double()
    xs = xs.movedim(axis, -1)
    n = xs.shape[-1]
    y = torch.zeros_like(xs)
    for k, hk in enumerate(h.tolist()):
        s = offset - k                      # y[i] += h[k] x[i + s]
        if s >= 0:
            y[..., :n - s] += hk * xs[..., s:]
        else:
            y[..., -s:] += hk * xs[..., :n + s]
    return y.movedim(-1, axis)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "r03_bench_convolve.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = card()
    g = torch.Generator(device="cuda").manual_seed(0)
    rows = []
    cases = [(torch.float32, ax, nh) for ax in (-1, 0) for nh in (5, 11, 21, 41, 81)]
    cases += [(torch.float64, ax, 41) for ax in (-1, 0)]
    bufs = {}
    for dt, axis, nh in cases:
        if dt not in bufs:
            bufs.clear()
            torch.cuda.empty_cache()
            bufs[dt] = (torch.randn(DIMS, generator=g, device="cuda", dtype=dt), torch.empty(DIMS, device="cuda", dtype=dt))
        x, y = bufs[dt]
        n = x.numel()
        esz = x.element_size()
        h = np.random.default_rng(nh).standard_normal(nh)
        offset = nh // 2
        C = pm.local.Convolve1D(DIMS, h, offset=offset, axis=axis, dtype=dt)
        xf = x.reshape(-1)
        yf = y.reshape(-1)
        C.matvec(xf, out=yf)
        ref = reference_slice(x, h, offset, axis)
        got = (y[:2] if axis == -1 else y[:, :4, :1024]).double()
        err = float(torch.linalg.vector_norm(got - ref) / torch.linalg.vector_norm(ref))
        assert err < (1e-5 if dt == torch.float32 else 1e-13), (dt, axis, nh, err)

        # library baseline: cuDNN cross-correlation with the flipped filter and symmetric padding (odd nh, centred)
        w = torch.as_tensor(h[::-1].copy(), device="cuda", dtype=dt)
        if axis == -1:
            xin, wt = x.view(-1, 1, DIMS[-1]), w.view(1, 1, nh)
            lib = lambda: F.conv1d(xin, wt, padding=nh // 2)                         # noqa: E731
        else:
            xin, wt = x.view(1, 1, DIMS[0], -1), w.view(1, 1, nh, 1)
            lib = lambda: F.conv2d(xin, wt, padding=(nh // 2, 0))                    # noqa: E731
        yl = lib()
        lerr = float(torch.linalg.vector_norm(yl.reshape(DIMS).double() - y.double()) / torch.linalg.vector_norm(y.double()))
        del yl
        t_conv = timed(lambda: C.matvec(xf, out=yf), args.iters)
        t_copy = timed(lambda: y.copy_(x), args.iters)
        t_lib = timed(lib, args.iters)
        gbs = 2 * n * esz / t_conv / 1e9
        row = {"dtype": str(dt).split(".")[-1], "axis": axis, "nh": nh, "elements": n, "kernel_ms": t_conv * 1e3,
               "kernel_GBps": gbs, "kernel_TFMAps": n * nh / t_conv / 1e12, "copy_ms": t_copy * 1e3,
               "copy_GBps": 2 * n * esz / t_copy / 1e9, "share_of_copy": t_copy / t_conv,
               "torch_conv_ms": t_lib * 1e3, "speedup_vs_torch_conv": t_lib / t_conv, "rel_err_vs_fp64": err,
               "torch_conv_rel_diff": lerr}
        rows.append(row)
        print(json.dumps(row), flush=True)
    out = {"card": info, "dims": DIMS, "iters": args.iters, "timing": "CUDA events, 3 warm-up launches",
           "bytes": "2 * elements * sizeof(T) per apply (algorithmic)", "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
