#!/usr/bin/env python
"""Benchmark of the pylops-mpi hot path on B200 (contract: see the task brief).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--no-extras] [--dump-outputs DIR]

Headline (BASELINE.json metric "... GB/s (FirstDerivative)"): one *step* is one
``MPIFirstDerivative.matvec`` (centered, order 3, float32) over the (65536, 8192)
float32 array of SURVEY 8(d) / BASELINE.md 1b, row-block partitioned over the N
GPUs (STRONG scaling: 2 GiB in + 2 GiB out in total; per-GPU blocks >= 256 MiB,
above the 126 MB L2), inputs resident in HBM.  ``value`` = algorithmic bytes
(2 * 4 B per element) / time.  ``e2e`` = the same operator through the
host-buffer plugin entry (``b2_first_derivative_host``: pinned host arrays in
and out, H2D + kernel + D2H inside the timed region).  Before any timing every
rank runs the parity set of tests/parity_checks.py against the oracle at THIS
world size (``parity`` in the line; a failure aborts the timing).
``secondary`` = the MatrixMult half of BASELINE's metric (GF/s on the 32768^2
bf16 config, with its own roofline and a 256-sampled-rows parity check) and the
weak-scaling curve of the stencil; ``extra`` = the other BASELINE configs.

``--dump-outputs DIR`` writes, after the timed steps, a fixed seeded sample of what the last timed step returned
(whole rows of the (65536, 8192) result, float32) and their row indices (float64) as DIR/*.npy.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.

``--impl reference`` times the reference's CPU algorithm for the same operator
on the same global workload (the NumPy restatement in oracle/, one OS process
per host core, each applying the per-rank stencil code to its own row block).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

# rank 0 must print exactly ONE JSON line on stdout: keep NCCL's banner / debug text off it
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

GLOBAL_ROWS = 65536            # SURVEY 8(d) C1-throughput / BASELINE.md 1b: dims (65536, 8192) float32, split over G
NCOLS = 8192
METRIC = "MPIFirstDerivative matvec GB/s (algorithmic bytes, centered-3 float32)"
METRIC2 = "MPIMatrixMult matvec GF/s (bf16 -> fp32, 32768 x 32768, M = 4096)"
HBM_FALLBACK = 6650.0
DUMP_ROWS = 1024               # rows of the headline output written by --dump-outputs: 1024 x 8192 float32 = 32 MiB


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": HBM_FALLBACK, "bf16_tflops": 1590.0}, "fallback"


# --------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------
# CPU reference arm (oracle port, one process per core)
# --------------------------------------------------------------------------
def _cpu_rank_main(conn, rows, ncols, seed):
    """one simulated CPU rank: owns its row block (created ONCE, outside the timed passes) and applies the
    reference's per-rank stencil code to it every time the parent says go"""
    import pylops_mpi_oracle as o
    x = np.random.default_rng(seed).standard_normal((rows, ncols), dtype=np.float32)
    flat = [x.ravel()]
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg is None:
            break
        t0 = time.perf_counter()
        y = o.first_derivative(flat, (rows, ncols), 1.0, "centered", False, 3, False, dtype=np.float32)
        conn.send((time.perf_counter() - t0, float(y[0][ncols + 1])))


class CpuRanks:
    """`cores` OS processes, each a simulated rank of the reference's NumPy path"""

    def __init__(self, cores: int, rows_per_proc: int, ncols: int):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.cores = cores
        self.conns, self.procs = [], []
        for i in range(cores):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_rank_main, args=(b, rows_per_proc, ncols, 42 + i), daemon=True)
            p.start()
            self.conns.append(a)
            self.procs.append(p)
        for c in self.conns:
            c.recv()

    def step(self) -> float:
        """one pass: every rank applies the stencil to its block concurrently; wall-clock seconds"""
        t0 = time.perf_counter()
        for c in self.conns:
            c.send("go")
        for c in self.conns:
            c.recv()
        return time.perf_counter() - t0

    def close(self):
        for c in self.conns:
            c.send(None)
        for p in self.procs:
            p.join(timeout=10)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


def cpu_split():
    """the CPU arm runs the WHOLE (65536, 8192) workload: one process per host core, rows split evenly"""
    cores = min(os.cpu_count() or 1, 64)
    while GLOBAL_ROWS % cores:
        cores -= 1
    return cores, GLOBAL_ROWS // cores


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores, rows_per_proc = cpu_split()
    with CpuRanks(cores, rows_per_proc, NCOLS) as pool:
        for _ in range(max(1, args.warmup // 2)):
            pool.step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.step()
        dt = time.perf_counter() - t0
    nbytes = 2 * 4 * GLOBAL_ROWS * NCOLS * args.steps
    val = nbytes / dt / 1e9
    sample = (f"the full ({GLOBAL_ROWS} x {NCOLS}) float32 workload per step: {cores} processes x ({rows_per_proc} x {NCOLS}) rows "
              "(oracle restatement of FirstDerivative.py:201-219 per rank; the same global workload for every --gpus N)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(n):
    return {"workload": "MPIFirstDerivative matvec, kind=centered order=3 edge=False sampling=1, float32, "
                        f"dims=({GLOBAL_ROWS}, {NCOLS}) global, row-block partition over N={n} GPUs (strong scaling; "
                        "SURVEY 8d C1 / BASELINE.md 1b)",
            "global_rows": GLOBAL_ROWS, "ncols": NCOLS, "rows_per_gpu": GLOBAL_ROWS // n,
            "l2": f"per-GPU input {GLOBAL_ROWS // n * NCOLS * 4 >> 20} MiB + output of the same size > 126 MB L2 (no flush needed)",
            "parallelism": f"rows{n}"}


# --------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------
def time_loop(fn, steps, warmup, comm=None):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if comm is not None:
        comm.Barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_cpu = time.perf_counter()
    for _ in range(steps):
        fn()
    time_loop.last_enqueue_ms = (time.perf_counter() - t_cpu) * 1e3 / max(steps, 1)
    e1.record()
    torch.cuda.synchronize()
    if comm is not None:
        comm.Barrier()
    ms = e0.elapsed_time(e1)
    if comm is not None and comm.Get_size() > 1:
        ms = comm.allreduce(ms, "max")
    return ms


def dump_outputs(out_dir, y, comm, nloc):
    """write DUMP_ROWS rows of the headline output ``y`` (global shape (GLOBAL_ROWS, NCOLS)): the first and last row
    of every rank's block, where the halo exchange acts, and the rest drawn with a fixed seed"""
    import torch
    rank, size = comm.Get_rank(), comm.Get_size()
    edges = {r * nloc for r in range(size)} | {(r + 1) * nloc - 1 for r in range(size)}
    pool = np.setdiff1d(np.arange(GLOBAL_ROWS), sorted(edges))
    rows = np.union1d(sorted(edges), np.random.default_rng(0).choice(pool, DUMP_ROWS - len(edges), replace=False))
    mine = rows[(rows >= rank * nloc) & (rows < (rank + 1) * nloc)]
    yl = y.local_array.reshape(nloc, NCOLS)
    local = yl[torch.as_tensor(mine - rank * nloc, device=yl.device)].cpu().numpy()
    parts = comm.allgather(local)
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "first_derivative_y_rows.npy"), np.concatenate(parts).astype(np.float32))
        np.save(os.path.join(out_dir, "first_derivative_y_row_index.npy"), rows.astype(np.float64))


def numa_bind_to_gpu(dev: int):
    """pin this process (and, by first touch, its pinned host buffers) to the NUMA node the GPU hangs off:
    with 8 ranks the e2e host<->device pipelines otherwise cross the inter-socket link for half of the GPUs"""
    try:
        import torch
        prop = torch.cuda.get_device_properties(dev)
        bus = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return {"numa_node": None, "pci": bus}
        cpus = set()
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus_bound": len(cpus), "pci": bus}
    except Exception as exc:
        return {"numa_node": None, "error": repr(exc)[:120]}


def run_gpu_arm(args):
    import torch
    import pylops_mpi_b200 as pm
    from pylops_mpi_b200 import _lib as L

    comm = pm.get_comm_world()
    rank, size = comm.Get_rank(), comm.Get_size()
    numa = numa_bind_to_gpu(torch.cuda.current_device())
    if size != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but world size {size}", file=sys.stderr)
    peaks, peak_kind = load_peaks()
    dev = torch.cuda.current_device()
    if GLOBAL_ROWS % size:
        raise SystemExit(f"world size {size} does not divide {GLOBAL_ROWS} rows")
    N = GLOBAL_ROWS
    dims = (N, NCOLS)
    nloc = N // size
    elem_loc = nloc * NCOLS
    bytes_loc = 2 * 4 * elem_loc

    # ---- parity preamble: the multi-rank paths against the oracle at THIS world size, before any timing ----------
    parity = None
    if not args.no_check:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import parity_checks
        parity = parity_checks.run_all(pm, comm, full_size=True)
        torch.cuda.synchronize()
        # a failed check on the HEADLINE path (the stencil and its halo exchange) aborts the run: no timing of a wrong
        # result.  A failure elsewhere is reported in the line (parity.failed > 0, parity.failures) and the sections that
        # depend on the failed component are skipped instead of timed.
        failed_names = [n for n, dtl in parity["details"].items() if any(n in f for f in parity["failures"])]
        parity["failed_checks"] = failed_names
        critical = [n for n in failed_names if "Derivative" in n]
        if parity["failed"] and (critical or not failed_names):
            if rank == 0:      # no timing of a wrong result: report and stop
                print(json.dumps({"metric": METRIC, "value": 0.0, "unit": "GB/s", "n_gpus": size, "steps": 0,
                                  "warmup": 0, "ms_per_step": None, "higher_is_better": True, "scaling": "strong",
                                  "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                                  "config": workload_config(size), "parity": parity,
                                  "error": "parity check failed: timing aborted"}))
            sys.exit(1)

    # a CUDA-graph capture that died half-way (seen once at 8 ranks) leaves torch's generator flagged as capturing and
    # every later RNG call raises: probe, and clear the flag with one empty capture if needed
    try:
        torch.empty(4, device="cuda").normal_()
        rng_note = None
    except RuntimeError as exc:
        from pylops_mpi_b200.optimization.cls_basic import _reset_capture_state
        _reset_capture_state()
        rng_note = f"torch CUDA generator was stuck in capture mode ({repr(exc)[:80]}): reset"
        torch.empty(4, device="cuda").normal_()

    # ---- inputs resident in HBM --------------------------------------------------
    g = torch.Generator(device="cuda").manual_seed(42 + rank)
    x = pm.DistributedArray(global_shape=N * NCOLS, dtype=np.float32)
    assert x.local_shape == (elem_loc,)
    x.local_array.normal_(generator=g)
    Fop = pm.MPIFirstDerivative(dims, kind="centered", order=3, dtype=np.float32)
    holder = {}

    def step():
        holder["y"] = Fop.matvec(x)

    sampler = ClockSampler(dev)
    sampler.start()                      # samples cover warm-up, the timed region and the kernel-only loop
    for _ in range(args.warmup):
        step()
    ms = time_loop(step, args.steps, 0, comm)
    enqueue_ms = time_loop.last_enqueue_ms     # host time to enqueue one step (GPU-bound if << ms_per_step)
    value = bytes_loc * size * args.steps / (ms * 1e-3) / 1e9
    fused_halo = size > 1 and comm.halo is not None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, holder["y"], comm, nloc)

    # ---- roofline of the dominant kernel: live CUDA-event timing of the kernel alone --------
    xl = x.local_array
    yl = torch.empty_like(xl)
    st = L.stream()

    def kern():
        L.check(L.lib.b2_first_derivative(L.ctx(), xl.data_ptr(), yl.data_ptr(), None, 0, None, 0, nloc, NCOLS,
                                          0, nloc, L.FD_CENTERED, 3, 0, 1.0, 0, L.F32, st))
    kms = time_loop(kern, args.steps, max(3, args.warmup), None) / args.steps
    achieved = bytes_loc / (kms * 1e-3) / 1e9
    # the timed region is only a few ms: keep the same kernel running ~0.7 s so that the 100 ms
    # nvidia-smi sampler sees clocks / throttle reasons under this exact load
    t_load = time.perf_counter()
    while True:
        for _ in range(20):
            kern()
        torch.cuda.synchronize()
        waited = time.perf_counter() - t_load
        # at least 0.7 s; on an 8-GPU box nvidia-smi needs seconds to deliver its first sample: keep the load up
        # until a few samples exist (bounded at 8 s)
        if waited >= 0.7 and (len(sampler.lines) >= 5 or waited > 8.0):
            break
    clocks = sampler.stop()
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
            per_elem = tj.get("stencil_vec_kernel_f32_centered3_bytes_per_element")
            traffic = per_elem * elem_loc if per_elem else None
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "stencil_vec_kernel<float, taps{-1,+1}>", "achieved": achieved,
                "peak": peaks["hbm_gbs"], "peak_kind": f"{peak_kind} copy bandwidth (burst)", "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                "algorithmic_bytes_per_launch": bytes_loc, "us_per_launch": kms * 1e3,
                "note": "algorithmic = 8 B per float32 element (read x once, write y once) x the rows one launch owns"}

    # ---- e2e: host buffers through the plugin entry (H2D + kernel + D2H in the timed region) --
    # each rank owns rows [rank*nloc, (rank+1)*nloc) of the replicated host array; only its block
    # (+2 halo rows each side) is materialised, addressed through a virtual global base pointer
    lo = 2 if rank > 0 else 0
    hi = 2 if rank < size - 1 else 0
    xh = torch.empty((nloc + lo + hi, NCOLS), dtype=torch.float32).pin_memory()
    xh.normal_()
    yh = torch.empty((nloc, NCOLS), dtype=torch.float32).pin_memory()
    row_bytes = NCOLS * 4
    x_base = xh.data_ptr() - (rank * nloc - lo) * row_bytes
    y_base = yh.data_ptr() - (rank * nloc) * row_bytes

    def e2e_step():
        L.check(L.lib.b2_first_derivative_host(L.ctx(), x_base, y_base, N, NCOLS, rank * nloc, (rank + 1) * nloc,
                                               L.FD_CENTERED, 3, 0, 1.0, 0, L.F32), "b2_first_derivative_host")
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    comm.Barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if size > 1:
        e2e_s = comm.allreduce(e2e_s, "max")
    e2e_val = bytes_loc * size * e2e_steps / e2e_s / 1e9
    # the host-buffer result must equal the device-resident path on the same rows (same kernel, same data)
    nchk = 64
    xd = xh[:lo + nchk + 2].cuda()
    yd = torch.empty(nchk, NCOLS, device="cuda")
    L.check(L.lib.b2_first_derivative(L.ctx(), xd[lo:].data_ptr(), yd.data_ptr(), xd.data_ptr() if lo else None, lo,
                                      xd[lo + nchk:].data_ptr(), 2, nchk, NCOLS, rank * nloc, N, L.FD_CENTERED, 3, 0, 1.0,
                                      0, L.F32, L.stream()), "e2e check")
    e2e_diff = float((yd.cpu() - yh[:nchk]).abs().max())
    e2e = {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": (nloc + lo + hi) * row_bytes * size,
           "d2h_bytes_per_step": nloc * row_bytes * size, "steps": e2e_steps,
           "per_gpu_pcie_GB/s_each_way": nloc * row_bytes * e2e_steps / e2e_s / 1e9,
           "api": "b2_first_derivative_host (pinned host in/out, 3-stream chunk pipeline)",
           "numa": numa, "limiter": "PCIe (H2D + D2H of every byte; the kernel itself runs at the HBM roofline)",
           "check_vs_device_path": {"rows": nchk, "max_abs_diff": e2e_diff, "equal": e2e_diff == 0.0}}
    del xh, yh, xd, yd

    secondary, extra = {}, {}
    if not args.no_extras:
        bad = (parity or {}).get("failed_checks", [])
        if any("MatrixMult" in n for n in bad):
            secondary = {"skipped": "a MPIMatrixMult parity check failed at this world size: not timed", "failed_checks": bad}
        else:
            try:
                secondary = run_secondary(pm, L, comm, peaks, args)
            except Exception as exc:
                secondary = {"error": repr(exc)}
        if bad and not any("MatrixMult" in n for n in bad):
            extra = {"skipped": "a parity check of a component timed here failed: not timed", "failed_checks": bad}
        else:
            try:
                extra = run_extras(pm, L, comm, peaks, args)
            except Exception as exc:  # extras must never kill the headline line
                extra = {"error": repr(exc)}

    cpu_baseline = None
    if rank == 0 and size == 1 and not args.no_cpu:
        cores, rows_per_proc = cpu_split()
        with CpuRanks(cores, rows_per_proc, NCOLS) as pool:
            pool.step()
            reps = 0
            t0 = time.perf_counter()
            while time.perf_counter() - t0 < 10.0 and reps < 50:
                pool.step()
                reps += 1
            dt = time.perf_counter() - t0
        cpu_baseline = {"value": 2 * 4 * GLOBAL_ROWS * NCOLS * reps / dt / 1e9, "unit": "GB/s",
                        "cores": cores, "kind": "port",
                        "sample": f"{reps} passes over the full ({GLOBAL_ROWS} x {NCOLS}) float32 workload: {cores} processes x "
                                  f"({rows_per_proc} x {NCOLS}) (oracle restatement of FirstDerivative.py:201-219 per rank)"}

    if rank == 0:
        launches = 1 if (size == 1 or fused_halo) else 3
        line = {"metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": size, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(size), "roofline": roofline, "cpu_baseline": cpu_baseline,
                "e2e": e2e, "gpu_launches": args.steps * launches,
                "halo": ("peer-memory push + flags inside the stencil kernel (1 launch / apply)" if fused_halo else
                         ("none (single rank)" if size == 1 else "grouped ncclSend/Recv on a side stream (3 launches / apply)")),
                "clocks": clocks, "host_enqueue_ms_per_step": enqueue_ms, "parity": parity, "rng_note": rng_note,
                "secondary": secondary, "extra": extra}
        print(json.dumps(line))


def run_secondary(pm, L, comm, peaks, args):
    """second half of BASELINE's metric: MPIMatrixMult GF/s on config 4 (32768 x 32768 bf16 -> fp32) through the
    operator, plus the weak-scaling curve of the headline stencil.  Each figure carries its own roofline."""
    import torch
    rank, size = comm.Get_rank(), comm.Get_size()
    out = {"metric": METRIC2, "unit": "GF/s"}
    hbm, tpk = peaks["hbm_gbs"], peaks.get("bf16_tflops", 1590.0)
    grids = {1: (1, 1), 2: (1, 2), 4: (2, 2), 8: (2, 4)}
    if size in grids:
        Pr, Pc = grids[size]
        Ng = Kg = 32768
        Mg = 4096
        bn, bkA, bkX, bm = Ng // Pr, Kg // Pc, Kg // Pr, Mg // Pc

        def a_tile(r):
            return (torch.randn(bn, bkA, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1 + r)) / 181).to(torch.bfloat16)

        def x_tile(r):
            return torch.randn(bkX, bm, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1001 + r))
        At = a_tile(rank)
        modes = {}
        import parity_checks
        for name, kw in (("stationary", {"stationary": True}), ("summa", {}), ("replicated", {"replicate": True})):
            if size == 1 and name != "summa":
                continue
            try:
                Sop = pm.MPIMatrixMult(At, Mg, kind="summa", dtype="bfloat16", grid=(Pr, Pc), **kw)
            except TypeError:
                continue
            xs = pm.DistributedArray(global_shape=Kg * Mg, local_shapes=[bkX * bm] * size, dtype=np.float32)
            xs.local_array.copy_(x_tile(rank).reshape(-1))
            y = Sop.matvec(xs)
            torch.cuda.synchronize()
            ok, det = parity_checks.sampled_rows_check(pm, comm, Sop, a_tile, x_tile, y, Ng, Kg, Mg, Pr, Pc, nrows=256)
            oks = comm.allgather(bool(ok)) if size > 1 else [bool(ok)]
            ms = time_loop(lambda: Sop.matvec(xs), 5, 2, comm)
            fl = 2.0 * Ng * Kg * Mg
            tf = fl * 5 / (ms * 1e-3) / 1e12
            ms2 = time_loop(lambda: Sop.rmatvec(y), 3, 1, comm)
            modes[name] = {"GF/s": tf * 1e3, "TF/s": tf, "ms": ms / 5, "adjoint_ms": ms2 / 3,
                           "frac_of_N_x_burst_peak": tf / (size * tpk),
                           "frac_of_N_x_sustained_peak": tf / (size * peaks.get("bf16_tflops_sustained", tpk)),
                           "parity_256_sampled_rows_vs_fp64": {"ok": all(oks), "detail": det}}
            del Sop, xs, y
        best = "stationary" if "stationary" in modes else "summa"
        out["value"] = modes[best]["GF/s"]
        out["layout"] = f"{best}: one copy of A per GPU on a {Pr} x {Pc} grid (the reference's 2-D tile layout)"
        out["config"] = {"workload": f"MPIMatrixMult 32768 x 32768 bf16 -> fp32, M = 4096 columns, grid {Pr}x{Pc}",
                         "flop_per_apply": 2.0 * Ng * Kg * Mg}
        tp = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tp = json.load(f).get("gemm_bf16_tc2_tensor_pipe_pct")
        except Exception:
            pass
        out["roofline"] = {"bound": "tensor", "kernel": "gemm_bf16_tc2_kernel (tcgen05 cta_group::2, 256x256x64 tiles)",
                           "achieved": modes[best]["TF/s"] / size, "peak": tpk, "unit": "TFLOP/s per GPU",
                           "frac": modes[best]["TF/s"] / (size * tpk), "tensor_pipe_pct_ncu": tp,
                           "peak_kind": "measured cuBLAS bf16 8192^3 burst (MEASURED_PEAKS.json)"}
        out["modes"] = modes
        del At
        # config 4 (i), the literal "32768-vec": single right-hand side, HBM-bound GEMV through the operator
        try:
            At1 = (torch.randn(Ng // size, Kg, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1 + rank)) / 181).to(torch.bfloat16)
            Sop = pm.MPIMatrixMult(At1, 1, kind="summa", dtype="bfloat16", grid=(size, 1), replicate=True)
            xs = pm.DistributedArray(global_shape=Kg, local_shapes=[Kg // size] * size, dtype=np.float32)
            xs.local_array.normal_()
            torch.cuda.synchronize()
            time.sleep(0.5)
            ms = time_loop(lambda: Sop.matvec(xs), 20, 10, comm)
            gb = 2.0 * Ng * Kg * 20 / (ms * 1e-3) / 1e9
            out["m1_32768_vec"] = {"us": ms / 20 * 1e3, "GB/s_A": gb, "GF/s": gb, "frac_hbm": gb / (size * hbm),
                                   "host_enqueue_us": time_loop.last_enqueue_ms * 1e3,
                                   "layout": f"1-D row panels, grid {size}x1: one-shot peer all-gather of x + row-splitting GEMV",
                                   "bound": "hbm (1 flop/B)"}
            del Sop, xs, At1
        except Exception as exc:
            out["m1_32768_vec"] = {"error": repr(exc)}
    # weak-scaling curve of the headline stencil (the N = 1 block on every GPU)
    nloc = GLOBAL_ROWS
    xw = pm.DistributedArray(global_shape=nloc * size * NCOLS, dtype=np.float32)
    xw.local_array.normal_()
    Fw = pm.MPIFirstDerivative((nloc * size, NCOLS), kind="centered", order=3, dtype=np.float32)
    hold = {}

    def stepw():
        hold["y"] = Fw.matvec(xw)
    ms = time_loop(stepw, 10, 3, comm)
    v = 2 * 4 * nloc * NCOLS * size * 10 / (ms * 1e-3) / 1e9
    out["fd_weak_scaling"] = {"GB/s": v, "rows_per_gpu": nloc, "ms_per_step": ms / 10, "frac_hbm_per_gpu": v / size / hbm,
                              "scaling": "weak"}
    return out


def run_extras(pm, L, comm, peaks, args):
    """other BASELINE configs, each timed with CUDA events after warm-up (short loops)"""
    import torch
    rank, size = comm.Get_rank(), comm.Get_size()
    out = {}
    K, W = 10, 3
    hbm = peaks["hbm_gbs"]

    def gbs(nbytes, ms_total, k=K):
        return nbytes * k / (ms_total * 1e-3) / 1e9

    # --- FirstDerivative variants (per-GPU kernel, device resident) -------------------
    nloc, ncols = 32768, NCOLS
    for name, dt, code, kind, order, adj in (("fd_centered3_adj_f32", torch.float32, L.F32, L.FD_CENTERED, 3, 1),
                                             ("fd_centered5_f32", torch.float32, L.F32, L.FD_CENTERED, 5, 0),
                                             ("fd_forward_f32", torch.float32, L.F32, L.FD_FORWARD, 3, 0),
                                             ("fd_centered3_f64", torch.float64, L.F64, L.FD_CENTERED, 3, 0)):
        rows = nloc if dt is torch.float32 else nloc // 2
        xl = torch.randn(rows, ncols, device="cuda", dtype=dt)
        yl = torch.empty_like(xl)

        def kern():
            L.check(L.lib.b2_first_derivative(L.ctx(), xl.data_ptr(), yl.data_ptr(), None, 0, None, 0, rows, ncols,
                                              0, rows, kind, order, 0, 1.0, adj, code, L.stream()))
        ms = time_loop(kern, K, W)
        v = gbs(2 * xl.element_size() * xl.numel(), ms)
        out[name] = {"GB/s": v, "frac_hbm": v / hbm}
        del xl, yl

    # --- config 2: local reductions (dot 8 B/elem, norm 4 B/elem) ------------------------
    n = 1 << 28
    a = pm.DistributedArray(global_shape=n * size, dtype=np.float32)
    b = pm.DistributedArray(global_shape=n * size, dtype=np.float32)
    a.local_array.normal_()
    b.local_array.normal_()
    ms = time_loop(lambda: a._dot_device(b), K, W, comm)
    out["dot_f32_2^28_per_gpu"] = {"GB/s": gbs(8 * n * size, ms), "frac_hbm": gbs(8 * n, ms) / hbm, "us": ms / K * 1e3}
    ms = time_loop(lambda: a._norm_device(2), K, W, comm)
    out["norm2_f32_2^28_per_gpu"] = {"GB/s": gbs(4 * n * size, ms), "frac_hbm": gbs(4 * n, ms) / hbm, "us": ms / K * 1e3}
    # --- "next" row: fused ISTA / FISTA model update (ISTA: 2 reads + 1 write, FISTA: 3 reads + 2 writes per elem) ---
    from pylops_mpi_b200.optimization.cls_sparsity import _sparse_update
    sums = torch.zeros(4, dtype=torch.float64, device="cuda")
    xa, ga = a.local_array, b.local_array
    ms = time_loop(lambda: _sparse_update(xa, ga, 1e-3, xa, 1e-4, L.THRESH_SOFT, xa, None, 0.0, sums), K, W)
    out["ista_update_f32_2^28"] = {"GB/s": gbs(12 * n, ms), "frac_hbm": gbs(12 * n, ms) / hbm, "us": ms / K * 1e3}
    za = torch.randn_like(xa)
    ms = time_loop(lambda: _sparse_update(za, ga, 1e-3, xa, 1e-4, L.THRESH_SOFT, xa, za, 0.3, sums), K, W)
    out["fista_update_f32_2^28"] = {"GB/s": gbs(20 * n, ms), "frac_hbm": gbs(20 * n, ms) / hbm, "us": ms / K * 1e3}
    del za
    small = pm.DistributedArray(global_shape=10000 * size, dtype=np.float32)
    small.local_array.normal_()
    ms = time_loop(lambda: small.dot(small), 50, 5, comm)
    out["dot_f32_1e4_host_result_us"] = ms / 50 * 1e3
    if size > 1:
        from pylops_mpi_b200.Distributed import allreduce_
        sweep = {}
        big = torch.zeros(10 ** 9, dtype=torch.float32, device="cuda")      # 4 GB: config 2 sweeps 1e4 .. 1e9 elements
        for ne in (10 ** 4, 10 ** 5, 10 ** 6, 10 ** 7, 10 ** 8, 10 ** 9):
            buf = big[:ne]
            ms = time_loop(lambda: allreduce_(comm, buf), 10, 3, comm)
            us = ms / 10 * 1e3
            alg = 4 * ne / (us * 1e-6) / 1e9
            sweep[str(ne)] = {"us": us, "algbw_GB/s": alg, "busbw_GB/s": alg * 2 * (size - 1) / size,
                              "path": "peer-memory one-shot" if 4 * ne <= 64 * 1024 and comm.peer_vec is not None else "nccl"}
        out["allreduce_f32_sweep"] = sweep
        del big
    del a, b

    # --- config 3: BlockDiag of one 4096^2 f32 block per GPU + cgls ------------------------
    nb = 4096
    A = torch.randn(nb, nb, device="cuda", generator=torch.Generator(device="cuda").manual_seed(100 + rank)) / 128
    A += 2 * torch.eye(nb, device="cuda")
    blk = pm.MatrixMult(A)
    xv = torch.randn(nb, device="cuda")
    yv = torch.empty(nb, device="cuda")
    ms = time_loop(lambda: blk.matvec(xv, out=yv), 50, 10)
    out["gemv_f32_4096_N"] = {"GB/s": gbs(4 * nb * nb, ms, 50), "us": ms / 50 * 1e3,
                              "note": "A (64 MiB) fits the 126 MB L2: >100% of HBM peak means L2 hits"}
    ms = time_loop(lambda: blk.rmatvec(xv, out=yv), 50, 10)
    out["gemv_f32_4096_T"] = {"GB/s": gbs(4 * nb * nb, ms, 50), "us": ms / 50 * 1e3}
    Op = pm.MPIBlockDiag([blk])
    xt = pm.DistributedArray(global_shape=nb * size, dtype=np.float32)
    xt.local_array.normal_()
    yd = Op.matvec(xt)
    x0 = xt.zeros_like()
    pm.cgls(Op, yd, x0=x0, niter=5, tol=0.0)
    torch.cuda.synchronize()
    comm.Barrier()
    t0 = time.perf_counter()
    solver = pm.CGLS(Op)
    xinv, istop, iit, r1, r2, cost = solver.solve(yd, x0=x0, niter=50, tol=0.0)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if size > 1:
        dt = comm.allreduce(dt, "max")
    err = (xinv - xt).norm()[0] / xt.norm()[0]
    # steady-state cost of one iteration: slope between a 50- and a 450-iteration solve (the 50-iteration wall time
    # also carries setup, two eager warm-up iterations and the one-off graph capture)
    torch.cuda.synchronize()
    comm.Barrier()
    t0 = time.perf_counter()
    pm.CGLS(Op).solve(yd, x0=x0, niter=450, tol=0.0)
    torch.cuda.synchronize()
    dt2 = time.perf_counter() - t0
    if size > 1:
        dt2 = comm.allreduce(dt2, "max")
    out["cgls_blockdiag_4096_f32_50it"] = {"iters_per_s": 50 / dt, "ms_per_iter": dt / 50 * 1e3, "rel_err_vs_xtrue": float(err),
                                           "ms_per_iter_steady_state": (dt2 - dt) / 400 * 1e3,
                                           "cuda_graph_replays": getattr(solver, "graph_replays", 0),
                                           "cuda_graph_capture_ms": getattr(solver, "graph_capture_ms", None),
                                           "cuda_graph_capture_breakdown_ms": getattr(solver, "graph_capture_breakdown_ms", None),
                                           "cuda_graph_error": getattr(solver, "graph_error", None)}
    # HBM-bound GEMV (A = 1 GiB)
    A2 = torch.randn(32768, 8192, device="cuda")
    big = pm.MatrixMult(A2)
    xb, yb = torch.randn(8192, device="cuda"), torch.empty(32768, device="cuda")
    ms = time_loop(lambda: big.matvec(xb, out=yb), K, W)
    out["gemv_f32_32768x8192_N"] = {"GB/s": gbs(4 * A2.numel(), ms), "frac_hbm": gbs(4 * A2.numel(), ms) / hbm}
    xb2, yb2 = torch.randn(32768, device="cuda"), torch.empty(8192, device="cuda")
    ms = time_loop(lambda: big.rmatvec(xb2, out=yb2), K, W)
    out["gemv_f32_32768x8192_T"] = {"GB/s": gbs(4 * A2.numel(), ms), "frac_hbm": gbs(4 * A2.numel(), ms) / hbm}
    del A2, big
    # config 4 (i): bf16 matrix, single right-hand side (GEMV, HBM-bound)
    Ab = (torch.randn(32768, 16384, device="cuda") / 181).to(torch.bfloat16)
    bop = pm.MatrixMult(Ab)
    xb, yb = torch.randn(16384, device="cuda"), torch.empty(32768, device="cuda")
    ms = time_loop(lambda: bop.matvec(xb, out=yb), K, W)
    v = gbs(2 * Ab.numel(), ms)
    out["gemv_bf16_32768x16384_N"] = {"GB/s": v, "frac_hbm": v / hbm, "GF/s": 2 * Ab.numel() * K / (ms * 1e-3) / 1e9}
    # config 4 (ii): bf16 tile product on tensor cores, if the kernel is available
    try:
        m = n_ = k = 8192
        Am = (torch.randn(m, k, device="cuda") / 90).to(torch.bfloat16)
        Bm = (torch.randn(k, n_, device="cuda") / 90).to(torch.bfloat16)
        Cm = torch.empty(m, n_, device="cuda")

        def mm():
            L.check(L.lib.b2_gemm_bf16(L.ctx(), Am.data_ptr(), k, Bm.data_ptr(), n_, Cm.data_ptr(), n_, m, n_, k,
                                       L.OP_N, 0, L.stream()), "b2_gemm_bf16")
        ms = time_loop(mm, K, W)
        tf = 2.0 * m * n_ * k * K / (ms * 1e-3) / 1e12
        out["gemm_bf16_8192^3"] = {"TF/s": tf, "GF/s": tf * 1e3, "frac_tensor": tf / peaks.get("bf16_tflops", 1590.0)}
        del Am, Bm, Cm
    except Exception as exc:
        out["gemm_bf16_8192^3"] = {"unavailable": repr(exc)}
    del Ab, bop
    # --- config 5: Fredholm1 (64 slices per GPU, 256 x 256 x 64, complex64) -------------------
    nsl, ns, nr, nv = 64, 256, 256, 64
    G = torch.randn(nsl, ns, nr, device="cuda", dtype=torch.complex64)
    Fr = pm.MPIFredholm1(G, nz=nv, dtype=np.complex64, fused=False)
    xm = pm.DistributedArray(global_shape=nsl * size * nr * nv, partition=pm.Partition.BROADCAST, dtype=np.complex64)
    xm.local_array.normal_()
    ms = time_loop(lambda: Fr.matvec(xm), K, W, comm)
    fl = 8.0 * nsl * size * ns * nr * nv
    out["fredholm1_c64_64x256x256x64_per_gpu"] = {"GF/s": fl * K / (ms * 1e-3) / 1e9, "us": ms / K * 1e3,
                                                  "mode": "product kernel + NCCL all-gather"}
    if size > 1:
        Ff = pm.MPIFredholm1(G, nz=nv, dtype=np.complex64, fused=True)
        ms = time_loop(lambda: Ff.matvec(xm), K, W, comm)
        out["fredholm1_fused_peer_c64_64x256x256x64_per_gpu"] = {
            "GF/s": fl * K / (ms * 1e-3) / 1e9, "us": ms / K * 1e3,
            "mode": "ONE kernel: product + all-gather via P2P stores into IPC-mapped peer buffers"}
    # --- MDD (tutorials/mdd.py:108-120, 190-194 shapes): MPIMDC + 50 CGLS iterations, ns = nr = 256, nt = 1024
    #     (one-sided: nfft = 513, 512 slices in the band at 8 GPUs = 64 per GPU), nv = 64, float32 / complex64 -------
    try:
        import warnings
        nt, nf_loc = 1024, 64
        gen = torch.Generator(device="cuda").manual_seed(5)
        gt = torch.randn(nt, ns, nr, device="cuda", generator=gen) * 0.05          # real kernels -> physical spectrum
        Gf = torch.fft.rfft(gt, n=nt, dim=0)[rank * nf_loc:(rank + 1) * nf_loc].contiguous()
        del gt
        mm = pm.DistributedArray(global_shape=nt * nr * nv, partition=pm.Partition.BROADCAST, dtype=np.float32)
        mm.local_array.copy_(torch.randn(nt * nr * nv, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6)))
        res = {}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sols = {}
            for dom in ("time", "frequency"):
                Mop = pm.MPIMDC(Gf, nt=nt, nv=nv, nfreq=nf_loc * size, dt=0.004, dr=1.0, twosided=False, data_domain=dom)
                dd = Mop @ mm
                x0 = mm.zeros_like()
                pm.cgls(Mop, dd, x0=x0, niter=2, tol=0.0)
                torch.cuda.synchronize()
                comm.Barrier()
                t0 = time.perf_counter()
                xinv, istop, iit, r1, r2, cost = pm.cgls(Mop, dd, x0=x0, niter=50, tol=0.0)
                torch.cuda.synchronize()
                dt_s = time.perf_counter() - t0
                if size > 1:
                    dt_s = comm.allreduce(dt_s, "max")
                sols[dom] = xinv
                res[dom] = {"ms_per_iter": dt_s / 50 * 1e3, "iterations": int(iit), "cost_first": float(cost[0]),
                            "cost_last": float(cost[-1]), "rel_err_vs_m_true": float((xinv - mm).norm()[0] / mm.norm()[0]),
                            "allgathers_per_iteration": 2 if dom == "time" else 1}
                del Mop, dd
            res["iterates_agree_rel"] = float((sols["time"] - sols["frequency"]).norm()[0] / sols["time"].norm()[0])
        res["config"] = f"ns=nr=256, nt={nt} one-sided, nv=64, {nf_loc} frequency slices per GPU, float32/complex64, cgls 50 it"
        out["mdd_cgls50"] = res
    except Exception as exc:
        out["mdd_cgls50"] = {"error": repr(exc)[:300]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the multi-rank parity preamble")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of the last step's output to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
