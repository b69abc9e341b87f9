#!/usr/bin/env python
"""Benchmark of the torchcde_b200 hot path against BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one fused fixed-step solve ``cdeint(CubicSpline(hermite coeffs), linear func, z0,
t=[0, L-1], method='rk4', options={'step_size': 1})`` over one synthetic batch at BASELINE
config 3: batch 65536 per GPU, length 256, 8 input channels, 32 hidden channels, fp32.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what every key means.

``--dump-outputs DIR`` writes what the last timed step returned on rank 0 -- the whole
``cdeint`` output, (65536, 2, 32) float32, 16 MB -- as ``DIR/cdeint_out.npy``.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.

Timing rules: inputs resident in HBM for ``value`` (CUDA events, max over ranks, barrier +
synchronize both sides); the coefficient tensor is 2.1 GB per GPU, far larger than the 126 MB
L2, so no flush is needed between iterations.  ``e2e`` runs the user pipeline from pinned HOST
series through ``torchcde_b200.hostio.cdeint_from_host_series`` (H2D of x and z0, fused gap fill +
Hermite coefficients on the device, fused solve, D2H) with the copies inside the timed region.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the tree may be read-only: leave no __pycache__ behind in it

import torch  # noqa: E402

BATCH, LENGTH, CHANNELS, HIDDEN = 65536, 256, 8, 32
METRIC = "sequences/s for cdeint RK4 (batch=65536,len=256,ch=8,hid=32)"
# SURVEY.md 8(d) / BASELINE.md 4: algorithmic work per sequence of the fused RK4 solve
BYTES_PER_SEQ = 255 * 3 * CHANNELS * 4 + HIDDEN * 4 + 2 * HIDDEN * 4           # 24,864 B
FLOPS_PER_SEQ = 255 * (4 * (2 * HIDDEN * HIDDEN * CHANNELS + HIDDEN * CHANNELS + 2 * HIDDEN * CHANNELS + 4 * CHANNELS) + 320)
HERMITE_BYTES_PER_SEQ = LENGTH * CHANNELS * 4 + (LENGTH - 1) * 4 * CHANNELS * 4   # 40,832 B
WORKLOAD = ("cdeint rk4 step_size=1 (255 steps, 1020 stage evals), CubicSpline(hermite bdiff coeffs), linear func "
            "Linear(32,256).view(32,8), batch=65536 per GPU, len=256, ch=8, hid=32, adjoint=False")




def config_for(world):
    return {"workload": WORKLOAD, "parallelism": "batch-sharded x{}".format(world), "global_batch": world * BATCH,
            "l2": "inputs (2.1 GB coeffs per GPU) exceed the 126 MB L2; no flush"}


_T0 = time.perf_counter()


def note(msg):
    """Progress marker on stderr (the JSON line on stdout stays alone)."""
    sys.stderr.write("[bench {:7.1f}s] {}\n".format(time.perf_counter() - _T0, msg))
    sys.stderr.flush()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "sm_max_mhz": p.get("sm_max_mhz", 1965.0),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0,
            "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------- synthetic data
def synthetic(batch, device, seed):
    """SURVEY.md 8(d): bounded random walk x = cumsum(randn)/sqrt(L); Linear(32, 256) default init; z0 ~ N(0,1)."""
    import torchcde_b200 as cde
    gen = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(batch, LENGTH, CHANNELS, generator=gen, device=device).cumsum(1) / math.sqrt(LENGTH)
    z0 = torch.randn(batch, HIDDEN, generator=gen, device=device)
    torch.manual_seed(1)
    func = cde.LinearVectorField(HIDDEN, CHANNELS).to(device)
    return x, z0, func


class ClockSampler:
    """nvidia-smi in the background from the start of the run (its start-up takes longer than the
    timed region); afterwards only the samples whose timestamps fall inside the timed window count."""
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        self.window = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.file,
                                         stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def wait_ready(self, timeout=20.0):
        """Block until nvidia-smi has written its first sample (its start-up on a fresh box can take seconds, longer
        than the whole timed region -- BENCH_r01 had 'no samples' for that reason)."""
        if self.proc is None:
            return False
        deadline = time.time() + timeout
        while time.time() < deadline:
            try:
                if os.path.getsize(self.file.name) > 0:
                    return True
            except OSError:
                pass
            if self.proc.poll() is not None:
                return False
            time.sleep(0.05)
        return False

    def mark(self, t_begin, t_end):
        self.window = (t_begin, t_end)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.file.flush()
        self.file.seek(0)
        import datetime
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.file:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                stamp = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((stamp, float(parts[1]), float(parts[2]), [n for n, v in zip(names, parts[4:8]) if v == "Active"]))
            except ValueError:
                continue
        self.file.close()
        os.unlink(self.file.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        picked, where = rows, "whole run"
        if self.window is not None:
            lo, hi = self.window
            inside = [r for r in rows if lo - 0.02 <= r[0] <= hi + 0.02]
            if inside:
                picked, where = inside, "timed region"
            else:
                mid = 0.5 * (lo + hi)
                picked, where = sorted(rows, key=lambda r: abs(r[0] - mid))[:3], "nearest to the timed region"
        sm = sorted(r[1] for r in picked)
        reasons = sorted({n for r in picked for n in r[3]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[2] for r in picked), "reasons": reasons,
                "samples": len(picked), "window": where}


_LOCAL_MS = {}


def time_loop(fn, steps, warmup, device, dist=None):
    """W untimed + exactly K timed calls, CUDA events on the current stream, barrier + sync both sides."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(device)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(device)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        fn()
    end.record()
    torch.cuda.synchronize(device)
    if dist is not None:
        dist.barrier()
    ms = start.elapsed_time(end)
    _LOCAL_MS["last"] = ms                        # this rank's own device time (before the MAX over ranks)
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


# ------------------------------------------------------------------------------- CPU arm
CPU_SAMPLE_PATHS = 8192      # FIXED sample (never calibrated): per-sequence CPU cost depends on the batch size


def host_threads():
    """Threads the CPU arm uses: one per physical core the process may run on (cpu_count // 2 on an SMT-2 host),
    set explicitly so that torchrun's OMP_NUM_THREADS=1 does not silently turn the arm single-threaded."""
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count() or 1
    return max(1, usable // 2)


def cpu_reference_solver(sample_paths):
    """The reference's OWN ``cdeint`` (unmodified torchcde from /root/reference or oracle/_ref: its
    ``_check_compatability``, ``_VectorField.forward`` with 63 aten calls and 4 ``item()`` per evaluation,
    ``CubicSpline.derivative``, output permute) on host cores.  torchdiffeq, which it dispatches to at
    solver.py:226-227, is not installable offline: ``oracle/odeint_port.py`` stands in for it (kind "_ref+port").
    Falls back to the streamlined oracle port only if no reference tree is present at all (kind "port")."""
    from oracle import cde_oracle as O
    from oracle import reference_loader
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(sample_paths, LENGTH, CHANNELS, generator=gen).cumsum(1) / math.sqrt(LENGTH)
    z0 = torch.randn(sample_paths, HIDDEN, generator=gen)
    torch.manual_seed(1)
    lin = torch.nn.Linear(HIDDEN, HIDDEN * CHANNELS)
    t = torch.tensor([0.0, LENGTH - 1.0])
    if reference_loader.reference_available():
        ref = reference_loader.load_reference()

        class ReadmeField(torch.nn.Module):          # README.md:42-49
            def __init__(self):
                super().__init__()
                self.linear = lin

            def forward(self, t, z):
                return self.linear(z).view(*z.shape[:-1], HIDDEN, CHANNELS)

        func = ReadmeField()
        with torch.no_grad():
            coeffs = ref.hermite_cubic_coefficients_with_backward_differences(x)
            X = ref.CubicSpline(coeffs)

        def run():
            with torch.no_grad():
                return ref.cdeint(X=X, func=func, z0=z0, t=X.interval, adjoint=False, method="rk4",
                                  options={"step_size": 1.0})
        kind = "_ref+port"
        what = ("the reference's own torchcde.cdeint ({} tree), torchdiffeq replaced by oracle/odeint_port.py"
                .format(reference_loader.reference_kind()))
    else:
        knots = O.knot_times(LENGTH, torch.float32)
        with torch.no_grad():
            coeffs = O.hermite_backward_difference_coeffs(x)

        def run():
            with torch.no_grad():
                return O.cdeint_linear(coeffs, knots, lin.weight, lin.bias, z0, t, "rk4", 1.0)
        kind = "port"
        what = "oracle port of the reference op sequence (no reference tree on this machine)"
    return run, kind, what


def cpu_baseline(reps=4):
    threads = host_threads()
    torch.set_num_threads(threads)
    run, kind, what = cpu_reference_solver(CPU_SAMPLE_PATHS)
    run()
    t0 = time.perf_counter()
    for _ in range(reps):
        run()
    dt = (time.perf_counter() - t0) / reps
    note("cpu baseline ({}): {} paths in {:.2f}s on {} threads".format(kind, CPU_SAMPLE_PATHS, dt, threads))
    return {"value": CPU_SAMPLE_PATHS / dt, "unit": "sequences/s", "cores": torch.get_num_threads(), "kind": kind,
            "host_cpus": os.cpu_count(), "seconds_per_sample": dt,
            "sample": "FIXED {} of 65536 paths, full 255 RK4 steps (1020 field evaluations), fp32, {}; mean of {} runs "
                      "after 1 warm-up, torch.set_num_threads({})".format(CPU_SAMPLE_PATHS, what, reps, threads)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    torch.set_num_threads(threads)
    run, kind, what = cpu_reference_solver(CPU_SAMPLE_PATHS)
    for _ in range(max(1, args.warmup)):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    total = time.perf_counter() - t0
    value = CPU_SAMPLE_PATHS * args.steps / total
    base = {"value": value, "unit": "sequences/s", "cores": torch.get_num_threads(), "kind": kind,
            "host_cpus": os.cpu_count(),
            "sample": "each step = FIXED {} of 65536 paths, full 255 RK4 steps, fp32, {}; torch.set_num_threads({})"
                      .format(CPU_SAMPLE_PATHS, what, threads)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "sequences/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_for(args.gpus),     # the SAME config as the GPU arm; what was sampled is in cpu_baseline
            "host": {"threads": threads, "sample_paths_per_step": CPU_SAMPLE_PATHS},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------- GPU arm
def run_gpu_arm(args):
    import torchcde_b200 as cde
    from torchcde_b200 import _lib, hostio

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # Keep stdout clean for the ONE JSON line: libraries (NCCL prints its version banner to fd 1) get
    # stderr; the JSON is written to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    _lib.load()
    if args.variant is not None:
        _lib.call("tcde_set_solve_variant", args.variant)

    sampler = ClockSampler(local_rank)       # every rank watches its own GPU; rank 0 reports its own and a per-rank summary
    sampler.start()
    note("rank {} of {}: generating synthetic data".format(rank, world))
    x, z0, func = synthetic(BATCH, device, seed=1000 + rank)
    if dist is not None:
        from torchcde_b200.distributed import broadcast_field
        broadcast_field(func, src=0)          # the one collective of the job: 8,448 floats over NCCL
    options = {"step_size": 1.0}
    with torch.no_grad():
        coeffs = cde.hermite_cubic_coefficients_with_backward_differences(x)
        X = cde.CubicSpline(coeffs)
        t = torch.tensor([0.0, LENGTH - 1.0])      # == X.interval, kept on the host: no sync per call
        holder = {}

        def step():
            holder["out"] = cde.cdeint(X, func, z0, t, adjoint=False, method="rk4", options=options)

        note("timing {} solves".format(args.steps))
        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize(device)
        sampler.wait_ready()
        wall_begin = time.time()
        ms = time_loop(step, args.steps, 0, device, dist)
        wall_end = time.time()
        sampler.mark(wall_begin, wall_end)
        clocks = sampler.stop()
        if dist is not None:
            # per-rank device time and clocks of the same timed region: `value` uses the slowest rank (time_loop's MAX)
            mine = {"rank": rank, "ms_per_step": _LOCAL_MS.get("last", 0.0) / args.steps, "sm_mhz": clocks.get("sm_mhz"),
                    "reasons": clocks.get("reasons")}
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            if rank == 0:
                clocks["per_rank"] = gathered
        if rank != 0:
            clocks = None
        assert bool(torch.isfinite(holder["out"]).all())
        if args.dump_outputs and rank == 0:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "cdeint_out.npy"), holder["out"].float().cpu().numpy())

        note("device-resident: {:.3f} ms per solve".format(ms / args.steps))
        # ---- end to end from pinned host buffers (copies inside the timed region) ------------
        coeffs_host = torch.empty(coeffs.shape, dtype=coeffs.dtype, pin_memory=True)
        coeffs_host.copy_(coeffs)
        z0_host = torch.empty(z0.shape, dtype=z0.dtype, pin_memory=True)
        z0_host.copy_(z0)
        out_host = torch.empty(BATCH, 2, HIDDEN, dtype=z0.dtype, pin_memory=True)
        chunk = 4096
        pipe = hostio.HostPipeline(device, chunk, tuple(coeffs.shape[1:]), HIDDEN, 2, coeffs.dtype)

        def e2e_step():
            hostio.cdeint_from_host(coeffs_host, func, z0_host, t, out_host=out_host, chunk_paths=chunk,
                                    pipeline=pipe, device=device, method="rk4", options=options)

        note("pinned host buffers ready; timing end to end")
        e2e_steps = max(2, min(args.steps, 5))
        e2e_ms = time_loop(e2e_step, e2e_steps, 1, device, dist)
        torch.cuda.synchronize(device)
        e2e_ok = torch.equal(out_host.to(device), holder["out"])
        e2e_h2d = coeffs_host.numel() * 4 + z0_host.numel() * 4
        del coeffs_host, pipe

        # the same result from the RAW series on the host (coefficients rebuilt on the device)
        x_host = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
        x_host.copy_(x)
        out_host2 = torch.empty(BATCH, 2, HIDDEN, dtype=z0.dtype, pin_memory=True)

        def e2e_series_step():
            hostio.cdeint_from_host_series(x_host, func, z0_host, t, out_host=out_host2, chunk_paths=8192,
                                           device=device, method="rk4", options=options)

        series_ms = time_loop(e2e_series_step, e2e_steps, 1, device, dist)
        torch.cuda.synchronize(device)
        series_ok = torch.equal(out_host2.to(device), holder["out"])

        note("end to end: {:.3f} ms per solve, matches={}".format(e2e_ms / e2e_steps, bool(e2e_ok)))
        # ---- secondary kernels (rank 0, N=1 only): the HBM-bound coefficient builders ---------
        # ms = one public-API call (allocation, launch, and for the linear / natural builders the NaN-flag read-back that
        # picks the reference's branch: a host sync; the Hermite builder reads nothing back); kernel_ms = the C-ABI
        # launch alone, 10 back to back (inputs + outputs are 5-20x the L2, so nothing is served from cache).
        # The roofline fraction is the kernel's; the API time is what a caller of the Python function sees.
        extra = {}
        if rank == 0:
            from torchcde_b200 import _lib
            peaks = measured_peaks()
            code = _lib.dtype_code(x.dtype)
            stream = _lib.stream_of(x)
            flags = torch.zeros(1, dtype=torch.int32, device=device)
            rows = torch.empty(BATCH, LENGTH - 1, 4 * CHANNELS, dtype=x.dtype, device=device)
            ws = torch.empty(4 * LENGTH + 8, dtype=x.dtype, device=device)
            xn = x.clone()
            hole = torch.rand(x.shape, device=device) < 0.3
            hole[:, 0] = False
            hole[:, -1] = False
            xn[hole] = float("nan")
            del hole
            fill_bytes = 2 * LENGTH * CHANNELS * 4
            cases = (
                ("hermite_bdiff_coeffs", HERMITE_BYTES_PER_SEQ,
                 lambda: cde.hermite_cubic_coefficients_with_backward_differences(x),
                 lambda: _lib.call("tcde_hermite_bdiff_coeffs", _lib.ptr(x), None, _lib.ptr(rows), BATCH, LENGTH,
                                   CHANNELS, code, _lib.ptr(flags), stream), None),
                ("natural_cubic_coeffs", HERMITE_BYTES_PER_SEQ,
                 lambda: cde.natural_cubic_coeffs(x),
                 lambda: _lib.call("tcde_natural_cubic_coeffs", _lib.ptr(x), None, _lib.ptr(rows), _lib.ptr(ws), BATCH,
                                   LENGTH, CHANNELS, code, _lib.ptr(flags), stream),
                 "two launches: the batch-independent Thomas elimination (1 CTA) + the per-path kernel"),
                ("linear_interpolation_coeffs_30pct_nan", fill_bytes,
                 lambda: cde.linear_interpolation_coeffs(xn),
                 lambda: _lib.call("tcde_linear_fill", _lib.ptr(xn), None, _lib.ptr(rows), BATCH, LENGTH, CHANNELS,
                                   code, _lib.ptr(flags), stream),
                 "one launch: tcde_linear_fill reports the NaN flag itself (8,192 R + 8,192 W per sequence)"),
                ("hermite_bdiff_coeffs_30pct_nan", HERMITE_BYTES_PER_SEQ,
                 lambda: cde.hermite_cubic_coefficients_with_backward_differences(xn),
                 lambda: _lib.call("tcde_hermite_bdiff_coeffs_series", _lib.ptr(xn), None, _lib.ptr(rows), BATCH, LENGTH,
                                   CHANNELS, code, None, stream),
                 "one launch, no flag read-back: the gap fill happens in the warp's shared-memory tile "
                 "(tcde_hermite_bdiff_coeffs_series; round 1: NaN-flag sync + fill + Hermite = 3 launches)"),
            )
            for name, nbytes, api_fn, abi_fn, remark in cases:
                api_ms = time_loop(api_fn, 5, 3, device) / 5
                k_ms = time_loop(abi_fn, 10, 3, device) / 10
                gbs = BATCH * nbytes / (k_ms * 1e-3) / 1e9
                extra[name] = {"ms": api_ms, "kernel_ms": k_ms, "sequences_per_s": BATCH / (api_ms * 1e-3),
                               "bound": "hbm", "achieved_gbs": gbs, "peak_gbs": peaks["hbm_gbs"],
                               "frac": gbs / peaks["hbm_gbs"], "algorithmic_bytes_per_seq": nbytes}
                if remark:
                    extra[name]["note"] = remark
            del xn, rows
            # training step at the same shapes: cdeint(adjoint=True) forward + backward (fused adjoint stage kernel)
            try:
                def train_step():
                    zz = z0.clone().requires_grad_(True)
                    func.zero_grad()
                    with torch.enable_grad():
                        res = cde.cdeint(X, func, zz, t, adjoint=True, method="rk4", options=options)
                        res[:, -1].sum().backward()

                train_step()                                          # allocates the two 8.6 GB stage trajectories once
                t_ms = min(time_loop(train_step, 1, 0, device) for _ in range(3))
                extra["cdeint_rk4_forward_plus_adjoint_backward"] = {
                    "ms": t_ms, "sequences_per_s": BATCH / (t_ms * 1e-3), "bound": "tensor (bf16 / f16 MMAs)", "runs": "best of 3",
                    "note": "backward = two tensor-core solves that keep their stage inputs + one tcgen05 GEMM for dL/dW, dL/db "
                            "(tcde_cdeint_fixed_linear_stages x2, tcde_linear_field_param_grads); not the headline"}
            except Exception as exc:      # never lose the headline line over the extra
                extra["cdeint_rk4_forward_plus_adjoint_backward"] = {"error": repr(exc)}
            # SURVEY 8(f)1: a generic (non-linear) func through this package's stage loop -- the MLP + tanh field of
            # example/time_series_classification.py:37-51 (hidden 8, 3 input channels), batch 65536, length 256, rk4 step 1
            try:
                class MlpField(torch.nn.Module):
                    def __init__(self):
                        super().__init__()
                        self.linear1 = torch.nn.Linear(8, 128)
                        self.linear2 = torch.nn.Linear(128, 24)

                    def forward(self, tt, z):
                        z = self.linear2(self.linear1(z).relu()).tanh()
                        return z.view(*z.shape[:-1], 8, 3)

                torch.manual_seed(2)
                mlp = MlpField().to(device)
                Xg = cde.CubicSpline(cde.hermite_cubic_coefficients_with_backward_differences(x[..., :3].contiguous()))
                zg = z0[:, :8].contiguous()
                g_rows = {}
                for label, opts in (("kernel_loop", {"step_size": 1.0}), ("cuda_graph", {"step_size": 1.0, "cuda_graph": True})):
                    fn = lambda: cde.cdeint(Xg, mlp, zg, t, adjoint=False, method="rk4", options=opts)  # noqa: E731
                    g_ms = time_loop(fn, 2, 1, device) / 2
                    g_rows[label] = {"ms": g_ms, "sequences_per_s": BATCH / (g_ms * 1e-3)}
                extra["generic_mlp_field_rk4"] = dict(g_rows, note="func = Linear(8,128)-ReLU-Linear(128,24)-tanh (the reference example's "
                                                     "field), CubicSpline control with 3 channels; 12 launches per stage: dX/dt of a "
                                                     "step in one tcde_spline_eval launch, every Runge-Kutta combination one "
                                                     "tcde_linear_combination launch; func itself stays torch operators")
                del Xg, zg
            except Exception as exc:
                extra["generic_mlp_field_rk4"] = {"error": repr(exc)}
            # BASELINE config 4: the reference's default call (dopri5, adjoint=True) at the same shapes
            config4 = {}
            try:
                def fwd4():
                    holder["c4"] = cde.cdeint(X, func, z0, t, adjoint=True)          # no grad needed: forward only

                f_ms = time_loop(fwd4, 2, 1, device) / 2
                st4 = dict(cde.cdeint.last_stats)
                config4 = {"workload": "cdeint(X, func, z0, X.interval) -- torchdiffeq defaults: dopri5, rtol 1e-4, atol 1e-6, "
                                       "adjoint=True -- batch 65536, len 256, ch 8, hid 32",
                           "forward": {"ms": f_ms, "sequences_per_s": BATCH / (f_ms * 1e-3), "accepted_steps": st4.get("n_accepted"),
                                       "rejected_steps": st4.get("n_rejected"), "launches": st4.get("launches"),
                                       "device_controlled": st4.get("device_controlled"),
                                       "kernel": "dopri5_attempt_kernel: one launch per attempted step, controller and dense "
                                                 "output on the device, one host read per 48 launches"}}

                def train4():
                    zz = z0.clone().requires_grad_(True)
                    func.zero_grad()
                    with torch.enable_grad():
                        res = cde.cdeint(X, func, zz, t, adjoint=True)
                        res[:, -1].sum().backward()

                t0 = time.perf_counter()
                train4()
                torch.cuda.synchronize(device)
                b_s = time.perf_counter() - t0
                t0 = time.perf_counter()
                train4()                                                  # second run: the trajectory slots are allocated
                torch.cuda.synchronize(device)
                b_s = min(b_s, time.perf_counter() - t0)
                config4["forward_plus_adjoint_backward"] = {
                    "ms": b_s * 1e3, "sequences_per_s": BATCH / b_s, "runs": "best of 2",
                    "adjoint_stats": getattr(cde.cdeint, "last_adjoint_stats", None),
                    "note": "backward = dopri5 on (z, adjoint state) as one virtual batch with the controller on the device "
                            "(tcde_dopri5_linear_paired_attempts), dL/dW, dL/db by quadrature over the accepted steps' stage "
                            "inputs (one tcgen05 GEMM per 256 accepted steps); round 1 / host-driven: ~1.4 s"}
            except Exception as exc:
                config4["error"] = repr(exc)
            extra["config4_dopri5_adjoint"] = config4

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    ms_step = ms / args.steps
    value = world * BATCH * args.steps / (ms * 1e-3)
    kernel_s = ms_step * 1e-3                       # one launch per step: the step IS the kernel
    achieved_gbs = BATCH * BYTES_PER_SEQ / kernel_s / 1e9
    achieved_tf = BATCH * FLOPS_PER_SEQ / kernel_s / 1e12
    fp32_peak_tf = 148 * 128 * 2 * peaks["sm_max_mhz"] * 1e6 / 1e12
    e2e_value = world * BATCH * e2e_steps / (e2e_ms * 1e-3)
    variant = (args.variant if args.variant is not None else 0) & 15
    tensor_kernel = variant != 1
    fp16_split = variant in (0, 4, 5)
    mmas_per_stage = 7 if fp16_split else 13        # 128 x 256 x (16 halves | 8 tf32) each: the same 2 * 128 * 256 * 16 / 2 ... flops per cycle-slot
    mma_flops = BATCH / 128 * 255 * 4 * mmas_per_stage * 2 * 128 * 256 * (16 if fp16_split else 8)
    mma_peak = peaks["bf16_tflops"] if fp16_split else peaks["bf16_tflops"] / 2
    kernel_name = {0: "cdeint_tc_kernel<1> (tcgen05.mma kind::f16, 2xFP16 split, TMA rows, persistent)", 2: "cdeint_umma_kernel<8> (round 1, 3xTF32)",
                   3: "cdeint_tc_kernel<0> (3xTF32)", 4: "cdeint_tc_kernel<1> (2xFP16)", 5: "cdeint_tc_kernel<1> (2xFP16)",
                   6: "cdeint_tc_kernel<0> (3xTF32)"}.get(variant, "?")
    secondary = dict(extra)
    config4 = secondary.get("config4_dopri5_adjoint")
    line = {
        "metric": METRIC, "value": value, "unit": "sequences/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_for(world),
        "clocks": clocks,
        # end to end from HOST buffers through the package's public pipeline: the raw series and z0 leave pinned host memory
        # every step (H2D inside the timed region), the Hermite coefficients are built on the device (hot path (i)), the
        # fused solve runs (hot path (ii)), the result returns to pinned host memory (D2H inside the timed region)
        "e2e": {"value": world * BATCH * e2e_steps / (series_ms * 1e-3), "unit": "sequences/s",
                "h2d_bytes_per_step": x_host.numel() * 4 + z0_host.numel() * 4, "d2h_bytes_per_step": out_host2.numel() * 4,
                "ms_per_step": series_ms / e2e_steps, "matches_device_result": bool(series_ok),
                "api": "torchcde_b200.hostio.cdeint_from_host_series (pinned host x + z0 -> chunked H2D / gap fill + Hermite "
                       "coefficients on device / fused solve / D2H, 4 streams)",
                "from_coefficients": {"value": e2e_value, "unit": "sequences/s", "ms_per_step": e2e_ms / e2e_steps,
                                      "h2d_bytes_per_step": e2e_h2d, "d2h_bytes_per_step": out_host.numel() * 4,
                                      "matches_device_result": bool(e2e_ok),
                                      "api": "torchcde_b200.hostio.cdeint_from_host (pinned host COEFFICIENTS + z0: 4x the "
                                             "PCIe bytes; what a user who stores coefficients as the dataset pays)"}},
        "gpu_launches": args.steps,
        "roofline": ({
            "bound": "tensor", "achieved": achieved_tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": achieved_tf / peaks["bf16_tflops"], "traffic": 2225915168, "peak_source": peaks["source"],
            "kernel": kernel_name,
            "algorithmic_flops_per_launch": BATCH * FLOPS_PER_SEQ,
            "note": "achieved = ALGORITHMIC flops (17.6 MFLOP/seq) / time against the measured dense bf16 peak, as the "
                    "contract asks. fp32 accuracy on the tensor pipe costs a 2-way operand split: 3 partial products + 1 bias "
                    "block = 7 FP16 MMAs (13 TF32 MMAs in round 1) per 128 x 256 x 32 product, so the kernel's own ceiling is "
                    "peak * 2 / 7; see mma below (executed MMA flops against the same peak). The pace is set by the serial "
                    "chain MMA -> TMEM read -> Runge-Kutta -> operand split of the two tiles TMEM can hold, not by the pipe "
                    "(profiles/README.md). traffic = dram bytes of one launch from the ncu capture in profiles/ "
                    "(algorithmic bytes: 1.63e9; whole 128-byte coefficient rows are fetched).",
            "mma": {"executed_mma_tflops": mma_flops / kernel_s / 1e12, "peak_tflops": mma_peak,
                    "frac": mma_flops / kernel_s / 1e12 / mma_peak, "mmas_per_tile_stage": mmas_per_stage,
                    "peak_source": "measured dense bf16 (kind::f16 rate)" if fp16_split else "measured dense bf16 / 2 (tf32 rate)"},
            "hbm": {"achieved_gbs": achieved_gbs, "peak_gbs": peaks["hbm_gbs"], "frac": achieved_gbs / peaks["hbm_gbs"],
                    "note": "the north_star's HBM framing: this solve is ~700 flop/B, compute bound by ~60x"},
            "secondary": secondary,
        } if tensor_kernel else {
            "bound": "hbm", "achieved": achieved_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved_gbs / peaks["hbm_gbs"], "traffic": 2176804000, "peak_source": peaks["source"],
            "kernel": "cdeint_simt_kernel<float,8,8>", "algorithmic_bytes_per_launch": BATCH * BYTES_PER_SEQ,
            "note": "this kernel is FP32-FMA bound (708 flop/B), not HBM bound; see fp32 below and DESIGN.md",
            "fp32": {"achieved_tflops": achieved_tf, "peak_tflops": fp32_peak_tf, "frac": achieved_tf / fp32_peak_tf,
                     "peak_source": "148 SMs x 128 FMA lanes x 2 x clocks.max.sm"},
            "secondary": secondary}),
        "config4": config4,
    }
    if world == 1:
        line["cpu_baseline"] = cpu_baseline()
    if dist is not None:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", type=int, default=None, help="solve kernel: 1 = CUDA-core, 2 = tcgen05 (default: the library's choice)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (rank 0) as DIR/cdeint_out.npy, float32")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the output of the CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
