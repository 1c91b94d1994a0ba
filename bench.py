#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 raster backend.

Metric (BASELINE.json): Mcells/s of slope + hillshade + focal.mean on a float32 DEM, with the
fraction of the HBM roofline, at 1/2/4/8 GPUs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--raster R] [--dump-outputs DIR]

N = 1   : 32768 x 32768 synthetic fBm-like DEM resident on the GPU (BASELINE configs[1]).
N > 1   : launched by torchrun, one rank per GPU; a 65536 x 65536 DEM (configs[4]) is row-striped
          over the ranks, every step exchanges the 1-row halos with NCCL send/recv and runs the
          three operators on the stripe (strong scaling: the raster is fixed, Mcells/s is
          size-normalised so it compares directly with the N = 1 line).
A step = slope, hillshade and focal.mean (one pass) each once over the whole raster:
3 * H * W cells.  Inputs are 4-16 GiB (>> the 126 MB L2), so no L2 flush is needed.

JSON line: value (device-resident throughput, CUDA events, max over ranks), e2e (same three
operators through the public API on numpy/pinned HOST rasters: H2D + kernels + D2H inside
the timed region), roofline of the dominant kernel, cpu_baseline (the CPU oracle, i.e. the
reference's algorithm restated in C, on the box's host cores over a bounded sample), clocks,
and
  parity_gate     N = 1: the three operators on a 2048^2 window vs the CPU oracle;
                  N > 1: every stripe boundary -- the rank above recomputes a 4096-row band that
                  straddles the boundary as ONE raster and compares it bit for bit with the two
                  stripes' outputs (the reference's numpy == dask invariant,
                  tests/general_checks.py:124-131) -- plus a striped zonal.stats(comm=WORLD) whose
                  counts must equal the closed form of the 32 x 32 block zones;
  ops             BASELINE.json configs 2-4 one operator at a time: aspect, curvature, the fused
                  suite, convolve_2d k = 3 / 9 / 25 (uniform and mixed weights), zonal.stats with
                  1024 zones (at N > 1 striped, AllReduce inside the timing), each with ms,
                  Mcells/s, fraction of the measured HBM peak and its own parity check;
  n1_same_raster  (N = 1) the 65536^2 raster of the N > 1 runs on ONE GPU, so the 1 -> 8 curve has
                  a same-raster anchor.

--impl reference times that CPU oracle instead (all host threads, bounded sample per step).

--dump-outputs DIR (N = 1) writes the slope, hillshade and mean rasters of the last timed step as
DIR/<name>.npy (float32), on a fixed, seeded grid of at most 2048 interior rows x 2048 interior
columns (48 MiB in all).  The edge rows and columns are NaN by design and are not written.  The DEM is
a pure function of its seed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "Mcells/s slope+hillshade+focal.mean f32"
RES = (30.0, 30.0)
ALG_BYTES_PER_CELL = 8.0  # 4 B read + 4 B written per cell for each 3x3 float32 operator


# ----------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons every 20 ms.  The process is started before the warm-up
    steps (its start-up takes longer than a short timed region); `mark()` is called when the timed
    region begins and `stop()` right after it ends, and only the rows printed in between are
    reported.  If the timed region is shorter than two samples, the warm-up rows (same kernels,
    same load) are included and `window` says so."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index
        self.i0 = 0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def wait_first(self, timeout=2.0):
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        self.i0 = len(self.rows)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        i1 = len(self.rows)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows, window = self.rows[self.i0:i1], "timed region"
        if len(rows) < 2:
            rows, window = self.rows[:max(i1, 1)], "warm-up + timed region (timed region shorter than two samples)"
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "window": window,
                "reasons": sorted(reasons)}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------- CPU arm
def cpu_steps(sample, threads, steps, warmup):
    """Time slope + hillshade + focal.mean of the oracle on `sample`; returns seconds per step."""
    import oracle
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        oracle.slope(sample, RES[0], RES[1], nthreads=threads)
        oracle.hillshade(sample, 225, 25, nthreads=threads)
        oracle.focal_mean(sample, nthreads=threads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return times


def host_threads():
    """All host cores this process may use (torchrun pins OMP_NUM_THREADS=1, so ask the OS)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def synth_sample(rows, cols):
    """The top-left rows x cols window of the benchmark DEM from the oracle's HOST twin of the
    generator (oracle/xrs_oracle.c xo_synth_terrain_f32: the same function of (seed, row, col) as
    csrc/synth.cu) -- the CPU arms never map the CUDA library."""
    import oracle
    z = oracle.synth_terrain(rows, cols, 0, 0, 1235, 0.0, 4000.0, nthreads=host_threads())
    return z, "top-left %d x %d window of the benchmark DEM (host generator, seed 1235)" % (rows, cols)


def run_reference_arm(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself is
    pure Python/Numba and cannot travel to the GPU box) on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    threads = host_threads()
    rows = cols = args.cpu_sample
    sample, sample_desc = synth_sample(rows, cols)
    times = cpu_steps(sample, threads, args.steps, args.warmup)
    dt = float(np.mean(times))
    value = 3.0 * rows * cols / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mcells/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "slope+hillshade+focal.mean on a float32 fBm-like DEM, res=(30,30): CPU oracle "
                               "(C restatement of the reference's Numba/NumPy kernels, which cannot travel to "
                               "this box), bounded sample per step",
                   "sample": sample_desc, "arithmetic": "Horn sums in f64 as Numba promotes them"},
        "cpu_baseline": {"value": value, "unit": "Mcells/s", "cores": threads, "kind": "port",
                         "sample": sample_desc + ", all three operators, OpenMP over rows"},
        "e2e": {"value": value, "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
def synth_into(t, row0, seed=1235, lo=0.0, hi=4000.0):
    import ctypes
    import torch
    from xrspatial_b200 import _lib
    _lib.call("xrs_synth_terrain_f32", ctypes.c_void_p(t.data_ptr()), t.stride(0) * 4, t.shape[0], t.shape[1], row0, 0,
              seed, lo, hi, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))


def block_zones(rows, W, row0, H, dev, n=32):
    """int32 zones of an n x n block grid over the GLOBAL H x W raster, rows [row0, row0 + rows)
    (mirrors benchmarks/benchmarks/zonal.py:44-48)."""
    import torch
    yy = (torch.arange(row0, row0 + rows, device=dev, dtype=torch.int64) // (H // n)).clamp_(max=n - 1)
    xx = (torch.arange(W, device=dev, dtype=torch.int64) // (W // n)).clamp_(max=n - 1)
    return (yy[:, None] * n + xx[None, :]).to(torch.int32).contiguous()


def event_times(fn, steps, warmup=3):
    """median / all CUDA-event times (ms) of `steps` calls of fn on the current stream."""
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    t = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    return float(np.median(t)), t


DUMP_SIDE = 2048   # sampled rows x columns per array: 3 float32 arrays of 2048^2 are 48 MiB


def dump_sample(n, side=DUMP_SIDE, seed=0):
    """Sorted indices of a fixed, seeded sample of at most `side` of the interior indices 1 .. n - 2.
    The first and last row and column are left out: the 3x3 operators make them NaN by design (the
    reference's raster-edge rule, which the test suite checks), and the dump holds finite values only."""
    inner = np.arange(1, n - 1)
    if len(inner) <= side:
        return inner
    return np.sort(np.random.default_rng(seed).choice(inner, side, replace=False))


def dump_outputs(out_dir, outs):
    """--dump-outputs: the arrays of the last timed step, as out_dir/<name>.npy, sampled on a fixed grid
    of interior rows x columns, the same for every run and build."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outs.items():
        rows = torch.from_numpy(dump_sample(t.shape[0])).to(t.device)
        cols = torch.from_numpy(dump_sample(t.shape[1])).to(t.device)
        a = t[rows[:, None], cols[None, :]].cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def rel_err(got, ref, rtol=1e-5, atol=1e-6, circular=False):
    """worst |got - ref| / (rtol |ref| + atol) with identical NaN masks (raises otherwise)."""
    g = np.asarray(got, dtype=np.float64)
    r = np.asarray(ref, dtype=np.float64)
    if not np.array_equal(np.isnan(g), np.isnan(r)):
        raise AssertionError("NaN masks differ")
    m = ~np.isnan(r)
    d = np.abs(g[m] - r[m])
    if circular:
        if not np.array_equal(g == -1, r == -1):
            raise AssertionError("flat (-1) masks differ")
        d = np.minimum(d, 360.0 - d)
    return float((d / (rtol * np.abs(r[m]) + atol)).max()) if m.any() else 0.0


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    import xrspatial_b200 as xb
    from xrspatial_b200 import _lib
    from xrspatial_b200.stripes import RowStripes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    side = args.raster or (32768 if n_gpus == 1 else 65536)
    H = W = side
    stripes = RowStripes(H, W, radius=1, device=dev)
    lib = _lib.lib()
    # synthetic DEM: pure function of (seed, global row, col) -> identical for any striping
    synth_into(stripes.interior, stripes.y0)
    torch.cuda.synchronize()

    attrs = {"res": RES}
    hp = stripes.buf.shape[0]
    agg = xb.DataArray(stripes.buf, dims=("y", "x"), attrs=attrs)
    outs = {}

    def step(events=None):
        stripes.exchange()
        if events is not None:
            events[0].record()
        outs["slope"] = xb.slope(agg).data
        if events is not None:
            events[1].record()
        outs["hillshade"] = xb.hillshade(agg).data
        if events is not None:
            events[2].record()
        outs["mean"] = xb.mean(agg).data
        if events is not None:
            events[3].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity = None
    if n_gpus == 1:
        if not args.skip_host:
            parity = run_parity_gate(xb, stripes, attrs)     # before any timing
    else:
        step()
        parity = run_stripe_parity_gate(xb, stripes, outs, attrs, dist, dev, step=step)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()           # before the warm-up: nvidia-smi needs ~0.1 s to print its first row
        sampler.wait_first()
    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    assert lib.xrs_debug_last_used_tma() == 1, "TMA kernels were not selected"

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    t_begin = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark()
    t_begin.record()
    for i in range(args.steps):
        step(ev[i])
    t_end.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs)
    total_ms = t_begin.elapsed_time(t_end)
    kt = np.array([[e[j].elapsed_time(e[j + 1]) for j in range(3)] for e in ev])  # ms per kernel
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        k = torch.tensor(kt.mean(0), dtype=torch.float64, device=dev)
        dist.all_reduce(k, op=dist.ReduceOp.MAX)
        kmean = k.cpu().numpy()
    else:
        kmean = kt.mean(0)
    ms_per_step = total_ms / args.steps
    cells_step = 3.0 * H * W
    value = cells_step / (ms_per_step * 1e-3) / 1e6

    # roofline of the dominant (slowest) kernel, per launch, algorithmic bytes only
    names = ["slope", "hillshade", "focal.mean"]
    dom = int(np.argmax(kmean))
    peak, peak_src = measured_peak_gbs()
    rows_launch = hp  # the kernel processes the padded stripe
    alg_bytes = ALG_BYTES_PER_CELL * rows_launch * W
    achieved = alg_bytes / (kmean[dom] * 1e-3) / 1e9
    # dram__bytes_read.sum + dram__bytes_write.sum per launch: STATIC, from the committed ncu --set full
    # capture of these kernels on a 32768 x 32768 launch (profiles/dram_traffic.json names the report),
    # scaled to the rows of this launch -- ncu cannot run inside a timed benchmark
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as f:
            tj = json.load(f)
        traffic = tj.get(names[dom])
        traffic_src = "static: " + str(tj.get("source", "committed ncu capture"))
        if traffic is not None:
            traffic = traffic * (float(rows_launch) * W) / (32768.0 * 32768.0)
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "per_kernel_ms": dict(zip(names, [float(x) for x in kmean])),
                "per_kernel_frac": dict(zip(names, [float(alg_bytes / (x * 1e-3) / 1e9 / peak) for x in kmean]))}

    del outs["slope"], outs["hillshade"], outs["mean"]
    torch.cuda.empty_cache()
    ops = None
    if not args.skip_ops:
        ops = run_ops_record(xb, stripes, attrs, args, peak, dist if world > 1 else None, dev)

    same = None
    e2e = None
    cpu = None
    if n_gpus == 1:
        if not args.skip_ops and not args.raster:
            same = run_same_raster_anchor(xb, args, dev)
        e2e = None if args.skip_host else run_e2e(xb, stripes, H, W, attrs, args)
        cpu = None if args.skip_host else run_cpu_baseline(stripes, args)
    elif not args.skip_host:
        e2e = run_e2e_striped(xb, stripes, attrs, args, dist, dev)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mcells/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "slope+hillshade+focal.mean on a %d x %d float32 fBm-like DEM, res=(30,30)%s"
                                   % (H, W, "" if n_gpus == 1 else ", row-striped over %d GPUs with 1-row NCCL "
                                      "halo exchange per step" % n_gpus),
                       "raster": [H, W], "cells_per_step": cells_step, "parallelism": "rows/%d" % n_gpus,
                       "arithmetic": "f32 in/out; Horn sums and focal sums in f64 like the reference's Numba kernels",
                       "l2": "inputs (%.1f GiB per GPU) are larger than L2, no flush" % (hp * W * 4 / 2 ** 30)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "parity_gate": parity,
            "ops": ops, "n1_same_raster": same,
            "gpu_launches": 3 * args.steps,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _stripe_boundary_mismatches(xb, stripes, outs, attrs, dist, dev, band):
    """One pass of the boundary check: per-operator counts of cells that differ (this rank's lower
    boundary), plus the number of halo cells that differ from the regenerated DEM rows."""
    import torch
    rank, world = stripes.rank, stripes.world
    W, h = stripes.W, stripes.h
    B = int(min(band, h - 1))
    own = {k: v[stripes.top:stripes.top + h] for k, v in outs.items()}       # the rows this rank owns
    names = ["slope", "hillshade", "mean"]
    send_in = stripes.interior[:B + 1].contiguous() if rank > 0 else None
    send_out = [own[k][:B].contiguous() for k in names] if rank > 0 else []
    recv_in = torch.empty((B + 1, W), dtype=torch.float32, device=dev) if rank < world - 1 else None
    recv_out = [torch.empty((B, W), dtype=torch.float32, device=dev) for _ in names] if rank < world - 1 else []
    reqs = []
    if rank > 0:
        for t in [send_in] + send_out:
            reqs.append(dist.P2POp(dist.isend, t, rank - 1))
    if rank < world - 1:
        for t in [recv_in] + recv_out:
            reqs.append(dist.P2POp(dist.irecv, t, rank + 1))
    for r in dist.batch_isend_irecv(reqs):
        r.wait()
    bad = [0, 0, 0, 0]                                # slope, hillshade, mean, halo cells
    # the halo rows of the stripe buffer against the generator (a pure function of the coordinates)
    for lo, n, y in ((0, stripes.top, stripes.y0 - stripes.top), (stripes.top + h, stripes.bot, stripes.y1)):
        if n:
            ref = torch.empty((n, W), dtype=torch.float32, device=dev)
            synth_into(ref, y)
            bad[3] += int((stripes.buf[lo:lo + n].view(torch.int32) != ref.view(torch.int32)).sum().item())
    if rank < world - 1:
        band_in = torch.cat([stripes.interior[h - B - 1:h], recv_in], dim=0)      # rows y1-B-1 .. y1+B
        bagg = xb.DataArray(band_in, dims=("y", "x"), attrs=attrs)
        for i, (k, fn) in enumerate(zip(names, (xb.slope, xb.hillshade, xb.mean))):
            got = fn(bagg).data[1:2 * B + 1]
            exp = torch.cat([own[k][h - B:h], recv_out[i]], dim=0)
            bad[i] = int((got.view(torch.int32) != exp.view(torch.int32)).sum().item())
        del band_in
    t = torch.tensor(bad, dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return [int(x) for x in t.tolist()], B


def run_stripe_parity_gate(xb, stripes, outs, attrs, dist, dev, band=2048, step=None):
    """N > 1, before timing.  For every stripe boundary (rank r | r + 1) rank r receives the first
    `band` + 1 input rows and the first `band` output rows of rank r + 1, recomputes the band of
    2 x `band` rows around the boundary as ONE raster on its own GPU and compares it BIT FOR BIT with
    the two stripes' outputs of the benchmark step: the partition-invariance the reference asserts
    between its numpy and dask backends (tests/general_checks.py:124-131).  The halo rows are also
    compared with the regenerated DEM rows.  Then a striped zonal.stats(comm=WORLD) over 32 x 32 block
    zones, whose counts have a closed form.

    The gate never suppresses the bench line: a mismatch is counted per operator, the step is run and
    checked once more (`retried`), and the record says `ok: false` if the second pass differs too."""
    import sys
    world = stripes.world
    names = ["slope", "hillshade", "focal.mean", "halo_rows"]
    first, B = _stripe_boundary_mismatches(xb, stripes, outs, attrs, dist, dev, band)
    final, retried = first, False
    if any(first) and step is not None:
        retried = True
        step()
        final, B = _stripe_boundary_mismatches(xb, stripes, outs, attrs, dist, dev, band)
    ok = not any(final)
    if any(first) and stripes.rank == 0:
        sys.stderr.write("parity gate: cells differing at the stripe boundaries (all ranks) first pass %r, "
                         "after re-running the step %r\n" % (dict(zip(names, first)), dict(zip(names, final))))
    # striped zonal.stats: exact integer counts, zone ids 0..1023
    zones = block_zones(stripes.h, stripes.W, stripes.y0, stripes.H, dev)
    df = xb.zonal_stats(xb.DataArray(zones, dims=("y", "x")), xb.DataArray(stripes.interior, dims=("y", "x")),
                        stats_funcs=["count", "min", "max", "mean"], comm=dist.group.WORLD)
    cells = (stripes.H // 32) * (stripes.W // 32)
    zonal_ok = bool(np.array_equal(np.asarray(df["zone"]), np.arange(1024)) and
                    np.array_equal(np.asarray(df["count"]), np.full(1024, float(cells))))
    if not zonal_ok and stripes.rank == 0:
        sys.stderr.write("parity gate: striped zonal.stats counts differ from the closed form\n")
    return {"checked": True, "ok": bool(ok and zonal_ok),
            "kind": "stripe boundaries recomputed as one raster, bit-exact; halo rows == generator; striped "
                    "zonal.stats counts == closed form (general_checks.py:124-131)",
            "boundaries": world - 1, "band_rows": 2 * B, "operators": ["slope", "hillshade", "focal.mean"],
            "mismatching_cells": dict(zip(names, final)),
            "retried": retried, "mismatching_cells_first_pass": dict(zip(names, first)) if retried else None,
            "zonal_counts_exact": zonal_ok, "zones": 1024, "cells_per_zone": cells}


def run_ops_record(xb, stripes, attrs, args, peak, dist, dev):
    """BASELINE.json configs 2-4, one operator at a time on the benchmark raster (this rank's stripe):
    CUDA-event median of `--steps` launches + a parity check of each operator on a 1024^2 window
    against the CPU oracle (N = 1).  At N > 1 only the striped zonal.stats (AllReduce included, wall
    clock between barriers, max over ranks) is recorded -- the stencil kernels are the same binaries."""
    import torch
    import oracle
    from xrspatial_b200.convolution import convolve_2d
    rows = []
    W, h = stripes.W, stripes.h
    world = stripes.world
    steps = max(3, min(args.steps, 10))

    def add(name, ms, bpc, cells, parity=None, note=None):
        gbs = cells * bpc / (ms * 1e-3) / 1e9
        r = {"op": name, "ms": ms, "mcells_s": cells / (ms * 1e-3) / 1e6, "alg_bytes_per_cell": bpc,
             "gbs": gbs, "frac": gbs / peak, "parity": parity}
        if note:
            r["note"] = note
        rows.append(r)

    zones = block_zones(h, W, stripes.y0, stripes.H, dev)
    zagg = xb.DataArray(zones, dims=("y", "x"))
    vagg = xb.DataArray(stripes.interior, dims=("y", "x"))
    stats7 = ["mean", "max", "min", "sum", "std", "var", "count"]
    cells_zone = (stripes.H // 32) * (W // 32)

    def zonal_wall(fn, n):
        ts = []
        for i in range(n + 1):
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            df = fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if dist is not None:
                tt = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt.item())
            if i:
                ts.append(dt * 1e3)
        return float(np.median(ts)), df

    comm = dist.group.WORLD if dist is not None else None
    ms, df = zonal_wall(lambda: xb.zonal_stats(zagg, vagg, stats_funcs=stats7, comm=comm), steps)
    exact = bool(np.array_equal(np.asarray(df["count"]), np.full(1024, float(cells_zone))) and
                 np.array_equal(np.asarray(df["zone"]), np.arange(1024)))
    if not exact:
        raise AssertionError("zonal.stats counts differ from the closed form")
    add("zonal.stats 1024 block zones, 7 statistics%s" % ("" if world == 1 else " (striped, AllReduce inside)"),
        ms, 8, float(stripes.H) * W, {"counts_exact": exact, "zones": 1024},
        "whole public call incl. zone discovery, host finalisation%s; wall clock%s"
        % ("" if world == 1 else ", id all-gather + 5 AllReduce", "" if world == 1 else ", max over ranks"))
    if world > 1:
        return rows

    # ---- single GPU: the stencil operators of configs 2 and 3
    agg = xb.DataArray(stripes.interior, dims=("y", "x"), attrs=attrs)
    n = 1024
    win = stripes.interior[:n, :n].contiguous()
    hwin = win.cpu().numpy()
    wagg = xb.DataArray(win, dims=("y", "x"), attrs=attrs)
    th = host_threads()
    cells = float(h) * W

    def par(got, ref, **kw):
        e = rel_err(got.cpu().numpy(), ref, **kw)
        if e > 1.0:
            raise AssertionError("ops parity: %.3g x outside the tolerance" % e)
        return {"ok": True, "worst_err_over_tol": e, "window": [n, n]}

    add("slope", event_times(lambda: xb.slope(agg), steps)[0], 8, cells,
        par(xb.slope(wagg).data, oracle.slope(hwin, RES[0], RES[1], nthreads=th)))
    add("aspect", event_times(lambda: xb.aspect(agg), steps)[0], 8, cells,
        par(xb.aspect(wagg).data, oracle.aspect(hwin, nthreads=th), rtol=1e-5, atol=1e-4, circular=True))
    add("hillshade", event_times(lambda: xb.hillshade(agg), steps)[0], 8, cells,
        par(xb.hillshade(wagg).data, oracle.hillshade(hwin, 225, 25, nthreads=th)))
    cref = oracle.curvature(hwin, 30.0, nthreads=th)
    add("curvature", event_times(lambda: xb.curvature(agg), steps)[0], 8, cells,
        par(xb.curvature(wagg).data, cref, atol=1e-6 * float(np.nanmax(np.abs(cref)))))
    add("focal.mean", event_times(lambda: xb.mean(agg), steps)[0], 8, cells,
        par(xb.mean(wagg).data, oracle.focal_mean(hwin, nthreads=th)))
    suite = xb.surface_suite(wagg)
    e = max(rel_err(suite["slope"].data.cpu().numpy(), oracle.slope(hwin, RES[0], RES[1], nthreads=th)),
            rel_err(suite["aspect"].data.cpu().numpy(), oracle.aspect(hwin, nthreads=th), atol=1e-4, circular=True),
            rel_err(suite["hillshade"].data.cpu().numpy(), oracle.hillshade(hwin, 225, 25, nthreads=th)),
            rel_err(suite["curvature"].data.cpu().numpy(), cref, atol=1e-6 * float(np.nanmax(np.abs(cref)))))
    if e > 1.0:
        raise AssertionError("ops parity: suite %.3g x outside the tolerance" % e)
    add("surface suite: slope+aspect+curvature+hillshade fused (one read)", event_times(lambda: xb.surface_suite(agg), steps)[0],
        20, cells, {"ok": True, "worst_err_over_tol": e, "window": [n, n]}, "configs[1] as one kernel: 4 B read + 16 B written per cell")
    krng = np.random.default_rng(7)
    for k in (3, 9, 25):
        for kind in ("uniform", "mixed"):
            kern = np.ones((k, k)) / (k * k) if kind == "uniform" else krng.standard_normal((k, k))
            ref = oracle.convolve_2d(hwin, kern, nthreads=th)
            p = par(convolve_2d(win, kern), ref, atol=1e-6 * float(np.nanmax(np.abs(ref))))
            # mixed k = 25 is bound by the FP64 FMA rate (1250 flop / cell): a quarter of the rows keeps it short
            sub = stripes.interior if not (k == 25 and kind == "mixed") else stripes.interior[: h // 4]
            add("convolve_2d k=%d %s" % (k, kind), event_times(lambda: convolve_2d(sub, kern), max(3, steps // 2))[0], 8,
                float(sub.shape[0]) * W, p,
                "f64 accumulation like the reference; bound: HBM (k=3, uniform) or the FP64 FMA rate (mixed k>=9)")
    # the reference's own focal benchmark (benchmarks/benchmarks/focal.py FocalApply): apply(agg, np.ones((k, k)))
    from xrspatial_b200 import focal as xfocal
    for k in (5, 25):
        kern = np.ones((k, k))
        p = par(xfocal.apply(wagg, kern).data, oracle.focal_apply(hwin, kern, "mean", nthreads=th))
        add("focal.apply mean, np.ones((%d, %d))" % (k, k), event_times(lambda: xfocal.apply(agg, kern), max(3, steps // 2))[0],
            8, cells, p, "running box in NaN-skipping mode (clamped windows at the raster's edges)")
    # config 4 with the reference's default list (incl. majority) on a categorical raster
    cats = (stripes.interior * (16.0 / 4000.0)).floor_().clamp_(0, 15)
    cagg = xb.DataArray(cats, dims=("y", "x"))
    ms, df = zonal_wall(lambda: xb.zonal_stats(zagg, cagg), 3)
    add("zonal.stats 1024 block zones, default list incl. majority (16-class values)", ms, 8, cells,
        {"counts_exact": bool(np.array_equal(np.asarray(df["count"]), np.full(1024, float(cells_zone))))},
        "two passes: partials + (zone, value) pair histogram; wall clock")
    del cats
    return rows


def run_same_raster_anchor(xb, args, dev, side=65536):
    """N = 1 only: the same step on the 65536^2 raster of the N > 1 runs (16 GiB in, 3 x 16 GiB out), so
    the driver's 1 -> 8 curve can be anchored on one raster."""
    import torch
    try:
        free = torch.cuda.mem_get_info(dev)[0]
        if free < 70 * 2 ** 30:
            return {"skipped": "only %.0f GiB free" % (free / 2 ** 30)}
        big = torch.empty((side, side), dtype=torch.float32, device=dev)
        synth_into(big, 0)
        agg = xb.DataArray(big, dims=("y", "x"), attrs={"res": RES})

        def step():
            xb.slope(agg)
            xb.hillshade(agg)
            xb.mean(agg)
        steps = max(3, min(args.steps, 10))
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            step()
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / steps
        del big, agg
        torch.cuda.empty_cache()
        return {"raster": [side, side], "steps": steps, "ms_per_step": ms,
                "value": 3.0 * side * side / (ms * 1e-3) / 1e6, "unit": "Mcells/s"}
    except Exception as exc:  # an anchor must never take the headline down
        return {"skipped": "%s: %s" % (type(exc).__name__, exc)}


def run_e2e_striped(xb, stripes, attrs, args, dist, dev, max_rows=8192):
    """N > 1: the same three operators through the public API on HOST rasters, every rank feeding its own
    GPU over its own PCIe link from its own pinned stripe (rows of the benchmark DEM incl. one halo row per
    neighbour, so the stitched result is the single-raster result).  Bounded to `max_rows` rows per rank
    (10 GiB of pinned host memory per rank); wall clock between barriers, max over ranks."""
    import torch
    from xrspatial_b200 import _hostmem
    _hostmem.MAX_CACHED_BYTES = max(_hostmem.MAX_CACHED_BYTES, 24 << 30)   # keep the result blocks between steps
    W = stripes.W
    rows = int(min(stripes.h, max_rows))
    top, bot = stripes.top, stripes.bot
    try:
        z = _hostmem.empty((top + rows + bot, W), np.float32)
    except Exception as exc:
        z = None
        err = "%s: %s" % (type(exc).__name__, exc)
    ok = torch.tensor([1 if z is not None else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) == 0:
        return {"value": None, "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "could not allocate pinned host memory on every rank"} if stripes.rank == 0 else None
    # the first `rows` owned rows of the stripe plus their halos (the lower halo row is an owned row when the
    # sample is shorter than the stripe)
    torch.from_numpy(z).copy_(stripes.buf[0:top + rows + bot])
    torch.cuda.synchronize()
    hagg = xb.DataArray(z, dims=("y", "x"), attrs=attrs)

    def one():
        a = xb.slope(hagg).data
        b = xb.hillshade(hagg).data
        c = xb.mean(hagg).data
        return a[top:top + rows], b[top:top + rows], c[top:top + rows]

    res = one()
    assert isinstance(res[0], np.ndarray) and res[2].dtype == np.float64
    del res
    steps = max(1, min(args.steps, args.e2e_steps))
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = one()
        del res
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item()) / steps
    world = stripes.world
    cells = 3.0 * rows * W * world
    hp = top + rows + bot
    if stripes.rank != 0:
        return None
    return {"value": cells / dt / 1e6, "unit": "Mcells/s", "steps": steps, "ms_per_step": dt * 1e3,
            "h2d_bytes_per_step": int(3 * hp * W * 4) * world, "d2h_bytes_per_step": int(hp * W * (4 + 4 + 8)) * world,
            "raster": [rows * world, W], "links": world,
            "api": "xrspatial_b200.slope/hillshade/mean on numpy DataArrays in pinned host memory, one process and "
                   "one PCIe link per GPU (%d rows + halo per rank); wall clock, max over ranks" % rows}


def run_e2e(xb, stripes, H, W, attrs, args):
    """Same three operators through the public API on HOST (pinned) rasters."""
    import torch
    from xrspatial_b200 import _hostmem
    _hostmem.MAX_CACHED_BYTES = max(_hostmem.MAX_CACHED_BYTES, 40 << 30)   # keep the result blocks between steps
    # N = 1 means ONE GPU and one PCIe link, whatever else the box exposes (the numpy runners would
    # otherwise stripe over every visible GPU)
    os.environ["XRS_B200_DEVICES"] = str(torch.cuda.current_device())
    steps = max(1, min(args.steps, args.e2e_steps))
    eh = H
    z = None
    while eh >= 1024:
        try:
            z = _hostmem.empty((eh, W), np.float32)
            break
        except Exception:
            eh //= 2
    if z is None:
        return {"value": None, "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "could not allocate pinned host memory"}
    torch.from_numpy(z).copy_(stripes.interior[:eh])
    torch.cuda.synchronize()
    hagg = xb.DataArray(z, dims=("y", "x"), attrs=attrs)

    def one():
        a = xb.slope(hagg).data
        b = xb.hillshade(hagg).data
        c = xb.mean(hagg).data
        return a, b, c

    res = one()  # warm-up: allocates the pinned result blocks and the device slots
    assert isinstance(res[0], np.ndarray) and res[2].dtype == np.float64
    del res
    t0 = time.perf_counter()
    for _ in range(steps):
        res = one()
        del res
    dt = (time.perf_counter() - t0) / steps
    cells = 3.0 * eh * W
    return {"value": cells / dt / 1e6, "unit": "Mcells/s", "steps": steps, "ms_per_step": dt * 1e3,
            "h2d_bytes_per_step": int(3 * eh * W * 4), "d2h_bytes_per_step": int(eh * W * (4 + 4 + 8)),
            "raster": [eh, W],
            "api": "xrspatial_b200.slope/hillshade/mean on numpy DataArrays in pinned host memory "
                   "(xrs_host_stencil: chunked H2D -> kernel -> D2H pipeline); focal.mean returns float64 "
                   "like the reference's numpy path"}


def run_parity_gate(xb, stripes, attrs, n=2048):
    """SURVEY.md 8d: parity gate before timing -- the three benchmark operators on the top-left
    n x n window of the benchmark DEM against the CPU oracle (|gpu - ref| <= 1e-5 |ref| + 1e-6,
    identical NaN masks)."""
    import oracle
    oracle.build()
    n = int(min(n, stripes.h, stripes.W))
    win = stripes.interior[:n, :n].contiguous()
    host = win.cpu().numpy()
    agg = xb.DataArray(win, dims=("y", "x"), attrs=attrs)
    threads = host_threads()
    worst = 0.0
    for name, got, ref in (
            ("slope", xb.slope(agg).data, oracle.slope(host, RES[0], RES[1], nthreads=threads)),
            ("hillshade", xb.hillshade(agg).data, oracle.hillshade(host, 225, 25, nthreads=threads)),
            ("focal.mean", xb.mean(agg).data, oracle.focal_mean(host, nthreads=threads))):
        g = got.cpu().numpy().astype(np.float64)
        r = np.asarray(ref, dtype=np.float64)
        if not np.array_equal(np.isnan(g), np.isnan(r)):
            raise AssertionError("parity gate: NaN mask of %s differs from the oracle" % name)
        m = ~np.isnan(r)
        e = float((np.abs(g[m] - r[m]) / (1e-5 * np.abs(r[m]) + 1e-6)).max())
        if e > 1.0:
            raise AssertionError("parity gate: %s is %.3g x outside the tolerance" % (name, e))
        worst = max(worst, e)
    return {"checked": True, "window": [n, n], "operators": ["slope", "hillshade", "focal.mean"],
            "tolerance": "|gpu-ref| <= 1e-5*|ref| + 1e-6, NaN masks identical", "worst_err_over_tol": worst}


def run_cpu_baseline(stripes, args):
    import oracle
    oracle.build()
    n = min(args.cpu_sample, stripes.h, stripes.W)
    sample = stripes.interior[:n, :n].contiguous().cpu().numpy()
    threads = host_threads()
    t_all = float(np.mean(cpu_steps(sample, threads, 2, 1)))
    t_one = float(np.mean(cpu_steps(sample[: max(256, n // 4)], 1, 1, 1)))
    cells = 3.0 * n * n
    return {"value": cells / t_all / 1e6, "unit": "Mcells/s", "cores": threads, "kind": "port",
            "sample": "top-left %d x %d window of the benchmark DEM, slope+hillshade+focal.mean" % (n, n),
            "single_thread_value": 3.0 * max(256, n // 4) * n / t_one / 1e6,
            "note": "oracle/xrs_oracle.c (C restatement of the reference's Numba/NumPy kernels); "
                    "single_thread_value is what a stock numpy-backed xrspatial call does (ngjit is serial)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--raster", type=int, default=0, help="raster side (default 32768 at N=1, 65536 at N>1)")
    ap.add_argument("--cpu-sample", type=int, default=8192, help="side of the CPU-arm sample window")
    ap.add_argument("--e2e-steps", type=int, default=20, help="upper bound; the e2e leg runs min(--steps, this)")
    ap.add_argument("--skip-ops", action="store_true",
                    help="profiling runs only: skip the per-operator record and the 65536^2 anchor")
    ap.add_argument("--skip-host", action="store_true",
                    help="profiling runs only: skip the e2e (host-buffer) and CPU-baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy, sampled on a fixed, seeded "
                         "grid of at most %d interior rows x columns (the NaN edge rows and columns are left out)"
                         % DUMP_SIDE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs is supported on the single-GPU run only")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
