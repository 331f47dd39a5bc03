#!/usr/bin/env python
"""bench.py -- grid-cell-timesteps/s on the fused PV convert+aggregate path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload = the BASELINE.json north star: synthetic ERA5 1440 x 720 x 8760
(global 0.25 deg, one year hourly), cutout.pv(panel="CSi",
orientation="latitude_optimal") aggregated to 3000 NUTS-like shapes.  One
"step" = one full pass of the hot path over that cutout: 9.08e9
cell-timesteps, 181.6 GB (169.2 GiB) of float32 input, all of it resident in
HBM.  Inputs may take at most 80 % of the device memory (a full device stops
answering the box's health checks), so at N = 1 the year is processed as TWO
resident half-years one after the other -- each timed over its own `--steps`
passes with its own warm-up -- and the two times are summed (`config.parts`;
one launch per part through the operator's `t0` slab argument).

N > 1 (torchrun, one rank per GPU) is STRONG scaling: the same cutout, its
time axis sharded T/N per rank (atlite_b200.dist.shard_bounds; the synthetic
generator is seeded per absolute time block, so the shards ARE the single-GPU
cutout), and every step ends with the NCCL all-gather that re-assembles the
(time, bus) result on every rank.

`value`   : device-resident inputs, CUDA-event timed (memset + fused kernel + result gather).
`e2e`     : the public API (Cutout.pv) on HOST (pinned) arrays -- H2D streaming,
            kernels, D2H of the result inside the timed region; each rank streams
            a bounded slab (<= 1095 steps = the 1/8-year shard) of its own shard.
`roofline`: algorithmic bytes (20 B / cell-timestep, SURVEY.md section 8d) / the
            fused kernel's CUDA-event time, against MEASURED_PEAKS.json.
`cpu_baseline`: the NumPy oracle (restatement of the reference) on this box's
            cores (process pool), bounded sample, rank 0 at N = 1 only.
`extra`   : BASELINE configs[2] (wind) and configs[3] (heat demand) on the same
            grid and shards, same protocol (strong scaling at N > 1); at N = 1
            also configs[1], the non-default PV variants, config 4, the indicator matrix.

`--steps K` is the number of timed passes of the headline, of `e2e` and of the wind /
heat entries of `extra`; `--warmup W` untimed passes precede those of the headline and
of wind / heat.  `--dump-outputs DIR` then writes the (time, bus) results of the last
timed pass of the headline (`pv`) and of wind and heat demand as float32
`DIR/<name>.npy`, with the time steps they hold in `DIR/<name>_time_index.npy`, 64 MB
in all (see `dump_outputs`).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NX, NY, NT, NBUS = 1440, 720, 8760, 3000
X0, Y0 = -180.0, -90.0
PANEL, ORIENT, TURBINE = "CSi", "latitude_optimal", "Vestas_V112_3MW"
BYTES_PER_CELL_TS = 20.0  # 5 float32 fields (SURVEY.md section 8d)
E2E_MAX_STEPS = 1095  # host-streamed slab per rank (22.7 GB of pinned host memory)
VRAM_FRACTION = 0.80  # share of the device memory the resident inputs may take
DUMP_BYTES = 64_000_000  # --dump-outputs: every file together, headers included
DUMP_SEED = 0
WORKLOAD = (f"synthetic ERA5 {NX}x{NY}x{NT}, cutout.pv(panel=CSi, orientation=latitude_optimal) "
            f"-> {NBUS} shapes (BASELINE.json north star)")
METRIC = "grid-cell-timesteps/s on PV convert+aggregate"


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML, every
    ~2 ms; nvidia-smi -lms 200 is too coarse for millisecond steps)."""

    def __init__(self, index=0):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self.max_mhz = None

    def _run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            while not self._stop.is_set():
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((float(sm), int(rs)))
                self._stop.wait(0.002)
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)

    def __enter__(self):
        self._t.start()
        time.sleep(0.05)
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=10)

    def summary(self):
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                "sw_thermal_slowdown": 0x20}
        sm = [r[0] for r in self.rows]
        reasons = sorted({n for _, rs in self.rows for n, b in bits.items() if rs & b})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(sm), **({"error": self.error} if hasattr(self, "error") else {})}


# ----------------------------------------------------------------------------
# reference arm / cpu baseline: the NumPy oracle on host cores (process pool)
# ----------------------------------------------------------------------------


def _cpu_worker(wid, chunk_steps, barrier, results, n_rounds):
    """One host core of the CPU arm: builds its own chunk of the north-star cutout
    (`chunk_steps` hourly steps of 1440 x 720, daytime somewhere on the globe at every
    step), then, `n_rounds` times, waits at the barrier and runs the reference
    restatement (convert_pv + aggregate_matrix) on it -- the unit of work of the
    reference's dask graph (one time chunk through the whole ufunc chain and the
    sparse product, convert.py:198 + aggregate.py:24-32)."""
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    os.environ.setdefault("MKL_NUM_THREADS", "1")
    warnings.simplefilter("ignore")
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import atlite_oracle as O

    import atlite_b200 as ab
    from atlite_b200 import synthetic as syn

    ds = syn.make_dataset(NX, NY, chunk_steps, X0, Y0, kinds=("pv",), t_offset=24 * 150 + wid * chunk_steps)
    d = {k: np.asarray(ds.raw(k)) for k in ds.keys()}
    d.update(time=ds.coords["time"], lon=ds.coords["lon"], lat=ds.coords["lat"])
    m = syn.make_shapes(NX, NY, NBUS)
    panel, orient = ab.get_solarpanelconfig(PANEL), O.get_orientation(ORIENT)
    for _ in range(n_rounds):
        barrier.wait()
        t0 = time.perf_counter()
        res = O.aggregate_matrix(O.convert_pv(d, panel, orient), m)
        dt = time.perf_counter() - t0
        assert res.shape == (chunk_steps, NBUS)
        results.put((wid, dt))
        barrier.wait()


class CpuArm:
    """`workers` single-threaded processes, each holding one time chunk; a round = all
    of them convert+aggregate their chunk concurrently (wall clock of the slowest)."""

    def __init__(self, workers, chunk_steps, n_rounds):
        import multiprocessing as mp

        ctx = mp.get_context("spawn")  # never fork a process that holds a CUDA context
        self.workers, self.chunk_steps = workers, chunk_steps
        self.barrier = ctx.Barrier(workers + 1)
        self.results = ctx.Queue()
        self.procs = [ctx.Process(target=_cpu_worker, args=(w, chunk_steps, self.barrier, self.results, n_rounds),
                                  daemon=True) for w in range(workers)]
        for p in self.procs:
            p.start()

    def round(self):
        """Returns (wall seconds, per-worker seconds)."""
        self.barrier.wait(timeout=600)  # every worker has its data and is ready
        t0 = time.perf_counter()
        self.barrier.wait(timeout=1800)  # every worker is done
        wall = time.perf_counter() - t0
        per = [self.results.get(timeout=60)[1] for _ in range(self.workers)]
        return wall, per

    def close(self):
        for p in self.procs:
            p.join(timeout=30)
            if p.is_alive():
                p.kill()  # the exact processes this object started


def _host_limits():
    """(usable cores, usable bytes of RAM) of THIS container: the scheduler affinity mask and
    the cgroup CPU quota / memory limit when there are any, not the bare host's numbers -- a
    process pool sized for the host inside a smaller cgroup takes the whole box down."""
    import psutil

    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        cores = os.cpu_count() or 1
    avail = psutil.virtual_memory().available
    try:  # cgroup v2
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            cores = max(1, min(cores, int(float(quota) / float(period))))
    except Exception:  # noqa: BLE001
        pass
    for lim_f, use_f in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                         ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            with open(lim_f) as fh:
                lim = fh.read().strip()
            with open(use_f) as fh:
                use = int(fh.read().strip())
            if lim != "max" and int(lim) < (1 << 60):
                avail = min(avail, max(0, int(lim) - use))
            break
        except Exception:  # noqa: BLE001
            continue
    return cores, avail


def _cpu_plan(target_s):
    """Workers and chunk length of the CPU arm.  The reference computes in dask chunks of
    {"time": 100} (cutout.py:143) -- 4.0e6 elements per array at the 200 x 200 config.  On the
    1440 x 720 grid one step already is 1.04e6 cells, so the chunk is bounded by the time
    target and by host memory instead (never below 4 steps = 4.1e6 elements per array, the
    element count of the reference's own chunks at configs[1]).  A worker needs ~0.35 GB
    (interpreter, NumPy / SciPy / pandas, the 3000-shape matrix) plus ~0.12 GB per step of its
    chunk (inputs + the float64 temporaries alive at once; measured: 0.61 GB peak for 4 steps);
    the pool is sized to stay below a QUARTER of the memory this container may use."""
    cores, avail = _host_limits()
    budget = 0.25 * avail
    rate_guess = 3.0e6  # cell-ts/s/core with every core busy (3.6e6 measured on the 8-core build box)
    chunk = int(np.clip(target_s * rate_guess / (NX * NY), 4, 100))
    workers = cores
    while workers > 1 and workers * (0.35e9 + 0.12e9 * chunk) > budget:
        if chunk > 4:
            chunk = max(4, chunk // 2)
        else:
            workers = max(1, workers * 3 // 4)
    return workers, chunk


def cpu_measure(rounds, warmup, target_s=12.0):
    cores, chunk = _cpu_plan(target_s)  # cores = worker processes actually used
    arm = CpuArm(cores, chunk, rounds + warmup)
    try:
        for _ in range(warmup):
            arm.round()
        walls, pers = [], []
        for _ in range(rounds):
            w, per = arm.round()
            walls.append(w)
            pers.append(per)
    finally:
        arm.close()
    cell_ts = float(NX) * NY * chunk * cores
    per = np.asarray(pers)
    return {"walls": walls, "cell_ts_per_round": cell_ts, "cores": cores, "chunk_steps": chunk,
            "per_core_rate_under_load": float(NX * NY * chunk / per.mean()),
            "slowest_worker_s": float(per.max()), "fastest_worker_s": float(per.min())}


def cpu_baseline():
    warnings.simplefilter("ignore")
    r = cpu_measure(rounds=1, warmup=0)
    value = r["cell_ts_per_round"] / r["walls"][0]
    return {"value": value, "unit": "grid-cell-timesteps/s", "cores": r["cores"], "kind": "port",
            "per_core_rate_under_load": r["per_core_rate_under_load"],
            "efficiency_vs_cores_x_per_core_rate": value / (r["cores"] * r["per_core_rate_under_load"]),
            "sample": f"NumPy float64 oracle (restatement of the reference; xarray/dask absent), {r['cores']} "
                      f"single-threaded worker processes x one {r['chunk_steps']}-step chunk of the {NX}x{NY} cutout -> "
                      f"{NBUS} shapes ({r['cores'] * r['chunk_steps']} of {NT} steps), wall {r['walls'][0]:.1f} s "
                      f"(workers {r['fastest_worker_s']:.1f}-{r['slowest_worker_s']:.1f} s)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warnings.simplefilter("ignore")
    r = cpu_measure(rounds=args.steps, warmup=args.warmup, target_s=8.0)
    total = float(sum(r["walls"]))
    value = r["cell_ts_per_round"] * args.steps / total
    nsteps = r["cores"] * r["chunk_steps"]
    line = {
        "impl": "reference", "metric": METRIC,
        "value": value, "unit": "grid-cell-timesteps/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "sample": f"each step = {nsteps} of the {NT} time steps ({r['cores']} worker processes x one "
                             f"{r['chunk_steps']}-step chunk each)"},
        "cpu_baseline": {"value": value, "unit": "grid-cell-timesteps/s", "cores": r["cores"], "kind": "port",
                         "per_core_rate_under_load": r["per_core_rate_under_load"],
                         "sample": f"NumPy float64 oracle port of the reference CPU path (the reference itself needs "
                                   f"xarray/dask, absent here), {nsteps} of {NT} steps per step, process pool"},
        "e2e": {"value": value, "unit": "grid-cell-timesteps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------


def _timeit(torch, fn, n, warm=2):
    """Median and mean CUDA-event time (ms) of fn() on the current stream."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    ts = [a.elapsed_time(b) for a, b in ev]
    return float(np.median(ts)), float(np.mean(ts))


class Comm:
    """Rank plumbing of one bench process (torch.distributed over NCCL at N > 1)."""

    def __init__(self, torch, dist):
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa_bound = self._bind_to_gpu_node()
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def _bind_to_gpu_node(self):
        """One process per GPU: run this rank (its pinned allocations, its staging threads) on the
        CPUs next to its GPU, as `numactl --cpunodebind` would -- on a two-socket box half of the
        ranks otherwise stream their host slabs across the inter-socket link."""
        if self.world == 1:
            return False
        try:
            from atlite_b200 import _lib

            cpus = set(_lib.device_local_cpus(self.local_rank)) & set(os.sched_getaffinity(0))
            if cpus:
                os.sched_setaffinity(0, cpus)
                return True
        except Exception:  # noqa: BLE001
            pass
        return False

    def sync(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_scalars(self, x):
        if self.world == 1:
            return [float(x)]
        parts = [self.torch.zeros(1, dtype=self.torch.float64, device=self.dev) for _ in range(self.world)]
        self.dist.all_gather(parts, self.torch.tensor([x], dtype=self.torch.float64, device=self.dev))
        return [float(p.item()) for p in parts]


def measure_sharded(comm, shard, reduce_local, units_local, counts, steps, warmup, clock=None):
    """The timed region of one operator on this rank's shard: `steps` passes of
    memset + fused kernel, each followed (N > 1) by the all-gather of the (time, bus)
    result, issued asynchronously so the next pass overlaps the NVLink transfer; all
    gathers complete inside the region.  Returns step ms (max over ranks), kernel ms per
    rank (separate passes without the gather), the gather alone, and the last results."""
    torch = comm.torch
    pending = []

    def step():
        out = reduce_local()
        if shard is not None:
            full, work = shard.gather_time(out, counts=counts, async_op=True)
            if work is None:  # ragged shards: synchronous path
                return out, full
            pending.append(work)
            return out, full
        return out, out

    def drain():
        for w in pending:
            w.wait()  # the current stream waits for the gathers: the closing event covers them
        pending.clear()

    for _ in range(warmup):
        step()
    drain()
    comm.sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx = clock if clock is not None else _Null()
    with ctx:
        comm.sync()
        ev0.record()
        for _ in range(steps):
            local, full = step()
        drain()
        ev1.record()
        comm.sync()
        ms_total = ev0.elapsed_time(ev1)
        _, kern_ms = _timeit(torch, reduce_local, steps, warm=0)
    gather_ms = None
    if shard is not None:
        def g():
            o, w = shard.gather_time(local, counts=counts, async_op=True)
            if w is not None:
                w.wait()
        comm.sync()
        gather_ms, _ = _timeit(torch, g, 5, warm=1)
        gather_ms = comm.max(gather_ms)
    ms_step = comm.max(ms_total) / steps
    return {"ms_per_step": ms_step, "kernel_ms": kern_ms, "kernel_ms_per_rank": comm.gather_scalars(kern_ms),
            "gather_ms": gather_ms, "local": local, "full": full, "units_local": units_local}


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def check_gather(comm, res, lo, hi):
    """N > 1: the gathered (time, bus) tensor must hold this rank's local result in its
    rows, bit for bit, on every rank (and be finite)."""
    torch = comm.torch
    ok = bool(torch.equal(res["full"][lo:hi], res["local"])) and bool(torch.isfinite(res["full"]).all())
    t = torch.tensor([1 if ok else 0], device=comm.dev)
    if comm.world > 1:
        comm.dist.all_reduce(t, op=comm.dist.ReduceOp.MIN)
    if int(t.item()) != 1:
        raise SystemExit("bench: gathered result differs from the local shard results")
    return True


def dump_outputs(outdir, results):
    """Write each (time, bus) result as float32 `outdir/<name>.npy` and the time steps it holds
    as float64 `outdir/<name>_time_index.npy`, in at most DUMP_BYTES together.  Results are
    kept whole smallest first while they fit an equal share of what is left; a larger one keeps
    a sorted sample of its time steps drawn with DUMP_SEED, so the same shapes give the same
    sample on every run."""
    os.makedirs(outdir, exist_ok=True)
    left = DUMP_BYTES - 2 * 4096 * len(results)  # 4 KiB per .npy header is generous (NumPy writes 128 B)
    row_bytes = {k: v.shape[1] * 4 + 8 for k, v in results.items()}  # float32 row + its float64 index
    order = sorted(results, key=lambda k: results[k].shape[0] * row_bytes[k])
    for i, name in enumerate(order):
        v = results[name]
        n = v.shape[0]
        keep = min(n, left // (len(order) - i) // row_bytes[name])
        left -= keep * row_bytes[name]
        rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, keep, replace=False))
        np.save(os.path.join(outdir, f"{name}.npy"), np.ascontiguousarray(v[rows], dtype=np.float32))
        np.save(os.path.join(outdir, f"{name}_time_index.npy"), rows.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    import atlite_b200 as ab
    from atlite_b200 import _lib, engine, synthetic as syn
    from atlite_b200.convert import _HeatSpec, _PvSpec, _WindSpec
    from atlite_b200.dist import TimeShard, shard_bounds

    warnings.simplefilter("ignore")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    comm = Comm(torch, dist)
    world, rank, dev = comm.world, comm.rank, comm.dev
    shard = TimeShard() if world > 1 else None
    peak, peak_src = hbm_peak()

    x, y = syn.make_coords(NX, NY, X0, Y0)
    time_axis = syn.make_time(NT)
    S = float(NX) * NY
    lo, hi = shard_bounds(NT, world, rank)
    counts = [b - a for a, b in (shard_bounds(NT, world, r) for r in range(world))]
    shapes = syn.make_shapes(NX, NY, NBUS)
    plan = engine.get_plan(shapes, NY, NX)
    co = dict(x=x, y=y, lon=x, lat=y)

    # ---- PV north star: this rank's shard, resident in HBM (in `parts` when it cannot be)
    need = (hi - lo) * S * BYTES_PER_CELL_TS
    free, total_mem = torch.cuda.mem_get_info()
    # never fill the device: at most VRAM_FRACTION of it holds inputs (a box whose GPU memory is
    # exhausted stops answering its health checks); generation temporaries need ~3 GiB more
    usable = min(free - (6 << 30), VRAM_FRACTION * total_mem)
    parts = 1
    while need / parts > usable and parts < 16:
        parts += 1
    clk = ClockSampler(comm.local_rank)
    my_rows = (sum(counts[:rank]), sum(counts[:rank + 1]))

    def run_parts(parts):
        bounds = [(lo + (hi - lo) * p // parts, lo + (hi - lo) * (p + 1) // parts) for p in range(parts)]
        acc = {"ms_step": 0.0, "kern_ms": 0.0, "kern_ranks": [0.0] * world, "gather_ms": None, "last": []}
        for p, (a, b) in enumerate(bounds):
            f = syn.make_pv_fields_device(time_axis[a:b], x, y, dev, seed=0, t_offset=a)
            spec = _PvSpec(ab.Dataset(f, coords=dict(time=time_axis[a:b], **co)),
                           ab.get_solarpanelconfig(PANEL), ab.get_orientation(ORIENT))
            # parts > 1 only happens on a single GPU whose HBM cannot hold the year: resident
            # parts one after the other, their times summed
            res = measure_sharded(comm, shard if parts == 1 else None, lambda: spec.op.reduce(plan, spec.fields),
                                  (b - a) * S, counts if parts == 1 else None, args.steps, args.warmup,
                                  clock=clk if p == 0 else None)
            if world > 1:
                check_gather(comm, res, *my_rows)
            acc["ms_step"] += res["ms_per_step"]
            acc["kern_ms"] += res["kernel_ms"]
            acc["kern_ranks"] = [u + v for u, v in zip(acc["kern_ranks"], res["kernel_ms_per_rank"])]
            acc["gather_ms"] = res["gather_ms"]
            if args.dump_outputs:
                acc["last"].append(res["full"].cpu())
            del f, spec, res
            torch.cuda.empty_cache()
        return acc

    n0 = _lib.launch_count()
    while True:
        try:
            acc = run_parts(parts)
            break
        except torch.OutOfMemoryError:
            if world > 1 or parts >= 16:
                raise
            parts += 1
            torch.cuda.empty_cache()
    ms_step, kern_ms, kern_ranks, gather_ms = acc["ms_step"], acc["kern_ms"], acc["kern_ranks"], acc["gather_ms"]
    outputs = {"pv": torch.cat(acc["last"]).numpy()} if args.dump_outputs else None
    launches = _lib.launch_count() - n0
    value = S * NT / (ms_step * 1e-3)
    cell_ts_local = S * (hi - lo)
    achieved = cell_ts_local * BYTES_PER_CELL_TS / (kern_ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            tj = json.load(fh)
        ratio = tj.get("pv_fused_1440x720_traffic_over_algorithmic")
        if ratio:
            traffic = ratio * cell_ts_local * BYTES_PER_CELL_TS / parts
    except Exception:  # noqa: BLE001
        pass

    # ---- e2e through the public API on pinned host arrays: a bounded slab of this rank's shard
    # pinned host memory is charged to the container's memory cgroup: every rank of this box takes
    # at most its share of a quarter of what the container may still use
    _, host_avail = _host_limits()
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    ne = int(min(E2E_MAX_STEPS, hi - lo, max(24, 0.25 * host_avail / local_world // (S * BYTES_PER_CELL_TS))))
    fe = syn.make_pv_fields_device(time_axis[lo:lo + ne], x, y, dev, seed=0, t_offset=lo)
    spec = _PvSpec(ab.Dataset(fe, coords=dict(time=time_axis[lo:lo + ne], **co)),
                   ab.get_solarpanelconfig(PANEL), ab.get_orientation(ORIENT))
    dev_slab = spec.op.reduce(plan, spec.fields).float().cpu().numpy()
    host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in fe.items()}
    for k, v in fe.items():
        host[k].copy_(v)
    torch.cuda.synchronize()
    del fe, spec
    torch.cuda.empty_cache()
    cut_host = ab.Cutout(data=ab.Dataset({k: v.numpy() for k, v in host.items()},
                                         coords=dict(time=time_axis[lo:lo + ne], **co)))

    def step_e2e():
        return cut_host.pv(PANEL, ORIENT, matrix=shapes, aggregate_time=None)

    res = step_e2e()
    comm.sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step_e2e()
    torch.cuda.synchronize()
    e2e_s = comm.max(time.perf_counter() - t0)
    e2e_value = S * ne * world * args.steps / e2e_s
    api_res = np.asarray(res.values).T
    agree = float(np.max(np.abs(dev_slab - api_res) / (np.abs(api_res) + 1e-3)))
    del host, cut_host, res

    line = {
        "metric": METRIC,
        "value": value, "unit": "grid-cell-timesteps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "per_gpu": (f"time axis sharded {NT}/{world} steps per rank (the same cutout at every N); NCCL "
                               "all-gather of the (time,bus) result inside every step (asynchronous: overlaps the next "
                               "pass, all gathers complete inside the timed region)") if world > 1 else "single GPU",
                   "parts": parts, "hbm_free_gib_at_start": round(free / 2 ** 30, 1),
                   "input_gib_this_rank": round(need / 2 ** 30, 1),
                   "l2_policy": "inputs (>= 22 GB per pass and rank) larger than L2; no flush needed",
                   "kernel": "k_fused_reduce<PvPhys<true,true>> (+1 memset)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": f"MEASURED_PEAKS.json ({peak_src})",
                     "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": cell_ts_local * BYTES_PER_CELL_TS / parts,
                     "launches_per_step": parts,
                     **({"kernel_ms_per_rank": [round(k, 4) for k in kern_ranks], "gather_ms": gather_ms}
                        if world > 1 else {})},
        "e2e": {"value": e2e_value, "unit": "grid-cell-timesteps/s",
                "h2d_bytes_per_step": int(S * ne * BYTES_PER_CELL_TS),
                "d2h_bytes_per_step": int(ne * NBUS * 4), "steps": args.steps,
                "sample": f"each rank streams the first {ne} steps of its shard from pinned host memory "
                          f"({world * ne} of {NT} steps per pass)",
                "api": "atlite_b200.Cutout(data=<pinned host arrays>).pv('CSi','latitude_optimal',matrix=...,aggregate_time=None)",
                "rank_bound_to_gpu_numa_node": comm.numa_bound,
                "max_rel_diff_vs_device_path": agree},
        "gpu_launches": int(launches),
        "clocks": clk.summary(),
    }
    if world > 1:
        line["gather_check"] = "gathered (time,bus) tensor == local shard result on every rank (bitwise)"

    # ---- BASELINE configs[2] / configs[3] on the same grid and shards
    extra = {}
    if not args.no_extra:
        extra.update(wind_heat_sharded(comm, shard, plan, x, y, time_axis, args, peak, outputs))
        if world == 1:
            extra.update(extra_single_gpu(torch, dev, peak))
    if extra:
        line["extra"] = extra
    if rank == 0 and outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0 and world == 1:
        line["cpu_baseline"] = cpu_baseline()
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def wind_heat_sharded(comm, shard, plan, x, y, time_axis, args, peak, outputs=None):
    """BASELINE configs[2] (wind, Vestas V112 3 MW) and configs[3] (heat demand) on the
    1440 x 720 x 8760 cutout -> 3000 shapes: this rank's time shard resident in HBM, same
    timed region as the headline (strong scaling at N > 1).  Heat-demand shards are cut on
    day boundaries (dist.shard_bounds(align=24)), so they may differ by one day.  The full
    (time, bus) results of the last timed passes go into `outputs` when it is a dict."""
    import atlite_b200 as ab
    from atlite_b200 import synthetic as syn
    from atlite_b200.convert import _HeatSpec, _WindSpec
    from atlite_b200.dist import shard_bounds

    torch = comm.torch
    S = float(NX) * NY
    world, rank = comm.world, comm.rank
    out = {}

    def entry(r, n_local, bytes_per):
        return {"cell_ts_per_s": S * NT / (r["ms_per_step"] * 1e-3), "ms_per_step": r["ms_per_step"],
                "kernel_ms_per_rank": [round(k, 4) for k in r["kernel_ms_per_rank"]], "gather_ms": r["gather_ms"],
                "achieved_GBs": n_local * S * bytes_per / r["kernel_ms"] / 1e6,
                "frac_of_hbm_peak": n_local * S * bytes_per / r["kernel_ms"] / 1e6 / peak, "scaling": "strong"}

    lo, hi = shard_bounds(NT, world, rank)
    counts = [b - a for a, b in (shard_bounds(NT, world, r) for r in range(world))]
    co = dict(time=time_axis[lo:hi], x=x, y=y, lon=x, lat=y)
    f = syn.make_wind_fields_device(hi - lo, NY, NX, comm.dev, seed=1, t_offset=lo)
    ws = _WindSpec(ab.Dataset(f, coords=co), ab.get_windturbineconfig(TURBINE))
    r = measure_sharded(comm, shard, lambda: ws.op.reduce(plan, ws.wnd, ws.aux), (hi - lo) * S, counts,
                        args.steps, args.warmup)
    if shard is not None:
        check_gather(comm, r, sum(counts[:rank]), sum(counts[:rank + 1]))
    if outputs is not None:
        outputs["wind"] = r["full"].cpu().numpy()
    out["wind_c2_1440x720x8760_3000"] = entry(r, hi - lo, 8)
    if world == 1:
        # the same kernel on a quarter-year slab (what each rank of a 4-GPU run processes): the 72.6 GB
        # full-year launch sits under the power cap, shorter slabs do not (profiles/r2_wind_slab_length.jsonl)
        try:
            nq = min(2190, hi - lo)
            wq, aq = ws.wnd[:nq], ws.aux[:nq]
            ms, _ = _timeit(torch, lambda: ws.op.reduce(plan, wq, aq), 7)
            out["wind_c2_quarter_year_slab_1440x720x2190_3000"] = {
                "steps": nq, "kernel_ms": ms, "cell_ts_per_s": S * nq / ms * 1e3,
                "achieved_GBs": S * nq * 8 / ms / 1e6, "frac_of_hbm_peak": S * nq * 8 / ms / 1e6 / peak}
            del wq, aq
        except Exception as e:  # noqa: BLE001 -- an extra data point must never cost the bench line
            out["wind_c2_quarter_year_slab_1440x720x2190_3000"] = {"error": repr(e)[:200]}
    del ws, r, f
    torch.cuda.empty_cache()

    lo, hi = shard_bounds(NT, world, rank, align=24)
    dcounts = [(b - a) // 24 for a, b in (shard_bounds(NT, world, r, align=24) for r in range(world))]
    co = dict(time=time_axis[lo:hi], x=x, y=y, lon=x, lat=y)
    tf = syn.make_pv_fields_device(time_axis[lo:hi], x, y, comm.dev, seed=2, names=("temperature",), t_offset=lo)
    hs = _HeatSpec(ab.Dataset(tf, coords=co), 15.0, 1.0, 0.0, 0.0)
    r = measure_sharded(comm, shard, lambda: hs.op.reduce(plan, hs.temp, hs.day_start), (hi - lo) * S, dcounts,
                        args.steps, args.warmup)
    if shard is not None:
        check_gather(comm, r, sum(dcounts[:rank]), sum(dcounts[:rank + 1]))
    if outputs is not None:
        outputs["heat_demand"] = r["full"].cpu().numpy()
    out["heat_c3_1440x720x8760_3000"] = entry(r, hi - lo, 4)
    out["heat_c3_1440x720x8760_3000"]["days_per_rank"] = dcounts
    del hs, r, tf
    torch.cuda.empty_cache()
    return out


def extra_single_gpu(torch, dev, peak):
    """Kernel-only roofline points next to the headline (N = 1): BASELINE configs[1]
    (200 x 200 x 8760 -> 100), the non-default PV variants on the north-star grid
    (real ERA5 cutouts store the solar position as float64: 36 B per cell-step), config 4
    (per-cell capacity factors), and the indicator matrix."""
    import atlite_b200 as ab
    from atlite_b200 import engine, synthetic as syn
    from atlite_b200.convert import _PvSpec, _WindSpec

    out = {}
    # ---- BASELINE configs[1] (the round-1 headline)
    nx, ny, nt, nbus = 200, 200, 8760, 100
    x, y = syn.make_coords(nx, ny, 0.0, 30.0)
    tm = syn.make_time(nt)
    f = syn.make_pv_fields_device(tm, x, y, dev, seed=0)
    plan = engine.get_plan(syn.make_shapes(nx, ny, nbus), ny, nx)
    spec = _PvSpec(ab.Dataset(f, coords=dict(time=tm, x=x, y=y, lon=x, lat=y)),
                   ab.get_solarpanelconfig(PANEL), ab.get_orientation(ORIENT))
    ms, _ = _timeit(torch, lambda: spec.op.reduce(plan, spec.fields), 10)
    cts = float(nx) * ny * nt
    out["pv_c1_200x200x8760_100"] = {"kernel_ms": ms, "cell_ts_per_s": cts / ms * 1e3,
                                     "achieved_GBs": cts * 20 / ms / 1e6, "frac_of_hbm_peak": cts * 20 / ms / 1e6 / peak}
    del f, spec, plan

    # ---- non-default PV variants, 1440 x 720 x 219 slab -> 3000 shapes
    nx, ny, nt, nbus = NX, NY, 219, NBUS
    x, y = syn.make_coords(nx, ny, X0, Y0)
    tm = syn.make_time(nt + 24 * 170)[24 * 170:]
    co = dict(time=tm, x=x, y=y, lon=x, lat=y)
    f = syn.make_pv_fields_device(tm, x, y, dev, seed=7, t_offset=24 * 170)
    plan = engine.get_plan(syn.make_shapes(nx, ny, nbus), ny, nx)
    out["plan_1440x720_3000"] = {k: plan.info[k] for k in ("nnz", "n_active_tiles", "n_slots", "slots_per_active_tile", "fused")}
    cts = float(nx) * ny * nt
    from atlite_b200 import era5

    alt, az = era5.solar_position(tm, x, y, "0h", dev.index)  # float64, as stored in real ERA5 cutouts
    variants = {
        "stored_solar_f64": (dict(f, solar_altitude=alt, solar_azimuth=az), {}, 36),
        "stored_solar_f32": (dict(f, solar_altitude=alt.float(), solar_azimuth=az.float()), {}, 28),
        "hay_davies": (f, dict(trigon_model="other"), 20),
        "tracking_horizontal": (f, dict(tracking="horizontal"), 20),
        "tracking_dual": (f, dict(tracking="dual"), 20),
    }
    for name, (fields, kw, bpc) in variants.items():
        spec = _PvSpec(ab.Dataset(fields, coords=co), ab.get_solarpanelconfig(PANEL), ab.get_orientation(ORIENT), **kw)
        ms, _ = _timeit(torch, lambda: spec.op.reduce(plan, spec.fields), 5)
        out[f"pv_variant_{name}_1440x720_slab"] = {
            "steps": nt, "bytes_per_cell_ts": bpc, "kernel_ms": ms, "cell_ts_per_s": cts / ms * 1e3,
            "achieved_GBs": cts * bpc / ms / 1e6, "frac_of_hbm_peak": cts * bpc / ms / 1e6 / peak}
        del spec
    del alt, az, f, variants, plan
    torch.cuda.empty_cache()
    out["indicatormatrix_1440x720_3000"] = indicator_measurement(x, y, nbus)

    # ---- BASELINE configs[4]: Europe-scale 1000 x 800, per-cell pv + wind capacity factors (no shapes
    # reduction: the no-matrix branch, convert.py:200-211) -> k_cells time-sum kernels
    nx, ny, nt = 1000, 800, 240
    x, y = syn.make_coords(nx, ny, -12.0, 33.0, 0.05, 0.05)
    tm = syn.make_time(nt + 24 * 170)[24 * 170:]
    f = syn.make_pv_fields_device(tm, x, y, dev, seed=9, t_offset=24 * 170)
    co = dict(time=tm, x=x, y=y, lon=x, lat=y)
    spec = _PvSpec(ab.Dataset(f, coords=co), ab.get_solarpanelconfig(PANEL), ab.get_orientation(ORIENT))
    ws = _WindSpec(ab.Dataset(syn.make_wind_fields_device(nt, ny, nx, dev, seed=9), coords=co),
                   ab.get_windturbineconfig(TURBINE))
    cts = float(nx) * ny * nt
    ms_pv, _ = _timeit(torch, lambda: spec.cells(timesum=True), 5)
    ms_w, _ = _timeit(torch, lambda: ws.cells(timesum=True), 5)
    out["percell_cf_c4_1000x800_slab"] = {
        "steps": nt, "pv_kernel_ms": ms_pv, "wind_kernel_ms": ms_w,
        "cell_ts_per_s_combined": cts / (ms_pv + ms_w) * 1e3,
        "pv_frac_of_hbm_peak": cts * 20 / ms_pv / 1e6 / peak, "wind_frac_of_hbm_peak": cts * 8 / ms_w / 1e6 / peak,
        "combined_achieved_GBs": cts * 28 / (ms_pv + ms_w) / 1e6,
        "combined_frac_of_hbm_peak": cts * 28 / (ms_pv + ms_w) / 1e6 / peak}
    return out


def indicator_measurement(x, y, n_shapes):
    """The step in front of the path (SURVEY 8 f1): shapes -> indicator matrix, 3000
    Voronoi regions on the 1440 x 720 grid.  Wall time of the public call (host
    packing + H2D + kernels + CSR back on the host), with the oracle's clipping
    loop timed on a few shapes beside it."""
    from atlite_b200 import gis, synthetic as syn

    rings = syn.make_voronoi_shapes(x, y, n_shapes)
    gis.compute_indicatormatrix(x, y, rings[:8])  # warm-up (context, allocator)
    t0 = time.perf_counter()
    m = gis.compute_indicatormatrix(x, y, rings)
    dt = time.perf_counter() - t0
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import indicator_oracle as IO  # the checker, timed as the CPU stand-in for shapely's loop

    k = 6
    t0 = time.perf_counter()
    mo = IO.indicatormatrix(x, y, [gis.geometry_rings(r) for r in rings[:k]])
    dto = time.perf_counter() - t0
    err = float(abs(m[:k] - mo).max())
    return {"shapes": n_shapes, "nnz": int(m.nnz), "edges": int(sum(len(r) for r in rings)), "gpu_call_ms": dt * 1e3,
            "cpu_oracle_ms_per_shape": dto / k * 1e3, "cpu_oracle_extrapolated_ms": dto / k * n_shapes * 1e3,
            "max_abs_diff_on_sample": err, "column_sum_max_dev": float(abs(np.asarray(m.sum(0)).ravel() - 1).max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[2,3] / variant roofline points")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the (time, bus) results of the last timed pass to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
