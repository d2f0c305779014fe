#!/usr/bin/env python
"""bench.py -- constraint + Jacobian evals/sec of the Bezier hot path on B200.

Workload (BASELINE.json configs[3], "C4"): synthetic 1024-vehicle 3-D swarm,
degree 10, DEG_ELEV 100: one *eval* = the full constraint vector of one x
(523 776 pairs x 121 separation values + 1024 x 121 max-speed values = 508 MB).
One *step* = one pass over a batch of B such x (the base point and B-1
finite-difference perturbations of it, which is what SLSQP's Jacobian asks for).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU).  Sharding: the batch of
perturbed x is split across ranks (each rank evaluates its own B x over all
pairs, no data-path collective); the per-pair minimum (the active-pair source,
[B, P] fp64) is all-gathered over NCCL/NVLink so every rank holds the whole
min-distance matrix.  Weak scaling: B per rank is fixed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = dict(N=1024, dim=3, deg=10, elev=100)
SEED = 20261018
DUMP_BYTES = 64 * 10 ** 6   # --dump-outputs: at most this much in all
DUMP_PAIRS = 8192           # --dump-outputs: separation rows of this many pairs (fixed seeded sample)


def synthetic_swarm(N, deg, seed=SEED):
    """SURVEY 8(d) 'Synthetic inputs C4' (same generator as oracle/make_golden.py)."""
    rng = np.random.default_rng(seed)
    init = rng.uniform(0, 100, size=(N, 3))
    final = rng.uniform(0, 100, size=(N, 3))
    args = dict(numVeh=N, dimension=3, degree=deg, minimizeGoal='Euclidean',
                maxSep=0.9, maxSpeed=5, tf=20.0, initPoints=init, finalPoints=final)
    x = np.empty((N * 3, deg - 1))
    for i in range(N):
        for d in range(3):
            x[3 * i + d] = np.linspace(init[i, d], final[i, d], deg + 1)[1:-1]
    x = x + rng.normal(size=x.shape)
    return args, x.ravel()


def fd_batch(x, B, seed=1):
    """base x plus B-1 single-variable forward perturbations (SciPy's h)."""
    X = np.repeat(x[None, :], B, axis=0)
    rng = np.random.default_rng(seed)
    for b, k in enumerate(rng.choice(x.size, size=B - 1, replace=False), start=1):
        X[b, k] += 1.4901161193847656e-08
    return X


def dump_outputs(path, pairmin, sep, spd):
    """Writes what one step of the timed path returned, as float64 .npy files under `path`:
    pair_min [b, P] (per-pair minima), max_speed [b, N, L] (max-speed rows) and separation
    [b, DUMP_PAIRS, L] (the separation rows of a fixed, seeded sample of the pairs, in pair order).
    The full separation block is 2 GB per step, hence the sample; b is the number of leading
    evaluations of the batch that fit into DUMP_BYTES (all of them at the default batch)."""
    import torch
    P, L = sep.shape[1], sep.shape[2]
    idx = np.sort(np.random.default_rng(SEED).choice(P, size=min(P, DUMP_PAIRS), replace=False))
    b = min(sep.shape[0], DUMP_BYTES // (8 * (pairmin.shape[1] + spd.shape[1] * spd.shape[2] + idx.size * L)))
    arrays = {"pair_min": pairmin[:b], "max_speed": spd[:b],
              "separation": sep[:b].index_select(1, torch.as_tensor(idx, device=sep.device))}
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


# --------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled (NVML) during the timed region."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20,
               "hw_thermal_slowdown": 0x40, "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index, period=0.002):
        self.gpu, self.period = gpu_index, period
        self.sm, self.reasons, self.smax = [], set(), None
        self._stop = threading.Event()
        self._go = threading.Event()
        self.thread = None
        self.err = None

    def _open(self):
        import pynvml
        pynvml.nvmlInit()
        # NVML enumerates physical GPUs; honour CUDA_VISIBLE_DEVICES when it lists indices
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = self.gpu
        if vis and all(t.strip().isdigit() for t in vis.split(",")):
            idx = int(vis.split(",")[self.gpu])
        self._nvml = pynvml
        self._h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))

    def _run(self):
        try:
            pynvml, h = self._nvml, self._h
            self._go.wait()                # armed by go(): the first sample belongs to the timed region
            while not self._stop.is_set():
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                try:
                    mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                if self._stop.wait(self.period):
                    break
        except Exception as e:            # pragma: no cover
            self.err = repr(e)

    def open(self):
        """NVML is opened ahead of the timed region (and of the barrier in front of it: it takes
        milliseconds, on rank 0 only), so that short runs are sampled from their first step."""
        try:
            self._open()
        except Exception as e:            # pragma: no cover
            self.err = repr(e)

    def start(self, armed=True):
        """Starts the sampling thread.  With armed=False the thread is created (hundreds of microseconds on
        rank 0 only -- with a fused all-gather every rank's timed region absorbs that start skew) but samples
        nothing until go() is called right in front of the timed region."""
        if self.err is None and not hasattr(self, "_h"):
            self.open()
        if self.err is not None:
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        if armed:
            self._go.set()

    def go(self):
        self._go.set()

    def stop(self):
        self._stop.set()
        self._go.set()
        if self.thread is not None:
            self.thread.join(timeout=5)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smax,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.err:
            out["error"] = self.err
        return out


# --------------------------------------------------------------------------
def cpu_baseline(args, x, E, target_seconds=12.0, threads=0):
    """Times the plain-C restatement of the reference (oracle/bezier_oracle.c, all
    host threads) on a bounded, contiguous sample of the C4 pair list and
    extrapolates linearly to evals/s (pairs are independent and of equal cost).
    The Python reference itself cannot travel to the GPU box; in the authoring
    container it costs 23-34 us per pair per core (BASELINE.md section 2), about
    10x more than this port."""
    from oracle import bezier_oracle as O
    from oracle import c_oracle as C
    m = O.Model(**args)
    y = O.reshape_vector(m, x)
    N, dim = m.numVeh, m.dim
    P = N * (N - 1) // 2
    L = 2 * m.deg + E + 1
    threads = threads or C.max_threads()
    cal_pairs = min(P, 65536)
    out = np.empty(cal_pairs * L)
    C.temporal_separation(y, N, dim, m.maxSep, E, 0, cal_pairs, nthreads=threads, out=out)   # warm + calibrate
    t0 = time.perf_counter()
    C.temporal_separation(y, N, dim, m.maxSep, E, 0, cal_pairs, nthreads=threads, out=out)
    per_pair = (time.perf_counter() - t0) / cal_pairs
    chunk = min(P, 262144)
    out = np.empty(chunk * L)
    reps = max(1, int(target_seconds / (per_pair * chunk)))
    done = 0
    t0 = time.perf_counter()
    for r in range(reps):
        begin = (r * chunk) % max(1, P - chunk + 1)
        C.temporal_separation(y, N, dim, m.maxSep, E, begin, chunk, nthreads=threads, out=out)
        done += chunk
    t_speed0 = time.perf_counter()
    C.speed(y, N, dim, m.tf, E, -1.0, m.maxSpeed ** 2, nthreads=threads)
    t_speed = time.perf_counter() - t_speed0
    wall = time.perf_counter() - t0 - t_speed
    sec_per_eval = wall / done * P + t_speed
    return {"value": 1.0 / sec_per_eval, "unit": "evals/s", "cores": threads, "kind": "port",
            "sample": "%d pair evaluations drawn from the %d pairs of the C4 swarm (N=%d, deg %d, elev %d) + all %d speed rows, "
                      "%d threads, %.1f s wall; plain-C restatement of the reference "
                      "(oracle/bezier_oracle.c: sub -> normSquare -> elev), extrapolated linearly in pairs"
                      % (done, P, N, m.deg, E, N, threads, wall + t_speed)}, wall + t_speed


# --------------------------------------------------------------------------
def run_reference(opts):
    """Reference arm: the reference's own algorithm for the path (C restatement, all host
    threads) on the same workload; each step is a bounded sample of the C4 pair list, sized so
    that the whole --steps/--warmup run stays within about two minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import bezier_oracle as O
    from oracle import c_oracle as C
    args, x = synthetic_swarm(WORKLOAD["N"], WORKLOAD["deg"])
    E = WORKLOAD["elev"]
    m = O.Model(**args)
    y = O.reshape_vector(m, x)
    N, dim = m.numVeh, m.dim
    P = N * (N - 1) // 2
    L = 2 * m.deg + E + 1
    threads = C.max_threads()
    cal = min(P, 65536)
    out = np.empty(cal * L)
    C.temporal_separation(y, N, dim, m.maxSep, E, 0, cal, nthreads=threads, out=out)          # warm
    t0 = time.perf_counter()
    C.temporal_separation(y, N, dim, m.maxSep, E, 0, cal, nthreads=threads, out=out)
    per_pair = (time.perf_counter() - t0) / cal
    t0 = time.perf_counter()
    C.speed(y, N, dim, m.tf, E, -1.0, m.maxSpeed ** 2, nthreads=threads)
    t_speed = time.perf_counter() - t0
    total_steps = max(1, opts.steps + opts.warmup)
    per_step = max(0.2, min(15.0, 110.0 / total_steps))
    chunk = int(min(P, max(4096, per_step / per_pair)))
    out = np.empty(chunk * L)
    vals, walls, done = [], [], 0
    for s in range(total_steps):
        begin = (s * chunk) % max(1, P - chunk + 1)
        t0 = time.perf_counter()
        C.temporal_separation(y, N, dim, m.maxSep, E, begin, chunk, nthreads=threads, out=out)
        wall = time.perf_counter() - t0
        if s >= opts.warmup:
            vals.append(1.0 / (wall / chunk * P + t_speed))
            walls.append(wall)
            done += chunk
    v = float(np.mean(vals))
    cb = {"value": v, "unit": "evals/s", "cores": threads, "kind": "port",
          "sample": "%d steps x %d pair evaluations drawn from the %d pairs of the C4 swarm (N=%d, deg %d, elev %d) "
                    "+ all %d speed rows timed once, %d threads, %.1f s of CPU wall in the timed steps; plain-C "
                    "restatement of the reference (oracle/bezier_oracle.c: sub -> normSquare -> elev), extrapolated "
                    "linearly in pairs" % (len(vals), chunk, P, N, m.deg, E, N, threads, float(np.sum(walls)))}
    line = {"impl": "reference", "metric": "constraint+Jacobian evals/sec", "value": v, "unit": "evals/s",
            "n_gpus": opts.gpus, "steps": opts.steps, "warmup": opts.warmup,
            "ms_per_step": 1e3 * float(np.mean(walls)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(), "evals_per_step_per_gpu": None, "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config():
    """The same dict on both arms (the driver compares them); per-arm details such as the
    batch per step or the gather implementation are top-level keys of the line."""
    return {"workload": "C4 synthetic swarm: N=1024 vehicles, dim 3, degree 10, DEG_ELEV 100, "
                        "all 523776 pairs x 121 separation values + 1024 x 121 max-speed values per eval",
            "sharding": "FD-perturbation batch split across ranks; all-gather of the [B,P] per-pair minimum",
            "l2_policy": "outputs (508 MB/eval) >> 126 MB L2, streaming stores; inputs 270 KB"}


# --------------------------------------------------------------------------
def _dist_env():
    return (int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")),
            int(os.environ.get("LOCAL_RANK", "0")))


def _bind_to_gpu_numa_node(local):
    """Binds this rank's host threads to the CPUs of its GPU's NUMA node (NVML affinity), so
    that pinned staging buffers and the copy threads sit next to the GPU's PCIe root."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = int(vis.split(",")[local]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else local
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def _peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _time_events(fn, reps, torch):
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b_ in evs:
        a.record()
        fn()
        b_.record()
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b_) for a, b_ in evs]))


def run_ours(opts):
    import torch
    import torch.distributed as dist
    from optimalbeziertrajectorygeneration_b200 import optimization as gopt
    from optimalbeziertrajectorygeneration_b200 import sharding
    from optimalbeziertrajectorygeneration_b200.engine import num_pairs

    world, rank, local = _dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    numa_cpus = _bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    strong = opts.scaling == "strong"

    N, deg, E = WORKLOAD["N"], WORKLOAD["deg"], WORKLOAD["elev"]
    B = opts.batch
    args, x = synthetic_swarm(N, deg)
    if strong:                      # one batch of B evaluations, the pair list cut into `world` ranges
        Xall = fd_batch(x, B)
        X = Xall
    else:                           # weak: every rank evaluates its own B perturbed x over all pairs
        Xall = fd_batch(x, B * world)
        X = Xall[rank * B:(rank + 1) * B]
    bezopt = gopt.BezOptimization(**args)
    eng = bezopt._engine(True)
    P = num_pairs(N)
    L = 2 * deg + E + 1
    p_lo, p_hi = sharding.pair_range(N, world, rank) if strong else (0, P)
    v_lo, v_hi = sharding.block_range(N, world, rank) if strong else (0, N)
    Pr, Nr = p_hi - p_lo, v_hi - v_lo
    d_x = eng.upload(X)
    # Consecutive steps alternate between two launch streams with their own output buffers: the
    # kernels of step k+1 are already queued when the persistent pair kernel of step k drains, so
    # its CTAs fill the SMs as they free up (no launch gap, no idle tail between steps).
    nlanes = 1 if opts.single_stream else 2
    lanes = [torch.cuda.Stream(device=eng.device) for _ in range(nlanes)]
    # the speed rows of a step only need the assembled control points: they run on a side stream of their launch
    # stream, next to (in practice: at the tail of) the previous persistent pair kernel, and never in front of
    # their own step's pair kernel
    aux = [torch.cuda.Stream(device=eng.device) for _ in range(nlanes)]

    def speed_aside(i, cpts, tf, ospd, **kw):
        ready = torch.cuda.Event()
        ready.record(lanes[i])
        with torch.cuda.stream(aux[i]):
            aux[i].wait_event(ready)
            eng.speed(cpts, tf, E, -1.0, max_speed2, out=ospd, **kw)
            done = torch.cuda.Event()
            done.record(aux[i])
        return done
    out_seps = [torch.empty((B, Pr, L), dtype=torch.float64, device=eng.device) for _ in range(nlanes)]
    out_spds = [torch.empty((B, Nr, L), dtype=torch.float64, device=eng.device) for _ in range(nlanes)]
    pairmins = [torch.empty((B, Pr), dtype=torch.float64, device=eng.device) for _ in range(nlanes)]
    out_sep, out_spd, pairmin = out_seps[0], out_spds[0], pairmins[0]
    max_speed2 = float(args["maxSpeed"]) ** 2
    step_no = [0]

    # The one collective of the path: every rank ends up with the whole per-pair minimum
    # (active-pair) matrix -- [world*B, P] (weak) or [B, P] (strong).  Preferred: fused into the
    # pair kernel (NVLink peer stores into symmetric memory, sharding.PeerMinima); fallback:
    # NCCL all-gather on its own stream.
    gatherer, peer, gather_mode = None, None, "none (1 GPU)"
    if world > 1 and opts.no_gather:       # diagnostic: N independent replicas, no exchange at all
        gather_mode = "none (diagnostic --no-gather)"
    if world > 1 and not opts.nccl_gather and not opts.no_gather:
        try:
            peer = sharding.PeerMinima(B, P, eng.device, layout="pairs" if strong else "batch")
            gather_mode = ("fused: in-kernel NVLink %s into symmetric memory; signal-pad barrier on a "
                           "high-priority side stream, three rotating matrices"
                           % ("multicast stores (NVSwitch replicates to every rank)" if peer.mc_ptr else "peer stores"))
        except Exception as e:                      # symmetric memory not available on this box
            if rank == 0:
                print("PeerMinima unavailable (%r); falling back to NCCL all-gather" % (e,), file=sys.stderr)
    if peer is None and not strong and not opts.no_gather:
        gatherer = sharding.PairMinimaGatherer(B, P, eng.device)
        if world > 1:
            gather_mode = "NCCL all_gather_into_tensor on a side stream"
    if peer is None and strong and world > 1:
        gather_mode = "NCCL padded all-gather (sharding.gather_pair_minima, mode 'pairs')"

    def step():
        i = step_no[0] % nlanes
        step_no[0] += 1
        osep, ospd, opm = out_seps[i], out_spds[i], pairmins[i]
        with torch.cuda.stream(lanes[i]):
            cpts, tf = eng.assemble(d_x, E)
            if peer is not None:
                pm, peers = peer.targets()
                sdone = speed_aside(i, cpts, tf, ospd, veh_begin=v_lo, nveh=Nr)
                eng.separation(cpts, E, args["maxSep"], pair_begin=p_lo, npairs=Pr, out=osep, pairmin=pm,
                               peer_ptrs=peers, min_pitch=P if strong else None)
                lanes[i].wait_event(sdone)
                # (the speed rows go first: behind the persistent pair kernel they would find no SM until the NEXT
                # pair kernel, already queued on the other launch stream, has drained)
                gathered = peer.complete()
                return gathered, osep
            if strong:
                sdone = speed_aside(i, cpts, tf, ospd, veh_begin=v_lo, nveh=Nr)
                eng.separation(cpts, E, args["maxSep"], pair_begin=p_lo, npairs=Pr, out=osep, pairmin=opm)
                lanes[i].wait_event(sdone)
                return sharding.gather_pair_minima(opm, mode="pairs", total=P), osep
            if gatherer is None:
                sdone = speed_aside(i, cpts, tf, ospd)
                eng.separation(cpts, E, args["maxSep"], out=osep, pairmin=opm)
                lanes[i].wait_event(sdone)
                return opm, osep
            pm = gatherer.local_buffer()
            sdone = speed_aside(i, cpts, tf, ospd)
            eng.separation(cpts, E, args["maxSep"], out=osep, pairmin=pm)
            lanes[i].wait_event(sdone)
            return gatherer.gather(), osep
    launches_per_step = 3       # assemble, speed kernel, fused pair kernel (values + per-pair min)

    def fork():
        """the launch streams start behind everything queued on the default stream"""
        for st in lanes:
            st.wait_stream(torch.cuda.current_stream())

    def finish():
        for st in lanes:
            with torch.cuda.stream(st):
                if gatherer is not None:
                    gatherer.finish()
                if peer is not None:
                    peer.wait()     # the last step's barrier (side stream) belongs to the timed region
        for st in lanes:
            torch.cuda.current_stream().wait_stream(st)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(v):
        t = torch.tensor([v], dtype=torch.float64, device=eng.device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    fork()
    for _ in range(max(3, opts.warmup)):
        step()
    finish()
    sampler = ClockSampler(local, period=opts.clock_period)
    if rank == 0:
        sampler.open()
        sampler.start(armed=False)
    barrier()
    if rank == 0:
        sampler.go()
    prof = None
    if opts.timeline and rank == 0:        # diagnostic: CUPTI kernel timeline of the timed region (distorts the timing)
        from torch.profiler import ProfilerActivity, profile
        prof = profile(activities=[ProfilerActivity.CUDA])
        prof.__enter__()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fork()
    t_host0 = time.perf_counter()
    for _ in range(opts.steps):
        gathered, last_sep = step()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / opts.steps     # host time to enqueue one step
    finish()
    ev1.record()
    barrier()
    if prof is not None:
        prof.__exit__(None, None, None)
        evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
        with open(opts.timeline, "w") as f:
            for e in evs:
                f.write("%10.1f us  +%8.1f us  %s\n" % (e.time_range.start - evs[0].time_range.start,
                                                         e.time_range.end - e.time_range.start, e.name[:90]))
    ms = maxreduce(ev0.elapsed_time(ev1))
    if world > 1 and not opts.no_gather:
        # self-check of the collective (outside the timed region): the gathered matrix of the
        # last step must equal a plain NCCL all-gather of the per-rank minima, bit for bit
        mine = last_sep.min(dim=2).values.contiguous()
        if strong:
            ref = sharding.gather_pair_minima(mine, mode="pairs", total=P)
        else:
            ref = torch.empty((world * B, P), dtype=torch.float64, device=eng.device)
            dist.all_gather_into_tensor(ref, mine)
        torch.cuda.synchronize()
        assert torch.equal(ref, gathered), "gathered per-pair minima differ from the NCCL all-gather"
    if opts.dump_outputs and rank == 0:
        # the last timed step's results, before anything below reuses its buffers (rank 0's share)
        dump_outputs(opts.dump_outputs, gathered, last_sep, out_spds[(step_no[0] - 1) % nlanes])

    # dominant kernel alone (pair kernel over this rank's pairs), CUDA events on its stream
    cpts, tf = eng.assemble(d_x, E)
    torch.cuda.synchronize()
    kms = _time_events(lambda: eng.separation(cpts, E, args["maxSep"], pair_begin=p_lo, npairs=Pr, out=out_sep,
                                              pairmin=pairmin), opts.steps, torch)
    # ... and with the fused all-gather's peer / multicast stores (no barrier): what the exchange costs inside the kernel
    kms_peer = None
    if peer is not None:
        pm_, peers_ = peer.targets()
        kms_peer = _time_events(lambda: eng.separation(cpts, E, args["maxSep"], pair_begin=p_lo, npairs=Pr, out=out_sep,
                                                       pairmin=pm_, peer_ptrs=peers_, min_pitch=P if strong else None),
                                opts.steps, torch)
        barrier()
    # the same kernel in the production launch pattern: back-to-back launches alternating between the
    # two launch streams, so that the CTAs of launch k+1 fill the SMs as launch k drains
    kms_pipe = None
    if nlanes > 1:
        fork()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record()
        fork()
        for i in range(opts.steps):
            with torch.cuda.stream(lanes[i % nlanes]):
                eng.separation(cpts, E, args["maxSep"], pair_begin=p_lo, npairs=Pr, out=out_seps[i % nlanes],
                               pairmin=pairmins[i % nlanes])
        for st in lanes:
            torch.cuda.current_stream().wait_stream(st)
        b_.record()
        torch.cuda.synchronize()
        kms_pipe = a_.elapsed_time(b_) / opts.steps
    clocks = sampler.stop() if rank == 0 else None
    line = None
    peak, peak_src = _peak()
    if rank == 0:
        alg_bytes = 8.0 * B * (Pr * L + Pr + 34 * N)    # rows + per-pair minima written, control-point rows read
        achieved = alg_bytes / (kms * 1e-3) / 1e9
        # measured DRAM traffic of the same launch shape from the committed ncu --set full capture
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "pair_kernel_traffic.json")
        if os.path.exists(tpath) and not strong:
            tj = json.load(open(tpath))
            if tj.get("evals_per_launch") == B:
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
        evals = (B if strong else B * world) * opts.steps
        line = {"metric": "constraint+Jacobian evals/sec", "value": evals / (ms * 1e-3), "unit": "evals/s",
                "n_gpus": world, "steps": opts.steps, "warmup": max(3, opts.warmup),
                "ms_per_step": ms / opts.steps, "higher_is_better": True, "scaling": opts.scaling,
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(), "evals_per_step_per_gpu": B if not strong else B / world,
                "gather": gather_mode,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                             "kernel": "sq_elev_ws_kernel<10,3,min,rows>: warp-specialised pair kernel (producer warps: TMA row "
                                       "fetch + stage 1; consumer warps: DMMA.8x8x4 stage 2, fused minimum, TMA bulk-store epilogue)",
                             "kernel_ms": kms, "kernel_ms_with_peer_stores": kms_peer,
                             "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                             "pipelined": None if kms_pipe is None else {
                                 "ms_per_launch": kms_pipe, "achieved": alg_bytes / (kms_pipe * 1e-3) / 1e9,
                                 "frac": alg_bytes / (kms_pipe * 1e-3) / 1e9 / peak,
                                 "note": "same kernel, back-to-back launches alternating between two streams (the "
                                         "production launch pattern of the step loop): total time / launches; "
                                         "`frac` above is the conservative figure from isolated launches"}},
                "gpu_launches": launches_per_step * opts.steps, "clocks": clocks,
                "host_enqueue_ms_per_step": host_enqueue_ms}
        if strong:
            line["config"] = dict(workload_config(), sharding="one FD batch; the pair list cut into contiguous "
                                  "ranges per rank (vehicle blocks for the speed rows); fused gather into one [B,P] matrix")
        if numa_cpus:
            line["host_cpus_bound_per_rank"] = numa_cpus

    if strong:                      # the strong-scaling line carries the device-timed figures only
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    # ----------------------------------------------------------------------------------
    # End to end through the public host API: host X (pinned) -> H2D -> kernels (every row
    # materialised in HBM) -> D2H of the step's result.
    #  (a) evaluate_sweep_active: result = packed active-pair bitmask + compacted (pair, min)
    #      list + per-vehicle max-speed minima and bitmask           <- the headline e2e
    #  (b) evaluate_sweep: result = the fp64 per-pair minimum matrix + all max-speed rows
    #  (c) evaluate_reduced: (b) one call per step, strictly serial
    #  (d) the reference-facing closures: the full 508 MB constraint vector per x
    gopt.DEG_ELEV = E
    bezopt.zero_copy_results = True
    nS = max(16, min(2 * opts.steps, 64))
    Xs = np.concatenate([X] * nS, axis=0)
    for _ in range(2):
        act = bezopt.evaluate_sweep_active(Xs, elev=E, chunk=B)
    barrier()
    t0 = time.perf_counter()
    act = bezopt.evaluate_sweep_active(Xs, elev=E, chunk=B)
    dt_act = maxreduce(time.perf_counter() - t0)
    d2h_act = int((act.pair_bufs.shape[1] + act.veh_bufs.shape[1]) * 8 + B * N * 8)
    nM = max(4, min(opts.steps, 24))
    Xm = Xs[:nM * B]
    for _ in range(2):
        sw = bezopt.evaluate_sweep(Xm, elev=E, chunk=B)
    barrier()
    t0 = time.perf_counter()
    sw = bezopt.evaluate_sweep(Xm, elev=E, chunk=B)
    dt_sweep = maxreduce(time.perf_counter() - t0)
    # the reduced result is consistent with the minimum matrix
    flags, ev_i, pair_i, val = act.pairs(0)
    assert np.array_equal(flags, sw["pairmin"][:B] < 0) and np.array_equal(val, sw["pairmin"][:B][flags])
    vmin, vflags = act.vehicles(0)
    assert np.array_equal(vmin, sw["maxspeed"][:B].reshape(B, N, L).min(axis=2))
    nE = max(3, min(opts.steps, 10))
    for _ in range(2):
        red = bezopt.evaluate_reduced(X, elev=E)
    barrier()
    t0 = time.perf_counter()
    for _ in range(nE):
        red = bezopt.evaluate_reduced(X, elev=E)
    torch.cuda.synchronize()
    dt_red = maxreduce(time.perf_counter() - t0)
    sepf, spdf = bezopt.temporalSeparationConstraints, bezopt.maxSpeedConstraints
    nF = 2
    r1 = sepf(X[0]); r2 = spdf(X[0])
    barrier()
    t0 = time.perf_counter()
    for s_ in range(nF):
        r1 = sepf(X[s_ % B]); r2 = spdf(X[s_ % B])
    torch.cuda.synchronize()
    dt_full = maxreduce(time.perf_counter() - t0)
    full_bytes = int((r1.size + r2.size) * 8)
    del r1, r2
    e2e = {"value": nS * B * world / dt_act, "unit": "evals/s",
           "h2d_bytes_per_step": int(X.size * 8), "d2h_bytes_per_step": d2h_act, "steps_timed": nS,
           "active_pairs_per_eval": float(act.pair_counts().mean() / B),
           "note": "BezOptimization.evaluate_sweep_active(X_host[steps*B, nvar], chunk=B): per step (chunk of B rows) "
                   "pinned H2D of X -> assemble -> fused pair kernel (all P*L values written to HBM, per-pair minimum "
                   "matrix kept in HBM, packed active bitmask + compacted (pair, min) list from the epilogue) -> speed "
                   "kernel (rows + per-vehicle minima + bitmask) -> D2H of bitmask, list, speed minima into pinned "
                   "host memory; two device workspaces, the D2H of step k overlaps the kernels of step k+1; wall "
                   "clock incl. Python",
           "minima_matrix": {"value": nM * B * world / dt_sweep, "unit": "evals/s", "steps_timed": nM,
                             "d2h_bytes_per_step": int((sw["pairmin"][:B].size + sw["maxspeed"][:B].size) * 8),
                             "note": "round-1 e2e: evaluate_sweep, D2H of the fp64 per-pair minimum matrix [B,P] and "
                                     "all max-speed rows"},
           "serial_call": {"value": nE * B * world / dt_red, "unit": "evals/s", "steps_timed": nE,
                           "note": "one evaluate_reduced(X_host[B,nvar]) call per step, H2D -> kernels -> D2H "
                                   "strictly in sequence with a host synchronisation per call"},
           "full_vector": {"value": nF * world / dt_full, "unit": "evals/s", "d2h_bytes_per_eval": full_bytes,
                           "note": "temporalSeparationConstraints(x)+maxSpeedConstraints(x) returning the full "
                                   "508 MB constraint vector to host memory (PCIe-bound)"}}
    gopt.DEG_ELEV = 0
    bezopt._sweep_ws = bezopt._active_ws = bezopt.workspace = None
    del sw, act, red
    torch.cuda.empty_cache()

    # Sparse-aware FD sweep (SURVEY 8(d)(ii)): the whole Jacobian of the separation block of ONE x
    # (what SLSQP obtains from nvar+1 = 27 649 full evals) in closed form, sweep layout
    # [variable][partner curve][L] = only the rows that depend on the variable (27.4 GB).
    sweep = None
    if not opts.no_sweep:
        J = eng.jac_separation(x, E, dense=False)
        for _ in range(2):
            eng.jac_separation(x, E, dense=False, out=J)
        torch.cuda.synchronize()
        sms = _time_events(lambda: eng.jac_separation(x, E, dense=False, out=J), 3, torch)
        sweep = {"value": (bezopt.nvar + 1) * world / (sms * 1e-3), "unit": "evals/s",
                 "ms_per_jacobian": sms, "bytes_per_jacobian": int(J.numel() * 8),
                 "hbm_frac": int(J.numel() * 8) / (sms * 1e-3) / 1e9 / peak,
                 "note": "closed-form FD Jacobian of the separation block of one x (all %d variables x %d partner "
                         "curves x %d values), equivalent to nvar+1 full evals of the reference; every rank "
                         "computes the Jacobian of its own x" % (bezopt.nvar, N - 1, L)}
        del J
        torch.cuda.empty_cache()
    del out_sep, out_spd, pairmin, out_seps, out_spds, pairmins, last_sep
    torch.cuda.empty_cache()

    # BASELINE configs[4] (C5) and configs[1], [2] (C2 Example1, C3 swarm) in the same line
    c5 = None if opts.no_c5 else c5_measure(opts, world, rank, local, steps=max(3, min(opts.steps, 10)))
    slsqp = None
    if rank == 0 and not opts.no_slsqp:
        slsqp = slsqp_measure(full=opts.slsqp_full)
    barrier()

    if rank == 0:
        line["e2e"] = e2e
        if sweep is not None:
            line["jacobian_sweep"] = sweep
        if c5 is not None:
            line["c5"] = c5
        if slsqp is not None:
            line["slsqp_c2"], line["slsqp_c3"] = slsqp["c2"], slsqp["c3"]
        if world == 1 and not opts.no_cpu:
            cb, _ = cpu_baseline(args, x, E, target_seconds=12.0)
            line["cpu_baseline"] = cb
            pyref = cpu_baseline_python(args, x, E)
            if pyref is not None:
                line["cpu_baseline_python"] = pyref
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------
def cpu_baseline_python(args, x, E, npairs=2048):
    """The unmodified Python reference (numpy + numba) timed on this host, when a copy of it
    travelled with the repository (baseline/_ref, written by __graft_entry__.build() in the
    authoring container; git-ignored).  One thread, a bounded sample: the first vehicles of the
    C4 swarm whose pair count reaches `npairs`, through the reference's own
    _temporalSeparationConstraints."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref_root, "bezier.py")):
        return None
    try:
        from oracle import ref_loader
        from oracle import bezier_oracle as O
        ref_loader.REFERENCE_ROOT = ref_root
        ref = ref_loader.load()
        m = O.Model(**args)
        y = O.reshape_vector(m, x)
        nveh = 2
        while nveh * (nveh - 1) // 2 < npairs:
            nveh += 1
        ys = np.ascontiguousarray(y[:nveh * 3])
        ref.optimization.DEG_ELEV = E
        try:
            ref.optimization._temporalSeparationConstraints(ys, nveh, 3, m.maxSep)      # JIT + table caches
            t0 = time.perf_counter()
            c = ref.optimization._temporalSeparationConstraints(ys, nveh, 3, m.maxSep)
            dt = time.perf_counter() - t0
        finally:
            ref.optimization.DEG_ELEV = 0
        pairs = nveh * (nveh - 1) // 2
        P = m.numVeh * (m.numVeh - 1) // 2
        return {"value": 1.0 / (dt / pairs * P), "unit": "evals/s", "cores": 1, "kind": "reference",
                "us_per_pair": 1e6 * dt / pairs,
                "sample": "%d pairs (the first %d vehicles of the C4 swarm) through the unmodified reference's "
                          "_temporalSeparationConstraints (numpy + numba, 1 thread, warm caches), %.2f s; extrapolated "
                          "linearly to the %d pairs of one eval (speed rows not included)" % (pairs, nveh, dt, P),
                "check": float(np.abs(np.asarray(c)).max())}
    except Exception as e:          # pragma: no cover
        return {"unavailable": repr(e)}


# --------------------------------------------------------------------------
def _example1_problem(mod, veh_only=False):
    kw = dict(numVeh=2, dimension=2, degree=10, minimizeGoal='TimeOpt', maxSep=1, maxSpeed=5, maxAngRate=1,
              initPoints=[(0, 5), (3, 0)], finalPoints=[(8, 4), (7, 10)], initSpeeds=[1, 1], finalSpeeds=[1, 1],
              initAngs=[0, np.pi / 2], finalAngs=[0, np.pi / 2])
    if not veh_only:
        kw["pointObstacles"] = [[3, 2], [6, 7]]
    return kw


def slsqp_measure(full=False):
    """BASELINE configs[1] and [2]: wall seconds of scipy.optimize.minimize(method='SLSQP') with
    (i) the GPU closures (SciPy forms the Jacobians with nvar+1 calls), (ii) the GPU closures +
    their *_jac closures + objectiveFunction_jac (one batched launch per Jacobian), (iii) the
    restatement of the reference's callables on the host (C2: oracle.bezier_oracle, numpy;
    C3: oracle/bezier_oracle.c behind numpy's reshapeVector).
    C2 = Examples/Example1_DubinsCarTimeOptimal.py:95-148 at elev 0 (reference: tf =
    2.4276431891903045, nit 22); C3 = Examples/SwarmOfAerialVehicles.py:137-166 (36 vehicles,
    nvar 432, one separation constraint block of 6930 values).  The host arm of C3 costs minutes
    per run, so unless --slsqp-full is given arms (i) and (iii) of C3 are capped at `cap` major
    iterations (same cap for both; arm (ii) always runs to convergence)."""
    import scipy.optimize as sop
    from oracle import bezier_oracle as O
    from optimalbeziertrajectorygeneration_b200 import optimization as gopt

    def run(fun, x0, cons, jac=None, maxiter=250):
        t0 = time.perf_counter()
        res = sop.minimize(fun, x0=x0, method='SLSQP', jac=jac, constraints=cons, options={'maxiter': maxiter})
        return {"wall_s": time.perf_counter() - t0, "fun": float(res.fun), "nit": int(res.nit),
                "nfev": int(res.nfev), "success": bool(res.success), "maxiter": maxiter}

    out = {}
    # ---- C2 ----
    gopt.DEG_ELEV = 0
    b = gopt.BezOptimization(**_example1_problem(gopt))
    vo = gopt.BezOptimization(**_example1_problem(gopt, veh_only=True))     # the example's own separation closure
    x0 = b.generateGuess(std=0)
    last = lambda v: v[-1]
    cons = [{'type': 'ineq', 'fun': vo.temporalSeparationConstraints}, {'type': 'ineq', 'fun': b.maxSpeedConstraints},
            {'type': 'ineq', 'fun': b.maxAngularRateConstraints}, {'type': 'ineq', 'fun': last}]
    consj = [dict(c) for c in cons]
    consj[0]['jac'] = vo.temporalSeparationConstraints_jac
    consj[1]['jac'] = b.maxSpeedConstraints_jac
    consj[2]['jac'] = b.maxAngularRateConstraints_jac
    run(b.objectiveFunction, x0, consj, jac=b.objectiveFunction_jac, maxiter=2)          # warm-up (plans, tables)
    c2 = {"gpu_closures": run(b.objectiveFunction, x0, cons),
          "gpu_closures_jac": run(b.objectiveFunction, x0, consj, jac=b.objectiveFunction_jac)}
    mo = O.Model(**_example1_problem(gopt))
    fo, fv = O.make_callables(mo, 0), O.make_callables(O.Model(**_example1_problem(gopt, veh_only=True)), 0)
    c2["host_oracle"] = run(last, x0, [{'type': 'ineq', 'fun': fv['sep']}, {'type': 'ineq', 'fun': fo['maxspeed']},
                                       {'type': 'ineq', 'fun': fo['angrate']}, {'type': 'ineq', 'fun': last}])
    c2["reference_tf"] = 2.4276431891903045
    c2["problem"] = "Example1: 2 Dubins vehicles, degree 10, time-optimal, nvar 29, elev 0; constraints 21 + 42 + 82 + 1"
    out["c2"] = c2
    # ---- C3 ----
    g = np.load(os.path.join(ROOT, "tests", "golden", "constraints.npz"))
    kw = dict(numVeh=36, dimension=3, degree=5, minimizeGoal='Euclidean', maxSep=0.9,
              initPoints=g["swarm_initPts"], finalPoints=g["swarm_finalPts"])
    b = gopt.BezOptimization(**kw)
    x0 = g["swarm_x0"]
    cons = [{'type': 'ineq', 'fun': b.temporalSeparationConstraints}]
    consj = [{'type': 'ineq', 'fun': b.temporalSeparationConstraints, 'jac': b.temporalSeparationConstraints_jac}]
    run(b.objectiveFunction, x0, consj, jac=b.objectiveFunction_jac, maxiter=1)
    cap = 250 if full else 3
    c3 = {"gpu_closures_jac": run(b.objectiveFunction, x0, consj, jac=b.objectiveFunction_jac),
          "gpu_closures": run(b.objectiveFunction, x0, cons, maxiter=cap)}
    # host arm: the plain-C restatement (oracle/bezier_oracle.c, all host threads) behind numpy's
    # reshapeVector -- the numpy restatement needs 0.2 s per eval here (340 s for 3 iterations)
    from oracle import c_oracle as C
    mo = O.Model(**kw)
    obj = lambda v: O.euclidean_objective(O.reshape_vector(mo, v), 36, 3)
    hsep = lambda v: C.temporal_separation(O.reshape_vector(mo, v), 36, 3, 0.9, 0)
    c3["host_oracle"] = run(obj, x0, [{'type': 'ineq', 'fun': hsep}], maxiter=cap)
    c3["host_oracle"]["threads"] = C.max_threads()
    t0 = time.perf_counter()
    Jt = b.temporalSeparationConstraints_jac(x0)
    c3["jacobian_ms_gpu"] = 1e3 * (time.perf_counter() - t0)
    c3["jacobian_shape"] = list(Jt.shape)
    # the latency-bound regime: one closure call = H2D of x, assemble, pair kernel (630 x 11 values), D2H, sync
    f = b.temporalSeparationConstraints
    f(x0)
    t0 = time.perf_counter()
    for _ in range(433):
        f(x0)
    dt = time.perf_counter() - t0
    c3["closure_calls_per_s"] = 433 / dt
    c3["fd_jacobian_by_433_calls_ms"] = 1e3 * dt
    t0 = time.perf_counter()
    for _ in range(20):
        hsep(x0)
    c3["host_closure_calls_per_s"] = 20 / (time.perf_counter() - t0)
    c3["problem"] = ("SwarmOfAerialVehicles: 36 vehicles, 3-D, degree 5, nvar 432, DEG_ELEV 0, 630 pairs x 11 values; "
                     "objective at x0 = 382.0101330471013")
    out["c3"] = c3
    return out


# --------------------------------------------------------------------------
def c5_measure(opts, world, rank, local, steps):
    """BASELINE.json configs[4] (SURVEY 8(d) "C5"): independent Dubins time-optimal problems
    (1 vehicle, degree 10, DEG_ELEV 100, 16 point obstacles each); one step = one FD sweep
    (nvar+1 = 16 evals) of every problem of this rank's block.  Problems are dealt out in
    contiguous blocks (no collective).  Returns the measurement dict on rank 0."""
    import torch
    import torch.distributed as dist
    from optimalbeziertrajectorygeneration_b200 import optimization as gopt
    from optimalbeziertrajectorygeneration_b200 import sharding
    from optimalbeziertrajectorygeneration_b200.batch import ProblemBatch

    Mtot = opts.problems * world                                # weak scaling: problems per rank fixed
    lo, hi = sharding.block_range(Mtot, world, rank)
    M, E, nobs, deg = hi - lo, 100, 16, 10
    template = dict(numVeh=1, dimension=2, degree=deg, minimizeGoal='TimeOpt', maxSep=1, maxSpeed=3,
                    maxAngRate=np.pi / 2, initPoints=[(0, 0)], finalPoints=[(12, 8)], initSpeeds=[1],
                    finalSpeeds=[1], tf=8, initAngs=[np.pi / 2], finalAngs=[0])
    sets = np.stack([np.random.default_rng(p).uniform(1.0, 11.0, size=(nobs, 2)) for p in range(lo, hi)])
    pb = ProblemBatch(template, sets)
    guess = gopt.BezOptimization(**template).generateGuess(std=0)
    X = guess[None, :] + np.stack([np.random.default_rng(10 ** 6 + p).normal(size=guess.size) * 0.5
                                   for p in range(lo, hi)])
    X[:, -1] = np.abs(X[:, -1]) + 4.0                            # tf stays positive
    Xp, dx = pb.fd_points(X)
    nv1 = pb.nvar + 1
    d_X = Xp.view(M * nv1, pb.nvar)

    def step():
        return pb.evaluate(d_X, nv1, elev=E)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(3):
        F = step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        F = step()
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=pb.eng.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # per-block kernel times (CUDA events) to name the dominant kernel
    cpts, tf = pb.eng.assemble(d_X, E, obst_sets=pb.d_obst, evals_per_set=nv1)
    parts = {}
    for name, fn in (("separation", lambda: pb.eng.separation(cpts, E, 1.0, pair_begin=0, npairs=pb.npairs_x)),
                     ("maxspeed", lambda: pb.eng.speed(cpts, tf, E, -1.0, 9.0)),
                     ("angrate", lambda: pb.eng.angrate(cpts, tf, E, -1.0, (np.pi / 2) ** 2))):
        fn()
        parts[name] = _time_events(fn, 3, torch)
    del F, cpts, tf
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    L, A = 2 * deg + E + 1, 4 * (deg + E) + 1
    evals = M * nv1 * world * steps
    alg_eval = 8.0 * (pb.npairs_x * L + L + A + 2 * (deg + 1) + 1)       # SURVEY 8(d): 20 168 B
    peak, _ = _peak()
    m_ = deg + E
    fma_eval = 4 * (m_ + 1) ** 2 + 2 * (2 * m_ + 1) ** 2                    # SURVEY 8(d): 146 966 MAC
    return {"value": evals / (ms * 1e-3), "unit": "evals/s", "problems_per_gpu": M, "evals_per_problem": nv1,
            "steps": steps, "ms_per_step": ms / steps, "kernel_ms": parts,
            "hbm_frac_whole_step": alg_eval * M * nv1 / (ms / steps * 1e-3) / 1e9 / peak,
            "angrate_fp64_frac": fma_eval * M * nv1 / (parts["angrate"] * 1e-3) / (64 * 148 * 1.965e9),
            # rows written + the control-point rows of every evaluation read once (16 obstacle rows + the
            # vehicle row per evaluation: the 392 MB input of 131 072 evaluations does not stay in L2)
            "separation_hbm_frac": 8.0 * (pb.npairs_x * L + (pb.npairs_x + 1) * 2 * (deg + 1)) * M * nv1
                                   / (parts["separation"] * 1e-3) / 1e9 / peak,
            "separation_hbm_frac_rows_only": 8.0 * pb.npairs_x * L * M * nv1 / (parts["separation"] * 1e-3) / 1e9 / peak,
            "gpu_launches": 4 * steps,
            "workload": "C5 synthetic Dubins batch: %d problems per GPU x (nvar+1 = %d) FD points, 1 vehicle + 16 "
                        "point obstacles, dim 2, degree 10, DEG_ELEV 100: 16 separation rows + max-speed row + "
                        "angular-rate row per eval; contiguous blocks of problems per rank, no collective" % (M, nv1),
            "note": "fp64 peak = 64 FMA/clk/SM x 148 SMs x 1.965 GHz (tools/pipe_bench.cu)"}


def run_c5(opts):
    """`--workload c5`: the C5 measurement as its own line (the default line carries it as the key `c5`)."""
    import torch
    import torch.distributed as dist
    world, rank, local = _dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    sampler = ClockSampler(local, period=opts.clock_period)
    if rank == 0:
        sampler.open()
        sampler.start()
    c5 = c5_measure(opts, world, rank, local, steps=opts.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peak, _ = _peak()
        line = {"metric": "constraint+Jacobian evals/sec", "value": c5["value"], "unit": "evals/s",
                "n_gpus": world, "steps": opts.steps, "warmup": 3, "ms_per_step": c5["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": c5["workload"]}, "kernel_ms": c5["kernel_ms"],
                "roofline": {"bound": "fp64 (angular rate) / hbm (separation rows)",
                             "hbm_frac_whole_step": c5["hbm_frac_whole_step"],
                             "angrate_fp64_frac": c5["angrate_fp64_frac"],
                             "separation_hbm_frac": c5["separation_hbm_frac"], "peak": peak, "unit": "GB/s",
                             "note": c5["note"]},
                "gpu_launches": c5["gpu_launches"], "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0,
                    help="evals (x vectors) per step: per GPU with --scaling weak (default 4), in total with "
                         "--scaling strong (default 32 = the work of 8 weak-scaling ranks)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--clock-period", type=float, default=0.002, help="NVML sampling period in seconds")
    ap.add_argument("--nccl-gather", action="store_true",
                    help="multi-GPU: use the NCCL all-gather instead of the fused in-kernel peer stores")
    ap.add_argument("--no-sweep", action="store_true", help="skip the closed-form Jacobian sweep leg")
    ap.add_argument("--timeline", default=None, help="diagnostic: write the kernel timeline of the timed region to this file")
    ap.add_argument("--no-gather", action="store_true",
                    help="diagnostic: with N > 1 run N independent replicas without the all-gather of the per-pair minima")
    ap.add_argument("--workload", default="c4", choices=["c4", "c5"],
                    help="c4 = the headline swarm (default); c5 = batch of independent Dubins problems")
    ap.add_argument("--problems", type=int, default=8192, help="c5: problems per GPU")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default): B evals per GPU per step; strong: one batch of B evals, the pair list "
                         "cut into contiguous ranges per rank")
    ap.add_argument("--single-stream", action="store_true",
                    help="launch every step on one stream (round-1 behaviour) instead of two alternating ones")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 key of the default line")
    ap.add_argument("--no-slsqp", action="store_true", help="skip the slsqp_c2 / slsqp_c3 keys")
    ap.add_argument("--slsqp-full", action="store_true",
                    help="run every SLSQP arm of C3 to convergence (the host arm takes minutes)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps write what the last one computed to DIR/<name>.npy (float64, at most "
                         "64 MB: per-pair minima, max-speed rows, separation rows of a fixed seeded sample of pairs)")
    opts = ap.parse_args()
    if opts.steps < 1:
        ap.error("--steps must be at least 1")
    if opts.dump_outputs and (opts.impl != "ours" or opts.workload != "c4"):
        ap.error("--dump-outputs applies to the default workload (--impl ours --workload c4)")
    if opts.batch <= 0:
        opts.batch = 32 if opts.scaling == "strong" else 4
    if opts.impl == "reference":
        run_reference(opts)
    elif opts.workload == "c5":
        run_c5(opts)
    else:
        run_ours(opts)


if __name__ == "__main__":
    main()
