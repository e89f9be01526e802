#!/usr/bin/env python
"""bench.py — headline benchmark: local_laplacian (8 levels, alpha=1, beta=1) on synthetic uint16
frames, Mpixels/s (1 Mpx = 1e6 output pixels W*H, channels not counted).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Default workload = the north-star configuration of BASELINE.json: ONE 16384x16384x3 uint16 frame, levels=8,
alpha=1/7 (the harness passes alpha/(levels-1), apps/local_laplacian/process.cpp:31), beta=1.  At N=1 the whole
frame is filtered on one GPU; for N>1 (launched by torchrun, one rank per GPU) the SAME frame is row-sharded into
N bands of 16384/N rows ("strong" scaling: total work fixed): rank r owns rows [r*H/N, (r+1)*H/N), fetches a halo of
input rows from its neighbours and gathers one coarse pyramid level (halide_b200_local_laplacian_sharded).
`--workload local_laplacian_4k` times BASELINE.json configs[1] (3840x2160x3) the same way.

One JSON line on stdout (rank 0).  `value` is device-resident throughput (inputs in HBM), timed with CUDA events on
the launch stream over exactly K steps, max over ranks; `e2e` is the same metric through the C ABI with HOST
(pinned) buffers, H2D + D2H inside the timed region, one caller thread (the same form at every N).
`--dump-outputs DIR` writes what the last timed step returned to DIR/output.npy (DIR/output_rank<r>.npy per rank when
sharded) as float32: the whole output frame when it is small enough, else a fixed seeded sample of its elements.  The
inputs are seeded too, so two builds run with the same arguments can be compared output for output.
`--impl reference` times the CPU oracle (a port of the reference's algorithm — libHalide needs LLVM and cannot be
built in this image) on the box's host cores for the same config, on a bounded sample of the frame.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LEVELS = 8
ALPHA = 1.0 / 7.0   # alpha=1 divided by (levels-1), as process.cpp:31 does
BETA = 1.0
BYTES_PER_PX = 12   # SURVEY.md §8(d): 3 ch x 2 B in + 3 ch x 2 B out
DUMP_ELEMENTS = 15 << 20   # float32 values --dump-outputs writes over all ranks: 60 MB, within a 64 MB budget

WORKLOADS = {
    # name: (W, H) of the whole frame
    "local_laplacian_16k": (16384, 16384),
    "local_laplacian_8k": (7680, 4320),
    "local_laplacian_16k_quarter": (16384, 4096),   # what one rank of four sees (diagnostics)
    "local_laplacian_4k": (3840, 2160),
}
DEFAULT_WORKLOAD = "local_laplacian_16k"
CPU_FLAGS = "g++ -O3 -mavx2 -fopenmp -ffp-contract=off -fno-fast-math (oracle/Makefile)"
# The reference's own published number for its manual CPU schedule (apps/local_laplacian/local_laplacian_generator.cpp:139-140:
# 21.4 ms on the 1536x2560 harness frame, i9-9960X, 32 threads) — other hardware, printed for context only.
PUBLISHED_HALIDE_CPU = {"value": 1536 * 2560 / 1e6 / 21.4e-3, "unit": "Mpixels/s",
                        "what": "Halide manual CPU schedule, 21.4 ms on 1536x2560x3, i9-9960X 32 threads (generator :139-140); other hardware"}


def make_config(workload, world):
    """The `config` object — identical in both arms (ours / reference) for the same command line."""
    W, H = WORKLOADS[workload]
    return {"workload": workload, "levels": LEVELS, "alpha": 1, "beta": 1, "frame": [W, H, 3],
            "frame_per_gpu": [W, H // world, 3],
            "parallelism": "single GPU" if world == 1 else f"one frame row-sharded x{world} (strong scaling): input-row halo exchange + one gathered pyramid level",
            "l2": "frame pairs larger than the 126 MB L2 (rotating sets when one pair is not)",
            "input": "uniform random uint16, worst case for the remap-table gathers"}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """Samples SM clock / throttle reasons with NVML while the GPU is busy."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = [("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                 ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                 ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                 ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")]
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for label, attr in names:
                    bit = getattr(nv, attr, None)
                    if bit is not None and (r & bit):
                        self.reasons.add(label)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self._stop.clear()
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        if self._t is not None:
            self._stop.set()
            self._t.join()
            self._t = None

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(workload, kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel from the committed
    `ncu --set full` capture of this workload (profiles/traffic.json names the capture); (None, None) when there is none."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p))
        v = d.get(workload, {}).get(kernel)
        return (float(v), d.get("_source")) if v is not None else (None, None)
    except Exception:
        return None, None


def best_thread_count(img, candidates=None):
    """The oracle's OpenMP scaling flattens on very wide hosts (many small parallel regions over the coarse
    pyramid levels): time one frame at a few thread counts and keep the fastest — 'all the host threads it can use'."""
    from oracle import pyoracle
    ncores = pyoracle.use_all_cores()
    cands = sorted({c for c in (candidates or [8, 16, 32, 64, ncores]) if c <= ncores} | {min(ncores, 8)})
    best_n, best_t = cands[0], float("inf")
    for n in cands:
        pyoracle.set_threads(n)
        pyoracle.local_laplacian(img, LEVELS, ALPHA, BETA)
        t0 = time.perf_counter()
        pyoracle.local_laplacian(img, LEVELS, ALPHA, BETA)
        t = time.perf_counter() - t0
        if t < best_t:
            best_n, best_t = n, t
    pyoracle.set_threads(best_n)
    return best_n


def sample_rows(W, H, max_px=3840 * 2160):
    """Rows of the bounded CPU sample: the top rows of the frame, at most ~one 4K frame worth of pixels."""
    rows = H
    while rows > 64 and W * rows > max_px:
        rows //= 2
    return rows


def cpu_oracle_rate(W, H, budget_s=12.0, max_steps=8):
    """Time the CPU oracle on a bounded sample of the workload (full width, the top rows)."""
    import numpy as np
    from oracle import pyoracle
    rows = sample_rows(W, H)
    rng = np.random.default_rng(0)
    img = rng.integers(0, 65536, (3, rows, W), dtype=np.uint16)
    threads = best_thread_count(img)
    times = []
    t_all = time.perf_counter()
    while len(times) < max_steps and time.perf_counter() - t_all < budget_s:
        t0 = time.perf_counter()
        pyoracle.local_laplacian(img, LEVELS, ALPHA, BETA)
        times.append(time.perf_counter() - t0)
    best = min(times)
    return {"value": W * rows / 1e6 / best, "unit": "Mpixels/s", "cores": threads, "kind": "port",
            "sample": f"{len(times)} runs of a {W}x{rows}x3 band (the frame's top rows), best of; oracle/oracle_local_laplacian.cpp, "
                      f"{CPU_FLAGS}, {threads} OpenMP threads (fastest of a sweep up to all host cores)",
            "ms": best * 1e3, "published_reference": PUBLISHED_HALIDE_CPU}


def dump_outputs(directory, out, rank, world):
    """Saves one rank's output frame (uint16 on the device) as float32: whole when it fits this rank's share of
    DUMP_ELEMENTS, else the elements at a fixed seeded set of flat positions (the same set for the same shape)."""
    import numpy as np
    import torch
    flat = out.view(torch.int16).reshape(-1)   # (uint16 tensors support few ops; int16 carries the same bits)
    limit = DUMP_ELEMENTS // world
    if flat.numel() > limit:
        idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), limit))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    values = flat.cpu().numpy().view(np.uint16).astype(np.float32)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "output.npy" if world == 1 else f"output_rank{rank}.npy"), values)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port) on the host cores."""
    if rank != 0:
        return
    import numpy as np
    from oracle import pyoracle
    W, H = WORKLOADS[args.workload]
    rows = sample_rows(W, H)   # bounded sample so that the whole run stays within a few minutes
    rng = np.random.default_rng(0)
    img = rng.integers(0, 65536, (3, rows, W), dtype=np.uint16)
    threads = best_thread_count(img)
    for _ in range(max(1, args.warmup)):
        pyoracle.local_laplacian(img, LEVELS, ALPHA, BETA)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = pyoracle.local_laplacian(img, LEVELS, ALPHA, BETA)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        import torch
        dump_outputs(args.dump_outputs, torch.from_numpy(out.view(np.int16)), 0, 1)
    val = W * rows / 1e6 / dt
    sample = f"{args.steps} steps of a {W}x{rows}x3 band ({'full frame' if rows == H else 'the top rows of the frame'})"
    line = {"impl": "reference", "metric": "local_laplacian Mpixels/s", "value": val, "unit": "Mpixels/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 internal, u16 I/O",
            "data": "synthetic", "config": make_config(args.workload, max(1, args.gpus)),
            "cpu_baseline": {"value": val, "unit": "Mpixels/s", "cores": threads, "kind": "port",
                             "sample": sample + f"; {CPU_FLAGS}; {threads} OpenMP threads (fastest of a sweep up to all host cores)",
                             "published_reference": PUBLISHED_HALIDE_CPU},
            "e2e": {"value": val, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import halide_b200
    from halide_b200 import HalideBuffer, filters
    import halide_b200.lib as hlib

    torch.cuda.set_device(local_rank)
    halide_b200.capi.halide_b200_set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = td

    W, H = WORKLOADS[args.workload]
    if H % world:
        raise SystemExit(f"bench: frame height {H} is not divisible by {world} ranks")
    band_h = H // world          # strong scaling: the same frame, N bands
    dev = torch.device("cuda", local_rank)
    nbytes = 3 * band_h * W * 2
    # rotate frame pairs so that the working set exceeds the 126 MB L2 (one pair is enough for big frames)
    NSETS = max(1, min(4, -(-300_000_000 // (2 * nbytes))))
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    ins, outs = [], []
    for _ in range(NSETS):
        t = torch.randint(-32768, 32768, (3, band_h, W), dtype=torch.int16, device=dev, generator=gen).view(torch.uint16)
        ins.append(t)
        outs.append(torch.zeros((3, band_h, W), dtype=torch.uint16, device=dev))
    bins = [HalideBuffer.from_torch(t) for t in ins]
    bouts = [HalideBuffer.from_torch(t) for t in outs]

    comm = None
    if world > 1:
        from halide_b200 import dist as hdist
        sharder = hdist.RowSharder(rank, world, W, band_h)
        def step(i):
            sharder.local_laplacian(bins[i % NSETS], LEVELS, ALPHA, BETA, bouts[i % NSETS])
        # evidence of the communicator the data plane runs on (the library's own NCCL communicator, one rank per GPU)
        # and of the NVLink peer mapping, beside the driver's own comm_nranks check
        peers = [bool(torch.cuda.can_device_access_peer(local_rank, d)) if d != local_rank else None for d in range(torch.cuda.device_count())]
        info = [None] * world
        dist.all_gather_object(info, {"rank": rank, "device": local_rank, "lib_rank": int(halide_b200.capi.halide_b200_dist_rank()),
                                      "lib_nranks": int(halide_b200.capi.halide_b200_dist_size()), "rows": [sharder.lo, sharder.hi],
                                      "peer_access": peers})
        comm = {"backend": "nccl (library communicator, bootstrapped over torch.distributed)", "nranks": world,
                "gathered_level": int(hdist.shard_plan_level(W, H, world)), "ranks": info}
    else:
        def step(i):
            filters.local_laplacian(bins[i % NSETS], LEVELS, ALPHA, BETA, bouts[i % NSETS])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    # ---- device-resident timing ---------------------------------------------------------------
    for i in range(args.warmup):
        step(i)
    barrier()
    n0 = halide_b200.capi.halide_b200_kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    e0.record()
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    host_enqueue_ms = (time.perf_counter() - t_host0) / args.steps * 1e3   # host time to issue one step (async): must stay below ms_per_step
    e1.record()
    barrier()
    sampler.stop()
    launches = halide_b200.capi.halide_b200_kernel_launch_count() - n0
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs:   # (before anything below reuses the output buffers)
        dump_outputs(args.dump_outputs, outs[(args.steps - 1) % NSETS], rank, world)
    if dist is not None:
        tt = torch.tensor([ms_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt.item())
    ms_step = ms_total / args.steps
    total_px = W * H
    value = total_px / 1e6 / (ms_step / 1e3)

    # keep the GPU busy a little longer so the clock sampler has samples even for short runs
    # (a fixed step count: under sharding every rank must issue the same number of exchanges)
    need_more = len(sampler.samples) < 5
    if dist is not None:  # the decision must be collective: every rank issues the same number of exchanges
        tt = torch.tensor([1 if need_more else 0], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        need_more = bool(tt.item())
    if need_more:
        sampler.start()
        for i in range(max(20, int(300 / max(ms_step, 0.05)))):
            step(i)
        torch.cuda.synchronize()
        sampler.stop()

    # ---- context: the same step on a smooth frame (natural images are spatially coherent; the uniform-noise frame above
    # is the worst case for the LUT gathers and the per-pixel plane picks).  Reported as an extra, never as `value`.
    smooth_value = None
    if world == 1:
        yy = torch.arange(band_h, device=dev, dtype=torch.float32).view(1, band_h, 1)
        xx = torch.arange(W, device=dev, dtype=torch.float32).view(1, 1, W)
        t_s = torch.empty((3, band_h, W), dtype=torch.uint16, device=dev)
        for c in range(3):   # plane by plane: a 16K frame of f32 temporaries would be several GB
            sm = 0.5 + 0.45 * torch.sin(xx / (61.0 + c)) * torch.cos(yy / (83.0 - c)) + 0.01 * torch.rand((1, band_h, W), device=dev)
            t_s[c:c + 1].view(torch.int16).copy_((sm.clamp_(0, 1) * 65535.0).to(torch.int32).to(torch.int16))
            del sm
        b_s = HalideBuffer.from_torch(t_s)
        for _ in range(3):
            filters.local_laplacian(b_s, LEVELS, ALPHA, BETA, bouts[0])
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps_s = 10
        s0.record()
        for i in range(reps_s):
            filters.local_laplacian(b_s, LEVELS, ALPHA, BETA, bouts[i % NSETS])
        s1.record()
        torch.cuda.synchronize()
        smooth_value = W * H / 1e6 / (s0.elapsed_time(s1) / reps_s / 1e3)
        del b_s, t_s

    # ---- end-to-end through the C ABI with host buffers ------------------------------------------
    h_in = torch.empty((3, band_h, W), dtype=torch.uint16).pin_memory()
    h_in.view(torch.int16).copy_(ins[0].view(torch.int16))
    h_out = torch.empty((3, band_h, W), dtype=torch.uint16).pin_memory()
    b_hin, b_hout = HalideBuffer.from_torch(h_in), HalideBuffer.from_torch(h_out)
    b_hout.set_host_dirty(False)

    def e2e_step():
        b_hin.set_host_dirty(True)           # fresh host frame every step -> H2D inside the call
        if world > 1:
            sharder.local_laplacian(b_hin, LEVELS, ALPHA, BETA, b_hout)
        else:
            filters.local_laplacian(b_hin, LEVELS, ALPHA, BETA, b_hout)
        b_hout.copy_to_host()                 # D2H + stream sync: the result is on the host
    e2e_steps = max(3, min(args.steps, 20 if nbytes < 200_000_000 else 6))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if dist is not None:
        tt = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    e2e_value = total_px / 1e6 / e2e_s
    e2e = {"value": e2e_value, "unit": "Mpixels/s", "h2d_bytes_per_step": nbytes * world, "d2h_bytes_per_step": nbytes * world,
           "ms_per_step": e2e_s * 1e3, "steps": e2e_steps, "host_memory": "pinned",
           "mode": "one caller thread per rank: H2D, kernels, D2H back to back (the same form at every N)"}
    if world == 1:
        # Context only (not `e2e.value`): a caller with several frames in hand (video) keeps DEPTH frames in flight, one
        # thread + CUDA stream each (halide_b200.FramePipeline): every step still copies its own input up and its own
        # result down, but frame i's D2H overlaps frame i+1's kernels and frame i+2's H2D on the full-duplex link.
        from halide_b200 import FramePipeline
        try:
            DEPTH = 3 if nbytes < 200_000_000 else 2   # (a 16K frame in flight = 3.2 GB of pinned host memory + ~8 GB of device scratch)
            slots = []
            for k in range(DEPTH):
                hi = torch.empty((3, band_h, W), dtype=torch.uint16).pin_memory()
                hi.view(torch.int16).copy_(ins[k % NSETS].view(torch.int16))
                ho = torch.empty((3, band_h, W), dtype=torch.uint16).pin_memory()
                bi, bo = HalideBuffer.from_torch(hi), HalideBuffer.from_torch(ho)
                bo.set_host_dirty(False)
                slots.append((bi, bo, hi, ho))

            def job(k):
                bi, bo = slots[k][0], slots[k][1]
                bi.set_host_dirty(True)
                filters.local_laplacian(bi, LEVELS, ALPHA, BETA, bo)
                bo.copy_to_host()

            pipe_steps = 3 * e2e_steps if nbytes < 200_000_000 else 8
            with FramePipeline(DEPTH, device=local_rank) as fp:
                for t in [fp.submit(job, k % DEPTH, slot=k % DEPTH) for k in range(2 * DEPTH)]:
                    fp.result(t)
                t0 = time.perf_counter()
                for t in [fp.submit(job, k % DEPTH, slot=k % DEPTH) for k in range(pipe_steps)]:
                    fp.result(t)
                e2e_pipe_s = (time.perf_counter() - t0) / pipe_steps
            # the pipelined frames must be the same bits as the serial call's
            if not torch.equal(slots[0][3].view(torch.int16), h_out.view(torch.int16)):
                raise SystemExit("bench: pipelined e2e output differs from the serial call")
            e2e["pipelined"] = {"value": total_px / 1e6 / e2e_pipe_s, "ms_per_step": e2e_pipe_s * 1e3, "steps": pipe_steps,
                                "mode": "FramePipeline depth %d: %d caller threads, one CUDA stream each" % (DEPTH, DEPTH)}
        except (RuntimeError, MemoryError) as exc:   # (out of pinned / device memory: the serial number above stands)
            e2e["pipelined"] = {"error": str(exc)[:300]}

    # ---- per-kernel profile for the roofline (event-bracketed launches, separate pass) --------------
    roofline, kernels = None, {}
    hlib.profile(True)
    hlib.profile_reset()
    reps = 5
    for i in range(reps):   # every rank runs the pass (exchanges pair up); rank 0 reports
        step(i)
    torch.cuda.synchronize()
    rep = hlib.profile_report()
    hlib.profile(False)
    if rank == 0:
        kernels = {k: {"launches_per_step": c / reps, "ms_per_launch": ms / c, "ms_per_step": ms / reps} for k, (c, ms) in rep.items()}
        if rep:
            # dominant kernel = the largest single-launch mean (a name launched several times per step on levels of
            # different sizes must not win by its sum)
            name, (cnt, ms) = max(rep.items(), key=lambda kv: kv[1][1] / kv[1][0])
            avg_s = ms / cnt / 1e3
            peak, how = measured_peak()
            alg_bytes = BYTES_PER_PX * W * band_h  # 12 B/px x the pixels one launch of a full-resolution kernel covers on this rank
            achieved = alg_bytes / avg_s / 1e9
            pipe_ms = sum(v[1] for v in rep.values()) / reps
            traffic, traffic_src = recorded_traffic(args.workload, name) if world == 1 else (None, None)
            roofline = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": how,
                        "kernel_ms": avg_s * 1e3, "algorithmic_bytes": alg_bytes,
                        "step_kernel_ms": pipe_ms,
                        "step_frac": alg_bytes / (pipe_ms / 1e3) / 1e9 / peak,
                        "note": "achieved = 12 B/px x this rank's pixels / the dominant kernel's mean launch time; step_frac = the same bytes over "
                                "the sum of all kernel times of a step (what the north-star's 70 % asks about)"}

    if dist is not None:
        dist.barrier()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    cpu = cpu_oracle_rate(W, H)
    cfg = make_config(args.workload, world)   # (identical to the reference arm's for the same command line)
    line = {"metric": "local_laplacian Mpixels/s", "value": value, "unit": "Mpixels/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32 internal, u16 I/O", "data": "synthetic",
            "config": cfg, "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": sampler.summary(),
            "kernels": kernels, "comm": comm, "host_enqueue_ms_per_step": host_enqueue_ms,
            "l2_detail": f"rotating {NSETS} device-resident frame pair(s) per GPU ({NSETS * 2 * nbytes / 1e6:.0f} MB) > 126 MB L2",
            "extra": {"smooth_frame_Mpixels_per_s": smooth_value,
                      "note": "same call on a low-frequency synthetic frame (coherent LUT / plane gathers); context only"}}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        print(json.dumps({"error": f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks"}), flush=True)
        sys.exit(2)
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
