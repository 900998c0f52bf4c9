#!/usr/bin/env python
"""Benchmark of the mastering hot path (BASELINE.json metric): stereo samples/sec as x real-time.

  python bench.py --gpus N --steps K --warmup W                 # this repo's CUDA path, BASELINE config 2
  python bench.py --workload c3|c5 ...                          # BASELINE configs 3 and 5 (one GPU)
  python bench.py --impl reference --steps K --warmup W         # the reference's CPU algorithm (oracle port)
  python bench.py ... --dump-outputs DIR                        # also write the last timed step's result to DIR

Workloads (SURVEY.md 8d recipes, synthetic):
  c2  3-minute 44.1 kHz stereo track vs a 3-minute reference, full pipeline stages.main(need_default);
      one track per GPU per step (tracks shard one-per-GPU, NCCL only gathers the timings)   [headline]
  c3  10-minute 96 kHz stereo track vs a 10-minute reference, full pipeline
  c5  limiter.limit() alone on one hour of 44.1 kHz stereo

One JSON line on stdout (rank 0):
  value     device-resident throughput: inputs already in HBM, `--lanes` tracks in flight, CUDA events
  e2e       the same job through the repo's public API at the reference's own seam --
            stages.main(float64 numpy, pageable) -> float64 numpy (c5: limiter.limit) -- one synchronous
            call per step, host->device and device->host copies inside the timed region (wall clock between
            device synchronisations).  Beside it: the C batch entry with pinned float32 / int16 buffers
            (e2e.batch_f32, e2e.batch_pcm16), mgb_process_host (e2e.single_call_f32) and mg.process on
            16-bit WAV files (e2e.process_files).
  roofline  the dominant kernel's algorithmic bytes per launch / its CUDA-event duration / measured HBM peak
"""
from __future__ import annotations

import argparse
import atexit
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "stereo 44.1kHz samples/sec (x real-time)"
UNIT = "x real-time"

WORKLOADS = {
    "c2": dict(sample_rate=44100, seconds=180.0, kind="pipeline",
               text="config 2: 180-s stereo 44.1 kHz synthetic track vs 180-s reference, full pipeline "
                    "stages.main(need_default), one track per GPU per step"),
    "c3": dict(sample_rate=96000, seconds=600.0, kind="pipeline",
               text="config 3: 600-s stereo 96 kHz synthetic track vs 600-s reference, full pipeline "
                    "stages.main(need_default), Config(internal_sample_rate=96000)"),
    "c5": dict(sample_rate=44100, seconds=3600.0, kind="limiter",
               text="config 5: Hyrax limiter alone, limiter.limit() on a 3600-s stereo 44.1 kHz buffer"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--seconds", type=float, default=None, help="override the workload's track length (tuning runs only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-files", action="store_true", help="skip the mg.process-on-WAV-files leg")
    ap.add_argument("--reference-budget-s", type=float, default=360.0,
                    help="reference arm: wall-clock budget for all steps; the per-step sample shrinks to fit")
    ap.add_argument("--lanes", type=int, default=6, help="tracks in flight per GPU for the device-resident number")
    ap.add_argument("--opt", action="append", default=[], help="library switch name=value (A/B measurements)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline path computed to DIR/<name>.npy (see dump_sample)")
    return ap.parse_args()


def workload_config(args) -> dict:
    """The description both arms print as `config` (the GPU arm adds how it ran it)."""
    w = WORKLOADS[args.workload]
    seconds = args.seconds if args.seconds else w["seconds"]
    n = int(w["sample_rate"] * seconds)
    return {"workload": w["text"] if not args.seconds else w["text"] + f" [track length overridden: {seconds:.0f} s]",
            "name": args.workload, "sample_rate": w["sample_rate"], "frames_per_track": n,
            "l2": "inputs larger than the 126 MB L2 between timed iterations: "
                  + ("3 rotating tracks per GPU, ~290 MB touched per step" if args.workload == "c2"
                     else f"one track is {n * 8 / 1e6:.0f} MB per signal"),
            "precision": "GPU arm: float32 I/O and FFTs, float64 reductions / FIR design / IIR state; CPU arm: float64"}


def oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import port
    return port


# --------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi while the timed region runs
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 100 ms in a child process that is started EARLY (its start-up can take
    seconds on a cold box); the samples that count are the ones time-stamped inside the timed window."""
    QUERY = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.t_begin = self.t_end = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)  # the poller never outlives the benchmark, however it ends
        except (OSError, FileNotFoundError):
            self.proc = None

    def begin(self, wait_s: float = 15.0):
        """Start of the timed window; waits (bounded) until the poller has produced its first line."""
        if self.proc is not None:
            deadline = time.time() + wait_s
            while time.time() < deadline and os.path.getsize(self.path) == 0 and self.proc.poll() is None:
                time.sleep(0.05)
        self.t_begin = time.time()

    def end(self):
        self.t_end = time.time()

    @staticmethod
    def _stamp(text: str):
        import datetime
        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        if self.t_end is None:
            self.end()
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            for line in f:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 10:
                    continue
                try:
                    rows.append((self._stamp(parts[0]), float(parts[2]), float(parts[3]),
                                 [n for n, v in zip(names, parts[6:10]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
        os.unlink(self.path)
        lo, hi = (self.t_begin or 0.0) - 0.05, (self.t_end or time.time()) + 0.15
        inside = [r for r in rows if r[0] is not None and lo <= r[0] <= hi]
        scope = "timed window"
        if not inside:  # clock skew or an unparsable stamp: fall back to everything the poller saw
            inside, scope = rows, "whole run"
        sm = sorted(r[1] for r in inside)
        reasons = sorted({n for r in inside for n in r[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": inside[-1][2] if inside else None,
                "samples": len(sm), "scope": scope, "reasons": reasons}


# --------------------------------------------------------------------------------------------------
# the reference arm: the reference's CPU algorithm (oracle/port.py, numpy/scipy float64) on the host cores
# --------------------------------------------------------------------------------------------------
def usable_cores() -> int:
    """Hardware threads this process may really use: the affinity mask, cut by a cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            text = open(path).read().split()
            if path.endswith("cpu.max"):
                if text[0] != "max":
                    n = min(n, max(1, int(int(text[0]) / int(text[1]))))
            else:
                quota = int(text[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, quota // period))
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def physical_cores() -> int:
    """Distinct (socket, core) pairs among the CPUs of the affinity mask (hyperthread siblings count once:
    the port's numpy/scipy kernels are memory-bound and gain nothing from a second thread per core)."""
    try:
        allowed = os.sched_getaffinity(0)
        pairs, cpu, phys = set(), None, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id") and cpu in allowed:
                pairs.add((phys, int(line.split(":")[1])))
        return len(pairs) or len(allowed)
    except (OSError, ValueError):
        return os.cpu_count() or 1


def mem_available_gb() -> float:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / (1 << 20)
    except OSError:
        pass
    return 64.0


_WORKER_INPUTS = {}


def _reference_worker(job):
    """One worker masters one synthetic track (its own seed) with the oracle port; the inputs are cached
    per process: synthesising noise is not part of the measured path."""
    name, sample_rate, seconds = job
    os.environ["OMP_NUM_THREADS"] = "1"
    port = oracle()
    import numpy as np
    key = (name, seconds)
    if key not in _WORKER_INPUTS:
        _WORKER_INPUTS.clear()
        n = int(sample_rate * seconds)
        seed = os.getpid() % 1000
        if name == "c5":
            _WORKER_INPUTS[key] = (port.synth_limiter_input(n, seed).astype(np.float64),)
        else:
            _WORKER_INPUTS[key] = (port.synth_target(n, seed).astype(np.float64),
                                   port.synth_reference(n, 1000 + seed).astype(np.float64))
    data = _WORKER_INPUTS[key]
    cfg = port.OracleConfig(internal_sample_rate=sample_rate)
    t0 = time.perf_counter()
    if name == "c5":
        port.limit(data[0], cfg)
    else:
        port.main(data[0], data[1], cfg, True, False, False)
    return time.perf_counter() - t0


def run_reference(args) -> dict:
    """Reference arm.  /root/reference is pure Python over numpy/scipy and cannot travel to the GPU box, so
    this times oracle/port.py -- a float64 numpy/scipy restatement of the same algorithm (its own blocked
    sliding maxima and reshape+rfft STFT in place of scipy.ndimage / scipy.signal.stft; pinned to the
    unmodified reference at 1e-12 by tests/test_oracle_port.py) -- with one single-threaded worker process
    per usable physical core, every worker mastering one track of the workload per step.  The track is the
    workload's own length unless a calibration step shows that K+W such steps would not fit
    --reference-budget-s; then each step is a shorter track of the same recipe, and the line says so."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return {}
    wcfg = workload_config(args)
    name, sr = wcfg["name"], wcfg["sample_rate"]
    full_seconds = wcfg["frames_per_track"] / sr
    gb_per_worker = {"c2": 2.0, "c3": 14.0, "c5": 15.0}[name] * (full_seconds / WORKLOADS[name]["seconds"])
    workers = max(1, min(usable_cores(), physical_cores(), int(0.7 * mem_available_gb() / max(gb_per_worker, 0.1))))
    ctx = mp.get_context("fork")
    total_steps = args.steps + max(1, args.warmup)
    with ctx.Pool(workers) as pool:
        # calibration (untimed, outside the warm-up): a short track per worker; the port's cost is linear in length
        cal_seconds = min(full_seconds, 20.0)
        pool.map(_reference_worker, [(name, sr, cal_seconds)] * workers, chunksize=1)
        t0 = time.perf_counter()
        pool.map(_reference_worker, [(name, sr, cal_seconds)] * workers, chunksize=1)
        cal = time.perf_counter() - t0
        projected = cal * (full_seconds / cal_seconds) * total_steps
        sample = full_seconds
        if projected > args.reference_budget_s:
            sample = max(10.0, float(int(full_seconds * args.reference_budget_s / projected)))
        job = (name, sr, sample)
        for w in range(max(1, args.warmup)):  # also fills every worker's input cache
            pool.map(_reference_worker, [job] * workers, chunksize=1)
        t0 = time.perf_counter()
        for step in range(args.steps):
            pool.map(_reference_worker, [job] * workers, chunksize=1)
        elapsed = time.perf_counter() - t0
    frames = args.steps * workers * int(sr * sample)
    value = frames / elapsed / sr
    whole = sample == full_seconds
    desc = (f"{workers} single-threaded worker processes (host: {os.cpu_count()} hardware threads, {usable_cores()} usable, "
            f"{physical_cores()} physical cores, {mem_available_gb():.0f} GB free), each mastering one "
            f"{sample:.0f}-s track of the workload's recipe per step"
            + ("" if whole else f" (bounded sample: the full {full_seconds:.0f}-s track would need ~{projected:.0f} s for "
                                f"{total_steps} steps, over the {args.reference_budget_s:.0f}-s budget)")
            + "; oracle/port.py, float64 numpy/scipy")
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "samples_per_sec": frames / elapsed,
        "config": wcfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": desc,
                         "seconds_per_track": sample, "whole_workload_track": whole},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


# --------------------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------------------
ALGORITHMIC_BYTES_PER_FRAME = {
    # SURVEY.md section 8(d): compulsory HBM bytes per stereo frame of the signal a launch covers
    "analyze_kernel": 8,      # read L,R once
    "convolve_kernel": 16,    # read L,R, write result L,R
    "clip_sumsq_kernel": 4,   # re-read the mid plane
    "limiter_kernel": 16,     # read result, write final
}
# real FP32 operations per stereo frame of the two FFT kernels (DESIGN.md section 4), for the CUDA-core roof
FP32_OPS_PER_FRAME = {"convolve_kernel": 217.0, "analyze_kernel": 75.0}  # (convolution: 4F-point frames, 3F outputs; 290 with 2F frames)
DUMP_BYTES = 64 * 10 ** 6  # --dump-outputs writes at most this much in all


def dump_sample(y) -> dict:
    """--dump-outputs: a (frames, 2) float32 CUDA tensor -> {name: numpy array} to write as <name>.npy.  The
    whole array as "result" when it fits DUMP_BYTES (config 2's 3-minute track does); otherwise one frame
    drawn from each of equal stretches of the buffer by a fixed seed, as "result", and those frames' indices
    as "result_frames" (float64), so that two builds dump the same frames.  Two runs of one build agree to a
    float32 rounding step, not bit for bit (config 2 on a B200: 6e-8 max-abs)."""
    import numpy as np
    import torch
    room = DUMP_BYTES - 4096  # (two .npy headers)
    if y.numel() * y.element_size() <= room:
        return {"result": y.cpu().numpy()}
    n, m = y.shape[0], room // (y.shape[1] * y.element_size() + 8)
    edges = np.linspace(0, n, m + 1).astype(np.int64)
    frames = edges[:-1] + (np.random.default_rng(0).random(m) * np.diff(edges)).astype(np.int64)
    picked = y.index_select(0, torch.from_numpy(frames).to(y.device))
    return {"result": picked.cpu().numpy(), "result_frames": frames.astype(np.float64)}


def run_b200(args) -> dict:
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    sampler = ClockSampler(local_rank)  # (polls from now on; only samples inside the timed window are reported)
    if rank == 0:
        sampler.start()
    # every rank stays on the cores (and memory) next to its own GPU; the host transport's worker threads are
    # created later and inherit the mask.  Ranks that share a socket share its cores: divide the workers.
    from matchering_b200.sharding import bind_host_thread_near_gpu
    bound_cores = bind_host_thread_near_gpu(local_rank)
    if world > 1:
        # keep stdout for the one JSON line: NCCL prints its version banner there at VERSION level
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=device)
        mine = sorted(os.sched_getaffinity(0))
        everyone = [None] * world
        dist.all_gather_object(everyone, mine)
        sharing = sum(1 for other in everyone if other and other[0] == mine[0])  # ranks on this rank's socket
        if "MGB_HOST_THREADS" not in os.environ:
            # ranks whose GPUs hang off the same socket share its hardware threads: one worker per thread in all
            # (measured with four ranks on one 64-thread socket: 16 workers each 7.8 ms per call, 8 each 9.2 ms)
            # ... and all ranks share the container's CPU quota (usable_cores): leave the main threads their share
            budget = min(len(mine) // max(1, sharing), usable_cores() // world - 3)
            os.environ["MGB_HOST_THREADS"] = str(max(4, min(16, budget)))
        # The transport's two modes (csrc/hostio.cu): "streaming" (staging chunks written past the caches, every
        # staged byte crosses the socket's memory twice more; fastest for one or two ranks per socket) and "cached"
        # (ordinary stores into a 4 MB ring that stays in the cores' caches, results by one DMA: no staging traffic
        # in memory, what ranks that compete for one socket's memory bandwidth want).
        mode = os.environ.get("MGB_BENCH_SHARED_SOCKET_MODE", SHARED_SOCKET_MODE if sharing >= 3 else "streaming")
        if mode == "cached":
            os.environ.setdefault("MGB_HOST_NT", "0")
            os.environ.setdefault("MGB_DOWNLOAD_RING", "0")

    port = oracle()  # synthetic-input recipes + the cpu_baseline leg only
    import matchering_b200 as mg
    from matchering_b200 import _native, stages
    from matchering_b200.engine import HostIO, TrackSession, get_plan, limiter_params
    from matchering_b200.limiter import limit as mg_limit
    from matchering_b200.plan import limiter_constants

    wcfg = workload_config(args)
    name, sr, n = wcfg["name"], wcfg["sample_rate"], wcfg["frames_per_track"]
    is_limiter = WORKLOADS[name]["kind"] == "limiter"
    seconds = n / sr
    cfg = mg.Config(internal_sample_rate=sr)
    plan = get_plan(cfg, device)
    lib = plan.lib
    for item in args.opt:
        opt_name, opt_value = item.split("=")
        _native.check(lib, lib.mgb_set_option(opt_name.encode(), int(opt_value)))
    stream = torch.cuda.current_stream(device)
    sptr = C.c_void_p(stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed_events(fn, steps, warmup):
        for k in range(warmup):
            fn(k)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = lib.mgb_launch_count()
        e0.record(stream)
        for k in range(steps):
            fn(warmup + k)
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1), lib.mgb_launch_count() - launches0

    def timed_wall(fn, steps, warmup):
        """Synchronous host-API calls: wall clock between two device synchronisations (+ barrier)."""
        for k in range(warmup):
            fn(k)
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            fn(warmup + k)
        torch.cuda.synchronize(device)
        ms = (time.perf_counter() - t0) * 1e3
        barrier()
        return ms

    # ---- inputs: distinct tracks per rank, rotated, so no step finds its inputs in the 126 MB L2 (config 2:
    # three 64 MB tracks; configs 3 and 5: one buffer of 0.46 / 1.27 GB, several times the L2 by itself)
    n_sets = 3 if name == "c2" else 1
    host_t, host_r, dev_t, dev_r = [], [], [], []
    for k in range(n_sets):
        seed = rank * 16 + k
        if is_limiter:
            t = torch.from_numpy(port.synth_limiter_input(n, seed)).pin_memory()
            r = t
        else:
            t = torch.from_numpy(port.synth_target(n, seed)).pin_memory()
            r = torch.from_numpy(port.synth_reference(n, 1000 + seed)).pin_memory()
        host_t.append(t)
        host_r.append(r)
        dev_t.append(t.to(device))
        dev_r.append(dev_t[-1] if is_limiter else r.to(device))

    legs = {}
    # =============================================================================================
    # device-resident
    # =============================================================================================
    if is_limiter:
        params = limiter_params(limiter_constants(cfg))
        ws_bytes = int(lib.mgb_limiter_workspace_bytes(C.byref(params), n))
        lim_ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)
        lim_out = torch.empty((n, 2), dtype=torch.float32, device=device)
        lim_flag = torch.zeros(1, dtype=torch.int32, device=device)

        def step_device(k):
            _native.check(lib, lib.mgb_limit(C.byref(params), dev_t[k % n_sets].data_ptr(), lim_out.data_ptr(), n,
                                             lim_ws.data_ptr(), ws_bytes, lim_flag.data_ptr(), sptr))
        n_lanes = 1
    else:
        # `--lanes` tracks in flight on as many streams: one track's small latency-bound kernels (FIR design)
        # overlap another's streaming kernels
        n_lanes = max(1, args.lanes)
        sessions = [TrackSession(plan, n, n) for _ in range(n_lanes)]
        lane_streams = [torch.cuda.Stream(device=device) for _ in range(n_lanes)]
        lane_out = [torch.empty((n, 2), dtype=torch.float32, device=device) for _ in range(n_lanes)]
        session, out_dev = sessions[0], lane_out[0]
        p_plan = C.byref(plan.struct)

        def step_on(k, sess, out, stream_ptr):
            t, r = dev_t[k % n_sets], dev_r[k % n_sets]
            lay, w, s_ = C.byref(sess.layout), sess.workspace.data_ptr(), sess.state.data_ptr()
            _native.check(lib, lib.mgb_match_levels(p_plan, lay, t.data_ptr(), r.data_ptr(), w, s_, stream_ptr))
            _native.check(lib, lib.mgb_match_frequencies(p_plan, lay, t.data_ptr(), sess.result.data_ptr(), None, w, s_, stream_ptr))
            _native.check(lib, lib.mgb_correct_levels(p_plan, lay, w, s_, stream_ptr))
            _native.check(lib, lib.mgb_finalize(p_plan, lay, sess.result.data_ptr(), out.data_ptr(), None, None, w, s_, stream_ptr))

        def step_device(k):  # one stream, one track at a time (profiling pass, single-track latency)
            step_on(k, session, out_dev, sptr)

        def timed_lanes(steps, warmup):
            """K tracks, alternating over the lanes; CUDA events on the main stream bracket all of them."""
            for k in range(warmup):
                step_on(k, sessions[k % n_lanes], lane_out[k % n_lanes], C.c_void_p(lane_streams[k % n_lanes].cuda_stream))
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            launches0 = lib.mgb_launch_count()
            e0.record(stream)
            for ls in lane_streams:
                ls.wait_event(e0)
            for k in range(steps):
                lane = k % n_lanes
                step_on(warmup + k, sessions[lane], lane_out[lane], C.c_void_p(lane_streams[lane].cuda_stream))
            for ls in lane_streams:
                stream.wait_stream(ls)
            e1.record(stream)
            barrier()
            return e0.elapsed_time(e1), lib.mgb_launch_count() - launches0

    # =============================================================================================
    # end to end at the reference's seam: pageable float64 numpy in, float64 numpy out, one call per step
    # =============================================================================================
    io = HostIO.get()
    seam_t = [t.numpy().astype(np.float64) for t in host_t]                 # pageable, like soundfile's arrays
    seam_r = seam_t if is_limiter else [r.numpy().astype(np.float64) for r in host_r]
    if is_limiter:
        def step_seam(k):
            out = mg_limit(seam_t[k % n_sets], cfg)
            assert out.dtype == np.float64 and out.shape == (n, 2)
    else:
        def step_seam(k):
            out = stages.main(seam_t[k % n_sets], seam_r[k % n_sets], cfg)[0]
            assert out.dtype == np.float64 and out.shape == (n, 2)

    # ---- the C batch entry (three tracks in flight, pinned float32 / int16 buffers) and mgb_process_host
    pipe = None
    if not is_limiter and name == "c2":
        from matchering_b200.batch import MasteringPipeline
        depth = 3
        pipe = MasteringPipeline(cfg, n, n, depth, device)
        outs_host = [torch.empty((n, 2), dtype=torch.float32).pin_memory() for _ in range(depth)]
        s_h2d, _, s_d2h = (torch.cuda.ExternalStream(p, device=device) for p in pipe.streams())
        pcm_t = [torch.from_numpy((t.numpy() * 32767.0).round().astype(np.int16)).pin_memory() for t in host_t]
        pcm_r = [torch.from_numpy((r.numpy() * 32767.0).round().astype(np.int16)).pin_memory() for r in host_r]
        pcm_out = [torch.empty((n, 2), dtype=torch.int16).pin_memory() for _ in range(depth)]
        out_host = torch.empty((n, 2), dtype=torch.float32).pin_memory()
        stage_t = torch.empty((n, 2), dtype=torch.float32, device=device)
        stage_r = torch.empty((n, 2), dtype=torch.float32, device=device)

        def timed_pipeline(steps, warmup, pcm=False):
            if pcm:
                def submit(k, slot_k):
                    pipe.submit_pcm(pcm_t[k % n_sets], pcm_r[k % n_sets], pcm_out[slot_k % depth])
            else:
                def submit(k, slot_k):
                    pipe.submit(host_t[k % n_sets], host_r[k % n_sets], outs_host[slot_k % depth])
            for k in range(warmup):
                submit(k, k)
            pipe.wait_all()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s_h2d)
            for k in range(steps):
                submit(warmup + k, k)
            pipe.wait_all()
            e1.record(s_d2h)
            barrier()
            return e0.elapsed_time(e1)

        def step_host(k):
            _native.check(lib, lib.mgb_process_host(
                p_plan, C.byref(session.layout), host_t[k % n_sets].data_ptr(), host_r[k % n_sets].data_ptr(),
                out_host.data_ptr(), None, None, stage_t.data_ptr(), stage_r.data_ptr(), session.result.data_ptr(),
                out_dev.data_ptr(), session.workspace.data_ptr(), session.state.data_ptr(), None, sptr))

    # ---- mg.process on 16-bit WAV files (rank 0, config 2 only): file read, device mastering, file write
    files_dir = None
    if rank == 0 and name == "c2" and not args.no_files:
        from matchering_b200 import wavio
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        files_dir = tempfile.mkdtemp(dir=base)
        wavio.write(os.path.join(files_dir, "t.wav"), host_t[0].numpy(), sr, "PCM_16")
        wavio.write(os.path.join(files_dir, "r.wav"), host_r[0].numpy(), sr, "PCM_16")

        def step_files(k):
            mg.process(os.path.join(files_dir, "t.wav"), os.path.join(files_dir, "r.wav"),
                       [mg.pcm16(os.path.join(files_dir, "o.wav"))], config=cfg)

    # =============================================================================================
    # the timed region
    # =============================================================================================
    warm = max(3, args.warmup)
    dumped = None
    sampler.begin()
    if is_limiter:
        dev_ms, launches = timed_events(step_device, args.steps, warm)
        if args.dump_outputs and rank == 0:
            dumped = dump_sample(lim_out)
        dev_serial_ms = dev_ms
    else:
        dev_ms, launches = timed_lanes(args.steps, warm)
        if args.dump_outputs and rank == 0:  # (before the single-stream pass below reuses lane 0's buffer)
            dumped = dump_sample(lane_out[(args.steps - 1) % n_lanes])
        dev_serial_ms, _ = timed_events(step_device, args.steps, warm)
    seam_ms = timed_wall(step_seam, args.steps, warm)
    if pipe is not None:
        legs["single_call_f32"] = timed_events(step_host, args.steps, warm)[0]
        legs["batch_f32"] = timed_pipeline(args.steps, warm)
        legs["batch_pcm16"] = timed_pipeline(args.steps, warm, pcm=True)
    sampler.end()
    clocks = sampler.stop() if rank == 0 else None
    files_ms = None
    if files_dir is not None:  # outside the clock window: dominated by host file I/O
        files_steps = min(args.steps, 5)
        files_ms = timed_wall(step_files, files_steps, 2) / files_steps
    if pipe is not None:
        pipe.close()

    # max over ranks of the times
    keys = ["dev", "serial", "seam"] + sorted(legs)
    mine = [dev_ms, dev_serial_ms, seam_ms] + [legs[k] for k in sorted(legs)]
    if world > 1:
        tms = torch.tensor(mine, dtype=torch.float64, device=device)
        gathered = [torch.zeros_like(tms) for _ in range(world)]
        dist.all_gather(gathered, tms)
        mine = [max(float(g[i]) for g in gathered) for i in range(len(mine))]
    times = dict(zip(keys, mine))
    frames_total = world * args.steps * n
    xrt = lambda ms: frames_total / (ms * 1e-3) / sr

    result = None
    if rank == 0:
        # ---- per-kernel durations: a separate profiled pass (CUDA events around every launch) ----
        lib.mgb_profile_enable(1)
        prof_steps = 5
        for k in range(prof_steps):
            step_device(k)
        cap = 4096
        names = C.create_string_buffer(1 << 16)
        ms = (C.c_float * cap)()
        got = lib.mgb_profile_collect(names, len(names), ms, cap)
        lib.mgb_profile_enable(0)
        per_kernel = {}
        for kname, t in zip(names.value.decode().split("\n"), list(ms)[:got]):
            per_kernel.setdefault(kname, []).append(float(t))
        summary = {k: {"launches_per_step": len(v) / prof_steps, "avg_ms": sum(v) / len(v),
                       "ms_per_step": sum(v) / prof_steps} for k, v in per_kernel.items()}
        dominant = max(summary, key=lambda k: summary[k]["ms_per_step"])
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        bpf = ALGORITHMIC_BYTES_PER_FRAME.get(dominant)
        traffic_path = os.path.join(ROOT, "profiles", "traffic.json")
        traffic = None
        if os.path.exists(traffic_path):
            table = json.load(open(traffic_path))
            traffic = table.get(name, {}).get(dominant) if isinstance(table.get(name), dict) else (table.get(dominant) if name == "c2" else None)
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                    "traffic": traffic, "peak_source": peak_src, "avg_launch_ms": summary[dominant]["avg_ms"],
                    "algorithmic_bytes_per_launch": None}
        if bpf:
            alg = bpf * n
            ach = alg / (summary[dominant]["avg_ms"] * 1e-3) / 1e9
            roofline.update(achieved=ach, frac=ach / peak, algorithmic_bytes_per_launch=alg)
        per_kernel_frac = {}
        for kname, bytes_per_frame in ALGORITHMIC_BYTES_PER_FRAME.items():
            if kname in summary:
                per_kernel_frac[kname] = bytes_per_frame * n / (summary[kname]["avg_ms"] * 1e-3) / 1e9 / peak
        roofline["per_kernel_frac"] = per_kernel_frac
        fp32_ops = FP32_OPS_PER_FRAME.get(dominant)
        if fp32_ops:
            # the FFT kernels sit under the FP32 roof, not the HBM one (DESIGN.md section 4): reported next to the
            # HBM figure, not instead of it
            props = torch.cuda.get_device_properties(device)
            peak_ops = props.multi_processor_count * 128 * 1.965e9  # lanes x max SM clock
            ops = fp32_ops * n
            roofline["cuda_core"] = {"ops_per_launch": ops, "peak_top_per_s": peak_ops / 1e12,
                                     "frac": ops / (summary[dominant]["avg_ms"] * 1e-3) / peak_ops,
                                     "note": "non-FMA FP32 operations; floor of this kernel = ops / peak"}
        # the whole step against its compulsory bytes (pipeline: 56 T + 8 R; limiter alone: 16 T; SURVEY.md 8d)
        step_bytes = 16 * n if is_limiter else 56 * n + 8 * n
        step_ach = step_bytes / (times["dev"] / args.steps * 1e-3) / 1e9
        roofline["pipeline"] = {"algorithmic_bytes_per_step": step_bytes, "achieved": step_ach, "frac": step_ach / peak}

        cpu_baseline = None
        if not args.no_cpu_baseline and world == 1:
            # the oracle port, float64 numpy/scipy, one thread, on this box's host cores: a bounded sample of the
            # same workload (config 2: the whole 180-s track, ~10 s; configs 3 and 5: the first 60 s / 300 s)
            sample_s = {"c2": seconds, "c3": min(seconds, 60.0), "c5": min(seconds, 300.0)}[name]
            m = int(sr * sample_s)
            ocfg = port.OracleConfig(internal_sample_rate=sr)
            if is_limiter:
                x64 = seam_t[0][:m].copy()
                t0 = time.perf_counter()
                port.limit(x64, ocfg)
            else:
                t64, r64 = seam_t[0][:m].copy(), seam_r[0][:m].copy()
                t0 = time.perf_counter()
                port.main(t64, r64, ocfg, True, False, False)
            cpu_s = time.perf_counter() - t0
            cpu_baseline = {"value": sample_s / cpu_s, "unit": UNIT, "cores": 1, "kind": "port",
                            "sample": f"the first {sample_s:.0f} s of one {seconds:.0f}-s {name} track, oracle/port.py "
                                      f"(numpy/scipy float64, one thread), {cpu_s:.2f} s wall; host has "
                                      f"{os.cpu_count()} hardware threads"}
        ring_route = bool(lib.mgb_host_download_through_ring(2 * n))  # the result crosses the link as float32 / float64
        e2e = {"value": xrt(times["seam"]), "unit": UNIT, "ms_per_step": times["seam"] / args.steps,
               "h2d_bytes_per_step": (1 if is_limiter else 2) * n * 8, "d2h_bytes_per_step": n * (8 if ring_route else 16),
               "host_bytes_read_per_step": (1 if is_limiter else 2) * n * 16, "host_threads": io.threads,
               "api": ("matchering_b200.limiter.limit" if is_limiter else "matchering_b200.stages.main")
                      + "(float64 numpy in pageable memory) -> float64 numpy, one synchronous call per step: the library's "
                        "worker threads narrow the arrays to float32 into a pinned ring while the link copies them, the "
                        + ("result comes back as float32 chunks through the same ring and is widened by the workers into "
                           "pooled pinned memory" if ring_route else
                           "result is widened on the device and copied into pooled pinned memory by one DMA")
                        + "; wall clock between device synchronisations"}
        if "batch_f32" in times:
            e2e["batch_f32"] = {"value": xrt(times["batch_f32"]), "ms_per_step": times["batch_f32"] / args.steps,
                                "h2d_bytes_per_step": 2 * n * 8, "d2h_bytes_per_step": n * 8,
                                "api": "mgb_pipeline_submit/wait (C batch entry, 3 tracks in flight per GPU; pinned float32 host "
                                       "buffers in and out; copies inside the timed region; CUDA events)"}
            e2e["batch_pcm16"] = {"value": xrt(times["batch_pcm16"]), "ms_per_step": times["batch_pcm16"] / args.steps,
                                  "h2d_bytes_per_step": 2 * n * 4, "d2h_bytes_per_step": n * 4,
                                  "api": "mgb_pipeline_submit_pcm (int16 host buffers in and out, decoded / quantised on the device)"}
            e2e["single_call_f32"] = {"value": xrt(times["single_call_f32"]), "ms_per_step": times["single_call_f32"] / args.steps,
                                      "api": "mgb_process_host (one track per call, pinned float32, copies and kernels back to back)"}
        if files_ms is not None:
            e2e["process_files"] = {"value": seconds / (files_ms * 1e-3), "ms_per_step": files_ms,
                                    "api": "matchering_b200.process(t.wav, r.wav, [pcm16(o.wav)]): 16-bit WAV files in "
                                           + ("/dev/shm" if files_dir.startswith("/dev/shm") else "the temp dir")
                                           + ", read, decoded and checked on the device, mastered, quantised on the device, written; "
                                             "wall clock, one GPU"}
        run = {"tracks_per_step": world, "tracks_in_flight_per_gpu": n_lanes, "host_cores_bound_per_rank": bound_cores}
        result = {
            "metric": METRIC, "value": xrt(times["dev"]), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": times["dev"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "samples_per_sec": frames_total / (times["dev"] * 1e-3),
            "config": wcfg, "run": run,
            "single_track_latency": {"value": xrt(times["serial"]), "ms_per_step": times["serial"] / args.steps,
                                     "note": "one track at a time on one stream, device-resident"},
            "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "kernels": summary, "cpu_baseline": cpu_baseline, "clocks": clocks,
        }
    if files_dir is not None:
        import shutil
        shutil.rmtree(files_dir, ignore_errors=True)
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, key + ".npy"), arr)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result or {}


# transport mode of ranks that share a socket with two or more other ranks (tools/gpu_n4_transport.sh decides)
SHARED_SOCKET_MODE = "cached"


def main():
    args = parse_args()
    out = run_reference(args) if args.impl == "reference" else run_b200(args)
    if out:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
