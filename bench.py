#!/usr/bin/env python
"""bench.py -- headline measurement of the event -> voxel-grid hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one voxel-grid build over one batch of synthetic events:
  N=1 : BASELINE.json configs[1] -- 50 M uniform events -> 5-bin 640x480 grid, reference
        semantics (events_to_voxel_torch: temporal bilinear x spatial truncation).
  N>1 : BASELINE.json configs[4] shape -- every rank holds a contiguous 50 M-event time shard of a
        N*50 M-event stream (weak scaling), global (t0, dt), one NCCL sum all-reduce of the grid.
`value` is whole-job Mevents/s with the events resident in HBM, timed with CUDA events over
exactly K steps, max over ranks.  `e2e` is the same metric through the public python API with
pinned HOST tensors in and a host tensor out (H2D + D2H inside the timed region).
`--impl reference` times the library-op port of the reference's events_to_voxel_torch (oracle/ref_port.py)
on the host cores.
`--dump-outputs DIR` writes the grid of the last timed step to DIR/voxel.npy (float32, B x H x W); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_PER_GPU = int(os.environ.get("EVK_BENCH_EVENTS", 50_000_000))
B, H, W = 5, 480, 640
CPU_SAMPLE = int(os.environ.get("EVK_BENCH_CPU_SAMPLE", 5_000_000))
METRIC = "Mevents/s voxel-grid build (B=5, 640x480)"
HBM_FALLBACK_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_config(world, mg_kind=None):
    return {
        "workload": ("50M uniform events -> 5x480x640 voxel grid (events_to_voxel_torch semantics), 1xB200"
                     if world == 1 else
                     "%dM events -> 5x480x640 voxel grid sharded over %d GPUs (50M-event time shard per GPU), "
                     "one all-reduce of the grid per step" % (50 * world, world)),
        "events_per_gpu": N_PER_GPU, "bins": B, "height": H, "width": W,
        "layout": "SoA f32 x,y,t,p (16 B/event)",
        "seed": 2024,
        "l2_policy": "inputs (800 MB/step) larger than L2 (126 MB); no explicit flush",
        "parallelism": ("events sharded x%d, global t0/dt agreed up front" % world) + ((
            "; fold + all-reduce fused in one kernel over NVLink peer memory (symmetric memory, two cross-GPU barriers), step k's reduce overlapped with the scatter of step k+1 (2 buffers)"
            if mg_kind == "peer" else "; NCCL all-reduce of step k overlapped with the scatter of step k+1 (2 grid buffers)") if world > 1 else ""),
    }


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples the SM clock and the throttle reasons through NVML in a background thread.  NVML is
    initialised up front so that the first sample falls inside the (tens of ms) timed region; every
    sample is time-stamped and `summary(t0, t1)` reports the ones taken inside a window."""

    BITS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.samples, self.max_mhz, self.err = [], None, None
        self._stop, self.th, self.h, self.nv = threading.Event(), None, None, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:   # honour CUDA_VISIBLE_DEVICES: go through the UUID of the torch device
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.nv = nv
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, int(r)))
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            time.sleep(0.001)

    def start(self):
        if self.nv is None:
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self._stop.set()
        if self.th is not None:
            self.th.join(timeout=2)

    def summary(self, t0, t1):
        rows = [s for s in self.samples if t0 <= s[0] <= t1]
        reasons = sorted(n for n, b in self.BITS.items() if any(r[2] & b for r in rows))
        out = {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None, "sm_max_mhz": self.max_mhz,
               "samples": len(rows), "reasons": reasons}
        if self.err:
            out["error"] = self.err
        return out


# ------------------------------------------------------------------------------------------------
# synthetic events (SURVEY.md section 8d config 2 generator)
# ------------------------------------------------------------------------------------------------
def make_shard(n, rank, world, device):
    g = torch.Generator(device=device).manual_seed(2024 + rank)
    x = torch.rand(n, device=device, generator=g) * (W - 1)
    y = torch.rand(n, device=device, generator=g) * (H - 1)
    t = torch.sort(torch.rand(n, device=device, generator=g)).values
    t = (t + rank) / world                       # contiguous time shard of the global [0,1) stream
    p = (torch.randint(0, 2, (n,), device=device, generator=g) * 2 - 1).float()
    return x, y, t, p


# ------------------------------------------------------------------------------------------------
# CPU baseline (the reference's library-op sequence, oracle/ref_port.py)
# ------------------------------------------------------------------------------------------------
def cpu_sample_events(n):
    rng = np.random.default_rng(2024)
    x = (rng.random(n) * (W - 1)).astype(np.float32)
    y = (rng.random(n) * (H - 1)).astype(np.float32)
    t = np.sort(rng.random(n)).astype(np.float32)
    p = (rng.integers(0, 2, n) * 2 - 1).astype(np.float32)
    return x, y, t, p


def best_torch_threads(fn, candidates):
    """The reference's torch-CPU scatter (index_put_ accumulate) does not scale with threads and gets
    much SLOWER with many; give the reference arm the thread count it runs fastest with."""
    best, best_t = candidates[0], float("inf")
    for c in candidates:
        torch.set_num_threads(c)
        fn()                                   # warm-up at this thread count
        el = float("inf")
        for _ in range(2):
            s = time.perf_counter()
            fn()
            el = min(el, time.perf_counter() - s)
            if el > 3.0 * best_t:              # hopeless candidate: do not spend a second run on it
                break
        if el < best_t:
            best, best_t = c, el
    torch.set_num_threads(best)
    return best


def thread_candidates():
    cores = os.cpu_count() or 1
    return sorted(set(c for c in (1, 4, 8, 16, 32, 64, cores) if c <= cores))


def reference_functions():
    """(kind, voxel_torch(xs,ys,ts,ps) -> grid, voxel_numpy(xs_int,ys_int,ts,ps) -> grid): the library-op port of the
    reference's events_to_voxel_torch / events_to_voxel."""
    from oracle import ref_port
    return ("port", lambda xs, ys, ts, ps: ref_port.voxel_torch_cpu(xs, ys, ts, ps, B, (H, W)),
            lambda xs, ys, ts, ps: ref_port.voxel_numpy(xs, ys, ts, ps, B, (H, W)), "oracle/ref_port.py")


def time_cpu_port(n, repeats):
    kind, voxel_torch, voxel_numpy, where = reference_functions()
    cores = os.cpu_count() or 1
    x, y, t, p = cpu_sample_events(n)
    xt, yt, tt, pt = (torch.from_numpy(a) for a in (x, y, t, p))
    # calibrate on the full sample: the best thread count at 0.5 M events is not the best at 5 M
    threads = best_torch_threads(lambda: voxel_torch(xt, yt, tt, pt), thread_candidates())
    best_t = float("inf")
    for _ in range(repeats):
        s = time.perf_counter()
        voxel_torch(xt, yt, tt, pt)
        best_t = min(best_t, time.perf_counter() - s)
    xi, yi = x.astype(np.int64), y.astype(np.int64)
    t64, p64 = t.astype(np.float64), p.astype(np.float64)
    best_n = float("inf")
    for _ in range(max(1, repeats - 1)):
        s = time.perf_counter()
        voxel_numpy(xi, yi, t64, p64)
        best_n = min(best_n, time.perf_counter() - s)
    return {"torch_cpu_mevs": n / best_t / 1e6, "numpy_mevs": n / best_n / 1e6, "cores": cores,
            "torch_threads": threads, "kind": kind, "where": where}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args, rank, world):
    """--impl reference: the port of the reference's CPU path on the host cores (see reference_functions)."""
    if rank != 0:
        return
    kind, voxel_torch, _, where = reference_functions()
    cores = os.cpu_count() or 1
    # thread count: the reference's index_put_(accumulate=True) gets SLOWER with many threads; give it its best
    xs, ys, ts, ps = (torch.from_numpy(a) for a in cpu_sample_events(CPU_SAMPLE))
    best_torch_threads(lambda: voxel_torch(xs, ys, ts, ps), thread_candidates())
    s = time.perf_counter()
    voxel_torch(xs, ys, ts, ps)
    t_sample = time.perf_counter() - s
    # the whole 50 M-event workload per step if the run then ends within a few minutes, else a bounded sample of it
    budget_s = float(os.environ.get("EVK_BENCH_REF_BUDGET_S", 150.0))
    per_step = budget_s / max(1, args.steps + args.warmup)
    n = N_PER_GPU if t_sample * (N_PER_GPU / CPU_SAMPLE) <= per_step else int(CPU_SAMPLE * per_step / t_sample)
    n = max(1_000_000, min(N_PER_GPU, n // 1_000_000 * 1_000_000))
    if n != CPU_SAMPLE:
        del xs, ys, ts, ps
        xs, ys, ts, ps = (torch.from_numpy(a) for a in cpu_sample_events(n))
    for _ in range(args.warmup):
        voxel_torch(xs, ys, ts, ps)
    s = time.perf_counter()
    for _ in range(args.steps):
        res = voxel_torch(xs, ys, ts, ps)
    el = time.perf_counter() - s
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, voxel=res)
    value = n * args.steps / el / 1e6
    what = "events_to_voxel_torch library-op port (%s)" % where
    sample = ("%s, torch CPU f32, %d threads = the fastest of %s on this host; %s per step" % (
        what, torch.get_num_threads(), thread_candidates(),
        "the FULL 50M-event workload" if n == N_PER_GPU else
        "a %d-event sample of the 50M-event workload (bounded so that %d steps end within %.0f s)" % (n, args.steps + args.warmup, budget_s)))
    cfg = workload_config(args.gpus, "peer" if args.gpus > 1 else None)
    cfg["reference_events_per_step"] = n
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mevents/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "Mevents/s", "cores": torch.get_num_threads(), "host_cores": cores,
                         "kind": kind, "sample": sample, "cpu": cpu_model()},
        "e2e": {"value": value, "unit": "Mevents/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch.distributed as dist
    from event_utils_b200 import _lib
    from event_utils_b200.parallel import global_time_span
    from event_utils_b200.representations.voxel_grid import events_to_voxel_torch

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # bind the rank to its GPU's NUMA node before any pinned buffer exists (the e2e arm streams 800 MB per step per GPU)
    from event_utils_b200.parallel import bind_to_gpu_numa_node
    numa_cpus = bind_to_gpu_numa_node(local_rank) if os.environ.get("EVK_BENCH_NUMA_BIND", "1") == "1" else None
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner) write to
    # file descriptor 1 directly, so point it at stderr until the line is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    L = _lib.lib()
    n = N_PER_GPU
    x, y, t, p = make_shard(n, rank, world, device)
    t0, dt = global_time_span(t) if world > 1 else (float(t[0]), float((t[-1] - t[0]).item()))
    out = torch.empty((B, H, W), dtype=torch.float32, device=device)
    ws = torch.empty(L.evk_voxel_workspace_bytes(B, H, W, 0), dtype=torch.uint8, device=device)
    oob = torch.zeros(1, dtype=torch.int64, device=device)
    stream = _lib.stream()
    variant = _lib.VARIANT_AUTO

    # N > 1: double-buffered grids, the all-reduce of step k on a communication stream overlaps the
    # scatter of step k+1 (parallel.ShardedVoxelStream); every step still ends with its reduced grid.
    import event_utils_b200 as eu
    from event_utils_b200.parallel import PeerReducedVoxel, ShardedVoxelStream
    pipe_mg, mg_kind = None, None
    if world > 1 and os.environ.get("EVK_BENCH_ALLREDUCE", "peer") == "peer":
        # the product path: fold + all-reduce in one kernel over NVLink peer memory (symmetric memory)
        try:
            pipe_mg, mg_kind = PeerReducedVoxel(B, (H, W), device, depth=2), "peer"
        except Exception as exc:       # no symmetric-memory support on this box: say so and take the NCCL stream
            print("bench: PeerReducedVoxel unavailable (%r), using the NCCL stream" % (exc,), file=sys.stderr)
    if world > 1 and pipe_mg is None:
        pipe_mg, mg_kind = ShardedVoxelStream(B, (H, W), device), "nccl"
    eu.config.check_index_errors = False      # the bench reads the out-of-range counter once, after the timed region

    def step():
        nonlocal out
        if world > 1:
            out, _ = pipe_mg.submit(x, y, t, p, t0, dt)
        else:
            _lib.check(L.evk_voxel_f32(x.data_ptr(), y.data_ptr(), t.data_ptr(), p.data_ptr(), n, t0, dt, B, H, W,
                                       variant, out.data_ptr(), ws.data_ptr(), ws.numel(), oob.data_ptr(), stream))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    if pipe_mg is not None:
        pipe_mg.drain()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    L.evk_prof_enable(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_dev0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step()
    if pipe_mg is not None:
        pipe_mg.drain()                        # the last all-reduce is inside the timed region
    e1.record()
    barrier()
    t_dev1 = time.perf_counter()
    elapsed_ms = e0.elapsed_time(e1)
    kms, ktimed, klaunch = ctypes.c_double(0), ctypes.c_longlong(0), ctypes.c_longlong(0)
    L.evk_prof_collect(ctypes.byref(kms), ctypes.byref(ktimed), ctypes.byref(klaunch))
    L.evk_prof_enable(0)
    if world == 1:
        assert int(oob.item()) == 0
    # sanity inside the bench: every event deposits its polarity once
    total = float(out.double().sum())
    if world > 1:
        el = torch.tensor([elapsed_ms], device=device)
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
        elapsed_ms = float(el.item())
        psum = p.double().sum()
        dist.all_reduce(psum)
        expect = float(psum)
    else:
        expect = float(p.double().sum())
    assert abs(total - expect) <= 1e-6 * n * world + 4.0, (total, expect)
    if args.dump_outputs and rank == 0:        # every rank holds the same reduced grid
        dump_outputs(args.dump_outputs, voxel=out)

    value = n * world * args.steps / elapsed_ms / 1e3          # Mevents/s, whole job
    peak, peak_src = measured_peak()
    alg_bytes = 16.0 * n + 4.0 * B * H * W                       # SURVEY 8d: 16 B/event + the grid once
    k_ms = kms.value / max(1, ktimed.value)
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            traffic = json.load(f).get("voxel_scatter_dram_bytes_per_launch")
    except Exception:
        pass

    # ---- end to end through the public API: pinned host tensors in, host tensor out --------------
    hx, hy, ht, hp = (torch.empty(n, dtype=torch.float32, pin_memory=True) for _ in range(4))
    for h, d in ((hx, x), (hy, y), (ht, t), (hp, p)):
        h.copy_(d)
    torch.cuda.synchronize()
    if world == 1:
        def e2e_step():
            return events_to_voxel_torch(hx, hy, ht, hp, B, sensor_size=(H, W))
    else:
        # the product path end to end: pinned host shard -> H2D -> scatter into the symmetric-memory quad workspace ->
        # fused fold + all-reduce over NVLink peer memory (or the NCCL stream where symmetric memory is unavailable) ->
        # D2H of the reduced grid on every rank
        ghost = torch.empty((B, H, W), dtype=torch.float32, pin_memory=True)
        e2e_pipe = pipe_mg

        def e2e_step():
            x.copy_(hx, non_blocking=True); y.copy_(hy, non_blocking=True)
            t.copy_(ht, non_blocking=True); p.copy_(hp, non_blocking=True)
            grid, done = e2e_pipe.submit(x, y, t, p, t0, dt)
            torch.cuda.current_stream().wait_event(done)
            ghost.copy_(grid, non_blocking=True)
            torch.cuda.synchronize()
            return ghost
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        res = e2e_step()
    barrier()
    s = time.perf_counter()
    for _ in range(e2e_steps):
        res = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - s
    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(t_dev0, t_dev1)
        clocks["e2e_region"] = sampler.summary(s, s + e2e_s)
        if not clocks["samples"]:   # device region shorter than one NVML poll: fall back to the e2e region
            for k in ("sm_mhz", "reasons"):
                clocks[k] = clocks["e2e_region"][k]
            clocks["note"] = "device-timed region too short for an NVML sample; values from the e2e region"
    if world > 1:
        el = torch.tensor([e2e_s], device=device, dtype=torch.float64)
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
        e2e_s = float(el.item())
    assert abs(float(res.double().sum()) - expect) <= 1e-6 * n * world + 4.0
    e2e_value = n * world * e2e_steps / e2e_s / 1e6
    e2e_pageable = None
    if world == 1:
        # what a user of the drop-in sees: the reference's callers hand over ORDINARY (pageable) CPU tensors / numpy
        # arrays at every call (events_cmax.py:341, base_dataset.py:446-453)
        qx, qy, qt, qp = (h.clone() for h in (hx, hy, ht, hp))          # clone() of a pinned tensor is pageable
        assert not qx.is_pinned()
        for _ in range(4):          # the first call allocates the pinned bounce slots and starts the worker pool; the next ones
            events_to_voxel_torch(qx, qy, qt, qp, B, sensor_size=(H, W))      # still speed up (fresh pageable pages settling)
        each = []
        for _ in range(5):
            sq = time.perf_counter()
            resq = events_to_voxel_torch(qx, qy, qt, qp, B, sensor_size=(H, W))
            each.append(time.perf_counter() - sq)
        tq = sorted(each)[len(each) // 2]
        assert abs(float(resq.double().sum()) - expect) <= 1e-6 * n + 4.0
        e2e_pageable = {"value": n / tq / 1e6, "unit": "Mevents/s", "h2d_bytes_per_step": 16 * n, "d2h_bytes_per_step": 4 * B * H * W,
                        "api": "events_to_voxel_torch(ordinary pageable CPU tensors) -> CPU tensor", "steps": 5, "stat": "median",
                        "ms_each": [round(v * 1e3, 2) for v in each]}
        # the plain upload behind every numpy-input entry point (evk_host_upload) beside torch's pageable copy
        from event_utils_b200 import _lib as _evk_lib
        _evk_lib.upload([qx, qy, qt, qp], device)
        su = time.perf_counter()
        up = _evk_lib.upload([qx, qy, qt, qp], device)
        tu = time.perf_counter() - su
        del up
        su = time.perf_counter()
        up = [a.to(device) for a in (qx, qy, qt, qp)]
        torch.cuda.synchronize()
        tt = time.perf_counter() - su
        del up
        e2e_pageable["upload_GBps"] = 16 * n / tu / 1e9
        e2e_pageable["torch_pageable_copy_GBps"] = 16 * n / tt / 1e9
        del qx, qy, qt, qp
    del hx, hy, ht, hp
    e2e_packed = None
    if world == 1:
        # the same call from the reference's STORAGE layout (int16 x,y / float64 t / uint8 p, 13 B/event,
        # event_packagers.py:90-93): what a data loader would hand over without its host-side casts
        from event_utils_b200.representations.voxel_grid import events_to_voxel_packed
        px = torch.empty(n, dtype=torch.int16, pin_memory=True); px.copy_(x.to(torch.int16))
        py = torch.empty(n, dtype=torch.int16, pin_memory=True); py.copy_(y.to(torch.int16))
        pt_ = torch.empty(n, dtype=torch.float64, pin_memory=True); pt_.copy_(t.double() + 1.6e9)
        pp = torch.empty(n, dtype=torch.uint8, pin_memory=True); pp.copy_((p > 0).to(torch.uint8))
        torch.cuda.synchronize()
        for _ in range(2):
            resp = events_to_voxel_packed(px, py, pt_, pp, B, sensor_size=(H, W))
        sp = time.perf_counter()
        for _ in range(e2e_steps):
            resp = events_to_voxel_packed(px, py, pt_, pp, B, sensor_size=(H, W))
        tp = time.perf_counter() - sp
        assert abs(float(resp.double().sum()) - expect) <= 1e-6 * n + 4.0
        e2e_packed = {"value": n * e2e_steps / tp / 1e6, "unit": "Mevents/s", "h2d_bytes_per_step": 13 * n,
                      "d2h_bytes_per_step": 4 * B * H * W, "api": "events_to_voxel_packed(pinned int16/int16/float64/uint8) -> CPU tensor"}
        del px, py, pt_, pp

    extra, cpu = {}, None
    if rank == 0 and world == 1:
        cpu_t = time_cpu_port(CPU_SAMPLE, repeats=3)
        best = max(cpu_t["torch_cpu_mevs"], cpu_t["numpy_mevs"])
        used = cpu_t["torch_threads"] if cpu_t["torch_cpu_mevs"] >= cpu_t["numpy_mevs"] else 1
        cpu = {"value": best, "unit": "Mevents/s", "cores": used, "host_cores": cpu_t["cores"], "kind": cpu_t["kind"],
               "sample": "%d-event sample of the workload, best of 3; faster of the library-op port of events_to_voxel_torch "
                         "on torch-CPU (%.1f Mev/s, %d threads) and events_to_voxel on numpy (%.1f Mev/s, 1 thread); from %s"
                         % (CPU_SAMPLE, cpu_t["torch_cpu_mevs"], cpu_t["torch_threads"], cpu_t["numpy_mevs"], cpu_t["where"]),
               "cpu": cpu_model()}
        if not args.no_extra:
            del x, y, t, p
            torch.cuda.empty_cache()
            try:
                extra = secondary_metrics(L, _lib, device, peak)
            except Exception as exc:   # a secondary number must never cost the headline line
                extra = {"error": repr(exc)}

    if world > 1:
        m_chk = min(n, 2_500_000)
        x_chk, y_chk, t_chk, p_chk = (a[:m_chk].clone() for a in (x, y, t, p))
    if world > 1 and not args.no_extra:
        try:
            peer = peer_reduce_metric(device, x, y, t, p, t0, dt)
        except Exception as exc:   # a secondary number must never cost the headline line
            peer = {"error": repr(exc)}
        del x, y, t, p
        torch.cuda.empty_cache()
        try:
            sharded = sharded_cmax_metric(device, world, rank)
        except Exception as exc:
            sharded = {"error": repr(exc)}
        try:
            zipf = sharded_zipf_image_metric(device, world, rank)
        except Exception as exc:
            zipf = {"error": repr(exc)}
        if rank == 0:
            extra = {"cmax_sharded": sharded, "voxel_single_call_latency": peer, "image_zipf_sharded": zipf}
    if world > 1:
        # parity of the product kernels vs the oracle (runs with --no-extra too; an assertion failure fails the bench)
        oracle_check = peer_oracle_check(device, world, rank, x_chk, y_chk, t_chk, p_chk, t0, dt)
        if rank == 0:
            extra = dict(extra or {})
            extra["multi_gpu_parity"] = oracle_check

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mevents/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world, mg_kind),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Mevents/s", "h2d_bytes_per_step": 16 * n,
                    "d2h_bytes_per_step": 4 * B * H * W, "steps": e2e_steps,
                    "api": "events_to_voxel_torch(pinned CPU tensors) -> CPU tensor" if world == 1 else
                           ("pinned host shard -> H2D -> %s.submit (the device-timed product path) -> D2H of the reduced grid on every rank"
                            % type(pipe_mg).__name__),
                    "numa_bound_cpus": (len(numa_cpus) if numa_cpus else None)},
            "gpu_launches": int(klaunch.value),
            "max_rel_err_vs_oracle": ((extra or {}).get("multi_gpu_parity", {}).get("peer", {}) or {}).get("max_rel_err_vs_oracle")
            if world > 1 and isinstance((extra or {}).get("multi_gpu_parity", {}).get("peer"), dict) else None,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic,
                         "traffic_source": "profiles/ncu_summary.json (dram__bytes_read+write of this kernel from the committed ncu --set full capture; NOT measured in this run)",
                         "kernel": "voxel_scatter_kernel<QUAD> (one red.global.add.v4.f32 per event), chosen over the hot-pixel-table instantiation by the launch-level contention probe; the timed scope covers probe + both launches",
                         "kernel_ms": k_ms, "launches_timed": int(ktimed.value),
                         "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                         "step_frac": (alg_bytes / (elapsed_ms / args.steps * 1e-3) / 1e9) / peak,
                         # the limiter ncu shows is the L2 scattered-reduction rate, not HBM: report it beside the contract's HBM fraction
                         "l2_reduction_rate": {"achieved_gops": (n / (k_ms * 1e-3) / 1e9) if k_ms > 0 else None, "ceiling_gops": 190.0,
                                               "ceiling_source": "tools/exp/tma_red.cu: 50 M red.global.add.v4.f32 to random 16-B slots of 9.8 MB in 0.263 ms",
                                               "frac": (n / (k_ms * 1e-3) / 1e9 / 190.0) if k_ms > 0 else None}},
            "cpu_baseline": cpu,
        }
        if e2e_packed:
            extra = dict(extra or {})
            extra["e2e_storage_layout"] = e2e_packed
        if e2e_pageable:
            extra = dict(extra or {})
            extra["e2e_pageable"] = e2e_pageable
        if extra:
            line["extra"] = extra
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def peer_reduce_metric(device, x, y, t, p, t0, dt):
    """Latency of ONE sharded voxel build (not the pipelined stream of the headline): scatter + the fused
    fold / all-reduce kernel over NVLink peer memory (parallel.PeerReducedVoxel) against scatter + fold + NCCL
    all-reduce (parallel.events_to_voxel_sharded).  CUDA events, best of 10, max over ranks."""
    import torch.distributed as dist
    from event_utils_b200.parallel import PeerReducedVoxel, events_to_voxel_sharded
    fused = PeerReducedVoxel(B, (H, W), device)

    def timed(fn):
        for _ in range(3):
            fn()
        best = 1e9
        for _ in range(10):
            dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            el = torch.tensor([a.elapsed_time(b)], device=device)
            dist.all_reduce(el, op=dist.ReduceOp.MAX)
            best = min(best, float(el))
        return best

    ga = fused(x, y, t, p, t0, dt).clone()
    gb = events_to_voxel_sharded(x, y, t, p, B, (H, W), t0=t0, dt=dt)
    diff = float((ga - gb).abs().max() / gb.abs().max())
    ms_f = timed(lambda: fused(x, y, t, p, t0, dt))
    ms_n = timed(lambda: events_to_voxel_sharded(x, y, t, p, B, (H, W), t0=t0, dt=dt))
    return {"fused_fold_peer_allreduce_ms": ms_f, "fold_plus_nccl_allreduce_ms": ms_n, "max_rel_diff": diff,
            "what": "one call, %d M events per GPU; the fused kernel reads every rank's quad workspace and writes every rank's grid "
                    "over NVLink (symmetric memory), two cross-GPU barriers" % (N_PER_GPU // 1000000)}


def peer_oracle_check(device, world, rank, x, y, t, p, t0, dt):
    """Parity of the multi-GPU PRODUCT kernels against the CPU oracle on a sub-stream (VERDICT r1 weak #2): every rank
    contributes the first `m` events of its shard, the fused fold + all-reduce kernel (peer-pointer form, and the NVLS
    multimem form where the symmetric-memory backend offers multicast) builds their grid with the stream's global
    (t0, dt), the sub-shards are gathered and rank 0 runs oracle.voxel_f32 on the same events.  Checker only."""
    import torch.distributed as dist
    from event_utils_b200.parallel import PeerReducedVoxel
    m = max(1, min(int(x.shape[0]), (2_000_000 + world - 1) // world + 250_000))
    sub = [a[:m].contiguous() for a in (x, y, t, p)]
    out = {"events": m * world}
    grids = {}
    for name, mc in (("peer", False), ("nvls", True)):
        try:
            pr = PeerReducedVoxel(B, (H, W), device, multicast=mc)
            if mc and not pr.multicast:
                out[name] = "multicast addresses not available on this box"
                continue
            grids[name] = pr(sub[0], sub[1], sub[2], sub[3], t0, dt).clone()
        except Exception as exc:
            out[name] = "unavailable: %r" % (exc,)
    gathered = []
    for a in sub:
        parts = [torch.empty_like(a) for _ in range(world)] if rank == 0 else None
        dist.gather(a, parts, dst=0)
        gathered.append(parts)
    if rank == 0:
        from oracle import evk_oracle
        evk_oracle.build()
        ex, ey, et, ep = (torch.cat(parts).cpu().numpy() for parts in gathered)
        ref = evk_oracle.voxel_f32(ex, ey, et, ep, B, (H, W), t0=t0, dt=dt)
        scale = float(np.abs(ref).max())
        for name, g in grids.items():
            err = float(np.abs(g.cpu().numpy() - ref).max() / scale)
            out[name] = {"max_rel_err_vs_oracle": err}
            assert err <= 1e-5, "multi-GPU %s kernel vs oracle: %.3e" % (name, err)
    return out


def sharded_cmax_metric(device, world, rank):
    """Contrast-maximisation (f, g) evaluations of ONE stream sharded over the ranks (SURVEY 8e): per evaluation each
    rank splats its 50 M events; the product path (parallel.PeerCmax) fuses the all-reduce of the 3 x 181 x 241 partial
    images into the objective kernel over NVLink peer memory (one cross-GPU barrier, no NCCL call); the NCCL formulation
    (parallel.cmax_variance_sharded) is timed beside it.  Timed on the device, max over ranks."""
    import torch.distributed as dist
    from event_utils_b200.parallel import PeerCmax, cmax_variance_sharded
    n = N_PER_GPU
    g = torch.Generator(device=device)
    g.manual_seed(7000 + rank)
    span = 0.05
    x = torch.rand(n, generator=g, device=device) * 239.0
    y = torch.rand(n, generator=g, device=device) * 179.0
    t = torch.sort(torch.rand(n, generator=g, device=device) * (span / world))[0] + rank * (span / world)
    p = (torch.randint(0, 2, (n,), generator=g, device=device) * 2 - 1).float()
    t_rel = (t.double() - span).float()          # fast mode: stamps relative to the stream's last one, made once
    iters = 10

    def timed(fn):
        for _ in range(2):
            out = fn(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for i in range(iters):
            out = fn(i)
        e1.record()
        torch.cuda.synchronize()
        el = torch.tensor([e0.elapsed_time(e1)], device=device)
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
        return float(el.item()) / iters, out

    res = {"events_total": n * world}
    ms_nccl, (f_n, g_n) = timed(lambda i: cmax_variance_sharded((45.0 + i, -20.0), x, y, t, p, (180, 240), 1.0, t_ref=span))
    res["nccl_ms_per_eval"] = ms_nccl
    try:
        pc = PeerCmax(device)
        ms, (f, gr) = timed(lambda i: pc((45.0 + i, -20.0), x, y, t_rel, p, (180, 240), 1.0, ts_relative=True))
        res.update({"ms_per_eval": ms, "evals_per_s": 1e3 / ms, "Mevents_per_s": n * world / ms / 1e3, "f": f, "g": [float(gr[0]), float(gr[1])],
                    "rel_diff_vs_nccl_f": abs(f - f_n) / abs(f_n),
                    "what": "variance objective + gradient, linvel warp, f32 fast mode, %d M events per GPU; all-reduce of the 3x181x241 "
                            "partial images fused into the objective kernel over NVLink peer memory (PeerCmax: one cross-GPU barrier, "
                            "no NCCL call); result read back to the host every evaluation" % (n // 1000000)})
    except Exception as exc:
        res.update({"ms_per_eval": ms_nccl, "evals_per_s": 1e3 / ms_nccl, "Mevents_per_s": n * world / ms_nccl / 1e3, "f": f_n,
                    "g": [float(g_n[0]), float(g_n[1])], "what": "NCCL formulation (PeerCmax unavailable: %r)" % (exc,)})
    return res


def sharded_zipf_image_metric(device, world, rank):
    """Hot-spot (Zipf s = 1.0) event image over the ranks (BASELINE configs[3] shape at N GPUs): every rank scatters its
    50 M-event shard through the shared-memory table kernel, one NCCL sum all-reduce joins the 1280x720 images
    (parallel.events_to_image_sharded).  Device-timed, max over ranks; the total count is checked."""
    import torch.distributed as dist
    from event_utils_b200.parallel import events_to_image_sharded
    n, Hi, Wi = N_PER_GPU, 720, 1280
    g = torch.Generator(device=device).manual_seed(4000 + rank)
    npx = Hi * Wi
    w = 1.0 / torch.arange(1, npx + 1, device=device, dtype=torch.float64)
    cdf = torch.cumsum(w, 0) / w.sum()
    ranks = torch.searchsorted(cdf, torch.rand(n, device=device, generator=g, dtype=torch.float64)).clamp_(max=npx - 1)
    perm = torch.randperm(npx, device=device, generator=torch.Generator(device=device).manual_seed(99))    # the same hot pixels on every rank
    pix = perm[ranks]
    x, y, p = (pix % Wi).float(), (pix // Wi).float(), torch.ones(n, device=device)
    del w, cdf, ranks, perm, pix
    for _ in range(2):
        img = events_to_image_sharded(x, y, p, (Hi, Wi))
    best = 1e9
    for _ in range(5):
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); img = events_to_image_sharded(x, y, p, (Hi, Wi)); b.record()
        torch.cuda.synchronize()
        el = torch.tensor([a.elapsed_time(b)], device=device)
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
        best = min(best, float(el))
    assert abs(float(img.double().sum()) - n * world) < 1.0       # a count image: exact
    return {"ms": best, "mevents_per_s": n * world / best / 1e3, "events_total": n * world,
            "what": "Zipf(1.0) stream, %d M events per GPU -> 1280x720 nearest image: shared-memory table scatter per rank + one NCCL "
                    "all-reduce of the 3.7 MB image" % (n // 1000000)}


def secondary_metrics(L, _lib, device, peak):
    """Short, separately timed numbers for the rest of the hot path (reported, not the headline)."""
    out = {}
    n = N_PER_GPU

    def best_of(fn, iters=3):
        fn(); torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return min(ts)
    # fused cmax, f64 parity mode, uniform scene (BASELINE configs[2] shape)
    g = torch.Generator(device=device).manual_seed(7)
    x = torch.rand(n, device=device, generator=g, dtype=torch.float64) * 239
    y = torch.rand(n, device=device, generator=g, dtype=torch.float64) * 179
    t = torch.sort(torch.rand(n, device=device, generator=g, dtype=torch.float64)).values * 0.05
    p = (torch.randint(0, 2, (n,), device=device, generator=g) * 2 - 1).double()
    ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device=device)
    res = torch.empty(8, dtype=torch.float64, device=device)
    tl = float(t[-1])
    ms = best_of(lambda: _lib.check(L.evk_cmax_linvel_variance_f64(
        x.data_ptr(), y.data_ptr(), t.data_ptr(), p.data_ptr(), n, 1.0, 45.0, -20.0, tl, 180, 240, 180, 240, 1.0,
        _lib.CMAX_WANT_GRAD, res.data_ptr(), None, None, ws.data_ptr(), ws.numel(), _lib.stream())))
    out["cmax_f64"] = {"iter_per_s": 1e3 / ms, "ms_per_iter": ms, "events": n, "what": "one fused (f, g) evaluation, "
                       "linvel warp, 181x241 IWE, sigma=1, f64 inputs (32 B/event); IWE in shared memory "
                       "(cmax_onchip_kernel), derivative values one L2 vector reduction per event",
                       "roofline_frac": 32.0 * n / (ms * 1e-3) / 1e9 / peak}
    ms_f = best_of(lambda: _lib.check(L.evk_cmax_linvel_variance_f64(
        x.data_ptr(), y.data_ptr(), t.data_ptr(), p.data_ptr(), n, 1.0, 45.0, -20.0, tl, 180, 240, 180, 240, 1.0,
        0, res.data_ptr(), None, None, ws.data_ptr(), ws.numel(), _lib.stream())))
    out["cmax_f64_f_only"] = {"iter_per_s": 1e3 / ms_f, "ms_per_iter": ms_f, "events": n,
                              "what": "objective only (what a numeric-gradient / grid-search evaluation costs): no L2 reduction at all, "
                                      "the finished image leaves each SM by TMA bulk reduction",
                              "roofline_frac": 32.0 * n / (ms_f * 1e-3) / 1e9 / peak}
    ms_l2 = best_of(lambda: _lib.check(L.evk_cmax_linvel_variance_f64(
        x.data_ptr(), y.data_ptr(), t.data_ptr(), p.data_ptr(), n, 1.0, 45.0, -20.0, tl, 180, 240, 180, 240, 1.0,
        _lib.CMAX_WANT_GRAD | _lib.VARIANT_VECTOR_RED, res.data_ptr(), None, None, ws.data_ptr(), ws.numel(), _lib.stream())))
    out["cmax_f64"]["ms_per_iter_l2_block_accumulator"] = ms_l2
    # CPU port of one reference iteration (f then g) on a 1M-event sample
    try:
        from oracle import ref_port
        m = 1_000_000
        xs, ys, ts, ps = (a[:: n // m][:m].cpu().numpy() for a in (x, y, t, p))
        k = 100_000
        best_torch_threads(lambda: ref_port.cmax_fg_cpu((45.0, -20.0), xs[:k], ys[:k], ts[:k], ps[:k]), thread_candidates())
        s = time.perf_counter()
        ref_port.cmax_fg_cpu((45.0, -20.0), xs, ys, ts, ps)
        el = time.perf_counter() - s
        out["cmax_cpu_port"] = {"iter_per_s_at_sample": 1.0 / el, "sample_events": m, "torch_threads": torch.get_num_threads(),
                                "iter_per_s_extrapolated_to_workload": 1.0 / (el * n / m)}
    except Exception as e:  # pragma: no cover
        out["cmax_cpu_port"] = {"error": repr(e)}
    # the optimiser's view: variance_objective through the public API (numpy f64 in, python floats out),
    # the way scipy's BFGS calls it (events_cmax.py:341-345); each call is a new parameter point
    try:
        from event_utils_b200.contrast_max.objectives import variance_objective
        from event_utils_b200.contrast_max.warps import linvel_warp
        from oracle import ref_port
        m = 1_000_000
        xs, ys, ts, ps = (a[:: n // m][:m].cpu().numpy() for a in (x, y, t, p))
        obj, warp = variance_objective(), linvel_warp()
        args = (xs, ys, ts, ps, warp, (180, 240), 1.0)
        obj.evaluate_function((40.0, -20.0), *args)
        k = 200
        s = time.perf_counter()
        for i in range(k):
            prm = (40.0 + 0.01 * i, -20.0)
            obj.evaluate_function(prm, *args)
            obj.evaluate_gradient(prm, *args)
        el = (time.perf_counter() - s) / k
        out["cmax_api_1M"] = {"iter_per_s": 1.0 / el, "events": m,
                              "what": "evaluate_function + evaluate_gradient per new parameter point through the python API, the way "
                                      "the reference's optimize_contrast calls it: every call hashes all 32 MB of the four host arrays "
                                      "(cache identity = every byte), then one fused launch, result read back"}
        from event_utils_b200.contrast_max.objectives import pinned_events
        with pinned_events(xs, ys, ts, ps):
            s = time.perf_counter()
            for i in range(k):
                prm = (41.0 + 0.01 * i, -20.0)
                obj.evaluate_function(prm, *args)
                obj.evaluate_gradient(prm, *args)
            el_p = (time.perf_counter() - s) / k
        out["cmax_api_1M"]["iter_per_s_pinned_events"] = 1.0 / el_p
        out["cmax_api_1M"]["pinned_events"] = ("inside `with pinned_events(xs, ys, ts, ps)` (what this repo's optimize_contrast does): "
                                               "the caller promises frozen arrays, no per-call hash")
        best_torch_threads(lambda: ref_port.cmax_fg_cpu((45.0, -20.0), xs[:100000], ys[:100000], ts[:100000], ps[:100000]),
                           thread_candidates())
        s = time.perf_counter()
        ref_port.cmax_fg_cpu((45.0, -20.0), xs, ys, ts, ps)
        out["cmax_api_1M"]["cpu_port_iter_per_s"] = 1.0 / (time.perf_counter() - s)
    except Exception as e:  # pragma: no cover
        out["cmax_api_1M"] = {"error": repr(e)}
    del x, y, t, p
    torch.cuda.empty_cache()
    # event image on a hot-spot (Zipf) stream vs a uniform one (BASELINE configs[3] shape: 1280x720)
    Hi, Wi = 720, 1280
    g = torch.Generator(device=device).manual_seed(99)
    npx = Hi * Wi
    img = torch.empty((Hi, Wi), dtype=torch.float32, device=device)
    oob = torch.zeros(1, dtype=torch.int64, device=device)
    for name, s_exp in (("uniform", None), ("zipf_s1.0", 1.0), ("zipf_s1.2", 1.2)):
        if s_exp is None:
            xi = torch.rand(n, device=device, generator=g) * (Wi - 1)
            yi = torch.rand(n, device=device, generator=g) * (Hi - 1)
        else:
            w = 1.0 / torch.arange(1, npx + 1, device=device, dtype=torch.float64) ** s_exp
            cdf = torch.cumsum(w, 0) / w.sum()
            ranks = torch.searchsorted(cdf, torch.rand(n, device=device, generator=g, dtype=torch.float64)).clamp_(max=npx - 1)
            pix = torch.randperm(npx, device=device, generator=g)[ranks]
            xi, yi = (pix % Wi).float(), (pix // Wi).float()
            del w, cdf, ranks, pix
        pi = torch.ones(n, device=device)
        ms = best_of(lambda: _lib.check(L.evk_image_f32(xi.data_ptr(), yi.data_ptr(), pi.data_ptr(), n, Hi, Wi, 0.0, 0.0, 0, 0.0,
                                                        img.data_ptr(), None, 0, oob.data_ptr(), _lib.stream())))
        assert abs(float(img.double().sum()) - n) < 1.0      # count image: exact
        out["image_nearest_" + name] = {"mevents_per_s": n / ms / 1e3, "ms": ms, "events": n,
                                        "roofline_frac": (12.0 * n + 4.0 * npx) / (ms * 1e-3) / 1e9 / peak}
        del xi, yi, pi
    torch.cuda.empty_cache()
    return out


def dump_outputs(directory, **arrays):
    """Write each array as DIR/<name>.npy in float32."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a.detach().to("cpu", torch.float32).numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary (cmax) numbers")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the grid of the last timed step to DIR/voxel.npy")
    args = ap.parse_args()
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
