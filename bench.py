#!/usr/bin/env python
"""bench.py — upscaled Mpixels/s of the FSR 1.0 hot path (EASU+RCAS) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one synthetic frame through EASU -> RCAS.  Default workload = BASELINE.json configs[1]:
1920x1080 -> 3840x2160, RGBA16F, sharpness 0.25 stops.  With N > 1 (launched by torchrun, one rank per GPU)
the frame is N slabs tall (1920 x 1080N -> 3840 x 2160N), sharded by output row slab with the EASU input halo
moved between neighbouring ranks every step (direct NVLink stores through the C ABI's fsr1_shard_*, or NCCL with --halo nccl):
per-GPU work is fixed ("weak" scaling).  Every N runs the SAME schedule (fsr1_shard: RCAS of frame i overlaps EASU of frame i+1).
N > 1 lines carry "parity" (sharded == single GPU bit for bit, both data planes, oracle bands) and "halo" (what the exchange costs).

Timing rules followed: >= 3 warm-up steps; frames rotate through a ring of buffer sets larger than L2
(so no step finds its input or output in cache from the previous one); the timed region is bracketed by a
barrier + cuda synchronize, measured with CUDA events on the launching stream, max over ranks; SM clocks and
throttle reasons are sampled with nvidia-smi during the timed region.
Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (in_w, in_h, out_w, out_h, dtype, description)
    "1080p-4k-fp16": (1920, 1080, 3840, 2160, "f16", "1920x1080->3840x2160 EASU+RCAS RGBA16F (BASELINE configs[1])"),
    "1440p-4k-fp16": (2560, 1440, 3840, 2160, "f16", "2560x1440->3840x2160 EASU+RCAS RGBA16F (BASELINE configs[2])"),
    "uq-4k-fp16": (2953, 1661, 3840, 2160, "f16", "2953x1661->3840x2160 (true Ultra Quality 1.3x) RGBA16F"),
    "1080p-4k-fp32": (1920, 1080, 3840, 2160, "f32", "1920x1080->3840x2160 EASU+RCAS RGBA32F (BASELINE configs[3])"),
    "2160p-8k-fp16": (3840, 2160, 7680, 4320, "f16", "3840x2160->7680x4320 EASU+RCAS RGBA16F (BASELINE configs[4])"),
    "1080p-4k-unorm8": (1920, 1080, 3840, 2160, "u8", "1920x1080->3840x2160 EASU+RCAS R8G8B8A8_UNORM (the sample's formats, FSR_Filter.cpp:72-73)"),
}
SHARPNESS = 0.25
RING = 8
METRIC = "upscaled Mpixels/sec (EASU+RCAS)"
DUMP_PIXELS = 1 << 21                  # --dump-outputs: at most 2M RGBA float32 pixels (32 MB) over all ranks


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_issue():
    """ncu-derived issue-rate data per kernel (tools/ncu_summary.py writes it): inst/px, inst/cycle/SM, pipe utilisation."""
    p = os.path.join(ROOT, "profiles", "ncu_issue.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return {}


def load_traffic():
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return {}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML queried from a thread that is armed before the warm-up and
    released when the timed steps start (the region is 1.5-15 ms, too short for `nvidia-smi -lms`), nvidia-smi as fallback."""
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.t, self.err = index, [], False, None, None
        self.go = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv, self.err = None, repr(e)

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                pass
        return i

    def _poll(self):
        """First sample 1 ms into the timed region (a 20-step run lasts ~1.6 ms), then one every 5 ms: each sample is two driver
        queries against the timed GPU, and at N > 1 a hiccup on one rank's GPU is a hiccup of every rank (they run in lockstep
        through the halo hand-shake), so the region is sampled, not hammered."""
        nv = self.nv
        self.go.wait()                 # armed before the warm-up, released when the timed region starts (see trigger)
        time.sleep(0.001)
        n = 0
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0 if n % 4 == 0 else (self.samples[-1][2] if self.samples else 0.0)
                self.samples.append((sm, reasons, pw))
                n += 1
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                break
            time.sleep(0.005)

    def start(self):
        if self.nv is None:
            return
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()

    def trigger(self):
        """The timed region starts now (called on the launching thread right before the first timed step)."""
        self.go.set()

    def stop(self):
        if self.nv is None:
            return self._smi_once()
        self.stop_flag = True
        self.go.set()
        self.t.join(timeout=1)
        if not self.samples:                       # a region shorter than 1 ms: one sample right behind it
            try:
                self.samples.append((self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM),
                                     self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h), self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            except Exception:  # noqa: BLE001
                pass
        sm = sorted(s[0] for s in self.samples)
        reasons = set()
        for _, r, _ in self.samples:
            for bit, name in self.BITS.items():
                if r & bit:
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "sm_mhz_min": sm[0] if sm else None,
                "power_w_max": max((s[2] for s in self.samples), default=None), "samples": len(sm),
                "reasons": sorted(reasons), "how": "NVML sampled 1 ms into the timed region and every 5 ms after"}

    def _smi_once(self):
        try:
            out = subprocess.check_output(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                           "--format=csv,noheader,nounits"], text=True).strip().split(",")
            return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "samples": 1, "reasons": [],
                    "how": "nvidia-smi once after the timed region (NVML unavailable: %s)" % self.err}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["unavailable"]}


# ------------------------------------------------------------------------------------------- reference arm
def cpu_reference_runner():
    """Returns (kind, fn) timing the reference's own CPU-compilable source (oracle/_ref) when it was built, else the
    oracle port."""
    import oracle_lib as ol
    R = ol.ref()
    lib, kind = (R, "reference") if R is not None else (ol.oracle(), "port")

    def run(frame, ow, oh, y0, y1, econ, rcon, tmp_holder):
        e0, e1 = max(y0 - 1, 0), min(y1 + 1, oh)
        ih, iw = frame.shape[:2]
        tmp, out = tmp_holder
        P, Z = ctypes.c_void_p, ctypes.c_size_t
        ec, rc = (ctypes.c_uint32 * 16)(*econ), (ctypes.c_uint32 * 4)(*rcon)
        if kind == "reference":
            lib.fsr1ref_easu_f(P(frame.ctypes.data), iw, ih, Z(iw * 4), P(tmp.ctypes.data), ow, oh, Z(ow * 4), ec, e0, e1)
            lib.fsr1ref_rcas_f(P(tmp.ctypes.data), ow, oh, Z(ow * 4), P(out.ctypes.data), Z(ow * 4), rc, 0, y0, y1)
        else:
            lib.fsr1o_easu_f32(P(frame.ctypes.data), iw, ih, Z(iw * 4), P(tmp.ctypes.data), ow, oh, Z(ow * 4), ec, e0, e1)
            lib.fsr1o_rcas_f32(P(tmp.ctypes.data), ow, oh, Z(ow * 4), P(out.ctypes.data), Z(ow * 4), rc, 0, y0, y1)
    return kind, run, ol


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def omp_runtime():
    """libgomp of this process (the oracle libraries link it): team size query / override."""
    try:
        g = ctypes.CDLL("libgomp.so.1")
        g.omp_get_max_threads.restype = ctypes.c_int
        return g
    except OSError:
        return None


def time_cpu(wl, steps, warmup, budget_s, threads=None):
    """Times the CPU reference on bands of output rows of the workload with `threads` OpenMP threads (None = all the
    runtime gives).  Returns dict(value, cores, kind, sample, ...)."""
    import numpy as np
    import fsr1_b200 as F
    iw, ih, ow, oh = wl[:4]
    kind, run, ol = cpu_reference_runner()
    g = omp_runtime()
    all_threads = g.omp_get_max_threads() if g else int(os.environ.get("OMP_NUM_THREADS", os.cpu_count() or 1))
    if threads is not None and g:
        g.omp_set_num_threads(int(threads))
    team = g.omp_get_max_threads() if g else all_threads
    frame = F.to_half(F.uniform(iw, ih, 12345)).astype(np.float32)
    econ, rcon = ol.easu_con(iw, ih, ow, oh), ol.rcas_con(SHARPNESS)
    holder = (np.zeros((oh, ow, 4), np.float32), np.zeros((oh, ow, 4), np.float32))
    # calibrate on 32 rows
    t = time.perf_counter(); run(frame, ow, oh, 0, 32, econ, rcon, holder); per_row = (time.perf_counter() - t) / 32
    t = time.perf_counter(); run(frame, ow, oh, 64, 96, econ, rcon, holder); per_row = min(per_row, (time.perf_counter() - t) / 32)
    rows = int(max(8, min(oh, budget_s / max(per_row, 1e-9) / max(steps + warmup, 1))))
    bands = [(y, min(y + rows, oh)) for y in range(0, oh - rows + 1, rows)] or [(0, oh)]
    for i in range(warmup):
        y0, y1 = bands[i % len(bands)]
        run(frame, ow, oh, y0, y1, econ, rcon, holder)
    t0 = time.perf_counter()
    px = 0
    for i in range(steps):
        y0, y1 = bands[i % len(bands)]
        run(frame, ow, oh, y0, y1, econ, rcon, holder)
        px += (y1 - y0) * ow
    dt = time.perf_counter() - t0
    if threads is not None and g:
        g.omp_set_num_threads(all_threads)
    return {"value": px / dt / 1e6, "unit": "Mpix/s", "cores": team, "kind": kind,
            "sample": "%d steps x %d-row bands of the %dx%d output, fp32 F path, OpenMP over rows (%d threads)" % (steps, rows, ow, oh, team),
            "cpu_model": cpu_model(), "logical_cpus": os.cpu_count(), "omp_proc_bind": os.environ.get("OMP_PROC_BIND", "unset"),
            "seconds": dt, "ms_per_step": dt / steps * 1e3}


def cpu_baseline(wl):
    """All host threads (the headline cpu_baseline) and one thread (SURVEY 8(d) asks for both), same run."""
    allc = time_cpu(wl, steps=12, warmup=1, budget_s=12.0)
    one = time_cpu(wl, steps=6, warmup=1, budget_s=6.0, threads=1)
    for d in (allc, one):
        d.pop("seconds", None)
    allc["one_thread"] = {"value": one["value"], "unit": "Mpix/s", "cores": 1, "sample": one["sample"]}
    return allc


def bind_to_gpu_numa_node(local_rank):
    """N > 1: keep this rank's host thread (and so its pinned frame buffers: first touch) on the CPUs of the NUMA node its GPU
    hangs off — the end-to-end leg moves 83 MB per frame per rank through host memory, and eight unplaced ranks share one
    socket's memory controllers.  Best effort: returns a note for the JSON line, or None when the topology cannot be read."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        text = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in text.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if len(cpus) >= 8 and len(cpus) < len(allowed):      # never squeeze the rank (NCCL proxy, sampler) onto a few CPUs
            os.sched_setaffinity(0, cpus)
            return "rank bound to the %d CPUs local to GPU %s" % (len(cpus), bdf)
    except Exception:  # noqa: BLE001
        pass
    return None


# ------------------------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    global RING
    if args.frames > 0:
        RING = args.frames
    import numpy as np
    import torch
    import fsr1_b200 as F
    api = F.api
    wl = WORKLOADS[args.workload]
    iw, ih, ow, oh, dts = wl[:5]
    tdt = {"f16": torch.float16, "f32": torch.float32, "u8": torch.uint8}[dts]
    bpp = {"f16": 8, "f32": 16, "u8": 4}[dts]
    fmt = {"f16": api.FORMAT_RGBA16F, "f32": api.FORMAT_RGBA32F, "u8": api.FORMAT_RGBA8_UNORM}[dts]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    affinity = None
    if world > 1:
        affinity = bind_to_gpu_numa_node(local_rank)
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    K, W = args.steps, max(args.warmup, 3)

    def host_frame(seed):
        f = F.uniform(iw, ih, seed)
        if dts == "u8":
            return np.floor(f * 255.0 + 0.5).astype(np.uint8)
        return f.astype(np.float16) if dts == "f16" else f

    # The frame the job upscales.  N = 1: the workload's frame.  N > 1, default ("weak"): `world` such frames stacked
    # (1920 x 1080N -> 3840 x 2160N), rank r owning frame r of the stack; --shard-frame ("strong"): the workload's own
    # frame cut into `world` row slabs (BASELINE configs[4] at N = 8).
    strong = world > 1 and args.shard_frame
    H_in, H_out = (ih, oh) if (world == 1 or strong) else (ih * world, oh * world)

    def rank_rows(t, r, o0, o1):
        """input rows [o0,o1) of the tall frame t owned by rank r"""
        if world == 1 or strong:
            return host_frame(12345 + t)[o0:o1]
        return host_frame(12345 + t + 1000 * r)          # rank r's slab IS frame r of the stack

    stream = torch.cuda.current_stream()
    halo_mode = args.halo if world > 1 else "p2p"
    kflags = api.FLAG_FUSED if args.fused else 0
    up = F.ShardedUpscaler(iw, H_in, ow, H_out, world, rank, SHARPNESS, dtype=tdt, device=dev, slots=RING, halo=halo_mode,
                           one_stream=args.no_pipeline, flags=kflags, trace=args.trace and world > 1)
    plan = up.plan
    o0, o1 = plan.owned_in_rows(rank)
    e0, e1 = plan.easu_rows(rank)
    y0, y1 = plan.out_rows(rank)
    for t in range(RING):                                 # every frame's slab is resident in HBM before the clock starts
        up.input(t).copy_(torch.from_numpy(np.ascontiguousarray(rank_rows(t, rank, o0, o1))).to(dev))
    torch.cuda.synchronize()
    halo = plan.halo_bytes(rank, iw, bpp)
    total_out_px = ow * H_out

    if halo_mode == "p2p":
        def step(i):
            up.submit(i % RING, stream)                   # C ABI: halo push + EASU + RCAS, pipelined on the shard's streams

        def drain():
            for k in range(RING):
                up.wait(k, stream)
    else:
        # NCCL data plane (torch.distributed send/recv): the halo rows of frame i+1 travel on a second stream while
        # frame i is upscaled; kernels of frame i+1 wait on that exchange's event only
        comm = torch.cuda.Stream(device=dev)
        ready = [torch.cuda.Event() for _ in range(RING)]

        def prefetch(j):
            comm.wait_stream(stream)
            with torch.cuda.stream(comm):
                up._exchange(j % RING)
                ready[j % RING].record(comm)
        prefetch(0)
        frame_no = [0]

        def step(_):
            i = frame_no[0]
            frame_no[0] += 1
            prefetch(i + 1)
            stream.wait_event(ready[i % RING])
            up._launch(i % RING, stream)

        def drain():
            stream.wait_stream(comm)

    # N > 1: the device-side rendezvous in front of every timed region (see timed()).  8 MB rather than one element: the all_reduce then
    # crosses every NVLink link of every GPU a few microseconds before the clock starts.  The device trace of the 20-step 8-GPU run
    # (profiles/r02_startup_trace_n8_k20.txt) shows the first halo push after the barrier's idle gap taking 118 us on every rank (218 us
    # where the receiving GPU had not sent anything itself yet) against 8-16 us from the second frame on — links leaving their idle power
    # state — which is ~280 us of a 1.9 ms timed region; a stream of frames never idles the links, a barrier in front of 20 steps does.
    rendezvous = torch.zeros(2 * 1024 * 1024, device=dev) if dist is not None else None
    if dist is not None:
        dist.all_reduce(rendezvous)            # first use outside any timed region (NCCL sets up its channels for this size once)
        torch.cuda.synchronize()

    def timed(fn, n, post=None, on_start=None):
        """K steps between a barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks.
        N > 1: hosts leave a barrier milliseconds apart (measured: 7-10 ms on this stack), which at 20 steps would be most of the
        timed region — so the start event sits behind a DEVICE-side rendezvous (an all_reduce enqueued on the same
        stream): the clock of every rank starts when the last rank's GPU arrives, and every timed step is ordered after it."""
        import gc
        gc.disable()                       # no collector pause inside the timed region (collected before the warm-up)
        try:
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if dist is not None:
                dist.all_reduce(rendezvous)    # async w.r.t. the host; `stream` waits for it; also wakes every NVLink link (see above)
            a.record(stream)
            if on_start:
                on_start()
            for i in range(n):
                fn(i)
            if post:
                post()
            b.record(stream)
            torch.cuda.synchronize()
        finally:
            gc.enable()
        ms = a.elapsed_time(b)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(t.item())
        return ms

    # everything slow on the host happens BEFORE the warm-up (NVML initialisation is ~80 ms, a full collection tens of ms), so that
    # the timed steps follow the warm-up steps after a barrier only: the NVLink peer path is still warm (the first push after ~100 ms
    # of idle measured 120 us instead of 8, profiles/r02_handshake_trace.txt)
    import gc
    gc.collect()
    sampler = ClockSampler(local_rank)
    for i in range(W):
        step(i)
    drain()
    if rank == 0 and not os.environ.get("FSR1_BENCH_NO_SAMPLER"):
        sampler.start()
    launches0 = api.launch_count()
    ms = timed(step, K, post=drain, on_start=sampler.trigger if rank == 0 else None)
    launches = api.launch_count() - launches0
    clocks = (sampler.stop() if not os.environ.get("FSR1_BENCH_NO_SAMPLER") else sampler._smi_once()) if rank == 0 else None
    up.status()
    if args.dump_outputs:
        # the slot of the last timed step; the nccl step numbers frames on from the warm-up
        last = (K - 1) % RING if halo_mode == "p2p" else (frame_no[0] - 1) % RING
        dump_output(args.dump_outputs, "output" if world == 1 else "output_rank%d" % rank, up.output(last), DUMP_PIXELS // world)
    if args.trace and world > 1 and halo_mode == "p2p":
        tr = up.trace().astype(np.int64)
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        np.save(os.path.join(ROOT, "gpurun_out", "trace_rank%d_%s.npy" % (rank, os.environ.get("FSR1_TRACE_TAG", "t"))), tr)
        if len(tr) > 8:
            tr = tr[4:-2]
            wait = (tr[:, 1] - tr[:, 0]) / 1e3
            kern = (tr[:, 2] - tr[:, 0]) / 1e3
            period = np.diff(tr[:, 2]) / 1e3
            lead_u = (tr[:, 0] - tr[:, 4]) / 1e3      # my push (up) published this long BEFORE my own EASU of the same frame started
            lead_d = (tr[:, 0] - tr[:, 6]) / 1e3
            pdur_u, pdur_d = (tr[:, 4] - tr[:, 3]) / 1e3, (tr[:, 6] - tr[:, 5]) / 1e3
            def st(a):
                a = a[np.isfinite(a)]
                return "med %.1f p90 %.1f max %.1f" % (np.median(a), np.percentile(a, 90), a.max()) if len(a) else "-"
            sys.stderr.write("[trace rank %d] us: halo wait inside EASU %s | EASU kernel (wait+work) %s | frame period %s | push duration up %s down %s | "
                             "own push published before own EASU start: up %s down %s\n" % (rank, st(wait), st(kern), st(period), st(pdur_u), st(pdur_d), st(lead_u), st(lead_d)))
    value = total_out_px * K / (ms * 1e-3) / 1e6
    peak, peak_src = load_peaks()

    # ---- the same frames one at a time on one stream (no overlap of consecutive frames): latency view
    latency_ms = None
    if world == 1 and not args.no_pipeline:
        seq = F.ShardedUpscaler(iw, ih, ow, oh, 1, 0, SHARPNESS, dtype=tdt, device=dev, slots=RING, halo="p2p", one_stream=True, flags=kflags)
        for t in range(RING):
            seq.input(t).copy_(up.input(t))

        def seq_step(i):
            seq.submit(i % RING, stream)
        for i in range(W):
            seq_step(i)
        latency_ms = timed(seq_step, K, post=lambda: [seq.wait(k, stream) for k in range(RING)]) / K
        seq.close()

    # ---- per-kernel times on this rank's slab (max over ranks) and the roofline of the dominant kernel
    tmps = [torch.empty((e1 - e0, ow, 4), dtype=tdt, device=dev) for _ in range(RING)]
    win_imgs = [api.image(up.windows[t], height=H_in, row0=up._win0) for t in range(RING)]
    tmp_imgs = [api.image(tmps[t], height=H_out, row0=e0) for t in range(RING)]
    out_imgs = [api.image(up.outputs[t], height=H_out, row0=y0) for t in range(RING)]

    def step_easu(i):
        api.easu(win_imgs[i % RING], tmp_imgs[i % RING], up.econ, y0=e0, y1=e1, stream=stream)

    def step_rcas(i):
        api.rcas(tmp_imgs[i % RING], out_imgs[i % RING], up.rcon, y0=y0, y1=y1, stream=stream)
    Pin, Pout = iw * (o1 - o0), ow * (y1 - y0)
    alg = {"easu": bpp * (Pin + Pout), "rcas": bpp * 2 * Pout}
    kernels = {}
    for key, fn in (("easu", step_easu), ("rcas", step_rcas)):
        for i in range(W):
            fn(i)
        name = api.last_kernel()
        kms = timed(fn, K) / K
        gbs = alg[key] / (kms * 1e-3) / 1e9
        kernels[key] = {"kernel": name, "us": kms * 1e3, "algorithmic_bytes": alg[key], "GBps": gbs, "frac_of_hbm_peak": gbs / peak}
    fused_used = False
    if args.fused:
        def step_fused(i):
            api.upscale(win_imgs[i % RING], tmp_imgs[i % RING], out_imgs[i % RING], up.econ, up.rcon, y0=y0, y1=y1, flags=kflags, stream=stream)
        for i in range(W):
            step_fused(i)
        name = api.last_kernel()
        fused_used = name.startswith("fused")
        if fused_used:
            kms = timed(step_fused, K) / K
            fb = bpp * (Pin + Pout)          # the fused kernel is held to ITS compulsory bytes, never the two-pass figure (SURVEY 8(d))
            kernels = {"fused": {"kernel": name, "us": kms * 1e3, "algorithmic_bytes": fb, "GBps": fb / (kms * 1e-3) / 1e9,
                                 "frac_of_hbm_peak": fb / (kms * 1e-3) / 1e9 / peak},
                       "two_pass_for_comparison": kernels}
            alg = {"fused": fb}
    del tmps
    dom = max((k for k in kernels if "us" in kernels[k]), key=lambda k: kernels[k]["us"])
    traffic = load_traffic().get(kernels[dom]["kernel"])
    issue = load_issue().get(kernels[dom]["kernel"])
    roofline = {"bound": "hbm", "kernel": kernels[dom]["kernel"], "achieved": kernels[dom]["GBps"], "peak": peak,
                "unit": "GB/s", "frac": kernels[dom]["GBps"] / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg[dom], "us_per_launch": kernels[dom]["us"], "per": "GPU (max over ranks)",
                "issue": issue}
    path_bytes = alg["fused"] if fused_used else alg["easu"] + alg["rcas"]
    per_frame_us = ms / K * 1e3
    kernels["path"] = {"algorithmic_bytes": path_bytes, "us": per_frame_us, "GBps": path_bytes / (per_frame_us * 1e-6) / 1e9,
                       "frac_of_hbm_peak": path_bytes / (per_frame_us * 1e-6) / 1e9 / peak}

    # ---- N > 1: parity of the sharded result, and what the halo exchange costs
    parity, halo_info = None, None
    if world > 1:
        parity = check_sharded_parity(F, api, up, dist, dev, rank, world, iw, ih, ow, oh, H_in, H_out, tdt, rank_rows, halo_mode)
        nh = F.ShardedUpscaler(iw, H_in, ow, H_out, world, rank, SHARPNESS, dtype=tdt, device=dev, slots=RING, halo="p2p",
                               one_stream=args.no_pipeline, skip_halo=True, flags=kflags)
        for t in range(RING):
            nh.input(t).copy_(up.input(t))

        def nh_step(i):
            nh.submit(i % RING, stream)
        for i in range(W):
            nh_step(i)
        ms_nh = timed(nh_step, K, post=lambda: [nh.wait(k, stream) for k in range(RING)])
        nh.close()
        halo_info = {"mode": halo_mode, "recv_bytes_per_step_per_rank": halo, "us_per_step_without_exchange": ms_nh / K * 1e3,
                     "exposed_us_per_step": (ms - ms_nh) / K * 1e3,
                     "how": "same schedule re-timed with FSR1_SHARD_SKIP_HALO (no push / wait / credit kernels)"}

    # ---- end to end: host (pinned) -> device -> kernels -> host
    e2e = None
    Ke = max(3, min(K, 60))
    if world == 1:
        NS = 3
        ctxs = [api.HostContext(iw, ih, ow, oh, fmt) for _ in range(NS)]
        streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
        hin = [torch.from_numpy(host_frame(777 + t)).pin_memory() for t in range(NS)]
        hout = [torch.empty((oh, ow, 4), dtype=tdt).pin_memory() for t in range(NS)]

        def e2e_step(i):
            j = i % NS
            ctxs[j].upscale_host(hin[j], hout[j], SHARPNESS, stream=streams[j])
        how = "fsr1_context_upscale_host on pinned host frames, %d streams round-robin" % NS
    else:
        NS = min(3, RING)
        streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
        hin = [torch.from_numpy(np.ascontiguousarray(rank_rows(50 + t, rank, o0, o1))).pin_memory() for t in range(NS)]
        hout = [torch.empty((y1 - y0, ow, 4), dtype=tdt).pin_memory() for t in range(NS)]
        for st in streams:
            st.wait_stream(stream)

        def e2e_step(i):
            j = i % NS
            with torch.cuda.stream(streams[j]):
                up.input(j).copy_(hin[j], non_blocking=True)
                up.submit(j, streams[j])
                up.wait(j, streams[j])
                hout[j].copy_(up.output(j), non_blocking=True)
        how = "every rank: pinned host slab -> fsr1_shard input, fsr1_shard_submit/wait, output slab -> pinned host; %d slots round-robin" % NS
    for i in range(NS * 2):
        e2e_step(i)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(Ke):
        e2e_step(i)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    e2e = {"value": total_out_px * Ke / dt / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": iw * H_in * bpp,
           "d2h_bytes_per_step": ow * H_out * bpp, "steps": Ke, "ms_per_step": dt / Ke * 1e3, "how": how,
           "host_checksum": float(hout[0][::97, ::89, :3].float().sum())}   # the result is really read on the host
    if world == 1:
        for c in ctxs:
            c.close()
    up.status()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(wl)

    if rank == 0:
        shard_desc = "" if world == 1 else (" cut into %d row slabs" % world if strong else " x%d slabs tall, row-slab sharded" % world)
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": dts, "data": "synthetic",
            "config": {"workload": wl[5] + shard_desc, "sharpness_stops": SHARPNESS, "frame": "LCG uniform noise, seed 12345+t",
                       "l2": "ring of %d frame sets (%.0f MB per rank) > 126 MB L2" % (RING, RING * (iw * (o1 - o0) + 2 * ow * (y1 - y0)) * bpp / 1e6),
                       "parallelism": "1 GPU" if world == 1 else "row-slab x%d, %d B halo recv per rank per step, %s" % (
                           world, halo, "direct NVLink stores into the neighbour's window (CUDA IPC, fsr1_shard_*), no NCCL in the step"
                           if halo_mode == "p2p" else "NCCL send/recv one frame ahead on a second stream"),
                       "structure": ("ONE fused EASU->RCAS kernel per frame (FSR1_FLAG_FUSED), no intermediate image" if fused_used else
                                     "two kernels per frame through a display-sized fp16 intermediate, as FSR_Filter::Upscale"),
                       "pipelining": "none: one frame at a time on one stream" if args.no_pipeline else
                                     "whole frames on two streams in turn inside fsr1_shard: RCAS of frame i overlaps EASU of frame i+1; same schedule at every N"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels, "e2e": e2e,
        }
        if latency_ms is not None:
            line["unpipelined_ms_per_step"] = latency_ms
            line["unpipelined_value"] = total_out_px / (latency_ms * 1e-3) / 1e6
        if affinity:
            line["config"]["host_affinity"] = affinity
        if world > 1:
            line["config"]["start"] = ("barrier + synchronize on every rank, then an 8 MB all_reduce on the launching stream in front of the start "
                                       "event: every rank's clock starts when the last GPU arrives, with the NVLink links out of their idle state")
        if parity is not None:
            line["parity"] = parity
        if halo_info is not None:
            line["halo"] = halo_info
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
    up.close()
    if dist is not None:
        dist.destroy_process_group()


def dump_output(dirname, name, out, max_pixels):
    """Writes dirname/name.npy: the [rows, width, 4] image `out` as float32 [n, 4], the pixels in row-major order; above
    max_pixels a fixed sample of them (numpy default_rng(0)), so that two builds write the same pixels."""
    import numpy as np
    import torch
    rows, width = out.shape[:2]
    n = rows * width
    idx = np.arange(n) if n <= max_pixels else np.sort(np.random.default_rng(0).choice(n, max_pixels, replace=False))
    idx = torch.from_numpy(idx).to(out.device)
    pix = out[idx // width, idx % width].float().cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), pix)


def check_sharded_parity(F, api, up, dist, dev, rank, world, iw, ih, ow, oh, H_in, H_out, tdt, rank_rows, halo_mode):
    """Outside the timed region: frame 0 once more through the sharded path, every rank's slab sent to rank 0, which upscales the
    whole frame on its own GPU and compares bit for bit; then against the oracle on bands that straddle slab boundaries; then
    the OTHER halo data plane against this one."""
    import numpy as np
    import torch
    import oracle_lib as ol
    stream = torch.cuda.current_stream()
    plan = up.plan
    o0, o1 = plan.owned_in_rows(rank)
    up.input(0).copy_(torch.from_numpy(np.ascontiguousarray(rank_rows(0, rank, o0, o1))).to(dev))
    up.submit(0, stream)
    up.wait(0, stream)
    torch.cuda.synchronize()
    mine = up.output(0).contiguous().clone()
    # the other data plane, one frame, same input
    other_mode = "nccl" if halo_mode == "p2p" else "p2p"
    other = F.ShardedUpscaler(iw, H_in, ow, H_out, world, rank, SHARPNESS, dtype=tdt, device=dev, slots=1, halo=other_mode)
    other.input(0).copy_(up.input(0))
    other.submit(0, stream)
    other.wait(0, stream)
    torch.cuda.synchronize()
    same = torch.tensor([1 if torch.equal(other.output(0), mine) else 0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    other.close()
    result = {"%s_equals_%s" % (other_mode, halo_mode): bool(same.item())}
    if rank != 0:
        dist.send(mine, 0)
        return None
    slabs = [mine]
    for r in range(1, world):
        a, b = plan.out_rows(r)
        t = torch.empty((b - a, ow, 4), dtype=tdt, device=dev)
        dist.recv(t, r)
        slabs.append(t)
    full = np.concatenate([rank_rows(0, r, *plan.owned_in_rows(r)) for r in range(world)])
    full_t = torch.from_numpy(np.ascontiguousarray(full)).to(dev)
    tmp = torch.empty((H_out, ow, 4), dtype=tdt, device=dev)
    whole = torch.empty((H_out, ow, 4), dtype=tdt, device=dev)
    api.upscale(full_t, tmp, whole, up.econ, up.rcon)
    torch.cuda.synchronize()
    eq = all(torch.equal(slabs[r], whole[plan.out_rows(r)[0]:plan.out_rows(r)[1]]) for r in range(world))
    result["sharded_equals_single_gpu"] = bool(eq)
    # oracle on bands: the top of the frame and 32 rows around the first and last slab boundaries
    f32 = full.astype(np.float32) if full.dtype != np.uint8 else full.astype(np.float32) / 255.0
    got = torch.cat(slabs).cpu().numpy()
    got = got.astype(np.float32) if got.dtype != np.uint8 else got.astype(np.float32) / 255.0
    worst = 0.0
    bands = [(0, 32)] + [(plan.out_rows(r)[0] - 16, plan.out_rows(r)[0] + 16) for r in sorted({1, world - 1})]
    for (a, b) in bands:
        e = ol.easu(f32, ow, H_out, y0=max(a - 1, 0), y1=min(b + 1, H_out))
        want = ol.rcas(e, ol.rcas_con(SHARPNESS), y0=a, y1=b)
        worst = max(worst, float(np.abs(got[a:b] - want[a:b])[..., :3].max()))
    result["max_abs_vs_oracle"] = worst
    result["oracle_bands"] = bands
    result["tolerance"] = 1e-2 if tdt != torch.float32 else 1e-5
    return result


def run_reference(args, rank):
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is meant to use all host threads it can,
    # so restore the default BEFORE the OpenMP runtime of the oracle libraries is loaded
    if os.environ.get("WORLD_SIZE") and os.environ.get("OMP_NUM_THREADS") == "1":
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    wl = WORKLOADS[args.workload]
    r = time_cpu(wl, steps=args.steps, warmup=max(args.warmup, 1), budget_s=100.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "Mpix/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl[5], "sharpness_stops": SHARPNESS,
                       "note": "the reference ships no CPU pixel path; this is its own FsrEasuF/FsrRcasF source compiled "
                               "for the host (oracle/_ref) or, if that was not built, the oracle port"},
            "cpu_baseline": {"value": r["value"], "unit": "Mpix/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                             "cpu_model": r["cpu_model"], "logical_cpus": r["logical_cpus"]},
            "e2e": {"value": r["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="1080p-4k-fp16", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-pipeline", action="store_true", help="EASU and RCAS of each frame back to back on one stream (no frame overlap)")
    ap.add_argument("--frames", type=int, default=0, help="distinct synthetic frames resident in HBM (default 8; BASELINE configs[2] uses 120)")
    ap.add_argument("--shard-frame", action="store_true", help="multi-GPU: shard the workload's own frame by rows (strong scaling) instead of stacking one frame per rank")
    ap.add_argument("--fused", action="store_true", help="FSR1_FLAG_FUSED: EASU and RCAS in one kernel (intermediate in shared memory); roofline against bpp*(Pin+Pout)")
    ap.add_argument("--trace", action="store_true", help="multi-GPU p2p: print device-timestamp statistics of the halo hand-shake per rank (stderr)")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"], help="multi-GPU halo data plane: direct NVLink stores through the C ABI (default) or NCCL send/recv")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the upscaled frame of the last one as DIR/output.npy "
                    "(DIR/output_rank<r>.npy per rank with --gpus > 1): float32 [n, 4] RGBA pixels, a fixed seeded sample of 2M "
                    "pixels of a larger frame; the inputs are the same every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # the reference's OpenMP team: one thread per logical CPU, threads pinned (must be set before libgomp loads)
    os.environ.setdefault("OMP_PROC_BIND", "true")
    if args.impl == "reference":
        return run_reference(args, rank)
    if args.gpus > 1 and world == 1:
        # launched without torchrun: re-exec under it (one rank per GPU)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29400 + os.getpid() % 500), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
