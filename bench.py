#!/usr/bin/env python
"""bench.py — the headline measurement: 4K yuv420p -> rgb24 swscale frames/s (BASELINE.json configs[1]),
with the batched 8x8 IDCT (configs[2]) reported beside it, on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One step = one pass of the hot path over one batch of 256 synthetic 4K frames per GPU (weak scaling: every rank
converts its own batch, no data-path collective; the optional NCCL gather at the mux boundary is reported separately).
Rank 0 prints ONE JSON line.  `value` is device-resident throughput (CUDA events on the launching stream, max over
ranks); `e2e` is the same metric through the C-ABI host entry point with pinned HOST buffers, H2D and D2H copies inside
the timed region.  --impl reference times the reference's own CPU implementation (oracle/_ref/libffref.so when it was
built, else the oracle port) with all host threads on a bounded sample of the same workload.
--dump-outputs DIR writes what the headline's last timed step computed (rank 0's rgb24 frames) as DIR/*.npy, see dump_outputs().
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W4K, H4K = 3840, 2160
BATCH = 256
FRAME_BYTES_IN = W4K * H4K * 3 // 2           # 12 441 600
FRAME_BYTES_OUT = W4K * H4K * 3               # 24 883 200
FRAME_BYTES = FRAME_BYTES_IN + FRAME_BYTES_OUT  # 37 324 800 algorithmic bytes / frame (SURVEY.md 8d)
SWS_BICUBIC, SWS_ACCURATE_RND, SWS_BITEXACT = 4, 0x40000, 0x80000
FLAGS_FATE = SWS_BICUBIC | SWS_ACCURATE_RND | SWS_BITEXACT
MB_W, MB_H = 120, 68                          # 1080p macroblocks
IDCT_FRAMES = 256                             # frames of 48 960 blocks per step (of the 10 000-frame stream)
HEADLINE_KERNEL = "sws_vscale_rgb24_pair_kernel<RGB24, yuv420p> (two output lines per thread; the first and last line of a frame go to sws_vscale_rgb24_fast_kernel)"
METRIC = "4K frames/sec swscale yuv420p->rgb24; 8x8 IDCT blocks/sec; HBM GB/s vs peak"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel_key):
    """dram bytes per launch from the committed ncu summary (profiles/ncu_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel_key)
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (B200_PROFILING.md recipe): one streaming
    `nvidia-smi -lms 100` process, started before the first timed region and stopped after the last."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            rows = [[x.strip() for x in ln.split(",")] for ln in out.splitlines() if ln.strip()]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "", 1).isdigit()]
        reasons = set()
        for r in rows:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(rows)}


# ------------------------------------------------------------------------------------------------ CPU arms
def gpu_numa_cpus(index):
    """CPUs of the NUMA node the GPU hangs off (what `numactl --cpunodebind` would use), or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                     # nvml prints an 8-digit domain, sysfs uses 4
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        return cpus or None
    except Exception:
        return None


class near_gpu:
    """Run the block on the CPUs next to the GPU, so that pinned host buffers allocated inside land on that NUMA node."""
    def __init__(self, index):
        self.cpus = gpu_numa_cpus(index)

    def __enter__(self):
        self.old = None
        if self.cpus:
            try:
                self.old = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self.cpus & self.old or self.cpus)
            except Exception:
                self.old = None
        return self

    def __exit__(self, *a):
        if self.old:
            os.sched_setaffinity(0, self.old)


_STDOUT_FD = None


def emit_line(line):
    """The one JSON line, on the real stdout."""
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)


def cpu_lib():
    import cpulibs as cl
    if cl.have_ref():
        return cl.ref(), "reference", "ffref"
    return cl.oracle(), "port", "orc"


def usable_cpus():
    """Host threads this process can really run at once: the scheduler affinity mask capped by the cgroup CPU quota (a leased box
    often shows every core in os.cpu_count() while the container is limited to a fraction of them)."""
    import math
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    n = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return n, {"os_cpu_count": os.cpu_count(), "affinity": aff, "cgroup_quota_cpus": quota}


def run_threads(workers, seconds):
    """workers: one callable per thread, each call returns the units it processed (ctypes releases the GIL inside the library).
    Every thread loops until the deadline; returns (units per second, units, seconds)."""
    counts = [0.0] * len(workers)
    deadline = time.perf_counter() + seconds

    def loop(i):
        w = workers[i]
        while True:
            counts[i] += w()
            if time.perf_counter() >= deadline:
                break

    ts = [threading.Thread(target=loop, args=(i,)) for i in range(len(workers))]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    return sum(counts) / dt, sum(counts), dt


def cpu_sws_workers(flags, threads):
    import numpy as np
    import cpulibs as cl
    lib, kind, pre = cpu_lib()
    y, u, v = cl.yuv_frame(W4K, H4K, 1, "random")
    out = [np.empty((H4K, W4K * 3), np.uint8) for _ in range(threads)]
    if pre == "ffref":
        ctxs = [lib.ffref_sws_open(W4K, H4K, W4K, H4K, flags, 1) for _ in range(threads)]
    else:
        ctxs = [lib.orc_sws_open(W4K, H4K, W4K, H4K, flags) for _ in range(threads)]

    def mk(i):
        def one():
            if pre == "ffref":
                lib.ffref_sws_scale(ctxs[i], cl.ptr(y), W4K, cl.ptr(u), W4K // 2, cl.ptr(v), W4K // 2, 0, H4K, cl.ptr(out[i]), W4K * 3)
            else:
                lib.orc_sws_scale(ctxs[i], cl.ptr(y), W4K, cl.ptr(u), W4K // 2, cl.ptr(v), W4K // 2, cl.ptr(out[i]), W4K * 3)
            return 1
        return one

    def close():
        for c in ctxs:
            (lib.ffref_sws_close if pre == "ffref" else lib.orc_sws_close)(c)
    return [mk(i) for i in range(threads)], close, "4K frames"


def cpu_idct_workers(threads, op=1):
    import numpy as np
    import cpulibs as cl
    from cases import idct_blocks
    lib, kind, pre = cpu_lib()
    n = MB_W * MB_H * 6
    blk0 = idct_blocks("dense", n, 1)
    off = (np.arange(n) * 8).astype(np.int64)
    fn = lib.ffref_idct_batch if pre == "ffref" else lib.orc_idct_batch
    bufs = [(blk0.copy(), np.zeros((8, n * 8), np.uint8)) for _ in range(threads)]

    def mk(i):
        def one():
            b, d = bufs[i]
            b[:] = blk0                                 # the reference clobbers the coefficients
            fn(op, cl.ptr(b, cl.i16p), n, cl.ptr(d), n * 8, cl.ptr(off, cl.i64p))
            return n
        return one
    return [mk(i) for i in range(threads)], (lambda: None), "8x8 blocks (one 1080p frame of 48 960 per call)"


def cpu_qpel_workers(threads):
    """one 1080p frame of 8160 16x16 operations per call: random quarter-pel position, put / avg, vectors within +-16 px"""
    import numpy as np
    import cpulibs as cl
    lib, kind, pre = cpu_lib()
    W, H, apron = 1920, 1088, 32
    PW, PH = W + 2 * apron, H + 2 * apron
    rng = np.random.default_rng(3)
    src = rng.integers(0, 256, (PH, PW), dtype=np.uint8)
    by, bx = np.meshgrid(np.arange(H // 16), np.arange(W // 16), indexing="ij")
    base = (by * 16 + apron) * PW + bx * 16 + apron
    dx, dy = rng.integers(-16, 17, base.shape), rng.integers(-16, 17, base.shape)
    doff = base.reshape(-1).astype(np.int64)
    soff = (base + dy * PW + dx).reshape(-1).astype(np.int64)
    ops = (rng.integers(0, 2, doff.size) | (rng.integers(0, 16, doff.size) << 3)).astype(np.uint8)
    n = int(doff.size)
    fn = lib.ffref_h264qpel_batch if pre == "ffref" else lib.orc_h264qpel_batch
    dsts = [rng.integers(0, 256, (PH, PW), dtype=np.uint8) for _ in range(threads)]

    def mk(i):
        def one():
            fn(n, cl.ptr(ops), cl.ptr(dsts[i]), cl.ptr(doff, cl.i64p), cl.ptr(src), cl.ptr(soff, cl.i64p), PW)
            return n
        return one
    return [mk(i) for i in range(threads)], (lambda: None), "16x16 blocks (one 1080p frame of 8160 per call)"


def cpu_esa_workers(threads):
    """one macroblock row (240 blocks x up to 4225 candidates) of a 4K frame pair per call; 135 rows = one pair"""
    import numpy as np
    import cpulibs as cl
    lib, kind, pre = cpu_lib()
    rng = np.random.default_rng(4)
    cur = rng.integers(0, 256, (H4K, W4K), dtype=np.uint8)
    ref = np.ascontiguousarray(np.roll(cur, (7, -13), (0, 1)))
    rows = H4K // 16
    nmb = rows * (W4K // 16)
    fn = lib.ffref_esa_frame if pre == "ffref" else lib.orc_esa_frame
    outs = [(np.zeros((nmb, 2), np.int32), np.zeros(nmb, np.uint64)) for _ in range(threads)]
    nxt = [i % rows for i in range(threads)]

    def mk(i):
        def one():
            r = nxt[i]
            nxt[i] = (r + threads) % rows
            fn(cl.ptr(cur), cl.ptr(ref), W4K, W4K, H4K, 16, 32, r, r + 1, cl.ptr(outs[i][0], cl.i32p), cl.ptr(outs[i][1], cl.u64p))
            return 1.0 / rows
        return one
    return [mk(i) for i in range(threads)], (lambda: None), "4K frame pairs (one macroblock row = 1/135 pair per call)"


def cpu_tx_workers(threads, typ, n):
    """256 transforms per call; typ 0: forward complex FFT of n points, typ 1: inverse MDCT of len n (scale 1/n)"""
    import numpy as np
    import cpulibs as cl
    lib, kind, pre = cpu_lib()
    cnt = 256
    rng = np.random.default_rng(5)
    op, cls, run = (lib.ffref_tx_open, lib.ffref_tx_close, lib.ffref_tx_run) if pre == "ffref" else (lib.orc_tx_open, lib.orc_tx_close, lib.orc_tx_run)
    hs = [op(typ, 1 if typ == 1 else 0, n, 1.0 / n if typ == 1 else 1.0, 0) for _ in range(threads)]
    ie = 2 * n if typ == 0 else n
    xin = [rng.random((cnt, ie), dtype=np.float32) for _ in range(threads)]
    xout = [np.zeros((cnt, ie), np.float32) for _ in range(threads)]

    def mk(i):
        def one():
            run(hs[i], xout[i].ctypes.data, xin[i].ctypes.data, 8 if typ == 0 else 4, cnt, 4 * ie, 4 * ie)
            return cnt
        return one

    def close():
        for h in hs:
            cls(h)
    return [mk(i) for i in range(threads)], close, "transforms (256 per call)"


def cpu_arm(make, seconds_all, seconds_one, unit):
    """One path on all usable host threads and on one thread (SURVEY 8d); returns the cpu_baseline object."""
    _, kind, _ = cpu_lib()
    n, info = usable_cpus()
    res = {}
    for threads, secs in ((n, seconds_all), (1, seconds_one)):
        workers, close, what = make(threads)
        workers[0]()                                    # warm-up
        rate, units, dt = run_threads(workers, secs)
        close()
        res[threads] = (rate, f"{units:.4g} {what} on {threads} thread{'s' if threads > 1 else ''}, {dt:.1f} s")
        if n == 1:
            break
    out = {"value": res[n][0], "unit": unit, "cores": n, "kind": kind, "sample": res[n][1], "cpu_limits": info}
    one = res.get(1, res[n])
    out["single_thread"] = {"value": one[0], "unit": unit, "sample": one[1]}
    return out


def cpu_baselines_all(scale=1.0, with_sws=True):
    """The reference's CPU path for every BASELINE config, bounded samples (about 35 s in all at scale 1)."""
    out = {}
    if with_sws:
        out["sws"] = cpu_arm(lambda t: cpu_sws_workers(FLAGS_FATE, t), 10.0 * scale, 3.0 * scale, "frames/s")
    out["idct_put"] = cpu_arm(lambda t: cpu_idct_workers(t, 1), 2.5 * scale, 1.2 * scale, "blocks/s")
    out["idct_add"] = cpu_arm(lambda t: cpu_idct_workers(t, 2), 2.0 * scale, 1.0 * scale, "blocks/s")
    out["h264qpel"] = cpu_arm(cpu_qpel_workers, 2.5 * scale, 1.2 * scale, "16x16 blocks/s")
    out["me_esa"] = cpu_arm(cpu_esa_workers, 3.0 * scale, 1.5 * scale, "4K frame pairs/s")
    for typ, nm in ((0, "fft"), (1, "imdct")):
        for n in (1024, 2048):
            out[f"{nm}{n}"] = cpu_arm(lambda t: cpu_tx_workers(t, typ, n), 1.5 * scale, 0.8 * scale, "transforms/s")
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    n, info = usable_cpus()
    t_all = time.perf_counter()
    workers, close, what = cpu_sws_workers(FLAGS_FATE, n)
    for _ in range(min(args.warmup, 1)):
        workers[0]()
    steps = max(1, min(args.steps, 3))             # bounded: each step is itself a multi-second sample
    rates, frames, secs = [], 0.0, 0.0
    for _ in range(steps):
        r, u, dt = run_threads(workers, 6.0)
        rates.append(r); frames += u; secs += dt
    close()
    fps = sum(rates) / len(rates)
    _, kind, _ = cpu_lib()
    cb = {"value": fps, "unit": "frames/s", "cores": n, "kind": kind, "cpu_limits": info,
          "sample": f"{frames:.0f} 4K frames on {n} threads, {secs:.1f} s ({steps} steps)"}
    others = cpu_baselines_all(scale=0.7, with_sws=False)
    cb["others"] = {k: {"value": v["value"], "unit": v["unit"], "single_thread": v["single_thread"]["value"]} for k, v in others.items()}
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * BATCH / fps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"swscale {W4K}x{H4K} yuv420p->rgb24 flags=bicubic+accurate_rnd+bitexact, batch={BATCH} (bounded CPU sample per step)",
                   "timed_steps": steps},
        "cpu_baseline": cb,
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "idct": {"value": others["idct_put"]["value"], "unit": "blocks/s"},
        "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def host_timed(call, steps, barrier, reduce_max):
    """Wall-clock of `steps` calls of a synchronous HOST-buffer entry point (it returns after its last D2H), max over ranks."""
    import torch
    call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        call()
    torch.cuda.synchronize()
    return reduce_max(time.perf_counter() - t0) / steps


def pinned_like(t):
    import torch
    h = torch.empty(t.shape, dtype=t.dtype).pin_memory()
    h.copy_(t)
    return h


def extra_paths(args, dev, stream, g, world, barrier, reduce_max, peak, devidx):
    """The other rows of SURVEY.md 8(d): ESA motion search, H.264 qpel MC and float FFT / iMDCT, each on a bounded batch, each with
    its device-resident number, its roofline fraction and an end-to-end number through the HOST-buffer entry point."""
    import torch
    from ffmpeg_b200 import me_cmp, pel, tx, idctdsp
    out = {}
    steps = max(2, min(args.steps, 5))
    sm_count = torch.cuda.get_device_properties(devidx).multi_processor_count
    sm_max_mhz = 1965.0
    try:
        sm_max_mhz = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"])
    except Exception:
        pass

    def timed(call):
        with torch.cuda.stream(stream):
            for _ in range(2):
                call()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                call()
            e1.record(stream)
        barrier()
        return reduce_max(e0.elapsed_time(e1)) / steps

    def timed_with_prep(prep, call):
        """mean device time of `call` alone: every step runs `prep` (refills what the call consumes, then evicts it from L2 by writing a
        buffer larger than L2) outside the event pair, `call` inside it -- nothing is subtracted afterwards"""
        flush = torch.empty(192 << 20, dtype=torch.uint8, device="cuda")
        with torch.cuda.stream(stream):
            for _ in range(2):
                prep(); flush.fill_(1); call()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        with torch.cuda.stream(stream):
            for a, b in evs:
                prep(); flush.fill_(1)
                a.record(stream); call(); b.record(stream)
        barrier()
        stream.synchronize()
        del flush
        return reduce_max(sum(a.elapsed_time(b) for a, b in evs)) / steps

    # --- config 4: SAD full search 16x16, +-32, 4K luma pairs (integer-ALU bound; bytes are 16.6 MB per pair)
    npairs = 4
    with torch.cuda.stream(stream):
        cur = torch.randint(0, 256, (npairs, H4K, W4K), dtype=torch.uint8, device="cuda", generator=g)
        ref = torch.roll(cur, shifts=(7, -13), dims=(1, 2)).contiguous()
        nmb = (W4K // 16) * (H4K // 16)
        mv = torch.zeros((npairs, nmb, 2), dtype=torch.int32, device="cuda")
        cost = torch.zeros((npairs, nmb), dtype=torch.int64, device="cuda")
    ms = timed(lambda: me_cmp.me_esa_device(dev, cur, ref, W4K, W4K, H4K, W4K * H4K, npairs, 16, 32, mv, cost))
    # algorithmic work: every candidate the clipped windows hold (exact count; 4225 per block only away from the frame borders)
    cx = sum(min(W4K - 16, x + 32) - max(0, x - 32) + 1 for x in range(0, W4K, 16))
    cy = sum(min(H4K - 16, y + 32) - max(0, y - 32) + 1 for y in range(0, H4K, 16))
    absdiff = float(cx) * cy * 256                   # abs-diff-accumulates per pair (3.40e10; SURVEY's 3.50e10 ignores the clipping)
    # integer peak: VABSDIFF4.U8.ACC does 4 byte lanes per thread on the ALU pipe, 16 threads / clk / SM sub-partition = 64 / clk / SM
    ipeak = sm_count * 64 * 4 * sm_max_mhz * 1e6 / 1e12
    ach = absdiff * npairs / (ms / 1e3) / 1e12
    out["me_esa"] = {"value": world * npairs / (ms / 1e3), "unit": "4K frame pairs/s", "ms_per_step": ms,
                     "config": f"SAD full search 16x16 +-32, {npairs} 4K pairs per step",
                     "roofline": {"bound": "integer alu", "achieved": ach, "peak": ipeak, "unit": "T abs-diff/s", "frac": ach / ipeak,
                                  "peak_source": f"{sm_count} SMs x 64 VABSDIFF4/clk x 4 bytes x {sm_max_mhz:.0f} MHz (MEASURED_PEAKS sm_max_mhz)",
                                  "hbm_GBps": 2 * W4K * H4K * npairs / (ms / 1e3) / 1e9, "hbm_frac": 2 * W4K * H4K * npairs / (ms / 1e3) / 1e9 / peak}}
    try:
        hcur, href = pinned_like(cur.cpu()), pinned_like(ref.cpu())
        hmv = torch.zeros((npairs, nmb, 2), dtype=torch.int32).pin_memory()
        hcost = torch.zeros((npairs, nmb), dtype=torch.int64).pin_memory()
        dt = host_timed(lambda: me_cmp.me_esa_host(dev, hcur, href, W4K, W4K, H4K, W4K * H4K, npairs, 16, 32, hmv, hcost), 2, barrier, reduce_max)
        stream.synchronize()
        out["me_esa"]["e2e"] = {"value": world * npairs / dt, "unit": "4K frame pairs/s", "h2d_bytes_per_step": 2 * W4K * H4K * npairs,
                                "d2h_bytes_per_step": nmb * 16 * npairs, "api": "b200_me_esa_host",
                                "matches_device_path": bool(torch.equal(hmv, mv.cpu()) and torch.equal(hcost, cost.cpu()))}
        del hcur, href, hmv, hcost
    except Exception as ex:
        out["me_esa"]["e2e"] = {"value": None, "error": str(ex)[:160]}
    del cur, ref, mv, cost

    # --- config 3 (MC half): H.264 qpel 16x16, random quarter-pel vectors within +-16 px, random put/avg, 1080p frames
    nfr, W, H, apron = 64, 1920, 1088, 32
    PW, PH = W + 2 * apron, H + 2 * apron
    with torch.cuda.stream(stream):
        refp = torch.randint(0, 256, (nfr, PH, PW), dtype=torch.uint8, device="cuda", generator=g)
        dstp = torch.randint(0, 256, (nfr, PH, PW), dtype=torch.uint8, device="cuda", generator=g)
        fidx = torch.arange(nfr, device="cuda").view(-1, 1, 1)
        by = torch.arange(H // 16, device="cuda").view(1, -1, 1)
        bx = torch.arange(W // 16, device="cuda").view(1, 1, -1)
        base = fidx * (PH * PW) + (by * 16 + apron) * PW + bx * 16 + apron
        dx = torch.randint(-16, 17, base.shape, device="cuda", generator=g)
        dy = torch.randint(-16, 17, base.shape, device="cuda", generator=g)
        doff = base.reshape(-1).to(torch.int64).contiguous()
        soff = (base + dy * PW + dx).reshape(-1).to(torch.int64).contiguous()
        ops = (torch.randint(0, 2, (doff.numel(),), device="cuda", generator=g) |
               (torch.randint(0, 16, (doff.numel(),), device="cuda", generator=g) << 3)).to(torch.uint8)
    nops = doff.numel()
    ms = timed(lambda: pel.h264qpel_batch_device(dev, nops, ops, dstp, doff, refp, soff, PW))
    qbytes = 441 + 256 + 128                         # 21x21 reference window + 16x16 out (+ dst read for the avg half)
    out["h264qpel"] = {"value": world * nops / (ms / 1e3), "unit": "16x16 blocks/s", "ms_per_step": ms,
                       "config": f"{nfr} 1080p frames x 8160 MBs, random qpel position and put/avg",
                       "roofline": {"bound": "hbm", "achieved": qbytes * nops / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": qbytes * nops / (ms / 1e3) / 1e9 / peak, "bytes_per_block": qbytes}}
    try:
        hsrc, hdst0 = pinned_like(refp.cpu()), dstp.cpu()
        hdst = pinned_like(hdst0)
        hops, hdo, hso = ops.cpu().numpy(), doff.cpu().numpy(), soff.cpu().numpy()
        import numpy as np
        begin = (np.arange(nfr + 1, dtype=np.int64) * (nops // nfr))
        call = lambda: pel.h264qpel_frames_host(dev, nfr, PH * PW, begin, hops, hdst, hdo, hsrc, hso, PW)
        dt = host_timed(call, 3, barrier, reduce_max)
        hdst.copy_(hdst0)                               # avg operations accumulate: compare one fresh pass with one device pass
        call()
        with torch.cuda.stream(stream):
            dchk = hdst0.cuda()
            pel.h264qpel_batch_device(dev, nops, ops, dchk, doff, refp, soff, PW)
        stream.synchronize()
        out["h264qpel"]["e2e"] = {"value": world * nops / dt, "unit": "16x16 blocks/s", "h2d_bytes_per_step": 2 * nfr * PH * PW + 17 * nops,
                                  "d2h_bytes_per_step": nfr * PH * PW, "api": "b200_h264qpel_frames_host",
                                  "matches_device_path": bool(torch.equal(dchk.cpu(), hdst))}
        del hsrc, hdst, hdst0, dchk
    except Exception as ex:
        out["h264qpel"]["e2e"] = {"value": None, "error": str(ex)[:160]}
    del refp, dstp, doff, soff, ops

    # --- widening row (SURVEY 8f): the chroma half of the same stream, h264chroma mc8 8x8 on the two 960x544 chroma planes
    CW, CH, capron = W // 2, H // 2, 16
    CPW, CPH = CW + 2 * capron, CH + 2 * capron
    with torch.cuda.stream(stream):
        refc = torch.randint(0, 256, (2 * nfr, CPH, CPW), dtype=torch.uint8, device="cuda", generator=g)
        dstc = torch.randint(0, 256, (2 * nfr, CPH, CPW), dtype=torch.uint8, device="cuda", generator=g)
        fidx = torch.arange(2 * nfr, device="cuda").view(-1, 1, 1)
        by = torch.arange(CH // 8, device="cuda").view(1, -1, 1)
        bx = torch.arange(CW // 8, device="cuda").view(1, 1, -1)
        base = fidx * (CPH * CPW) + (by * 8 + capron) * CPW + bx * 8 + capron
        dx = torch.randint(-8, 9, base.shape, device="cuda", generator=g)
        dy = torch.randint(-8, 9, base.shape, device="cuda", generator=g)
        doff = base.reshape(-1).to(torch.int64).contiguous()
        soff = (base + dy * CPW + dx).reshape(-1).to(torch.int64).contiguous()
        ops = torch.randint(0, 2, (doff.numel(),), device="cuda", generator=g).to(torch.uint8)
        hs = torch.full((doff.numel(),), 8, dtype=torch.uint8, device="cuda")
        xys = torch.randint(0, 64, (doff.numel(),), device="cuda", generator=g).to(torch.uint8)
    nops = doff.numel()
    ms = timed(lambda: pel.h264chroma_batch_device(dev, nops, ops, hs, xys, dstc, doff, refc, soff, CPW))
    cbytes = 81 + 64 + 32                            # 9x9 reference window + 8x8 out (+ dst read for the avg half)
    out["h264chroma"] = {"value": world * nops / (ms / 1e3), "unit": "8x8 blocks/s", "ms_per_step": ms,
                         "config": f"{2 * nfr} 960x544 chroma planes x 8160 blocks, random eighth-pel phase and put/avg",
                         "roofline": {"bound": "hbm", "achieved": cbytes * nops / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                      "frac": cbytes * nops / (ms / 1e3) / 1e9 / peak, "bytes_per_block": cbytes}}
    del refc, dstc, doff, soff, ops, hs, xys

    # --- widening row (SURVEY 8f): H.264 residual add, 4x4 and 8x8 transforms over 1080p luma planes
    hn = 32
    with torch.cuda.stream(stream):
        planes_h = torch.randint(0, 256, (hn, H, W), dtype=torch.uint8, device="cuda", generator=g)
    h264r = {}
    for kind, N, nm in ((0, 4, "idct4_add"), (1, 8, "idct8_add")):
        nb = hn * (H // N) * (W // N)
        with torch.cuda.stream(stream):
            coef = torch.randint(-600, 601, (nb, N * N), dtype=torch.int16, device="cuda", generator=g)
            keep = coef.clone()
            bi = torch.arange(nb, device="cuda", dtype=torch.int64)
            per = (H // N) * (W // N)
            fr, r = bi // per, bi % per
            hdoff = (fr * (H * W) + (r // (W // N)) * (N * W) + (r % (W // N)) * N).contiguous()
            hboff = (bi * (N * N)).contiguous()

        # the transform clears its coefficients, like the reference: refilled (and evicted from L2) before every timed call
        ms = timed_with_prep(lambda: coef.copy_(keep), lambda: idctdsp.h264_idct_batch_device(dev, kind, nb, coef, hboff, planes_h, hdoff, W))
        bpb = 2 * N * N * 2 + 2 * N * N                # coefficients read + cleared, pixels read + written
        h264r[nm] = {"value": world * nb / (ms / 1e3), "unit": "blocks/s", "ms_per_step": ms, "blocks": nb,
                     "roofline": {"bound": "hbm", "achieved": bpb * nb / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": bpb * nb / (ms / 1e3) / 1e9 / peak, "bytes_per_block": bpb},
                     "note": "coefficients refilled and evicted from L2 before every timed call; the events bracket the transform alone"}
        del coef, keep, hdoff, hboff
    out["h264_idct"] = h264r
    del planes_h

    # --- config 5: float FFT and iMDCT, len 1024 and 2048
    txr = {}
    for n in (1024, 2048):
        cnt = (1 << 18) if n == 1024 else (1 << 17)
        with torch.cuda.stream(stream):
            x = torch.rand((cnt, 2 * n), device="cuda", generator=g)
            y = torch.empty_like(x)
        c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 0, n, device=dev)
        ms = timed(lambda: c.batch_device(y, x, 8, cnt, 8 * n, 8 * n))
        c.uninit()
        b = 16 * n
        txr[f"fft{n}"] = {"value": world * cnt / (ms / 1e3), "unit": "transforms/s", "ms_per_step": ms, "batch": cnt,
                          "roofline": {"bound": "hbm", "achieved": b * cnt / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                       "frac": b * cnt / (ms / 1e3) / 1e9 / peak, "bytes_per_transform": b}}
        ecnt = cnt // 4
        try:
            c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 0, n, device=dev)
            hx = pinned_like(x[:ecnt].cpu())
            hy = torch.empty_like(hx).pin_memory()
            dt = host_timed(lambda: c.batch_host(hy, hx, 8, ecnt, 8 * n, 8 * n), 3, barrier, reduce_max)
            with torch.cuda.stream(stream):
                c.batch_device(y, x, 8, ecnt, 8 * n, 8 * n)
            stream.synchronize()
            txr[f"fft{n}"]["e2e"] = {"value": world * ecnt / dt, "unit": "transforms/s", "h2d_bytes_per_step": 8 * n * ecnt,
                                     "d2h_bytes_per_step": 8 * n * ecnt, "api": "b200_tx_batch_host",
                                     "matches_device_path": bool(torch.equal(y[:ecnt].cpu(), hy))}
            c.uninit()
            c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, n, scale=1.0 / n, device=dev)
            hxi = pinned_like(x.view(-1)[:ecnt * n].view(ecnt, n).cpu())
            hyi = torch.empty_like(hxi).pin_memory()
            dt = host_timed(lambda: c.batch_host(hyi, hxi, 4, ecnt, 4 * n, 4 * n), 3, barrier, reduce_max)
            e2e_imdct = {"value": world * ecnt / dt, "unit": "transforms/s", "h2d_bytes_per_step": 4 * n * ecnt,
                         "d2h_bytes_per_step": 4 * n * ecnt, "api": "b200_tx_batch_host"}
            c.uninit()
            del hx, hy, hxi, hyi
        except Exception as ex:
            txr[f"fft{n}"]["e2e"] = {"value": None, "error": str(ex)[:160]}
            e2e_imdct = {"value": None, "error": str(ex)[:160]}
        c = tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 0, n, scale=1.0, device=dev)      # r2c: n floats -> n/2+1 complex
        ms = timed(lambda: c.batch_device(y, x, 4, cnt, 8 * n, 8 * n))
        c.uninit()
        b = 4 * n + 4 * (n + 2)
        txr[f"rdft_r2c{n}"] = {"value": world * cnt / (ms / 1e3), "unit": "transforms/s", "ms_per_step": ms, "batch": cnt,
                               "roofline": {"bound": "hbm", "achieved": b * cnt / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                            "frac": b * cnt / (ms / 1e3) / 1e9 / peak, "bytes_per_transform": b}}
        c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, n, scale=1.0 / n, device=dev)
        ms = timed(lambda: c.batch_device(y, x, 4, cnt, 4 * n, 4 * n))
        c.uninit()
        b = 8 * n
        txr[f"imdct{n}"] = {"value": world * cnt / (ms / 1e3), "unit": "transforms/s", "ms_per_step": ms, "batch": cnt,
                            "roofline": {"bound": "hbm", "achieved": b * cnt / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                         "frac": b * cnt / (ms / 1e3) / 1e9 / peak, "bytes_per_transform": b},
                            "e2e": e2e_imdct}
        del x, y
    out["tx"] = txr
    # --- widening rows (SURVEY 8f) that had no timing yet: 10-bit simple IDCT add, the compound MDCT of Opus CELT (15 x 64 = 960),
    # the int32 FFT of fixed-point AAC, vector_fmul_window (what follows every AAC iMDCT).  Device-resident, roofline fraction only.
    wid = {}
    try:
        nb = 1 << 20
        with torch.cuda.stream(stream):
            blk = torch.randint(-512, 513, (nb, 64), dtype=torch.int16, device="cuda", generator=g)
            dest = torch.randint(0, 1024, (8, nb * 8), dtype=torch.int16, device="cuda", generator=g)
            doff = (torch.arange(nb, device="cuda", dtype=torch.int64) * 16).contiguous()
        ms = timed(lambda: idctdsp.idct_hbd_batch_device(dev, 10, 2, blk, nb, dest, doff, None, nb * 16))
        b = 128 + 128 + 128
        wid["idct10_add"] = {"value": world * nb / (ms / 1e3), "unit": "blocks/s", "ms_per_step": ms,
                             "roofline": {"bound": "hbm", "achieved": b * nb / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                          "frac": b * nb / (ms / 1e3) / 1e9 / peak, "bytes_per_block": b}}
        del blk, dest, doff
    except Exception as ex:
        wid["idct10_add"] = {"error": str(ex)[:160]}
    for name, typ, inv, n, esz, inb, outb in (("mdct960_inv_15x64", tx.AV_TX_FLOAT_MDCT, 1, 960, 4, 4 * 960, 4 * 960),
                                              ("int32_fft1024", tx.AV_TX_INT32_FFT, 0, 1024, 8, 8 * 1024, 8 * 1024)):
        try:
            cnt = 1 << 16
            with torch.cuda.stream(stream):
                if typ == tx.AV_TX_INT32_FFT:
                    x = torch.randint(-(1 << 20), 1 << 20, (cnt, 2 * n), dtype=torch.int32, device="cuda", generator=g)
                else:
                    x = torch.rand((cnt, n), device="cuda", generator=g)
                y = torch.empty_like(x)
            c = tx.av_tx_init(typ, inv, n, scale=(1.0 / n if typ == tx.AV_TX_FLOAT_MDCT else None), device=dev)
            ms = timed(lambda: c.batch_device(y, x, esz, cnt, outb, inb))
            c.uninit()
            wid[name] = {"value": world * cnt / (ms / 1e3), "unit": "transforms/s", "ms_per_step": ms, "batch": cnt,
                         "roofline": {"bound": "hbm", "achieved": (inb + outb) * cnt / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                      "frac": (inb + outb) * cnt / (ms / 1e3) / 1e9 / peak, "bytes_per_transform": inb + outb}}
            del x, y
        except Exception as ex:
            wid[name] = {"error": str(ex)[:160]}
    try:
        from ffmpeg_b200 import float_dsp as fd
        nvec, length = 1 << 16, 1024
        with torch.cuda.stream(stream):
            dstw = torch.empty((nvec, 2 * length), device="cuda")
            s0 = torch.rand((nvec, length), device="cuda", generator=g)
            s1 = torch.rand((nvec, length), device="cuda", generator=g)
            win = torch.rand((2 * length,), device="cuda", generator=g)
        ms = timed(lambda: fd.float_dsp_batch_device(dev, 5, nvec, length, dstw, 2 * length, s0, length, s1, length, win, 0, 0.0))
        b = 4 * length * 4                              # two inputs of `length` floats, 2 * length floats out; the window stays in cache
        wid["vector_fmul_window_1024"] = {"value": world * nvec / (ms / 1e3), "unit": "vectors/s", "ms_per_step": ms,
                                          "roofline": {"bound": "hbm", "achieved": b * nvec / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                                       "frac": b * nvec / (ms / 1e3) / 1e9 / peak, "bytes_per_vector": b}}
        del dstw, s0, s1, win
    except Exception as ex:
        wid["vector_fmul_window_1024"] = {"error": str(ex)[:160]}
    # put_dct of an MPEG-2 intra stream: inverse quantiser + IDCT put, as two kernels (128 B + 128 B of extra coefficient traffic per block)
    # and as the fused kernel (coefficients dequantised in registers)
    try:
        from ffmpeg_b200 import mpegvideo
        fr = 64
        nbq = MB_W * MB_H * 6 * fr
        zz = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
              35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]
        perm, rend = mpegvideo.ff_init_scantable(list(range(64)), zz)
        prm = mpegvideo.unquant_params([8] + [16 + (i % 23) for i in range(1, 64)], [16] * 64, perm, rend, 8, 8)
        with torch.cuda.stream(stream):
            qb = torch.randint(-40, 41, (nbq, 64), dtype=torch.int16, device="cuda", generator=g)
            qwork = torch.empty_like(qb)
            qsc = torch.randint(1, 32, (nbq,), dtype=torch.uint8, device="cuda", generator=g)
            lastq = torch.full((nbq,), 63, dtype=torch.int8, device="cuda")
            pls = [torch.zeros((fr, MB_H * 16, MB_W * 16), dtype=torch.uint8, device="cuda"),
                   torch.zeros((fr, MB_H * 8, MB_W * 8), dtype=torch.uint8, device="cuda"),
                   torch.zeros((fr, MB_H * 8, MB_W * 8), dtype=torch.uint8, device="cuda")]
        lsq = [MB_W * 16, MB_W * 8, MB_W * 8]
        fsq = [MB_W * 16 * MB_H * 16, MB_W * 8 * MB_H * 8, MB_W * 8 * MB_H * 8]

        def two_kernels():
            mpegvideo.unquantize_batch_device(dev, 2, prm, qwork, nbq, None, qsc, lastq)      # the separate quantiser works in place
            idctdsp.idct_mb420_device(dev, 1, qwork, MB_W, MB_H, fr, pls, lsq, fsq)
        ms2 = timed_with_prep(lambda: qwork.copy_(qb), two_kernels)
        msf = timed_with_prep(lambda: None, lambda: mpegvideo.unquant_idct_mb420_device(dev, 2, prm, 1, qb, qsc, lastq, MB_W, MB_H, fr, pls, lsq, fsq))
        bq = 128 + 64 + 2
        wid["mpeg2_put_dct"] = {"fused": {"value": world * nbq / (msf / 1e3), "unit": "blocks/s", "ms_per_step": msf,
                                          "roofline": {"bound": "hbm", "achieved": bq * nbq / (msf / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                                       "frac": bq * nbq / (msf / 1e3) / 1e9 / peak, "bytes_per_block": bq},
                                          "api": "b200_mpv_unquant_idct_mb420_device"},
                                "two_kernels": {"value": world * nbq / (ms2 / 1e3), "unit": "blocks/s", "ms_per_step": ms2,
                                                "note": "b200_mpv_unquantize_batch_device + b200_idct_mb420_device; working copy refilled and L2 flushed before every timed call (both legs)"}}
        del qb, qwork, qsc, lastq, pls
    except Exception as ex:
        wid["mpeg2_put_dct"] = {"error": str(ex)[:160]}
    out["widening"] = wid
    return out



DUMP_SAMPLES = 1 << 22                         # bytes of the batch's rgb24 output sampled into the dump (16 MB as float32)


def dump_outputs(out_dir, OUT):
    """The headline's output batch [BATCH, H, W*3] uint8, too large to store whole (6.4 GB): frame 0 and frame BATCH-1 at 1/4 scale
    in both directions (every 4th row and pixel) and DUMP_SAMPLES bytes at fixed, seeded positions of the whole batch, as float32."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    px = OUT.view(BATCH, H4K, W4K, 3)
    for i in (0, BATCH - 1):
        np.save(os.path.join(out_dir, f"sws_rgb24_frame{i}_sub4.npy"), px[i, ::4, ::4].float().cpu().numpy())
    idx = torch.randint(0, OUT.numel(), (DUMP_SAMPLES,), generator=torch.Generator().manual_seed(1234)).sort().values
    np.save(os.path.join(out_dir, "sws_rgb24_batch_sample.npy"), OUT.view(-1)[idx.to(OUT.device)].float().cpu().numpy())
    np.save(os.path.join(out_dir, "sws_rgb24_batch_sample_index.npy"), idx.double().numpy())


def run_b200(args, rank, world, local_rank, placement=None):
    import torch
    import torch.distributed as dist
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import swscale as sw, idctdsp

    torch.cuda.set_device(local_rank)                     # local_rank here = the CUDA device index chosen for this rank (pick_devices)
    stream = torch.cuda.Stream()
    dev = fb.Device(local_rank, stream=stream.cuda_stream)
    peak, peak_src = measured_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    results = {}
    with torch.cuda.stream(stream):
        g = torch.Generator(device="cuda")
        g.manual_seed(1 + rank)
        Y = torch.randint(0, 256, (BATCH, H4K, W4K), dtype=torch.uint8, device="cuda", generator=g)
        U = torch.randint(0, 256, (BATCH, H4K // 2, W4K // 2), dtype=torch.uint8, device="cuda", generator=g)
        V = torch.randint(0, 256, (BATCH, H4K // 2, W4K // 2), dtype=torch.uint8, device="cuda", generator=g)
        OUT = torch.empty((BATCH, H4K, W4K * 3), dtype=torch.uint8, device="cuda")
    stream.synchronize()
    sstr = [W4K, W4K // 2, W4K // 2]
    sfs = [W4K * H4K, W4K * H4K // 4, W4K * H4K // 4]

    def timed_sws(flags, steps, warmup, sample_clocks, fmt=sw.AV_PIX_FMT_RGB24, out=None):
        ctx = sw.sws_getContext(dev, W4K, H4K, sw.AV_PIX_FMT_YUV420P, W4K, H4K, fmt, flags)
        out = OUT if out is None else out
        call = lambda: ctx.scale_batch_device([Y, U, V], sstr, sfs, out, W4K * ctx.bpp, W4K * H4K * ctx.bpp, BATCH)
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                call()
        barrier()
        l0 = fb.launch_count()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for a, b in evs:
                a.record(stream)
                call()
                b.record(stream)
            e1.record(stream)
        barrier()
        launches = fb.launch_count() - l0
        total_ms = reduce_max(e0.elapsed_time(e1))
        kern_ms = sum(a.elapsed_time(b) for a, b in evs) / steps
        ctx.free()
        return total_ms, kern_ms, launches

    # headline: FATE flags (full h/v pipeline semantics; same-size -> fused vertical+convert kernel)
    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms, kern_ms, launches = timed_sws(FLAGS_FATE, args.steps, args.warmup, True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, OUT)
    fps = world * BATCH * args.steps / (total_ms / 1e3)
    ach = FRAME_BYTES * BATCH / (kern_ms / 1e3) / 1e9
    roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
            "kernel": HEADLINE_KERNEL, "bytes_per_launch": FRAME_BYTES * BATCH,
            "launch_ms": kern_ms, "traffic": ncu_traffic("sws_vscale_rgb24_kernel"),
            "traffic_source": "constant from the committed ncu --set full capture (profiles/ncu_traffic.json), not measured in this run"}
    # variant: flags=bicubic only (the reference takes its unscaled LUT converter; different, cheaper arithmetic)
    t2, k2, _ = timed_sws(SWS_BICUBIC, max(3, args.steps // 2), args.warmup, False)
    fps2 = world * BATCH * max(3, args.steps // 2) / (t2 / 1e3)
    ach2 = FRAME_BYTES * BATCH / (k2 / 1e3) / 1e9
    results["variant_flags_bicubic"] = {"value": fps2, "unit": "frames/s", "roofline": {
        "bound": "hbm", "achieved": ach2, "peak": peak, "unit": "GB/s", "frac": ach2 / peak, "kernel": "sws_unscaled_kernel",
        "launch_ms": k2, "traffic": ncu_traffic("sws_unscaled_kernel")}}
    # variant: nv12 source (the decoder-output layout), FATE flags: interleaved chroma read straight by the vector kernel
    with torch.cuda.stream(stream):
        UV = torch.stack((U, V), dim=3).reshape(BATCH, H4K // 2, W4K).contiguous()
    ctxn = sw.sws_getContext(dev, W4K, H4K, sw.AV_PIX_FMT_NV12, W4K, H4K, sw.AV_PIX_FMT_RGB24, FLAGS_FATE)
    with torch.cuda.stream(stream):
        calln = lambda: ctxn.scale_batch_device([Y, UV], [W4K, W4K], [W4K * H4K, W4K * H4K // 2], OUT, W4K * 3, W4K * H4K * 3, BATCH)
        for _ in range(3):
            calln()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(5):
            calln()
        e1.record(stream)
    barrier()
    msn = reduce_max(e0.elapsed_time(e1)) / 5
    results["variant_nv12"] = {"value": world * BATCH / (msn / 1e3), "unit": "frames/s", "ms_per_step": msn, "roofline": {
        "bound": "hbm", "achieved": FRAME_BYTES * BATCH / (msn / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
        "frac": FRAME_BYTES * BATCH / (msn / 1e3) / 1e9 / peak, "kernel": "sws_vscale_rgb24_pair_kernel<RGB24, nv12>"}}
    ctxn.free()
    del UV
    # variant: the scaler proper, 4K -> 1080p with FATE flags (horizontal pass -> int16 lines -> vertical pass), yuv420p and rgb24 out
    NS = 32
    sc = {}
    for fmt, nm in ((sw.AV_PIX_FMT_YUV420P, "yuv420p"), (sw.AV_PIX_FMT_RGB24, "rgb24")):
        ctx = sw.sws_getContext(dev, W4K, H4K, sw.AV_PIX_FMT_YUV420P, 1920, 1080, fmt, FLAGS_FATE)
        with torch.cuda.stream(stream):
            if fmt == sw.AV_PIX_FMT_YUV420P:
                oy = torch.empty((NS, 1080, 1920), dtype=torch.uint8, device="cuda")
                ou = torch.empty((NS, 540, 960), dtype=torch.uint8, device="cuda")
                ov = torch.empty_like(ou)
                call = lambda: ctx.scale_batch_device_planar([Y, U, V], sstr, sfs, [oy, ou, ov], [1920, 960, 960],
                                                             [1920 * 1080, 960 * 540, 960 * 540], NS)
                obytes = 1920 * 1080 * 3 // 2
            else:
                o3 = torch.empty((NS, 1080, 1920 * 3), dtype=torch.uint8, device="cuda")
                call = lambda: ctx.scale_batch_device([Y, U, V], sstr, sfs, o3, 1920 * 3, 1920 * 1080 * 3, NS)
                obytes = 1920 * 1080 * 3
            for _ in range(3):
                call()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(5):
                call()
            e1.record(stream)
        barrier()
        msc = reduce_max(e0.elapsed_time(e1)) / 5
        ab = (FRAME_BYTES_IN + obytes) * NS
        sc[nm] = {"value": world * NS / (msc / 1e3), "unit": "frames/s", "ms_per_step": msc, "frames": NS,
                  "roofline": {"bound": "hbm", "achieved": ab / (msc / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                               "frac": ab / (msc / 1e3) / 1e9 / peak, "note": "not HBM-bound as built: fused tile kernel (horizontal pass on the tensor cores, vertical pass + writer on the CUDA cores), bound by instruction issue"}}
        ctx.free()
    results["variant_scale_4k_to_1080p"] = sc
    # variant: rgba output (SURVEY 8f row 2), FATE flags; 4 bytes per pixel out
    with torch.cuda.stream(stream):
        OUT4 = torch.empty((BATCH, H4K, W4K * 4), dtype=torch.uint8, device="cuda")
    t3, k3, _ = timed_sws(FLAGS_FATE, max(3, args.steps // 2), args.warmup, False, sw.AV_PIX_FMT_RGBA, OUT4)
    bytes4 = (W4K * H4K * 3 // 2 + W4K * H4K * 4) * BATCH
    results["variant_rgba"] = {"value": world * BATCH * max(3, args.steps // 2) / (t3 / 1e3), "unit": "frames/s", "roofline": {
        "bound": "hbm", "achieved": bytes4 / (k3 / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": bytes4 / (k3 / 1e3) / 1e9 / peak,
        "kernel": "sws_vscale_rgb24_pair_kernel<RGBA, yuv420p>", "launch_ms": k3, "bytes_per_frame": bytes4 // BATCH}}
    del OUT4

    # ---- IDCT put on the 1080p macroblock stream (configs[2]): 256 frames x 48 960 blocks per step
    nblk = MB_W * MB_H * 6 * IDCT_FRAMES
    with torch.cuda.stream(stream):
        blocks = torch.randint(-256, 257, (nblk, 64), dtype=torch.int16, device="cuda", generator=g)
        planes = [torch.zeros((IDCT_FRAMES, MB_H * 16, MB_W * 16), dtype=torch.uint8, device="cuda"),
                  torch.zeros((IDCT_FRAMES, MB_H * 8, MB_W * 8), dtype=torch.uint8, device="cuda"),
                  torch.zeros((IDCT_FRAMES, MB_H * 8, MB_W * 8), dtype=torch.uint8, device="cuda")]
    ls = [MB_W * 16, MB_W * 8, MB_W * 8]
    fs = [MB_W * 16 * MB_H * 16, MB_W * 8 * MB_H * 8, MB_W * 8 * MB_H * 8]
    idct = {}
    for kind, name, bpb in ((idctdsp.IDCT_PUT, "put", 192), (idctdsp.IDCT_ADD, "add", 256)):
        call = lambda: idctdsp.idct_mb420_device(dev, kind, blocks, MB_W, MB_H, IDCT_FRAMES, planes, ls, fs)
        with torch.cuda.stream(stream):
            for _ in range(args.warmup):
                call()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(args.steps):
                call()
            e1.record(stream)
        barrier()
        ms = reduce_max(e0.elapsed_time(e1))
        bps = world * nblk * args.steps / (ms / 1e3)
        a = bpb * nblk / (ms / args.steps / 1e3) / 1e9
        idct[name] = {"value": bps, "unit": "blocks/s", "ms_per_step": ms / args.steps,
                      "roofline": {"bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
                                   "kernel": f"idct_mb420_kernel<{name}>", "bytes_per_block": bpb,
                                   "traffic": ncu_traffic(f"idct8x8_{name}")}}
    # e2e: coefficient blocks in pinned host memory -> b200_idct_mb420_host -> reconstructed planes back in host memory
    EF = 64
    for kind, name in ((idctdsp.IDCT_PUT, "put"), (idctdsp.IDCT_ADD, "add")):
        try:
            per = MB_W * MB_H * 6
            hblk = pinned_like(blocks[:per * EF].cpu())
            hpl = [pinned_like(p[:EF].cpu()) for p in planes]
            hp0 = [h.clone() for h in hpl] if kind == idctdsp.IDCT_ADD else None
            call = lambda: idctdsp.idct_mb420_host(dev, kind, hblk.data_ptr(), MB_W, MB_H, EF, [h.data_ptr() for h in hpl], ls, fs)
            dt = host_timed(call, 3, barrier, reduce_max)
            if hp0 is not None:                            # add accumulates: compare one fresh pass
                for h, h0 in zip(hpl, hp0):
                    h.copy_(h0)
                call()
            with torch.cuda.stream(stream):
                chk = [(h0 if hp0 is not None else h).cuda() for h, h0 in zip(hpl, hp0 or hpl)]
                idctdsp.idct_mb420_device(dev, kind, blocks, MB_W, MB_H, EF, chk, ls, fs)
            stream.synchronize()
            pbytes = sum(fs) * EF
            idct[name]["e2e"] = {"value": world * per * EF / dt, "unit": "blocks/s", "h2d_bytes_per_step": per * EF * 128 + (pbytes if kind == idctdsp.IDCT_ADD else 0),
                                 "d2h_bytes_per_step": pbytes, "api": "b200_idct_mb420_host", "frames": EF,
                                 "matches_device_path": all(bool(torch.equal(c.cpu(), h)) for c, h in zip(chk, hpl))}
            del hblk, hpl, hp0, chk
        except Exception as ex:
            idct[name]["e2e"] = {"value": None, "error": str(ex)[:160]}
    del blocks, planes
    results.update(extra_paths(args, dev, stream, g, world, barrier, reduce_max, peak, local_rank))
    clocks = sampler.stop()

    # ---- mux boundary (N > 1 only): every rank's finished rgb24 frames are collected on rank 0 over NCCL / NVLink (SURVEY 8e:
    # throughput both without and with that gather).  The collect of batch k runs on a side stream while batch k+1 converts.
    mux = None
    if world > 1:
        from ffmpeg_b200.sharding import MuxGather
        ctx = sw.sws_getContext(dev, W4K, H4K, sw.AV_PIX_FMT_YUV420P, W4K, H4K, sw.AV_PIX_FMT_RGB24, FLAGS_FATE)
        with torch.cuda.stream(stream):
            OUT2 = torch.empty_like(OUT)
        outs = [OUT, OUT2]
        mg = MuxGather(BATCH, (H4K, W4K * 3), torch.uint8, torch.device("cuda", local_rank), dst=0)
        gsteps = max(2, min(args.steps, 4))

        def one(k):
            o = outs[k & 1]
            with torch.cuda.stream(stream):
                mg.wait(stream)                             # the buffer being overwritten two batches later was sent one batch ago
                ctx.scale_batch_device([Y, U, V], sstr, sfs, o, W4K * 3, W4K * H4K * 3, BATCH)
                ev = torch.cuda.Event()
                ev.record(stream)
            mg.start(o, after=ev)
        one(0)                                              # warm-up: communicator set-up
        mg.wait(stream)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
        for k in range(gsteps):
            one(k + 1)
        with torch.cuda.stream(stream):
            mg.wait(stream)
            e1.record(stream)
        barrier()
        gms = reduce_max(e0.elapsed_time(e1)) / gsteps
        ok = None
        if rank == 0:                                       # spot check: rank 0's own slot equals its last batch
            ok = bool(torch.equal(mg.out[BATCH - 1], outs[gsteps & 1][BATCH - 1]))
        mux = {"value_with_gather": world * BATCH / (gms / 1e3), "unit": "frames/s", "ms_per_step": gms, "steps": gsteps,
               "GBps_into_rank0": (world - 1) * BATCH * FRAME_BYTES_OUT / (gms / 1e3) / 1e9, "frames_per_rank": BATCH,
               "own_slot_matches": ok,
               "note": "every rank's 256 rgb24 frames per step land on rank 0 (NCCL send/recv on a side stream, overlapped with the next "
                       "batch); bounded by rank 0's NVLink ingest (measured peer copy 770 GB/s = 30.9 k 4K rgb24 frames/s), not by the kernels"}
        ctx.free()
        del mg, OUT2, outs

    # ---- e2e: the C-ABI host entry point with pinned host buffers (H2D + kernels + D2H inside the timed region)
    e2e = None
    try:
        with near_gpu(local_rank) as ng:                 # host buffers on the GPU's NUMA node (numactl-style placement)
            hY = torch.empty((BATCH, H4K, W4K), dtype=torch.uint8).pin_memory()
            hU = torch.empty((BATCH, H4K // 2, W4K // 2), dtype=torch.uint8).pin_memory()
            hV = torch.empty((BATCH, H4K // 2, W4K // 2), dtype=torch.uint8).pin_memory()
            hO = torch.empty((BATCH, H4K, W4K * 3), dtype=torch.uint8).pin_memory()
            hO.zero_()                                   # first touch here
        hY.copy_(Y.cpu()); hU.copy_(U.cpu()); hV.copy_(V.cpu())
        ctx = sw.sws_getContext(dev, W4K, H4K, sw.AV_PIX_FMT_YUV420P, W4K, H4K, sw.AV_PIX_FMT_RGB24, FLAGS_FATE)
        call = lambda: ctx.scale_batch_host([hY.data_ptr(), hU.data_ptr(), hV.data_ptr()], sstr, sfs, hO.data_ptr(),
                                            W4K * 3, W4K * H4K * 3, BATCH)
        call()
        e2e_steps = max(2, min(args.steps, 5))
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            call()
        torch.cuda.synchronize()
        dt = reduce_max(time.perf_counter() - t0)
        # spot check: e2e output equals the device-resident output of the same frames
        with torch.cuda.stream(stream):
            ctx.scale_batch_device([Y, U, V], sstr, sfs, OUT, W4K * 3, W4K * H4K * 3, BATCH)
        stream.synchronize()
        same = bool(torch.equal(OUT[BATCH - 1].cpu(), hO[BATCH - 1])) and bool(torch.equal(OUT[0].cpu(), hO[0]))
        ctx.free()
        e2e = {"value": world * BATCH * e2e_steps / dt, "unit": "frames/s", "h2d_bytes_per_step": FRAME_BYTES_IN * BATCH,
               "d2h_bytes_per_step": FRAME_BYTES_OUT * BATCH, "steps": e2e_steps, "matches_device_path": same,
               "api": "b200_sws_scale_batch_host (C ABI, pinned host buffers)",
               "host_buffers": "allocated on the GPU's NUMA node" if ng.cpus else "default placement"}
        del hY, hU, hV, hO
    except Exception as ex:                       # pinned allocation can fail on small hosts: report, do not fake
        e2e = {"value": None, "unit": "frames/s", "error": str(ex)[:200]}

    cpu = None
    cpu_all = {}
    if rank == 0 and world == 1:
        cpu_all = cpu_baselines_all()
        cpu = cpu_all.pop("sws")
        idct["put"]["cpu_baseline"] = cpu_all["idct_put"]
        idct["add"]["cpu_baseline"] = cpu_all["idct_add"]
        results["h264qpel"]["cpu_baseline"] = cpu_all["h264qpel"]
        results["me_esa"]["cpu_baseline"] = cpu_all["me_esa"]
        for k in ("fft1024", "fft2048", "imdct1024", "imdct2048"):
            results["tx"][k]["cpu_baseline"] = cpu_all[k]

    # the driver's record keeps the contract keys whole and only the names of the others: the five BASELINE configs are summarised
    # inside `roofline`, `cpu_baseline` and `e2e` (full entries stay under their own keys)
    def brief(d, keys):
        return {k: d[k] for k in keys if d and k in d}
    per_cfg = {"idct_put": idct["put"], "idct_add": idct["add"], "h264qpel": results["h264qpel"], "me_esa": results["me_esa"],
               "fft1024": results["tx"]["fft1024"], "fft2048": results["tx"]["fft2048"],
               "imdct1024": results["tx"]["imdct1024"], "imdct2048": results["tx"]["imdct2048"]}
    roof["others"] = {k: dict(brief(v["roofline"], ("bound", "achieved", "peak", "unit", "frac")), value=v["value"], value_unit=v["unit"])
                      for k, v in per_cfg.items()}
    if e2e is not None:
        e2e["others"] = {k: brief(v.get("e2e"), ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "matches_device_path", "error"))
                         for k, v in per_cfg.items()}
    if cpu is not None:
        cpu["others"] = {k: {"value": v["value"], "unit": v["unit"], "cores": v["cores"], "single_thread": v["single_thread"]["value"]}
                         for k, v in cpu_all.items()}

    if rank == 0:
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"swscale {W4K}x{H4K} yuv420p->rgb24 flags=bicubic+accurate_rnd+bitexact, batch={BATCH} frames per GPU",
                       "l2": "inputs (3.2 GB) and outputs (6.4 GB) per step exceed L2 (126 MB): no flush needed",
                       "sharding": "frames of the batch are independent; each rank converts its own batch, no collective on the data path"},
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "value_with_gather": mux["value_with_gather"] if mux else None, "placement": placement,
            "idct": idct, "mux_gather": mux, **results,
        }
        emit_line(line)
    dev.close()


def gpu_inventory():
    """[(cuda index, numa node, used MiB or None)] of every GPU this process may index, without creating a CUDA context."""
    import torch
    inv = []
    try:
        import pynvml
        pynvml.nvmlInit()
    except Exception:
        pynvml = None
    for i in range(torch.cuda.device_count()):
        pr = torch.cuda.get_device_properties(i)
        bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node, used = -1, None
        try:
            node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        except Exception:
            pass
        if pynvml is not None:
            try:
                h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
                used = pynvml.nvmlDeviceGetMemoryInfo(h).used // (1 << 20)
            except Exception:
                pass
        inv.append((i, node, used))
    return inv


def pick_devices(world):
    """Rank -> CUDA device for this node.  When more GPUs are visible than ranks (an 8-GPU box running N = 2 or 4), spread the ranks
    over the host's NUMA nodes so that the end-to-end legs use every socket's memory and PCIe root (ffmpeg_b200.sharding.spread_over_numa);
    GPUs that already hold memory (another tenant) are left alone.  Otherwise rank r uses device r.  B200_BENCH_SPREAD=0 disables it."""
    import torch
    from ffmpeg_b200.sharding import spread_over_numa
    ident = list(range(world))
    if os.environ.get("B200_BENCH_SPREAD", "1") == "0" or torch.cuda.device_count() <= world:
        return ident, "rank r -> device r"
    try:
        inv = gpu_inventory()
        free = [(i, node) for i, node, used in inv if used is not None and used < 2048]
        if len(free) < world or len({n for _, n in free}) < 2:
            return ident, "rank r -> device r (no second NUMA node with idle GPUs)"
        m = spread_over_numa(free, world)
        return m, "ranks spread over NUMA nodes: " + ", ".join(f"r{r}->gpu{d}(node {dict(free)[d]})" for r, d in enumerate(m))
    except Exception as ex:
        return ident, f"rank r -> device r (inventory failed: {str(ex)[:80]})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's last timed step's output (sampled) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the communicator comes up; stdout must carry the JSON line only, so
        # everything before that line goes to stderr (emit_line() switches back)
        global _STDOUT_FD
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)
        # rank 0 decides the placement before any CUDA context exists and tells the others over gloo; NCCL then comes up on the
        # chosen devices (one process per GPU, single node)
        dist.init_process_group("cpu:gloo,cuda:nccl")
        box = [pick_devices(world) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        mapping, placement = box[0]
        local_rank = int(mapping[rank])
        torch.cuda.set_device(local_rank)
    else:
        placement = "single GPU"
    try:
        run_b200(args, rank, world, local_rank, placement)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
