#!/usr/bin/env python
"""bench.py -- frames/s of the 832x624 composite modulate + demodulate hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # product (CUDA) arm
    python bench.py --impl reference --gpus N ...            # reference C on the host cores

A "step" is one pass of the hot path over one batch: every monitor of the batch gets one
crt_modulate + crt_demodulate pair (= one field = one "frame" of the metric, SURVEY.md 8d).
Workload (BASELINE.json configs[1]): NTSC, 832x624 BGRA in -> 832x624 BGRA out, interlaced (field
alternates every step), full colour, noise 0, blend 1, scanlines 1 -- the CLI's settings
(crt_main.c:221-255).  Synthetic seeded-random images, one distinct image per monitor.

What the one JSON line carries
  value       frames/s, whole job, images resident in HBM, CUDA events around exactly K steps, max over ranks
  sustained   the same loop kept running for >= 1 s with the clock / power sampler on (an issue-bound integer kernel
              runs at the SM clock: a 10 ms burst says nothing about seconds of load)
  e2e         the same metric through the crtx_frames_host C-ABI call with page-locked HOST buffers: every step moves
              its source rows host -> device and the rows it decoded device -> host inside the timed region
  roofline    the line kernel (crt_core.c:511-664) charged with the bytes IT moves (windows, blend read, row writes)
              over its mean CUDA-event launch duration, against MEASURED_PEAKS.json hbm_gbs; `demodulate` inside it
              is the whole crt_demodulate (SURVEY 8d's 2 553 512 B per field) over sync + line kernels
  cpu_baseline  the reference C code (oracle/_ref, else the oracle port), 1 pinned thread, bounded sample
  N > 1       allgather (north_star's exchange: all_gather of the decoded frames over NVLink, overlapped with the next
              half-batch on a second stream), gather_to_root, and config4 (BASELINE configs[3]: one video sequence,
              frame ranges per rank, seam exchange, bit-checked against the sequential loop on rank 0)
  dropin      informational (SURVEY 8d "drop-in fps"): crt_modulate + crt_demodulate of the reference's own interface
              on host buffers, one struct CRT, synchronous, wall clock; measured in a child process
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading
import time

# rank 0 prints exactly one line on stdout: keep NCCL's version banner (NCCL_DEBUG=VERSION) off it
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W_IN, H_IN, W_OUT, H_OUT = 832, 624, 832, 624
VARIANT = "ntsc"
METRIC = "frames/sec (832x624 modulate+demodulate)"
WORKLOAD = "NTSC 832x624 BGRA -> 832x624 BGRA, interlaced, colour, noise 0, blend 1, scanlines 1"  # BASELINE configs[1]


def workload_name():
    """the same string in both arms (the driver compares them)"""
    if VARIANT == "ntsc":
        return WORKLOAD
    return "%s -> 832x624 BGRA, noise %d, blend 1, scanlines 1 (informational run of another BASELINE config)" % (
        VARIANT, 24 if VARIANT == "vhs" else 0)


def rank_info():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def field_rows(field, scanlines=1, outh=H_OUT, lines=240):
    """(rows computed, rows written) by one crt_demodulate of the given field parity (crt_core.c:404-407, 428-432, 662-664)"""
    ratio = (((outh << 16) // lines) + 32768) >> 16
    off = (field & 1) * (ratio // 2)
    computed = written = 0
    for k in range(lines):
        beg = k * outh // lines + off
        end = (k + 1) * outh // lines + off
        if beg >= outh:
            continue
        end = min(end, outh)
        computed += 1
        written += max(1, end - scanlines - beg)
    return computed, written


def demod_bytes(field, blend=1, scanlines=1, outw=W_OUT, outh=H_OUT, bpp=4, lines=240, input_size=238420):
    """Algorithmic bytes of one crt_demodulate (SURVEY.md 8d): read analog, write inp, blend-read the
    240 computed rows, write computed + duplicated rows (crt_core.c:428-432, 584-608, 662-664)."""
    computed, written = field_rows(field, scanlines, outh, lines)
    return 2 * input_size + bpp * outw * (computed * blend + written)


def lines_bytes(field, av_len, blend=1, scanlines=1, outw=W_OUT, outh=H_OUT, bpp=4, lines=240):
    """Algorithmic bytes of the LINE KERNEL alone: each decoded line's AV_LEN-sample window of inp[] (crt_core.c:511,
    534-543), the blend read of its computed row and the rows it writes.  (analog -> inp belongs to the sync kernel's
    fused noise pass and is not charged here.)"""
    computed, written = field_rows(field, scanlines, outh, lines)
    return computed * av_len + bpp * outw * (computed * blend + written)


def source_rows_read(h=H_IN, desth=236):
    """distinct source rows one crt_modulate reads (crt_ntsc.c:258-266): one per picture line"""
    return desth if h >= desth else h


def library_source_hash():
    """sha256 over the CUDA sources of the product: ties a committed ncu capture (profiles/*traffic*.json) to a build"""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "ntsc-crt_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled through NVML while a timed region runs."""

    def __init__(self, index, period=0.001):
        super().__init__(daemon=True)
        self.index = index
        self.period = period
        self.samples = []
        self.power = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self._halt.wait(self.period)

    def finish(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        p = sorted(self.power)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s),
                "power_w": (round(p[len(p) // 2], 1) if p else None)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(index):
    """Pin this process to the cores of the NUMA node its GPU hangs off, BEFORE any page-locked allocation: the
    buffers the e2e path streams over PCIe then live in that node's memory (first touch), and N ranks stop sharing
    one node's memory controllers (r1: e2e scaled 0.56 at 8 GPUs with unbound ranks).  Returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return {"bound": False, "why": "numa_node -1 (single node or not reported)"}
        cpus = _parse_cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read())
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use:
            return {"bound": False, "why": "no allowed cpu on node %d" % node}
        os.sched_setaffinity(0, use)
        return {"bound": True, "node": node, "cpus": len(use), "pci": bus}
    except Exception as e:  # informational: never take the bench down
        return {"bound": False, "why": "%s: %s" % (type(e).__name__, e)}


def usable_cores():
    """host threads this process may really use: the affinity mask capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            t = open(path).read().split()
            if path.endswith("cpu.max"):
                if t[0] != "max":
                    quota = float(t[0]) / float(t[1])
            else:
                q = float(t[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    if quota is not None:
        n = max(1, min(n, int(quota)))
    return n, quota


# --------------------------------------------------------------------------------------------
# reference / cpu_baseline arm
# --------------------------------------------------------------------------------------------

def _cpu_engine():
    import support as S
    if S.have_ref(VARIANT):
        return "reference", (lambda: S.RefEngine(VARIANT, W_OUT, H_OUT))
    return "port", (lambda: S.OracleEngine(VARIANT, W_OUT, H_OUT))


_WORKER = {}


def _cpu_init(seed=1):
    """Per-process set-up (outside any timed region): one reference instance, one source image."""
    import support as S
    kind, make = _cpu_engine()
    eng = make()
    eng.set(blend=1, scanlines=1)
    _WORKER["eng"] = eng
    if VARIANT not in ("nes", "nes_p0", "nes_p1"):
        _WORKER["img"] = S.rand_image(W_IN, H_IN, seed=seed + os.getpid() % 97)
    else:
        _WORKER["img"] = S.nes_image(W_IN, H_IN, seed=seed + os.getpid() % 97)
    _WORKER["f"] = 0


def _cpu_pair(eng, img, f):
    from ntsc_crt_b200 import layout
    if VARIANT.startswith("nesrgb"):
        eng.modulate(img, format=layout.PIX_BGRA, dot_crawl_offset=f & 1, hue=0)
    elif not VARIANT.startswith("nes"):
        eng.modulate(img, format=layout.PIX_BGRA, as_color=1, field=f & 1, frame=(f >> 1) & 1)
    else:
        eng.modulate(img, dot_crawl_offset=f & 1, hue=0)


def _cpu_worker(fields):
    """Run `fields` modulate+demodulate pairs of the bench workload on this host thread."""
    if "eng" not in _WORKER:
        _cpu_init()
    eng, img = _WORKER["eng"], _WORKER["img"]
    t0 = time.perf_counter()
    for _ in range(fields):
        f = _WORKER["f"]
        _cpu_pair(eng, img, f)
        eng.demodulate(24 if VARIANT == "vhs" else 0)
        _WORKER["f"] = f + 1
    return time.perf_counter() - t0


def cpu_baseline_single(seconds=8.0):
    """Reference C path, ONE thread pinned to one core, on a bounded sample of the same workload (SURVEY 8d):
    20 warm-up fields, then at least 200 fields; crt_modulate and crt_demodulate are also timed separately
    (medians, file I/O does not exist here)."""
    import statistics
    import pkgload
    pkgload.load()
    kind, _ = _cpu_engine()
    pinned = None
    try:  # like `taskset -c`: keep the scheduler from migrating the measurement
        allowed = sorted(os.sched_getaffinity(0))
        pinned = allowed[len(allowed) // 2]
        os.sched_setaffinity(0, {pinned})
    except (AttributeError, OSError):
        allowed = None
    try:
        _cpu_worker(20)  # warm-up
        eng, img = _WORKER["eng"], _WORKER["img"]
        t_mod, t_dem = [], []
        fields, spent = 0, 0.0
        while spent < seconds or fields < min(200, max(20, int(25 * seconds))):
            f = _WORKER["f"]
            t0 = time.perf_counter()
            _cpu_pair(eng, img, f)
            t1 = time.perf_counter()
            eng.demodulate(24 if VARIANT == "vhs" else 0)
            t2 = time.perf_counter()
            _WORKER["f"] = f + 1
            t_mod.append(t1 - t0)
            t_dem.append(t2 - t1)
            spent += t2 - t0
            fields += 1
    finally:
        if allowed is not None:
            os.sched_setaffinity(0, set(allowed))
    return {"value": fields / spent, "unit": "frames/s", "cores": 1, "kind": kind,
            "sample": "%d fields of the bench workload (%s), 1 thread%s, %.1f s"
                      % (fields, workload_name(), " pinned to cpu %d" % pinned if pinned is not None else "", spent),
            "modulate_ms_median": 1e3 * statistics.median(t_mod), "demodulate_ms_median": 1e3 * statistics.median(t_dem),
            "host_cores": os.cpu_count()}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation on all the host cores it can use
    (one single-threaded instance per core: the library keeps its filter state in file statics,
    crt_core.c:158-164, so it is process- not thread-parallel).  The pool is sized from what this process may really
    run on -- affinity mask capped by the cgroup quota, not os.cpu_count() -- and the line says how many cores' worth
    of the single-thread rate the pool delivered, so that two boxes can be compared."""
    import multiprocessing as mp
    import pkgload
    pkgload.load()
    rank, local_rank, world = rank_info()
    if rank != 0:
        return
    kind, _ = _cpu_engine()
    cores, quota = usable_cores()
    single = cpu_baseline_single(2.0)  # same box, one pinned thread: the unit `effective_cores` is counted in
    _WORKER.clear()
    fields_per_worker = 16
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init) as pool:
        jobs = [fields_per_worker] * cores
        for _ in range(max(1, args.warmup)):
            pool.map(_cpu_worker, jobs, chunksize=1)
        t0 = time.perf_counter()
        busy = 0.0
        for _ in range(args.steps):
            busy += sum(pool.map(_cpu_worker, jobs, chunksize=1))
        dt = time.perf_counter() - t0
    frames = args.steps * cores * fields_per_worker
    value = frames / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32",
        "data": "synthetic",
        "config": {"workload": workload_name(), "batch_per_step": cores * fields_per_worker, "host_processes": cores},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind,
                         "sample": "%d processes x %d fields per step, %d steps" % (cores, fields_per_worker, args.steps),
                         "per_process_fps": value / cores,
                         # a process's own time inside its fields vs the wall clock: < 1 means the pool waited for cores
                         "busy_fraction": busy / (dt * cores),
                         "single_thread_fps": single["value"],
                         "effective_cores": value / single["value"],
                         "host_cores": os.cpu_count(), "affinity_cores": len(os.sched_getaffinity(0)),
                         "cgroup_cpu_quota": quota},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# product arm
# --------------------------------------------------------------------------------------------

def dropin_fps(seconds=2.0):
    """SURVEY 8d "drop-in fps": the reference's own seven-function interface on HOST buffers, exactly what the
    unmodified drivers call -- crt_modulate + crt_demodulate on one struct CRT, synchronous, strict coherence.
    Wall clock around the calls, like a caller sees it.  Informational: it never touches the contract's `value` /
    `e2e`, and a failure here is reported in the key instead of costing the line."""
    try:
        import support as S
        from ntsc_crt_b200 import layout
        eng = S.ProductEngine(VARIANT, W_OUT, H_OUT)
        eng.set(blend=1, scanlines=1)
        nes = VARIANT in ("nes", "nes_p0", "nes_p1")
        img = S.nes_image(W_IN, H_IN, seed=7) if nes else S.rand_image(W_IN, H_IN, seed=7)

        def pair(f):
            if nes:
                eng.modulate(img, dot_crawl_offset=f & 1, hue=0)
            elif VARIANT.startswith("nesrgb"):
                eng.modulate(img, format=layout.PIX_BGRA, dot_crawl_offset=f & 1, hue=0)
            else:
                eng.modulate(img, format=layout.PIX_BGRA, as_color=1, field=f & 1, frame=(f >> 1) & 1)
            eng.demodulate(24 if VARIANT == "vhs" else 0)
        for f in range(4):
            pair(f)
        n, t0 = 0, time.perf_counter()
        while True:
            pair(n)
            n += 1
            dt = time.perf_counter() - t0
            if (dt >= seconds and n >= 8) or n >= 20000:
                break
        return {"value": n / dt, "unit": "frames/s", "pairs": n, "wall_s": dt,
                "api": "crt_modulate + crt_demodulate (crt_core.h:100-139) on host buffers, one struct CRT, synchronous, strict coherence"}
    except Exception as e:  # informational key: never take the bench line down
        return {"value": None, "error": "%s: %s" % (type(e).__name__, e)}


def dropin_isolated(seconds=2.0):
    """dropin_fps in a child process (`bench.py --impl dropin`): the drop-in library abort()s when CUDA fails (its
    signatures have no error channel), and an informational figure must not be able to take this process with it."""
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "dropin", "--variant", VARIANT,
                            "--dropin-seconds", str(seconds)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=180)
        if r.returncode != 0:
            return {"value": None, "error": "child exit %d: %s" % (r.returncode, r.stderr.strip()[-200:])}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {"value": None, "error": "%s: %s" % (type(e).__name__, e)}


def config4_block(args, dev, rank, world, noise=0):
    """BASELINE configs[3] (extra/video_convert.c:244-277): ONE image sequence of 640x480 BGRA frames through one struct
    CRT -- blend 0, scanlines 1, the field toggling every frame -- cut into contiguous frame ranges, one per rank, each
    range into time-parallel segments with a two-frame halo; the seams between ranks are verified by exchanging the
    sync state and the last image (all_gather over NCCL) and repaired where the speculation failed
    (ntsc_crt_b200/video.py).  Strong scaling: the sequence length is fixed.  The result is compared BIT FOR BIT with
    the sequential loop (one monitor, frame after frame) that rank 0 runs over the whole sequence."""
    import torch
    import torch.distributed as dist
    from ntsc_crt_b200 import capi, layout, sharding, video
    total = args.config4_frames
    w, h, ow, oh = 640, 480, 640, 480
    lo, hi = sharding.shard_range(total, rank, world)

    def make_frames(a, b):
        """frames [a, b) of the synthetic sequence: bars moving one pixel per frame + seeded noise, so every frame
        differs; a pure function of the frame index (any rank can make any frame)"""
        out = torch.empty(b - a, h, w, 4, dtype=torch.uint8, device=dev)
        xs = torch.arange(w, device=dev)
        for i, f in enumerate(range(a, b)):
            g = torch.Generator(device=dev).manual_seed(9000 + f)
            bars = (((xs + f) // 40) % 8).to(torch.int32)
            base = torch.stack([(bars & 1) * 191, ((bars >> 1) & 1) * 191, ((bars >> 2) & 1) * 191, torch.full_like(bars, 255)], dim=-1)
            nz = torch.randint(0, 64, (h, w, 4), dtype=torch.int32, device=dev, generator=g)
            out[i] = (base[None, :, :] + nz).clamp_(0, 255).to(torch.uint8)
        return out

    frames = make_frames(lo, hi)
    # time-parallel segments per rank: ~8 frames each (a two-frame halo on top), at most one line-kernel wave (296 monitors)
    segs = args.config4_segments if args.config4_segments > 0 else max(16, min(296, (hi - lo) // 8))
    segs = max(1, min(segs, hi - lo))
    conv = video.VideoConverter("ntsc", ow, oh, noise=noise, scanlines=1, segments=segs)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    # warm-up: the same call once before the timed one, so that the allocations of the timed call (6 GB of decoded images
    # at N = 1, the segments' monitors, their images) come out of the caching allocator's pool instead of cudaMalloc
    warm = conv.convert(frames, first_frame=lo)
    del warm
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(torch.cuda.current_stream(dev))
    outs = conv.convert(frames, first_frame=lo)
    e1.record(torch.cuda.current_stream(dev))
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - t0
    ms = max(e0.elapsed_time(e1), 1e3 * wall)  # convert() synchronises to read sync states: the wall clock is the honest one
    ms = sharding.max_over_ranks([ms], device=dev)[0]
    recomputed = int(sharding.max_over_ranks([float(conv.recomputed)], device=dev)[0])

    # ---- the check: rank 0 runs the sequential loop over the WHOLE sequence and compares every rank's images with it
    mism = 0
    checked = 0
    seq_s = None
    counts = [sharding.shard_range(total, r, world) for r in range(world)]
    if rank == 0:
        t1 = time.perf_counter()
        b = capi.Batch("ntsc", 1)
        work = torch.zeros(oh, ow, 4, dtype=torch.uint8, device=dev)
        b.set_monitor(0, work, fmt=layout.PIX_BGRA, noise=noise, blend=0, scanlines=1)
        b.commit_monitors()
        seq = torch.empty(total, oh, ow, 4, dtype=torch.uint8, device=dev)
        chunk = 256
        for a in range(0, total, chunk):
            fr = frames[a:min(a + chunk, hi)] if (a + chunk <= hi and a >= lo) else make_frames(a, min(a + chunk, total))
            for i in range(fr.shape[0]):
                field, frame = video.frame_parity(a + i)
                b.set_source(0, fr[i], format=layout.PIX_BGRA, as_color=1, field=field, frame=frame)
                b.modulate()
                b.demodulate()
                seq[a + i].copy_(work)
        torch.cuda.synchronize(dev)
        seq_s = time.perf_counter() - t1
        b.close()
    for r in range(world):  # rank r's images travel to rank 0 (one broadcast per rank: plain NCCL, no gather list)
        a, e = counts[r]
        if world > 1:
            buf = outs if rank == r else torch.empty(e - a, oh, ow, 4, dtype=torch.uint8, device=dev)
            if r != 0:
                dist.broadcast(buf, src=r)
        else:
            buf = outs
        if rank == 0:
            same = (buf == seq[a:e]).flatten(1).all(dim=1)
            mism += int((~same).sum().item())
            checked += e - a
    flag = sharding.max_over_ranks([float(mism)], device=dev)[0]
    return {"workload": "NTSC video sequence, %d frames 640x480 BGRA -> 640x480 BGRA, blend 0, scanlines 1, noise %d, interlaced "
                        "(video_convert.c:244-277)" % (total, noise),
            "value": total / (ms / 1e3), "unit": "frames/s", "scaling": "strong", "frames": total, "ms": ms,
            "frames_per_rank": hi - lo, "segments_per_rank": segs, "halo_frames": 2,
            "segments_recomputed_max": recomputed,
            "exchange": "all_gather of 2 input frames + sync state + last image per rank (seam verification), NCCL" if world > 1 else "none (one rank)",
            "bit_identical_to_sequential_loop": bool(flag == 0), "frames_checked": checked if rank == 0 else None,
            "sequential_loop_s_rank0": seq_s}


DUMP_IMAGES = 6  # decoded images written in full by --dump-outputs (6 x 832x624x4 float32 = 50 MB)


def dump_outputs(where, out):
    """--dump-outputs (rank 0): what the last timed step left in the monitors' output images, as .npy files (under
    64 MB in all): `out` = DUMP_IMAGES whole images (n, H, W, BGRA; float32) of monitors drawn with a fixed seed,
    `out_index` = which monitors they are (float32), `out_sums` = the per-channel sum of every monitor's image (B, 4;
    float64, exact)."""
    import numpy as np
    import torch
    os.makedirs(where, exist_ok=True)
    pick = np.sort(np.random.default_rng(0).choice(out.shape[0], size=min(DUMP_IMAGES, out.shape[0]), replace=False))
    idx = torch.from_numpy(pick).to(out.device)
    np.save(os.path.join(where, "out.npy"), out.index_select(0, idx).float().cpu().numpy())
    np.save(os.path.join(where, "out_index.npy"), pick.astype(np.float32))
    np.save(os.path.join(where, "out_sums.npy"), out.sum(dim=(1, 2), dtype=torch.float64).cpu().numpy())


def run_product(args):
    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist
    import pkgload
    pkgload.load()
    from ntsc_crt_b200 import capi, layout, sharding

    rank, local_rank, world = rank_info()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    numa = bind_to_gpu_numa_node(physical_gpu_index(local_rank)) if not args.no_numa else {"bound": False, "why": "--no-numa"}
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)
    # inputs: one distinct image per monitor, BGRA; far larger than L2 in total (see config)
    nes = VARIANT in ("nes", "nes_p0", "nes_p1")
    noise = 24 if VARIANT == "vhs" else 0  # BASELINE configs[4]: VHS at noise 24
    if nes:
        src = torch.randint(0, 512, (B, H_IN, W_IN), dtype=torch.int16, generator=gen).to(dev)
    else:
        src = torch.randint(0, 256, (B, H_IN, W_IN, 4), dtype=torch.uint8, generator=gen).to(dev)
    out = torch.zeros(B, H_OUT, W_OUT, 4, dtype=torch.uint8, device=dev)
    batch = capi.Batch(VARIANT, B)
    batch.set_option("timing", 1)
    for kv in args.set:
        name, val = kv.split("=")
        batch.set_option(name, int(val))
    for i in range(B):
        batch.set_monitor(i, out[i], fmt=layout.PIX_BGRA, noise=noise, blend=1, scanlines=1)
    batch.commit_monitors()
    # two prebuilt source tables, even / odd field (crt_main.c:245-253 toggles field each pass)
    tables = []
    for field in (0, 1):
        t = (capi.Source * B)()
        for i in range(B):
            s = t[i]
            s.data = src[i].data_ptr()
            s.format, s.w, s.h = layout.PIX_BGRA, W_IN, H_IN
            s.raw, s.as_color, s.field, s.frame = 0, 1, field, 0
            s.dot_crawl_offset, s.reinit = field, 0
        tables.append(t)
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream

    def sub_table(t, first):
        return C.cast(C.byref(t, first * C.sizeof(capi.Source)), C.POINTER(capi.Source))

    def step(k, first=0, count=None, on=None):
        count = B - first if count is None else count
        on = sp if on is None else on
        batch._check(batch.lib.crtx_modulate(batch._ctx, first, count, sub_table(tables[k & 1], first), on))
        batch._check(batch.lib.crtx_demodulate(batch._ctx, first, count, on))

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    if nes or VARIANT.startswith("nesrgb"):  # first call of a NES stream writes the sync template (crt_nes.c:118-121)
        t0 = (capi.Source * B)()
        C.memmove(t0, tables[0], C.sizeof(t0))
        for i in range(B):
            t0[i].reinit = 1
        batch._check(batch.lib.crtx_modulate(batch._ctx, 0, B, t0, sp))
    for k in range(args.warmup):
        step(k)
    barrier()
    batch.timing()  # drop warm-up timings
    # ---- the timed region: exactly K steps, nothing else on the stream (the library's per-kernel event pairs are a
    # diagnostic of ours: they are switched on for a second pass of K steps below, which feeds `roofline` and
    # `kernel_ms_per_step` and is NOT what `value` is computed from)
    batch.set_option("timing", 0)
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    launches0 = batch.launches
    lines2_0 = batch.lines2_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for k in range(args.steps):
        step(args.warmup + k)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.finish()
    if args.dump_outputs and rank == 0:  # the last timed step's images, before the passes below overwrite them
        dump_outputs(args.dump_outputs, out)
    launches = batch.launches - launches0
    took_lines2 = batch.lines2_launches - lines2_0
    batch.set_option("timing", 1)
    ki0, ki1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ki0.record(stream)
    for k in range(args.steps):
        step(args.warmup + k)
    ki1.record(stream)
    barrier()
    ms_instrumented = ki0.elapsed_time(ki1)
    ktimes = batch.timing()

    # ---------------- sustained: the same step loop for >= args.sustained_seconds, clocks and power sampled under it
    sustained = None
    if args.sustained_seconds > 0:
        per_step = max(ms / max(1, args.steps), 1e-3)
        n_sus = int(min(200000, max(args.steps, (1e3 * args.sustained_seconds) / per_step * 1.05 + 1)))
        batch.set_option("timing", 0)  # (no per-kernel event pairs in a loop this long)
        s_sampler = ClockSampler(physical_gpu_index(local_rank), period=0.005)
        barrier()
        s_sampler.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for k in range(n_sus):
            step(k)
        s1.record(stream)
        barrier()
        s_ms = s0.elapsed_time(s1)
        s_clk = s_sampler.finish()
        batch.set_option("timing", 1)
        if world > 1:
            s_ms = sharding.max_over_ranks([s_ms], device=dev)[0]
        # (the batch is left with timing on afterwards, as the e2e loop expects)
        sustained = {"frames_per_s": world * B * n_sus / (s_ms / 1e3), "unit": "frames/s", "steps": n_sus, "seconds": s_ms / 1e3,
                     "ms_per_step": s_ms / n_sus, "sm_mhz_median": s_clk["sm_mhz"], "sm_max_mhz": s_clk["sm_max_mhz"],
                     "power_w_median": s_clk["power_w"], "reasons": s_clk["reasons"], "clock_samples": s_clk["samples"]}

    # ---------------- end to end through the host-buffer C-ABI call
    Be = min(args.e2e_batch, B)
    nstreams = max(1, min(args.e2e_streams, Be))
    per = Be // nstreams
    if nes:
        h_src = torch.randint(0, 512, (Be, H_IN, W_IN), dtype=torch.int16, generator=gen).pin_memory()
    else:
        h_src = torch.randint(0, 256, (Be, H_IN, W_IN, 4), dtype=torch.uint8, generator=gen).pin_memory()
    h_out = torch.zeros(Be, H_OUT, W_OUT, 4, dtype=torch.uint8).pin_memory()
    streams = [torch.cuda.Stream(dev) for _ in range(nstreams)]
    htables = []
    for field in (0, 1):
        t = (capi.Source * Be)()
        for i in range(Be):
            s = t[i]
            s.data = h_src[i].data_ptr()
            s.format, s.w, s.h = layout.PIX_BGRA, W_IN, H_IN
            s.raw, s.as_color, s.field, s.frame = 0, 1, field, 0
        htables.append(t)
    outp = (C.c_void_p * Be)(*[h_out[i].data_ptr() for i in range(Be)])

    def e2e_step(k):
        for q in range(nstreams):
            first = q * per
            batch._check(batch.lib.crtx_frames_host(
                batch._ctx, first, per, sub_table(htables[k & 1], first),
                C.cast(C.byref(outp, first * C.sizeof(C.c_void_p)), C.POINTER(C.c_void_p)),
                streams[q].cuda_stream))

    e2e_steps = max(2, min(4 * args.steps, 64))  # long enough that filling / draining the stream pipeline is noise
    for k in range(2):
        e2e_step(k)
    barrier()
    launches_e0 = batch.launches
    t0 = time.perf_counter()
    e0 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s_ in streams:
        s_.wait_stream(stream)
    for k in range(e2e_steps):
        e2e_step(k)
    ends = []
    for q in range(nstreams):
        e = torch.cuda.Event(enable_timing=True)
        e.record(streams[q])
        ends.append(e)
    barrier()
    e2e_ms = max(e0.elapsed_time(e) for e in ends)
    e2e_wall = time.perf_counter() - t0
    e2e_ms = max(e2e_ms, 0.0)
    launches_e2e = batch.launches - launches_e0
    batch.timing()
    frames_e2e = per * nstreams * e2e_steps
    # what crtx_frames_host moves per frame with page-locked 16-byte granular images (include/crtx_batch.h): the source
    # rows a field reads and the output rows it writes (mean of the two parities); whole images otherwise
    host_rows = not any(kv.split("=")[0] == "host_rows" and int(kv.split("=")[1]) == 0 for kv in args.set)
    bandlimited = not (VARIANT.startswith("nes") or VARIANT == "snes")
    if host_rows and bandlimited:
        h2d_frame = source_rows_read(H_IN, 236 if VARIANT != "ntsc_bloom" else 232) * W_IN * 4 + 32
    else:
        h2d_frame = W_IN * H_IN * (2 if nes else 4)
    d2h_frame = ((field_rows(0)[1] + field_rows(1)[1]) / 2.0 * W_OUT * 4 + 8) if host_rows else W_OUT * H_OUT * 4

    # ---------------- N > 1: the exchange north_star names -- all_gather of the decoded frames over NVLink
    gather = root = None
    if world > 1 and not args.no_allgather:
        g_steps = max(2, min(args.steps, 6))
        half = B // 2
        halves = ((0, half), (half, B - half))
        side = torch.cuda.Stream(dev)
        full = [torch.empty((world, n) + tuple(out.shape[1:]), dtype=torch.uint8, device=dev) for _, n in halves]

        def run_gather(kind):
            """per step: both half-batches advance one field on the compute stream while the other half's decoded
            images travel on `side`; a half is not touched again before its gather has read it"""
            done = [None, None]
            ready = [torch.cuda.Event(), torch.cuda.Event()]
            for k in range(g_steps):
                for hi_, (f0, n0) in enumerate(halves):
                    if done[hi_] is not None:
                        stream.wait_event(done[hi_])
                    step(k, f0, n0)
                    ready[hi_].record(stream)
                    side.wait_event(ready[hi_])
                    with torch.cuda.stream(side):
                        if kind == "allgather":
                            dist.all_gather_into_tensor(full[hi_].view(-1), out[f0:f0 + n0].view(-1))
                        else:
                            dist.gather(out[f0:f0 + n0], list(full[hi_].unbind(0)) if rank == 0 else None, dst=0)
                        done[hi_] = torch.cuda.Event()
                        done[hi_].record(side)
            stream.wait_stream(side)

        res = {}
        for kind in ("allgather", "gather_to_root"):
            run_gather(kind)  # warm-up (NCCL channel set-up)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            run_gather(kind)
            g1.record(stream)
            barrier()
            g_ms = sharding.max_over_ranks([g0.elapsed_time(g1)], device=dev)[0]
            recv = (world - 1) * B * H_OUT * W_OUT * 4  # bytes a receiving rank takes in per step
            res[kind] = {"value": world * B * g_steps / (g_ms / 1e3), "unit": "frames/s", "steps": g_steps, "ms_per_step": g_ms / g_steps,
                         "bytes_received_per_rank_per_step": recv,
                         "nvlink_gbs_into_a_rank": recv * g_steps / (g_ms / 1e3) / 1e9}
        gather, root = res["allgather"], res["gather_to_root"]
        del full

    # ---------------- config 4 (video sequence over frame ranges), every N
    cfg4 = None
    if VARIANT == "ntsc" and args.config4_frames > 0:
        try:
            cfg4 = config4_block(args, dev, rank, world)
        except Exception as e:  # a secondary block must not cost the line
            cfg4 = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---------------- max over ranks
    if world > 1:
        t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
    value = world * B * args.steps / (ms / 1e3)
    e2e_value = world * frames_e2e / (e2e_ms / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        lines_ms, lines_n = ktimes["lines"]
        sync_ms, sync_n = ktimes["sync"]
        noise_ms, _ = ktimes["noise"]
        isz, av_len = batch.spec.input_size, batch.spec.av_len
        conv = "_conv" in VARIANT
        # the line kernel, charged with what IT moves
        kern_bytes = B * (lines_bytes(0, av_len) + lines_bytes(1, av_len)) / 2.0
        launch_ms = lines_ms / max(1, lines_n)
        achieved = (kern_bytes / 1e9) / (launch_ms / 1e3) if lines_n else None
        # the whole crt_demodulate (SURVEY 8d) over every kernel it runs
        dem_bytes = B * (demod_bytes(0, input_size=isz) + demod_bytes(1, input_size=isz)) / 2.0
        dem_ms = (lines_ms + sync_ms + noise_ms) / max(1, args.steps)
        dem_achieved = (dem_bytes / 1e9) / (dem_ms / 1e3) if dem_ms > 0 else None
        kernel_share = {k: round(v[0] / ms_instrumented, 4) for k, v in ktimes.items()}
        # DRAM bytes of the line kernel per launch: from the committed ncu --set full capture, and only if that capture
        # was taken from THIS build of the kernels (profiles/make_traffic.py records the source hash)
        traffic, traffic_src = None, "no ncu capture of this build under profiles/ (see profiles/make_traffic.py)"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            ent = tj.get(VARIANT)
            if ent and ent.get("src_sha") == library_source_hash():
                traffic = ent["dram_bytes_per_field"] * B
                traffic_src = "profiles/r2_traffic.json: %s" % ent.get("capture", "")
            elif ent:
                traffic_src = "profiles/r2_traffic.json is from another build of the kernels (%s): not reported" % ent.get("src_sha")
        except Exception:
            pass
        cpu = cpu_baseline_single() if (world == 1 and not args.no_cpu_baseline) else None
        if conv:
            kname = "k_lines_fir (crt_demodulate line pass of the USE_CONVOLUTION build, crt_core.c:96-147,511-664)"
        elif took_lines2:
            kname = "k_lines2 (crt_demodulate line pass, crt_core.c:511-664; two monitors per CTA)"
        else:
            kname = "k_lines (crt_demodulate line pass, crt_core.c:511-664)"
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
            "config": {"workload": workload_name(),
                       "batch_per_gpu": B, "global_batch": B * world, "parallelism": "dp%d (frames sharded, no collective in the step)" % world,
                       "l2": "inputs larger than L2: %.0f MB of images + signals touched per step per GPU" % (B * 4.63)},
            "e2e": {"value": e2e_value, "unit": "frames/s",
                    "h2d_bytes_per_step": int(per * nstreams * h2d_frame),
                    "d2h_bytes_per_step": int(per * nstreams * d2h_frame),
                    "batch": per * nstreams, "steps": e2e_steps,
                    "api": "crtx_frames_host, page-locked host images, %d streams; %s" % (
                        nstreams, "only the rows a field reads / writes cross PCIe" if host_rows else "whole images both ways"),
                    "pcie_gbs_h2d": per * nstreams * h2d_frame * e2e_steps / (e2e_ms / 1e3) / 1e9 if e2e_ms > 0 else None,
                    "pcie_gbs_d2h": per * nstreams * d2h_frame * e2e_steps / (e2e_ms / 1e3) / 1e9 if e2e_ms > 0 else None,
                    "numa": numa, "wall_s": e2e_wall},
            "gpu_launches": int(launches),
            "gpu_launches_e2e": int(launches_e2e),
            # SURVEY 8d: the CLI accumulates 8 modulate + demodulate pairs per interlaced image (crt_main.c:242-255)
            "cli_images_per_s": value / 8.0,
            "roofline": {"bound": "hbm", "kernel": kname,
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": kern_bytes, "launch_ms": launch_ms,
                         "bytes": "kernel-only: per decoded line its AV_LEN-sample window + blend read + rows written",
                         "peak_source": peak_src,
                         "demodulate": {"achieved": dem_achieved, "frac": (dem_achieved / peak) if dem_achieved else None,
                                        "algorithmic_bytes_per_step": dem_bytes, "ms_per_step": dem_ms,
                                        "bytes": "SURVEY 8d: 2*INPUT_SIZE + bpp*outw*(rows_computed*blend + rows_written) per field",
                                        "kernels": "k_sync (noise pass fused) + line kernel"}},
            "kernel_ms_per_step": {k: round(v[0] / max(1, args.steps), 4) for k, v in ktimes.items()},
            "kernel_times_from": "a second pass of %d steps with the library's per-kernel CUDA events on (%.4f ms per step; the timed region above runs without them)" % (args.steps, ms_instrumented / max(1, args.steps)),
            "kernel_share_of_step": kernel_share,
            "clocks": clocks,
        }
        if sustained:
            sustained["vs_value"] = sustained["frames_per_s"] / value if value else None
            line["sustained"] = sustained
        if world == 1:
            line["dropin"] = dropin_isolated(0.3 if args.no_cpu_baseline else 2.0)
        if cpu:
            line["cpu_baseline"] = cpu
        if gather:
            bound = "allgather (NVLink)" if gather["value"] < 0.9 * value else "kernels"
            gather["bound_by"] = bound
            line["allgather"] = gather
            line["gather_to_root"] = root
        if cfg4:
            line["config4"] = cfg4
        print(json.dumps(line), flush=True)
    batch.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference", "dropin"],
                    help="dropin: only the informational drop-in figure (used by the product arm in a child process)")
    ap.add_argument("--dropin-seconds", type=float, default=2.0)
    ap.add_argument("--batch", type=int, default=296,
                    help="monitors (frames per step) per GPU; 296 = 148 SMs x the two monitors a line-kernel CTA decodes")
    ap.add_argument("--e2e-batch", type=int, default=128)
    ap.add_argument("--e2e-streams", type=int, default=4)
    ap.add_argument("--sustained-seconds", type=float, default=1.2, help="0: skip the sustained block")
    ap.add_argument("--config4-frames", type=int, default=4999,
                    help="length of the config-4 video sequence: video_convert.c with num_frames 5000 converts 4999 images (0: skip)")
    ap.add_argument("--config4-segments", type=int, default=0, help="time-parallel segments per rank (0: about 8 frames per segment)")
    ap.add_argument("--set", action="append", default=[], help="library option name=value (A/B testing)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the images the last timed step computed to DIR/*.npy (a seeded sample; see dump_outputs)")
    ap.add_argument("--no-allgather", action="store_true", help="N > 1: skip the all_gather / gather_to_root blocks")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the process to the GPU's NUMA node")
    ap.add_argument("--variant", default="ntsc", choices=["ntsc", "ntsc_conv", "ntsc_conv6", "ntsc_conv5", "ntsc_conv4", "nes", "nes_p0", "nes_p1", "snes", "nesrgb", "nesrgb_p0", "nesrgb_p1", "vhs", "template", "pv1k", "ntsc_bloom"],
                    help="informational runs of the other systems (the contract metric is the default, ntsc)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "product" else args.warmup
    global VARIANT, W_IN, H_IN
    VARIANT = args.variant
    if VARIANT.startswith("nes"):
        W_IN, H_IN = 256, 240  # PPU image (BASELINE configs[2])
    if args.impl == "dropin":
        import pkgload
        pkgload.load()
        print(json.dumps(dropin_fps(args.dropin_seconds)), flush=True)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
