#!/usr/bin/env python
"""bench.py — interpolated frames/s of the optical-flow interpolation hot path on B200.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): 3840x2160 P010 HDR,
23.976 -> 144 fps, full-resolution flow, search radius R = 16 (where the reference's auto-tuner saturates
on a fast GPU), deltaScalar 8, neighborScalar 6, levels 0/255, BlendedFrame output.

A step = one source frame through the reference's call sequence (HopperRender.cpp:953-1186):
updateFrame + calculateOpticalFlow + N x warpFrames, N from the filter's own schedule (6, occasionally 7).
  value : device-resident — frames already in HBM (a ring larger than L2), outputs left in HBM.
  e2e   : the same through the public blocking API with pinned HOST buffers: H2D of the source frame and
          a D2H downloadFrame of every output frame inside the timed region.
One process per GPU; each rank runs its own independent stream (no data-path collective) => weak scaling.

`--impl reference` times the reference's algorithm on the host CPU cores (the oracle port of the OpenCL
kernels, OpenMP on all cores; the reference itself needs an OpenCL device, which this box lacks) on a
bounded sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step computed (its output frames and the flow
field its search produced) as DIR/<name>.npy, so that two builds run with the same arguments can be compared output for
output: the inputs are seeded, the same from run to run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (W, H, hdr, maxCalcRes, target_frame_time)
    "cfg3": dict(W=3840, H=2160, hdr=True, maxres=2160, target=69444, desc="3840x2160 P010 HDR 23.976->144 fps, full-resolution flow"),
    "cfg2": dict(W=1920, H=1080, hdr=False, maxres=540, target=69444, desc="1920x1080 NV12 SDR 23.976->144 fps, half-resolution flow"),
    "cfg1": dict(W=1920, H=1080, hdr=False, maxres=270, target=166667, desc="1920x1080 NV12 SDR 24->60 fps, 270p flow"),
    "cfg4": dict(W=7680, H=4320, hdr=True, maxres=4320, target=69444, desc="7680x4320 P010 HDR 23.976->144 fps, full-resolution flow, ONE stream "
                 "split spatially over the GPUs (NVLink all-gather of the ingested stripes, per-GPU warp + egress of its stripe)"),
}
SEARCH_RADIUS = 16
METRIC = "interpolated frames/s at 4K P010 (flow + warp, R=16)"


def metric_name(workload):
    """BASELINE.json's metric is quoted on cfg3; the other workloads are named for what they are."""
    return METRIC if workload == "cfg3" else f"interpolated frames/s, workload {workload} (flow + warp)"

UNIT = "frames/s"


def _nolib(name):
    """hopperrender_b200/<name>.py loaded WITHOUT the package __init__ (which loads libhrb.so): the reference arm must not
    map the CUDA library.  synth.py and replay.py are plain numpy / python."""
    import importlib.util
    key = f"_hrb_nolib_{name}"
    if key in sys.modules:
        return sys.modules[key]
    spec = importlib.util.spec_from_file_location(key, os.path.join(ROOT, "hopperrender_b200", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[key] = mod
    spec.loader.exec_module(mod)
    return mod


def host_threads():
    """Threads the CPU legs may use: the cores this process is allowed on (launchers export OMP_NUM_THREADS=1; ignored)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this
    workload (profiles/ncu_traffic.json, written by tools/ncu_summary.py), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)[workload][kernel]["dram_bytes_per_launch"]
    except Exception:  # noqa: BLE001
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", os.environ.get("HRB_CLOCK_MS", "20")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 7 or not self.rows:
                continue
            try:
                sm.append(float(c[0]))
                mx.append(float(c[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_near_gpu(local):
    """Pin this process to the CPU cores (and so, by first touch, its pinned buffers to the memory) next to its GPU.
    Matters for the end-to-end numbers at N>1: eight ranks on one NUMA node share that node's memory bandwidth."""
    if os.environ.get("HRB_NO_BIND"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        return sorted(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return None


def init_dist(local):
    """NCCL by default (eager, bound to this rank's GPU); HRB_DIST_BACKEND=gloo and HRB_DIST_LAZY=1 exist for A/B runs of the
    effect of the communicator on the device-timed loop."""
    import torch
    import torch.distributed as dist
    backend = os.environ.get("HRB_DIST_BACKEND", "nccl")
    if backend == "nccl" and not os.environ.get("HRB_DIST_LAZY"):
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group(backend)


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


DUMP_SAMPLES = 1 << 20         # values kept of a larger array: a fixed, seeded sample
DUMP_BYTES = 64 * 1000 * 1000  # all arrays of one dump together


def dump_outputs(out_dir, calc, blends, hdr):
    """The arrays a caller of the timed step receives after it: the len(blends) output frames of warpFramesBatch, in order,
    as output<k>.npy, and the flow field the step's calculateOpticalFlowAsync produced, as flow.npy.  float32 (exact for
    the 8/16-bit samples and 16-bit offsets).  An array longer than the per-array share of DUMP_BYTES (at most
    DUMP_SAMPLES values) is stored as the values at sorted indices drawn with a fixed seed: the same positions in every
    run."""
    n_el = calc.outputFrameBytes // (2 if hdr else 1)
    arrays = {}
    for k in range(len(blends)):
        a = np.empty(n_el, np.uint16 if hdr else np.uint8)
        calc.downloadFrame(a)
        arrays[f"output{k}"] = a
    arrays["flow"] = calc.readFlow(latest=True).reshape(-1)
    cap = min(DUMP_SAMPLES, (DUMP_BYTES - 1024 * len(arrays)) // 4 // len(arrays))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def algorithmic_bytes(wl):
    """SURVEY.md §8(d): F = 1.5*W*H*bpp, L = lw*lh; warp (mode 2) = 3F + 4L per launch."""
    bpp = 2 if wl["hdr"] else 1
    rs = 0
    while (wl["H"] >> rs) > wl["maxres"]:
        rs += 1
    lw, lh = -(-wl["W"] // (1 << rs)), -(-wl["H"] // (1 << rs))
    F = wl["W"] * wl["H"] * 3 // 2 * bpp
    L = lw * lh
    ws = 1
    while ws < max(lw, lh):
        ws <<= 1
    iters = max(ws // 2, 1).bit_length() - 1
    return dict(F=F, L=L, warp=3 * F + 4 * L, blur=8 * L, copy=2 * F, passes=2 * iters, absdiff=3 * SEARCH_RADIUS * L * 2 * iters, lw=lw, lh=lh)


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_sample_rows(wl, budget_s):
    """Rows of a full-width band of the workload frame whose flow + warps cost about budget_s on this host."""
    synth = _nolib("synth")
    from oracle import OracleCalc
    W, hdr = wl["W"], wl["hdr"]
    probe = 128
    o = OracleCalc(probe, W, 0, 0, 8, 6, 0.0, 255.0, probe, hdr)
    o.setParams(searchRadius=SEARCH_RADIUS)
    fr = [synth.make_frame(W, probe, t, hdr=hdr, noise=False) for t in range(3)]
    for f in fr:
        o.updateFrame(f)
    t0 = time.perf_counter()
    o.calculateOpticalFlow()
    for _ in range(6):
        o.warpFrames(0.5, 2)
    dt = time.perf_counter() - t0
    o.close()
    rows = int(probe * budget_s / max(dt, 1e-6))
    rows = max(64, min(wl["H"], rows // 16 * 16))
    return rows


def cpu_step_runner(wl, rows):
    """Returns (fn, n_out): fn() runs one source-frame step (update + flow + N warps + downloads) on the CPU sample."""
    replay, synth = _nolib("replay"), _nolib("synth")
    from oracle import OracleCalc
    W, hdr = wl["W"], wl["hdr"]
    o = OracleCalc(rows, W, 0, 0, 8, 6, 0.0, 255.0, rows, hdr)
    o.setParams(searchRadius=SEARCH_RADIUS)
    ring = [synth.make_frame(W, rows, t, hdr=hdr, noise=False) for t in range(4)]
    for f in ring[:3]:
        o.updateFrame(f)
    out = np.zeros(o.outputFrameBytes, np.uint8)
    state = {"i": 3, "blend": 0.0}

    def step():
        o.updateFrame(ring[state["i"] % len(ring)])
        state["i"] += 1
        o.calculateOpticalFlow()
        n = replay.num_int_frames(state["blend"], wl["target"], replay.SOURCE_FRAME_TIME_23976)
        for _ in range(n):
            o.warpFrames(state["blend"], 2)
            o.downloadFrame(out)
            state["blend"] = replay.advance_blend(state["blend"], wl["target"], replay.SOURCE_FRAME_TIME_23976)
        return n

    return step


class _StdoutToStderr:
    """The reference's host classes print to stdout (opticalFlowCalc.cpp:104-107); the bench's stdout carries ONE JSON line, so
    while they run file descriptor 1 points at stderr."""
    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)
        return False


_JSON_OUT = None


def claim_stdout():
    """stdout carries ONE JSON line.  Libraries underneath print there too (NCCL's version banner, the reference's device
    report), so the process's file descriptor 1 is pointed at stderr for its whole life and the line goes to a private
    duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def reference_opencl_same_gpu(wl, steps=8, radius=SEARCH_RADIUS):
    with _StdoutToStderr():
        return _reference_opencl_same_gpu(wl, steps, radius)


def _reference_opencl_same_gpu(wl, steps, radius):
    """The reference ITSELF — unmodified HopperRender host classes + OpenCL kernel strings (oracle/_ref) — through the NVIDIA
    OpenCL driver on this box's GPU, with the filter's call sequence, its blocking transfers and its own event timers
    (opticalFlowCalcSDR.cpp:119-138, :32-41).  None when oracle/_ref is not built or no OpenCL device accepts it."""
    try:
        from oracle import RefCalc, ref_available
        if not ref_available():
            return None
        replay, synth = _nolib("replay"), _nolib("synth")
        W, H, hdr = wl["W"], wl["H"], wl["hdr"]
        r = RefCalc(H, W, 0, 0, 8, 6, 0.0, 255.0, wl["maxres"], hdr)
        r.setParams(searchRadius=radius)
        frames = [synth.make_frame(W, H, t, synth.SEED_BASE + 2, hdr, noise=False) for t in range(3)]
        ring = frames + [frames[1]]
        out = np.zeros(r.outputFrameBytes, np.uint8)
        for f in frames:
            r.updateFrame(f)
        sched = replay.output_schedule(steps + 4, wl["target"], replay.SOURCE_FRAME_TIME_23976)

        def step(i):
            r.updateFrame(ring[i % 4])
            r.calculateOpticalFlow()
            for b in sched[i]:
                r.warpFrames(b, 2)
                r.downloadFrame(out)
            return len(sched[i])

        step(0)
        t0 = time.perf_counter()
        n, flow_s, warp_s = 0, [], []
        for i in range(1, 1 + steps):
            n += step(i)
            st = r.state()
            flow_s.append(st.ofcCalcTime)
            warp_s.append(st.warpCalcTime)
        dt = time.perf_counter() - t0
        res = {"value": n / dt, "unit": UNIT, "ofc_ms": float(np.median(flow_s)) * 1e3, "warp_ms": float(np.median(warp_s)) * 1e3, "steps": steps,
               "device": r.deviceName(), "api": "reference's own blocking calls (pageable host buffers) and event timers; same GPU, NVIDIA OpenCL"}
        r.close()
        return res
    except Exception as e:  # noqa: BLE001
        return {"value": None, "unit": UNIT, "error": str(e)[:200]}


def run_reference(args, wl, wl_name):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    from oracle import set_num_threads
    cores = set_num_threads(host_threads())
    per_step = max(0.2, min(8.0, float(os.environ.get("HRB_REF_BUDGET_S", "150")) / max(args.steps + args.warmup, 1)))
    rows = cpu_sample_rows(wl, per_step)
    step = cpu_step_runner(wl, rows)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    frames = 0
    for _ in range(args.steps):
        frames += step()
    dt = time.perf_counter() - t0
    frac = rows / wl["H"]
    value = frames * frac / dt
    sample = (f"each step = one source frame (updateFrame + calculateOpticalFlow + N warpFrames + downloadFrame) on a full-width "
              f"{wl['W']}x{rows} band of the workload frame ({frac:.4f} of the pixels); value = frames x {frac:.4f} / time "
              f"(full-frame equivalent, linear in pixels)")
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": {"workload": f"{wl_name}: {wl['desc']}, R={SEARCH_RADIUS}", "search_radius": SEARCH_RADIUS},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_cpu_baseline:
        # beside the CPU port: the reference's own kernels on this box's GPU (BASELINE.md B3), when its OpenCL leg is usable here
        line["reference_opencl_b200"] = reference_opencl_same_gpu(wl, radius=SEARCH_RADIUS)
    emit(line)


def cpu_baseline(wl):
    """Bounded CPU sample for the main line (rank 0, N=1): ~15 s of oracle work."""
    from oracle import set_num_threads
    cores = set_num_threads(host_threads())
    rows = cpu_sample_rows(wl, 5.0)
    step = cpu_step_runner(wl, rows)
    step()
    t0 = time.perf_counter()
    frames = 0
    for _ in range(2):
        frames += step()
    dt = time.perf_counter() - t0
    frac = rows / wl["H"]
    return {"value": frames * frac / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"2 source-frame steps on a full-width {wl['W']}x{rows} band ({frac:.4f} of the pixels), scaled linearly to the full frame"}


# ------------------------------------------------------------------------------------------------------
# configs[3]: one 8K stream split spatially over the GPUs (strong scaling)
# ------------------------------------------------------------------------------------------------------
def run_split(args, wl):
    import torch
    import torch.distributed as dist

    import hopperrender_b200 as hr
    from hopperrender_b200 import replay, shard, synth
    from hopperrender_b200.split import SpatialSplitStream

    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    if world > 1:
        bind_near_gpu(local)
    if world > 1:
        init_dist(local)
    W, H, hdr = wl["W"], wl["H"], wl["hdr"]
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    s = SpatialSplitStream(cls, H, W, 8, 6, 0.0, 255.0, wl["maxres"], rank=rank, world_size=world)
    s.calc.m_opticalFlowSearchRadius = args.radius
    RING = 3
    host = [torch.from_numpy(synth.make_frame(W, H, t, synth.SEED_BASE + 4, hdr, noise=False).view(np.int16 if hdr else np.uint8)).pin_memory()
            for t in range(RING)]
    POOL = 10
    pool = [torch.empty_like(host[0]).pin_memory() for _ in range(POOL)]
    sched = replay.output_schedule(3 * (args.steps + args.warmup) + 16, wl["target"], replay.SOURCE_FRAME_TIME_23976)
    pending, k = [], [0]

    def step(i):
        s.update_frame(host[i % RING])
        s.calculate_optical_flow()
        for b in sched[i]:
            pending.append(s.warp_and_download(b, hr.BlendedFrame, pool[k[0] % POOL]))
            k[0] += 1
        while len(pending) > 7:
            s.wait(pending.pop(0))
        return len(sched[i])

    idx = 0
    for _ in range(max(args.warmup, 3)):
        step(idx)
        idx += 1
    while pending:
        s.wait(pending.pop(0))
    s.calc.synchronize()
    shard.barrier()
    torch.cuda.synchronize()
    launches0 = hr.kernel_launch_count()
    t0 = time.perf_counter()
    frames = 0
    for _ in range(args.steps):
        frames += step(idx)
        idx += 1
    while pending:
        s.wait(pending.pop(0))
    s.calc.synchronize()
    shard.barrier()
    torch.cuda.synchronize()
    ms = shard.combine(0, (time.perf_counter() - t0) * 1e3)[1]
    launches = shard.combine(hr.kernel_launch_count() - launches0, 0)[0]
    if rank == 0:
        value = frames / (ms * 1e-3)  # every rank delivers a stripe of the SAME frames: the stream's rate, not a sum
        line = {
            "metric": "interpolated frames/s of one 8K P010 stream (flow + warp, R=16), spatially split", "value": value, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"cfg4: {wl['desc']}, R={args.radius}", "stripe_rows": H // world,
                       "collective": "NCCL all-gather of the ingested frame stripes (2 per source frame); search replicated; no other exchange",
                       "realtime_factor_vs_144fps": value / 144.0},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": int(s.stripe_bytes()),
                    "d2h_bytes_per_step": int(round(frames / args.steps * s.stripe_bytes())), "note": "bytes per rank"},
            "gpu_launches": int(launches),
        }
        emit(line)
    s.close()
    if world > 1:
        dist.destroy_process_group()



# ------------------------------------------------------------------------------------------------------
# several independent streams per GPU (SURVEY.md section 8(e), cfg5): S handles per device, one host thread round-robin
# ------------------------------------------------------------------------------------------------------
def run_streams(args, wl):
    import torch
    import torch.distributed as dist

    import hopperrender_b200 as hr
    from hopperrender_b200 import replay, shard, synth

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — hopperrender_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        bind_near_gpu(local)
    if world > 1:
        init_dist(local)
    S = args.streams_per_gpu
    W, H, hdr = wl["W"], wl["H"], wl["hdr"]
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    tstreams = [torch.cuda.Stream() for _ in range(S)]
    calcs = [cls(H, W, 0, 0, 8, 6, 0.0, 255.0, wl["maxres"], device=local, stream=ts.cuda_stream) for ts in tstreams]
    for c in calcs:
        c.m_opticalFlowSearchRadius = args.radius
        if args.no_overlap:
            c.setFlowOverlap(False)
    NFR = 6
    PING = list(range(NFR)) + list(range(NFR - 2, 0, -1))   # frames played back and forth: every pair is one motion step
    RING = len(PING)
    tdt = torch.int16 if hdr else torch.uint8
    distinct = [synth.make_frame(W, H, t, synth.SEED_BASE + 2 + rank, hdr) for t in range(NFR)]
    pinned_d = [torch.from_numpy(f.view(np.int16) if hdr else f).pin_memory() for f in distinct]
    dev_d = [p.cuda() for p in pinned_d]
    pinned = [pinned_d[t] for t in PING]
    dev = [dev_d[t] for t in PING]
    torch.cuda.synchronize()
    sched = replay.output_schedule(5 * (args.warmup + args.steps) + 128, wl["target"], replay.SOURCE_FRAME_TIME_23976)
    POOL = 8
    n_el = calcs[0].outputFrameBytes // (2 if hdr else 1)
    pools = [[torch.empty(n_el, dtype=tdt).pin_memory() for _ in range(POOL)] for _ in range(S)]
    pending = [[] for _ in range(S)]
    counts = [0] * S

    def step_device(h, i):
        c = calcs[h]
        c.updateFrameDevice(dev[(i + h) % RING])
        c.calculateOpticalFlowAsync()
        c.warpFramesBatch(sched[i], hr.BlendedFrame)
        return len(sched[i])

    def step_e2e(h, i):
        c = calcs[h]
        c.updateFrame(pinned[(i + h) % RING])
        c.calculateOpticalFlowAsync()
        c.warpFramesBatch(sched[i], hr.BlendedFrame)
        for b in sched[i]:
            while len(pending[h]) >= POOL - 1:   # the pinned buffer about to be reused has been delivered (its ticket waited for)
                c.waitDownload(pending[h].pop(0))
            pending[h].append(c.downloadFrameAsync(pools[h][counts[h] % POOL]))
            counts[h] += 1
        return len(sched[i])

    def sync_all():
        for h, c in enumerate(calcs):
            while pending[h]:
                c.waitDownload(pending[h].pop(0))
            c.synchronize()
        torch.cuda.synchronize()
        shard.barrier()

    idx = 0
    for i in range(3):
        for h in range(S):
            calcs[h].updateFrameDevice(dev[(i + h) % RING])
    for _ in range(args.warmup):
        for h in range(S):
            step_device(h, idx)
        idx += 1
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = hr.kernel_launch_count()
    e0 = torch.cuda.Event(enable_timing=True)
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(S)]
    e0.record(torch.cuda.current_stream())   # the device is idle here: every stream's work starts after this point
    frames = 0
    for _ in range(args.steps):
        for h in range(S):
            frames += step_device(h, idx)
        idx += 1
    for h in range(S):
        calcs[h].joinFlow()
        ends[h].record(tstreams[h])
    sync_all()
    ms = shard.combine(0, max(e0.elapsed_time(e) for e in ends))[1]
    launches = shard.combine(hr.kernel_launch_count() - launches0, 0.0)[0]
    clocks = sampler.stop() if rank == 0 else None
    total_frames = shard.combine(frames, 0.0)[0]
    value = total_frames / (ms * 1e-3)

    esteps = min(args.steps, 50)
    for _ in range(2):
        for h in range(S):
            step_e2e(h, idx)
        idx += 1
    sync_all()
    t0 = time.perf_counter()
    eframes = 0
    for _ in range(esteps):
        for h in range(S):
            eframes += step_e2e(h, idx)
        idx += 1
    sync_all()
    wall_ms = shard.combine(0, (time.perf_counter() - t0) * 1e3)[1]
    e2e_value = shard.combine(eframes, 0.0)[0] / (wall_ms * 1e-3)
    if rank == 0:
        line = {"metric": metric_name(args.workload), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic",
                "config": {"workload": f"{args.workload}: {wl['desc']}, R={args.radius}", "search_radius": args.radius,
                           "streams_per_gpu": S, "flow_overlap": not args.no_overlap,
                           "note": "a step = one source frame of EVERY stream; S independent handles per GPU driven round-robin by one host thread",
                           "l2": "each stream's per-step working set (~265 MB at cfg3) exceeds the 126 MB L2"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(S * calcs[0].inputFrameBytes),
                        "d2h_bytes_per_step": int(round(eframes / esteps * calcs[0].outputFrameBytes)), "steps": esteps},
                "gpu_launches": int(launches), "clocks": clocks}
        emit(line)
    for c in calcs:
        c.close()
    if world > 1:
        dist.destroy_process_group()

# ------------------------------------------------------------------------------------------------------
# the CUDA arm
# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="keep the asynchronous flow calculation on the compute stream (A/B)")
    ap.add_argument("--no-batch", action="store_true", help="one warpFrames call per output frame, as the reference's loop does (A/B of warpFramesBatch)")
    ap.add_argument("--radius", type=int, default=SEARCH_RADIUS)
    ap.add_argument("--streams-per-gpu", type=int, default=1, help="independent video streams (handles) per GPU; >1 prints the multi-stream line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the output frames and the flow of the last timed "
                    "step to DIR/<name>.npy (float32, 64 MB at most; rank 0; single-stream CUDA path only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload == "cfg4" or args.streams_per_gpu > 1):
        ap.error("--dump-outputs applies to the single-stream CUDA path (--impl ours, one stream per GPU, not cfg4)")
    claim_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, args.workload)
        return
    if args.workload == "cfg4":
        run_split(args, wl)
        return
    if args.streams_per_gpu > 1:
        run_streams(args, wl)
        return

    import torch
    import torch.distributed as dist

    import hopperrender_b200 as hr
    from hopperrender_b200 import replay, synth

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — hopperrender_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        bind_near_gpu(local)
    if world > 1:
        init_dist(local)

    W, H, hdr = wl["W"], wl["H"], wl["hdr"]
    alg = algorithmic_bytes(wl)
    stream = torch.cuda.Stream()
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    calc = cls(H, W, 0, 0, 8, 6, 0.0, 255.0, wl["maxres"], device=local, stream=stream.cuda_stream)
    if args.no_overlap:
        calc.setFlowOverlap(False)
    calc.m_opticalFlowSearchRadius = args.radius

    # synthetic frames: a ring of distinct frames, device-resident and pinned-host copies
    # ring of distinct frames played back and forth (0 1 2 3 4 5 4 3 2 1 0 1 ...): every consecutive pair is one step of
    # the scene's motion, forward or backward — a wrap from the last frame to the first would be a scene cut every 6 frames
    NFR = 6
    PING = list(range(NFR)) + list(range(NFR - 2, 0, -1))
    RING = len(PING)
    dt_np = np.uint16 if hdr else np.uint8
    distinct = [synth.make_frame(W, H, t, synth.SEED_BASE + 2 + rank, hdr) for t in range(NFR)]
    tdt = torch.int16 if hdr else torch.uint8
    pinned_d = [torch.from_numpy(f.view(np.int16) if hdr else f).pin_memory() for f in distinct]
    dev_d = [p.cuda(non_blocking=False) for p in pinned_d]
    pinned = [pinned_d[t] for t in PING]
    dev = [dev_d[t] for t in PING]
    out_pinned = torch.empty(calc.outputFrameBytes // (2 if hdr else 1), dtype=tdt).pin_memory()
    torch.cuda.synchronize()

    total_steps = args.warmup + args.steps
    sched = replay.output_schedule(5 * total_steps + 128, wl["target"], replay.SOURCE_FRAME_TIME_23976)

    from hopperrender_b200 import shard

    def barrier():
        shard.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        return shard.combine(0, ms)[1]

    def sum_over_ranks(v):
        return shard.combine(v, 0.0)[0]

    # ---- device-resident loop ---------------------------------------------------------------------
    dbg_peak = bool(os.environ.get("HRB_DEBUG_PEAK"))

    def step_device(i):
        calc.updateFrameDevice(dev[i % RING])
        calc.calculateOpticalFlowAsync()
        if dbg_peak and i < 10:  # diagnostics: the flow peak the warp kernel is about to read (synchronizes)
            print(f"step {i}: flow peak (for warp, latest) {calc.readFlowPeak()} t {[round(float(b), 4) for b in sched[i]]}", file=sys.stderr)
        if args.no_batch:
            for b in sched[i]:
                calc.warpFrames(b, hr.BlendedFrame)
        else:
            calc.warpFramesBatch(sched[i], hr.BlendedFrame)   # the N output frames of this source frame in one pass
        return len(sched[i])

    def step_e2e_blocking(i):
        # the reference's own call sequence, every transfer blocking (HopperRender.cpp:953-1186)
        calc.updateFrame(pinned[i % RING])
        calc.calculateOpticalFlow()
        for b in sched[i]:
            calc.warpFrames(b, hr.BlendedFrame)
            calc.downloadFrame(out_pinned)
        return len(sched[i])

    E2E_DEPTH = int(os.environ.get("HRB_E2E_DEPTH", "8"))          # downloads left in flight when a step returns
    E2E_ASYNC_UP = bool(int(os.environ.get("HRB_E2E_ASYNC_UP", "0")))  # upload through update_frame_async (own stream, no host wait)
    POOL = max(16, E2E_DEPTH + 10)
    out_pool = [torch.empty_like(out_pinned).pin_memory() for _ in range(POOL)]
    pending = []
    dl_count = [0]

    def step_e2e(i):
        # same work through the asynchronous entry points: the upload of this frame and the downloads of its outputs
        # overlap the kernels; a consumer takes the delivered frames in order, at most ~one source frame behind
        if E2E_ASYNC_UP:
            calc.updateFrameAsync(pinned[i % RING])   # the ring of pinned source frames is 10 deep: no buffer is reused before its upload ended
        else:
            calc.updateFrame(pinned[i % RING])
        calc.calculateOpticalFlowAsync()
        if not args.no_batch:
            calc.warpFramesBatch(sched[i], hr.BlendedFrame)
        for b in sched[i]:
            if args.no_batch:
                calc.warpFrames(b, hr.BlendedFrame)
            while len(pending) >= POOL - 1:      # never hand a pinned buffer to a second download before its ticket was waited for
                calc.waitDownload(pending.pop(0))
            pending.append(calc.downloadFrameAsync(out_pool[dl_count[0] % POOL]))
            dl_count[0] += 1
        while len(pending) > E2E_DEPTH:
            calc.waitDownload(pending.pop(0))
        return len(sched[i])

    def drain():
        while pending:
            calc.waitDownload(pending.pop(0))

    for i in range(3):  # prime the three input slots (m_frameCount >= 3, HopperRender.cpp:955)
        calc.updateFrameDevice(dev[i % RING])
    calc.synchronize()

    idx = 0
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # sampled from before the warm-up to the end of the end-to-end loops: a short timed region still gets samples
    for _ in range(args.warmup):
        step_device(idx)
        idx += 1
    calc.synchronize()
    barrier()
    launches0 = hr.kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    frames = 0
    host_issue_ms = None
    with torch.cuda.stream(stream):
        e0.record(stream)
        th = time.perf_counter()
        for k in range(args.steps):
            frames += step_device(idx)
            idx += 1
            if k == 3:  # host time to ISSUE a step: the first four steps, before the handle's ring of four flow records makes the host wait for the GPU
                host_issue_ms = (time.perf_counter() - th) * 1e3 / 4
        calc.joinFlow()  # the last flow runs on the handle's flow stream: the end event waits for it too
        e1.record(stream)
    calc.synchronize()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = sum_over_ranks(hr.kernel_launch_count() - launches0)
    total_frames = sum_over_ranks(frames)
    value = total_frames / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, calc, sched[idx - 1], hdr)

    # ---- the same loop at the auto-tuner's lower bound R=5 (SURVEY.md section 8(d): "also report R = 5") ----
    r5 = None
    if args.radius != 5:
        calc.m_opticalFlowSearchRadius = 5
        for _ in range(3):
            step_device(idx)
            idx += 1
        calc.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r5_steps = min(args.steps, 100)
        r5_frames = 0
        with torch.cuda.stream(stream):
            r0.record(stream)
            for _ in range(r5_steps):
                r5_frames += step_device(idx)
                idx += 1
            calc.joinFlow()
            r1.record(stream)
        calc.synchronize()
        r5_ms = max_over_ranks(r0.elapsed_time(r1))
        r5 = {"value": sum_over_ranks(r5_frames) / (r5_ms * 1e-3), "unit": UNIT, "ms_per_step": r5_ms / r5_steps, "steps": r5_steps}
        calc.m_opticalFlowSearchRadius = args.radius
        for _ in range(2):
            step_device(idx)
            idx += 1
        calc.synchronize()

    # ---- per-kernel breakdown (same loop, CUDA events around every kernel class on the handle's stream) ----
    calc.setProfile(True)
    calc.profileReset()
    psteps = min(args.steps, 20)
    pframes = 0
    for _ in range(psteps):
        pframes += step_device(idx)
        idx += 1
    prof = calc.profileRead()
    calc.setProfile(False)

    # ---- end-to-end loop (public blocking API, pinned host buffers) ------------------------------------
    def time_e2e(step_fn, nsteps):
        nonlocal idx
        for _ in range(3):
            step_fn(idx)
            idx += 1
        drain()
        calc.synchronize()
        barrier()
        nframes = 0
        t0 = time.perf_counter()
        for _ in range(nsteps):
            nframes += step_fn(idx)
            idx += 1
        drain()             # every output frame of the timed steps is in host memory
        calc.synchronize()
        barrier()
        wall_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)   # host clock: the region ends when the last byte has landed
        return sum_over_ranks(nframes) / (wall_ms * 1e-3), nframes / nsteps

    esteps = min(args.steps, 100)
    e2e_value, mean_out = time_e2e(step_e2e, esteps)
    e2e_blocking_value, _ = time_e2e(step_e2e_blocking, min(args.steps, 30))

    # ---- link roofline of the end-to-end loop: the same bytes per step (1 frame up, N frames down) over the same pinned
    # buffers on two copy streams, no kernels — what the host link of this box gives all ranks at once ----
    def link_leg(nsteps):
        up, down = torch.cuda.Stream(), torch.cuda.Stream()
        dev_in = torch.empty_like(dev[0])
        dev_out = torch.empty(out_pinned.numel(), dtype=tdt, device="cuda")
        n_out = max(1, int(round(mean_out)))
        for _ in range(2):
            with torch.cuda.stream(up):
                dev_in.copy_(pinned[0], non_blocking=True)
            with torch.cuda.stream(down):
                out_pool[0].copy_(dev_out, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(nsteps):
            with torch.cuda.stream(up):
                dev_in.copy_(pinned[i % RING], non_blocking=True)
            with torch.cuda.stream(down):
                for k in range(n_out):
                    out_pool[(i * n_out + k) % POOL].copy_(dev_out, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        wall = max_over_ranks((time.perf_counter() - t0) * 1e3) * 1e-3
        h2d = sum_over_ranks(nsteps * calc.inputFrameBytes) / wall / 1e9
        d2h = sum_over_ranks(nsteps * n_out * calc.outputFrameBytes) / wall / 1e9
        return {"h2d_gbs": h2d, "d2h_gbs": d2h, "frames_per_s": sum_over_ranks(nsteps * n_out) / wall, "steps": nsteps,
                "what": "concurrent pinned H2D (1 frame) + D2H (N frames) per step on two copy streams, no kernels, all ranks at once"}

    link = link_leg(min(args.steps, 50))
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        pk, pk_kind = peaks()
        hbm_peak = float(pk.get("hbm_gbs", 6650.0))
        warp_ms = prof["ms_warp"] / max(prof["n_warp"], 1)
        blur_ms = max(prof["ms_blur"] / max(prof["n_blur"], 1), 1e-6)
        pack_ms = max(prof["ms_ingest"] / max(prof["n_ingest"], 1), 1e-6)
        search_ms_per_step = prof["ms_search"] / psteps
        n_out_mean = total_frames / world / args.steps
        # SURVEY.md section 8(d): 3F + 4L per output frame (two sources, one output, the flow), times the output frames one
        # launch produces.  The batched launch reads sources and flow once for all of them: its own compulsory traffic is
        # 2F + 4L + N*F, reported beside it (and `traffic` is what ncu saw).
        n_per_launch = 1.0 if args.no_batch else n_out_mean
        warp_bytes = int(alg["warp"] * n_per_launch)
        warp_min_bytes = alg["warp"] if args.no_batch else int(2 * alg["F"] + 4 * alg["L"] + n_out_mean * alg["F"])
        warp_gbs = warp_bytes / (warp_ms * 1e-3) / 1e9
        sad_peak = None
        try:
            sad_peak = hr.microbench_sad_peak(local)
        except Exception as e:  # noqa: BLE001
            print(f"bench.py: SAD microbenchmark failed: {e}", file=sys.stderr)
        absdiff_rate = 3.0 * args.radius * alg["L"] * alg["passes"] / (search_ms_per_step * 1e-3) / 1e9
        step_kernel_ms = (prof["ms_ingest"] + prof["ms_search"] + prof["ms_blur"] + prof["ms_warp"]) / psteps
        line = {
            "metric": metric_name(args.workload), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: {wl['desc']}, R={args.radius}", "search_radius": args.radius, "delta_scalar": 8,
                       "neighbor_scalar": 6, "frame_output": "BlendedFrame", "streams_per_gpu": 1,
                       "flow_overlap": not args.no_overlap,
                       "mean_outputs_per_source_frame": total_frames / world / args.steps,
                       "realtime_factor_vs_144fps": value / world / 144.0,
                       "frames": f"{NFR} distinct frames played back and forth (every consecutive pair is one motion step of the scene)",
                       "l2": f"inputs larger than L2: {NFR} distinct device frames of {alg['F']/1e6:.0f} MB; a step touches ~{(3*alg['F'] + 2*alg['F'] + 6*(alg['L']*4 + alg['F']))/1e6:.0f} MB (126 MB L2)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(calc.inputFrameBytes),
                    "d2h_bytes_per_step": int(round(mean_out * calc.outputFrameBytes)), "steps": esteps,
                    "api": "update_frame (pinned host) + calculate_optical_flow_async + N x (warp_frames + download_frame_async to pinned host) "
                           "+ wait_download; transfers on their own streams overlap the kernels",
                    "blocking_api_value": e2e_blocking_value,
                    "link": link, "link_peak_frames_per_s": link["frames_per_s"], "frac_of_link": e2e_value / link["frames_per_s"]},
            "gpu_launches": int(launches),
            "host_issue_ms_per_step": host_issue_ms,
            "clocks": clocks,
            # the dominant cost of a step is the search ladder (integer-ALU bound: SURVEY.md section 8d)
            "roofline": {"kernel": "search ladder: sadTileKernel (windows 8..2048) + sadCandKernel (windows 4, 2), %d passes per source frame" % alg["passes"],
                         "bound": "int_alu", "achieved": absdiff_rate, "peak": sad_peak, "unit": "G byte-absdiff/s",
                         "frac": (absdiff_rate / sad_peak) if sad_peak else None,
                         "traffic": ncu_traffic(args.workload, "search_pass"),
                         "peak_source": "hrb_microbench_sad_peak: VABSDIFF4.U8.ACC issue rate measured in this run (4 byte-abs-diffs per lane instruction)",
                         "algorithmic_absdiff_per_step": 3 * args.radius * alg["L"] * alg["passes"], "ms_per_step": search_ms_per_step,
                         "note": "achieved = 3 * R * L * passes byte-abs-diffs (SURVEY.md section 8d) / CUDA-event time of the ladder; traffic = DRAM bytes per pass (ncu)"},
            "roofline_warp": {"kernel": "warpKernel = warpFrames, %s" % ("one launch per output frame" if args.no_batch else "one batched launch per source frame (all its output frames)"), "bound": "hbm",
                              "achieved": warp_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": warp_gbs / hbm_peak,
                              "traffic": ncu_traffic(args.workload, "warpKernel"),
                              "peak_source": f"{pk_kind} (MEASURED_PEAKS.json hbm_gbs)", "algorithmic_bytes_per_launch": warp_bytes,
                              "output_frames_per_launch": n_per_launch, "bytes_per_output_frame": alg["warp"],
                              "compulsory_bytes_of_the_batched_launch": warp_min_bytes,
                              "frac_of_compulsory": warp_min_bytes / (warp_ms * 1e-3) / 1e9 / hbm_peak,
                              "avg_launch_ms": warp_ms,
                              "note": "achieved = (3F + 4L per output frame, SURVEY.md section 8d) x output frames per launch / launch time: the HBM rate "
                                      "the reference's one-launch-per-frame form would need for this frame rate; the batched launch shares the source and "
                                      "flow reads, so its own compulsory bytes (and the DRAM traffic ncu sees) are lower"},
            "roofline_blur": {"kernel": "blurFlowCellKernel", "bound": "hbm", "achieved": alg["blur"] / (blur_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                              "frac": alg["blur"] / (blur_ms * 1e-3) / 1e9 / hbm_peak, "traffic": ncu_traffic(args.workload, "blurFlowCellKernel"),
                              "algorithmic_bytes_per_launch": alg["blur"], "avg_launch_ms": blur_ms},
            "roofline_pack": {"kernel": "packPlanarKernel (ingest: raw frame -> 8-bit search planes)", "bound": "hbm",
                              "achieved": alg["F"] / (pack_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": alg["F"] / (pack_ms * 1e-3) / 1e9 / hbm_peak,
                              "traffic": ncu_traffic(args.workload, "packPlanarKernel"), "algorithmic_bytes_per_launch": alg["F"], "avg_launch_ms": pack_ms},
            "search_radius_5": r5,
            "breakdown_ms_per_step": {"ingest": prof["ms_ingest"] / psteps, "search": search_ms_per_step, "blur": prof["ms_blur"] / psteps,
                                      "warp": prof["ms_warp"] / psteps, "kernels_total": step_kernel_ms},
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline(wl)
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
            # the reference's own OpenCL kernels on this same GPU (BASELINE.md B3): the like-for-like numbers are
            # e2e.blocking_api_value vs its value (both blocking APIs) and breakdown_ms_per_step.search vs its ofc_ms
            line["reference_opencl_b200"] = reference_opencl_same_gpu(wl, radius=args.radius)
        emit(line)
    calc.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
