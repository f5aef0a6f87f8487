#!/usr/bin/env python
"""delivery_bench.py — ms per source frame of frame-rate conversion with and without the scene-change rule.

Three handles hold the same frames; each source frame goes through one arm on each, the arms alternating (in rotating
order) frame by frame in one process after warm-up.  Source frames are device planes (update_frame_planes), outputs go to
pitched device surfaces:
  (a) calculate_optical_flow_async + warp_frames_to: today's fast path, with no scene-change rule;
  (b) the same plus the rule on the host: get_state after the flow (a wait for the whole ladder), then warp_frames_to or
      copy_frame_to — what a host has to do without the library's delivery loop;
  (c) hrb_delivery_step_to: the rule decided on the GPU right after pass 0 of the flow.
A step is timed by the host clock from its first enqueue to the end of hrb_ofc_synchronize.  Six distinct frames are played
back and forth (0 1 2 3 4 5 4 3 2 1 ...), as bench.py does, so that the inputs of a run exceed the 126 MB L2 at cfg3.  The
auto-tuner is off (radius 16) in every arm.  The outputs of the three arms are compared byte for byte after every step.
Workloads: cfg3 (3840x2160 P010, full-resolution flow, 23.976 -> 144 fps) and cfg1 (1920x1080 NV12, 270p flow,
23.976 -> 60 fps), blended output.

Prints one JSON line with the device name and power limit read in the same run.

    python tools/delivery_bench.py [--frames 40] [--warmup 8] [--only cfg3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from collections import deque

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

R = 16
SRC = 417083
WORKLOADS = {"cfg3": (3840, 2160, True, 2160, 69444), "cfg1": (1920, 1080, False, 270, 166667)}
ARMS = ("a_no_rule", "b_host_rule", "c_delivery")


def device_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    name, power = (x.strip() for x in out.split(","))
    return name, power


def stats(ms):
    q = np.percentile(ms, [10, 90])
    return {"median_ms": round(statistics.median(ms), 4), "p10_ms": round(float(q[0]), 4), "p90_ms": round(float(q[1]), 4), "n": len(ms)}


def host_rule(hist, threshold=200):
    """replay.DeliveryLoop._scene_change on (frame, delta) entries."""
    n = len(hist)
    if n < 3:
        return False
    count = min(n - 2, 10)
    avg = sum(hist[n - 2 - i][1] for i in range(count)) // count
    cur, nxt = hist[n - 2][1], hist[n - 1][1]
    d1, d2 = cur - avg, cur - nxt
    return d1 >= threshold and d1 > 0 and d2 >= threshold and d2 > 0


def run(name, args):
    import torch

    import hopperrender_b200 as hr
    from hopperrender_b200 import replay, synth
    W, H, hdr, maxres, target = WORKLOADS[name]
    dt = torch.int16 if hdr else torch.uint8
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    n_src = args.warmup + args.frames
    sched = replay.output_schedule(n_src, target, SRC)
    src = []
    for t in range(6):
        f = synth.make_frame(W, H, t, synth.SEED_BASE + 5, hdr)
        full = torch.from_numpy(f.view(np.int16) if hdr else f).cuda().reshape(H + H // 2, W)
        src.append((full[:H], full[H:]))
    order = list(range(6)) + list(range(4, 0, -1))

    def surfaces(n):
        return [(torch.zeros((H, W + 128), dtype=dt, device="cuda")[:, :W], torch.zeros((H // 2, W + 256), dtype=dt, device="cuda")[:, :W]) for _ in range(n)]

    def make():
        c = cls(H, W, 0, 0, 8, 6, 0.0, 255.0, maxres)
        c.m_opticalFlowSearchRadius = R
        return c
    calcs = {a: make() for a in ARMS}
    dst = {a: surfaces(8) for a in ARMS}
    delivery = hr.Delivery(calcs["c_delivery"], source_frame_time=SRC, target_frame_time=target, frame_output=hr.BlendedFrame, auto_adjust=False)
    hist = deque()
    frames_in_3s = int(3.0 * 10000000.0 / SRC)

    def step_a(c, i, outs):
        c.updateFramePlanes(*src[order[i % len(order)]])
        if i + 1 >= 3:
            c.calculateOpticalFlowAsync()
            c.warpFramesTo(sched[i], hr.BlendedFrame, outs)
        else:
            for o in outs:
                c.copyFrameTo(o)

    def step_b(c, i, outs):
        c.updateFramePlanes(*src[order[i % len(order)]])
        scene = False
        if i + 1 >= 3:
            c.calculateOpticalFlowAsync()
            s = c._state()  # hrb_ofc_get_state: waits for the flow
            hist.append((s.frame_count, int(s.total_frame_delta)))
            while hist and s.frame_count - hist[0][0] > frames_in_3s:
                hist.popleft()
            scene = host_rule(hist)
        if i + 1 >= 3 and not scene:
            c.warpFramesTo(sched[i], hr.BlendedFrame, outs)
        else:
            for o in outs:
                c.copyFrameTo(o)

    def step_c(c, i, outs):
        infos = delivery.deliver_to(*src[order[i % len(order)]], outs)
        assert [f["blend"] for f in infos] == sched[i]

    steps = {"a_no_rule": step_a, "b_host_rule": step_b, "c_delivery": step_c}
    ms = {a: [] for a in ARMS}
    same = True
    for i in range(n_src):
        n = len(sched[i])
        for j in range(len(ARMS)):
            arm = ARMS[(i + j) % len(ARMS)]
            c = calcs[arm]
            t0 = time.perf_counter()
            steps[arm](c, i, dst[arm][:n])
            c.synchronize()
            if i >= args.warmup:
                ms[arm].append((time.perf_counter() - t0) * 1e3)
        for k in range(n):
            for a in ARMS[1:]:
                same = same and all(torch.equal(x, y) for x, y in zip(dst[a][k], dst[ARMS[0]][k]))
    delivery.close()
    return {"workload": name, "desc": f"{W}x{H} {'P010' if hdr else 'NV12'}, flow max_calc_res {maxres}, 23.976 -> {1e7 / target:.0f} fps, R {R}",
            "arms": {a: stats(ms[a]) for a in ARMS}, "outputs_identical": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("delivery_bench.py measures on a GPU; none is available")
    name, power = device_info()
    res = [run(w, args) for w in (["cfg3", "cfg1"] if not args.only else [args.only])]
    print(json.dumps({"device": name, "power_limit": power, "results": res}))


if __name__ == "__main__":
    main()
