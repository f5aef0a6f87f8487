#!/usr/bin/env python
"""flow_batch_bench.py — ms per round of S flows on one GPU: S lone handles against one FlowBatch of S handles.

Workloads: cfg1 (1920x1080 NV12, max_calc_res 270: a 480x270 flow) and cfg2 (max_calc_res 540: a 960x540 flow) at
S = 1, 4, 16 and 64 streams, and cfg3 (3840x2160 P010 at full resolution) at S = 8 for information; R = 16, deltaScalar
8, neighborScalar 6.  Every stream has its own seeded frames (a shared moving scene, shifted in value per stream), resident
on the device.  A round ingests the next frame on every stream (updateFrameDevice, then a synchronise, untimed) and then
computes one flow per stream:
  (A) every handle calls calculateOpticalFlowAsync on its own streams from this thread, as bench.py --streams-per-gpu does;
  (B) one FlowBatch over another S handles calls calculateOpticalFlowAsync once.
Each arm is timed by the host clock from the first enqueue to the end of a device synchronise of all its handles; the
arms alternate round by round in one process, after warm-up.  Reported per workload, one JSON line: median and mean ms
per round, flows/s, kernel launches per round (hrb_kernel_launch_count), whether the last flows of the two arms are bit
identical, and the device name and power limit read in the same run.

    python tools/flow_batch_bench.py [--rounds 30] [--warmup 3] [--only cfg1]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

R = 16
WORKLOADS = [("cfg1", 1920, 1080, False, 270, (1, 4, 16, 64)), ("cfg2", 1920, 1080, False, 540, (1, 4, 16, 64)),
             ("cfg3", 3840, 2160, True, 2160, (8,))]


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return [dict(zip(("index", "name", "power_limit"), (x.strip() for x in line.split(",")))) for line in out.strip().splitlines()]
    except Exception as e:  # the numbers stay meaningful with the torch device name below
        return [{"error": str(e)}]


def stream_frames(torch, synth, W, H, hdr, S):
    """[stream][3] device frames: three frames of a moving scene, shifted in value by a seeded amount per stream."""
    base = [torch.from_numpy(synth.make_frame(W, H, t, synth.SEED_BASE + 61, hdr).view(np.int16 if hdr else np.uint8)).cuda() for t in range(3)]
    rng = np.random.default_rng(2024)
    out = []
    for s in range(S):
        d = int(rng.integers(1, 200))
        if hdr:  # P010: 10 significant bits in the MSBs
            out.append([(((f.view(torch.int16).to(torch.int32) & 0xFFFF) + (d << 6)) & 0xFFC0).to(torch.int16) for f in base])
        else:
            out.append([((f.to(torch.int32) + d) & 0xFF).to(torch.uint8) for f in base])
    return out


def run(name, W, H, hdr, maxres, S, rounds, warmup, torch, hr, synth):
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    frames = stream_frames(torch, synth, W, H, hdr, S)
    arms = {}
    for arm in ("A", "B"):
        calcs = [cls(H, W, 0, 0, 8, 6, 0.0, 255.0, maxres) for _ in range(S)]
        for c in calcs:
            c.m_opticalFlowSearchRadius = R
        arms[arm] = calcs
    batch = hr.FlowBatch(arms["B"])
    t = {"A": [], "B": []}
    launches = {"A": 0, "B": 0}
    for r in range(warmup + rounds):
        for arm in ("A", "B") if r % 2 == 0 else ("B", "A"):
            calcs = arms[arm]
            for s, c in enumerate(calcs):
                c.updateFrameDevice(frames[s][r % 3])
            for c in calcs:
                c.synchronize()
            n0 = hr.kernel_launch_count()
            t0 = time.perf_counter()
            if arm == "A":
                for c in calcs:
                    c.calculateOpticalFlowAsync()
            else:
                batch.calculateOpticalFlowAsync()
            for c in calcs:
                c.synchronize()
            dt = time.perf_counter() - t0
            launches[arm] = hr.kernel_launch_count() - n0
            if r >= warmup:
                t[arm].append(dt * 1e3)
    same = all(np.array_equal(a.readFlow(latest=True), b.readFlow(latest=True)) and a.m_totalFrameDelta == b.m_totalFrameDelta
               for a, b in zip(arms["A"], arms["B"]))
    nonzero = any(np.any(b.readFlow(latest=True)) for b in arms["B"])
    g = arms["A"][0]
    res = dict(workload=name, frame=f"{W}x{H}", format="P010" if hdr else "NV12", max_calc_res=maxres,
               flow=f"{g.m_opticalFlowFrameWidth}x{g.m_opticalFlowFrameHeight}", R=R, streams=S, rounds=rounds)
    for arm, label in (("A", "lone"), ("B", "batch")):
        med = statistics.median(t[arm])
        res[f"{label}_ms_per_round"] = round(med, 4)
        res[f"{label}_ms_per_round_mean"] = round(statistics.mean(t[arm]), 4)
        res[f"{label}_flows_per_s"] = round(S / med * 1e3, 1)
        res[f"{label}_launches_per_round"] = launches[arm]
    res["batch_speedup"] = round(res["lone_ms_per_round"] / res["batch_ms_per_round"], 3)
    res["bit_identical"] = bool(same)
    res["flow_nonzero"] = bool(nonzero)
    batch.close()
    for calcs in arms.values():
        for c in calcs:
            c.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", default=None, help="run only this workload (cfg1, cfg2 or cfg3)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("flow_batch_bench.py measures on a CUDA device; none is available")
    import hopperrender_b200 as hr
    from hopperrender_b200 import synth
    info = device_info()
    for name, W, H, hdr, maxres, ss in WORKLOADS:
        if args.only and name != args.only:
            continue
        for S in ss:
            res = run(name, W, H, hdr, maxres, S, args.rounds, args.warmup, torch, hr, synth)
            res["device"] = torch.cuda.get_device_name(0)
            res["power_limit"] = info[0].get("power_limit") if info else None
            print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
