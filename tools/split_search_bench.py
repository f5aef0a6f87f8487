#!/usr/bin/env python
"""split_search_bench.py — ms per flow of one 8K stream whose search is split over 1, 2, 4 and 8 GPUs (SplitSearch).

Workload: 7680x4320 P010, full-resolution flow, R = 16, deltaScalar 8, neighborScalar 6, three seeded source frames
(hopperrender_b200.synth) resident on every device; the search pair is frames 1 and 2 of the moving scene.  For each
shard count n (capped at the device count, shard k on device k) the group's calculateOpticalFlow and a lone handle's on
device 0 are timed alternately in the same loop, host clock around the blocking call (which ends in a device
synchronise), after warm-up.  Reported: mean / median ms per flow of both, their ratio, the replicated / sharded pass
counts of the ladder, whether the last flow of every shard equals the lone handle's bit for bit, and that this flow is
not zero.  One JSON line on stdout; device name and power limit read in the same run.

    python tools/split_search_bench.py [--steps 50] [--warmup 5]
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

W, H, R, ALIGN = 7680, 4320, 16, 128


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return [dict(zip(("index", "name", "power_limit"), (x.strip() for x in line.split(",")))) for line in out.strip().splitlines()]
    except Exception as e:  # the numbers stay meaningful with the torch device name below
        return [{"error": str(e)}]


def pass_counts(lh, lw):
    m = max(lw, lh)
    ws = m if m and not (m & (m - 1)) else 1 << m.bit_length()
    ws //= 2
    wss = [ws >> i for i in range(int(np.log2(ws)))]
    return {"replicated": 2 * sum(w > ALIGN for w in wss), "sharded": 2 * sum(w <= ALIGN for w in wss)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch

    import hopperrender_b200 as hr
    from hopperrender_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("split_search_bench: no CUDA device (the library has no CPU fallback)")
    ndev = torch.cuda.device_count()
    frames = [synth.make_frame(W, H, t, synth.SEED_BASE + 5, True) for t in range(3)]  # three distinct frames
    dev_frames = {d: [torch.from_numpy(f.view(np.int16)).to(f"cuda:{d}") for f in frames] for d in range(min(ndev, 8))}

    def calc(d):
        c = hr.OpticalFlowCalcHDR(H, W, 0, 0, 8, 6, 0.0, 255.0, H, d)
        c.m_opticalFlowSearchRadius = R
        for f in dev_frames[d]:   # frames 0, 1, 2: the search pair is (1, 2), a moving scene
            c.updateFrameDevice(f)
        torch.cuda.synchronize(d)
        return c

    lone = calc(0)
    results, not_measured = [], [n for n in (2, 4, 8) if n > ndev]
    for n in [n for n in (1, 2, 4, 8) if n <= ndev]:
        shards = [calc(k) for k in range(n)]
        grp = hr.SplitSearch(shards)
        for _ in range(args.warmup):
            grp.calculateOpticalFlow()
            lone.calculateOpticalFlow()
        tg, tl = [], []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            grp.calculateOpticalFlow()
            t1 = time.perf_counter()
            lone.calculateOpticalFlow()
            t2 = time.perf_counter()
            tg.append((t1 - t0) * 1e3)
            tl.append((t2 - t1) * 1e3)
        want = (lone.readOffsetArray(), lone.readFlow(latest=True), lone.readFlowPeak()[1], lone.m_totalFrameDelta)
        moving = bool(np.any(want[1]))
        same = all(np.array_equal(s.readOffsetArray(), want[0]) and np.array_equal(s.readFlow(latest=True), want[1])
                   and s.readFlowPeak()[1] == want[2] and s.m_totalFrameDelta == want[3] for s in shards)
        results.append(dict(shards=n, devices=list(range(n)), stripes=[grp.stripe(k) for k in range(n)],
                            group_ms_mean=round(statistics.mean(tg), 4), group_ms_median=round(statistics.median(tg), 4),
                            lone_ms_mean=round(statistics.mean(tl), 4), lone_ms_median=round(statistics.median(tl), 4),
                            speedup_median=round(statistics.median(tl) / statistics.median(tg), 3), bit_identical=bool(same), flow_nonzero=moving))
        grp.close()
        for s in shards:
            s.close()
    lone.close()
    out = dict(workload=f"{W}x{H} P010, full-resolution flow, R {R}", steps=args.steps, warmup=args.warmup,
               timing="host clock around the blocking calculate, group and lone handle alternated",
               passes=pass_counts(H, W), device_count=ndev, torch_device=torch.cuda.get_device_name(0), gpus=device_info(),
               results=results, not_measured=[f"{n} shards: {ndev} device(s)" for n in not_measured])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
