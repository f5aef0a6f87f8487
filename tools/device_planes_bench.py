#!/usr/bin/env python
"""device_planes_bench.py — ms per source frame of a GPU pipeline that keeps frames in pitched decoder / encoder surfaces.

Two handles hold the same seeded frames; each source frame goes through one arm on each, the arms alternating frame by
frame in one process after warm-up.  A source frame arrives as a pitched two-plane surface (luma pitch and chroma pitch
padded, chroma in its own allocation) and its output frames must land in such surfaces:
  (a) today's zero-copy caller: cudaMemcpy2DAsync of both planes into a contiguous frame, update_frame_device,
      calculate_optical_flow_async, warp_frames_batch into the output ring, then two cudaMemcpy2DAsync per output frame
      (luma, chroma) from the ring slot into the caller's surface;
  (b) update_frame_planes, calculate_optical_flow_async, warp_frames_to straight into the caller's surfaces.
Everything runs on the handle's compute stream (hrb_ofc_stream); a step is timed by the host clock from its first
enqueue to the end of hrb_ofc_synchronize.  Workloads: cfg3 (3840x2160 P010, full-resolution flow, 23.976 -> 144 fps:
6 outputs per source frame) and cfg1 (1920x1080 NV12, 270p flow, 24 -> 60 fps: 2 or 3), R 16, blended output.

--ring-profile instead runs the ring path alone (update_frame_device, calculate_optical_flow_async, warp_frames_batch)
with hrb_ofc_profile on and reports ms_ingest and ms_warp per source frame (CUDA events around the kernels).

Prints one JSON line with the device name and power limit read in the same run.

    python tools/device_planes_bench.py [--frames 40] [--warmup 5] [--only cfg3] [--ring-profile]
"""
import argparse
import ctypes as C
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
WORKLOADS = {"cfg3": (3840, 2160, True, 2160, 69444), "cfg1": (1920, 1080, False, 270, 166667)}
PAD_Y, PAD_UV = 256, 512  # bytes of row padding of the pitched surfaces
D2D = 3                   # cudaMemcpyDeviceToDevice


def device_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    name, power = (x.strip() for x in out.split(","))
    return name, power


def stats(ms):
    q = np.percentile(ms, [10, 90])
    return {"median_ms": round(statistics.median(ms), 4), "p10_ms": round(float(q[0]), 4), "p90_ms": round(float(q[1]), 4), "n": len(ms)}


def run(name, args, cudart):
    import torch

    import hopperrender_b200 as hr
    from hopperrender_b200 import replay, synth
    W, H, hdr, maxres, target = WORKLOADS[name]
    es = 2 if hdr else 1
    dt = torch.int16 if hdr else torch.uint8
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    n_src = args.warmup + args.frames
    sched = replay.output_schedule(n_src + 8, target, replay.SOURCE_FRAME_TIME_23976)
    frames = [synth.make_frame(W, H, t, synth.SEED_BASE + 5, hdr) for t in range(4)]
    yp, up = W * es + PAD_Y, W * es + PAD_UV  # byte pitches

    def pitched():
        y = torch.empty(H * yp // es, dtype=dt, device="cuda").as_strided((H, W), (yp // es, 1))
        uv = torch.empty((H // 2) * up // es, dtype=dt, device="cuda").as_strided((H // 2, W), (up // es, 1))
        return y, uv
    src = []
    for f in frames:
        y, uv = pitched()
        t = torch.from_numpy(f.view(np.int16) if hdr else f).cuda().reshape(H + H // 2, W)
        y.copy_(t[:H])
        uv.copy_(t[H:])
        src.append((y, uv))
    dst = [pitched() for _ in range(8)]
    dev = [torch.from_numpy(f.view(np.int16) if hdr else f).cuda() for f in frames]

    def make():
        c = cls(H, W, 0, 0, 8, 6, 0.0, 255.0, maxres)
        c.m_opticalFlowSearchRadius = R
        return c
    ca, cb = make(), make()
    for c in (ca, cb):  # the same history on both: two frames and a flow
        c.updateFrameDevice(dev[2])
        c.updateFrameDevice(dev[3])
        c.calculateOpticalFlow()
    contig = torch.empty((H + H // 2) * W, dtype=dt, device="cuda")
    # the ring slots of (a): every warp, then a download, advances the ring by one; after 16 the cursor is back at slot 0,
    # and without downloads warp_frames_batch writes slots 0 .. n-1 every time
    host = np.zeros(ca.outputFrameBytes, np.uint8)
    slots = []
    for _ in range(16):
        ca.warpFrames(0.0, 0)
        slots.append(ca.outputDevicePtr())
        ca.downloadFrame(host)
    so = ca.m_outputStride * es
    sa = C.c_void_p(ca.streamHandle())

    def copy2d(d, dp, s, sp, rows):
        rc = cudart.cudaMemcpy2DAsync(C.c_void_p(d), C.c_size_t(dp), C.c_void_p(s), C.c_size_t(sp), C.c_size_t(W * es), C.c_size_t(rows), D2D, sa)
        assert rc == 0, rc

    def step_a(i):
        y, uv = src[i % 4]
        copy2d(contig.data_ptr(), W * es, y.data_ptr(), yp, H)
        copy2d(contig.data_ptr() + H * W * es, W * es, uv.data_ptr(), up, H // 2)
        ca.updateFrameDevice(contig)
        if i >= 1:
            ca.calculateOpticalFlowAsync()
            ca.warpFramesBatch(sched[i], hr.BlendedFrame)
            for k in range(len(sched[i])):
                copy2d(dst[k][0].data_ptr(), yp, slots[k], so, H)
                copy2d(dst[k][1].data_ptr(), up, slots[k] + H * so, so, H // 2)
        ca.synchronize()

    def step_b(i):
        cb.updateFramePlanes(*src[i % 4])
        if i >= 1:
            cb.calculateOpticalFlowAsync()
            cb.warpFramesTo(sched[i], hr.BlendedFrame, dst[:len(sched[i])])
        cb.synchronize()

    torch.cuda.synchronize()
    if args.ring_profile:
        ca.setProfile(True)
        for i in range(n_src):
            if i == args.warmup:
                ca.profileReset()
            ca.updateFrameDevice(dev[i % 4])
            ca.calculateOpticalFlowAsync()
            ca.warpFramesBatch(sched[i], hr.BlendedFrame)
            ca.synchronize()
        p = ca.profileRead()
        n = args.frames
        return {"workload": name, "ms_ingest_per_frame": round(p["ms_ingest"] / n, 4), "ms_warp_per_frame": round(p["ms_warp"] / n, 4),
                "n_ingest": p["n_ingest"], "n_warp": p["n_warp"], "frames": n}
    ta, tb = [], []
    for i in range(n_src):
        for step, out in ((step_a, ta), (step_b, tb)) if i % 2 == 0 else ((step_b, tb), (step_a, ta)):
            t0 = time.perf_counter()
            step(i)
            if i >= args.warmup:
                out.append((time.perf_counter() - t0) * 1e3)
    # both arms warped the same frames from the same flow: the last outputs must agree
    ts = [1 / 6, 0.5, 5 / 6]
    ca.warpFramesBatch(ts, hr.BlendedFrame)
    for k in range(len(ts)):
        copy2d(dst[k][0].data_ptr(), yp, slots[k], so, H)
    ca.synchronize()
    a_last = [d[0].cpu() for d in dst[:len(ts)]]
    cb.warpFramesTo(ts, hr.BlendedFrame, dst[:len(ts)])
    cb.synchronize()
    b_last = [d[0].cpu() for d in dst[:len(ts)]]
    same = all(bool(torch.equal(x, y)) for x, y in zip(a_last, b_last))
    ca.close()
    cb.close()
    outs = [len(sched[i]) for i in range(args.warmup, n_src)]
    return {"workload": name, "size": f"{W}x{H} {'P010' if hdr else 'NV12'}", "outputs_per_source_frame": round(statistics.mean(outs), 3),
            "a_repack_and_ring_copies": stats(ta), "b_planes": stats(tb), "median_speedup": round(statistics.median(ta) / statistics.median(tb), 4),
            "last_outputs_identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    ap.add_argument("--ring-profile", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("device_planes_bench: no CUDA device")
    cudart = C.CDLL("libcudart.so.12")  # the CUDA runtime torch has loaded
    cudart.cudaMemcpy2DAsync.restype = C.c_int
    gpu, power = device_info()
    results = [run(n, args, cudart) for n in (["cfg3", "cfg1"] if not args.only else [args.only])]
    print(json.dumps({"tool": "device_planes_bench", "gpu": gpu, "power_limit": power, "mode": "ring_profile" if args.ring_profile else "arms",
                      "results": results}))


if __name__ == "__main__":
    main()
