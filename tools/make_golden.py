#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE ITSELF (oracle/_ref: the unmodified HopperRender host
classes and OpenCL kernel strings) on an OpenCL device.  Run on the GPU box, where the NVIDIA driver's OpenCL
implementation executes the reference's kernels on the B200 (32-wide lock-step warps = the semantics the
reference's barrier-free reduction relies on):

    gpurun -- 'python tools/make_golden.py gpurun_out/golden'

Each case is two files: <case>.npz holds the input frames and, per search pass, the window sums / winning layers at
the window representatives and the offset array, then the blurred flow and m_totalFrameDelta; <case>.outputs.npz
holds the output frames.  tests/test_oracle_golden.py replays the same inputs through the CPU oracle and compares.
"""
import json
import os
import sys
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hopperrender_b200 import synth  # noqa: E402

# name: hdr, W, H, maxres, inS, outS, R, ds, ns, black, white, kind
CASES = {
    "sdr_64x48_r5_scene": (False, 64, 48, 270, 0, 0, 5, 8, 6, 0.0, 255.0, "scene"),
    "hdr_130x70_r16_random_strided": (True, 130, 70, 270, 192, 160, 16, 8, 6, 0.0, 255.0, "random"),
    "sdr_258x146_rs1_r11_scene": (False, 258, 146, 73, 272, 0, 11, 8, 6, 16.0, 235.0, "scene"),
    "hdr_384x224_rs2_r16_scene": (True, 384, 224, 56, 0, 0, 16, 8, 6, 0.0, 255.0, "scene"),
    "sdr_192x128_r16_identical": (False, 192, 128, 270, 0, 0, 16, 8, 6, 0.0, 255.0, "identical"),
    "sdr_320x200_r9_ramp": (False, 320, 200, 270, 0, 0, 9, 8, 6, 0.0, 255.0, "ramp"),
    "sdr_160x160_r16_random_wrap": (False, 160, 160, 270, 0, 0, 16, 12, 0, 0.0, 255.0, "random"),
    "hdr_256x160_r6_scene_levels": (True, 256, 160, 270, 0, 272, 6, 4, 10, 12.0, 230.5, "scene"),
}
# the larger cases keep only these outputs (fixture size)
KEEP_BIG = {"warp_m2_t0.1667", "warp_m2_t0.5000", "warp_m3_t0.4000", "warp_m6_t0.4000", "copy"}
WARPS = [(0.0, 2), (1.0 / 6.0, 2), (0.5, 2), (0.4, 0), (0.4, 1), (0.4, 3), (0.4, 4), (0.4, 5), (0.4, 6), (1.0, 2)]


def make_frames(kind, W, H, hdr, stride, n, seed):
    if kind == "scene":
        return [synth.make_frame(W, H, t, synth.SEED_BASE + seed, hdr, stride) for t in range(n)]
    if kind == "random":
        return [synth.make_random_frame(W, H, 1000 + seed + t, hdr, stride) for t in range(n)]
    if kind == "identical":
        f = synth.make_frame(W, H, 0, synth.SEED_BASE + seed, hdr, stride)
        return [f.copy() for _ in range(n)]
    if kind == "ramp":
        return [synth.make_ramp_frame(W, H, 5 * t, hdr, stride) for t in range(n)]
    raise ValueError(kind)


def run_case(calc_factory, name, spec, with_outputs=True):
    """Drive one calculator (reference or oracle) through the case; returns a dict of arrays."""
    hdr, W, H, maxres, inS, outS, R, ds, ns, black, white, kind = spec
    frames = make_frames(kind, W, H, hdr, inS or None, 4, sum(map(ord, name)) % 97)
    c = calc_factory(H, W, inS, outS, ds, ns, black, white, maxres, hdr)
    c.setParams(searchRadius=R)
    c.enableTaps(True)
    out = {"spec": np.array(json.dumps(spec))}
    for i, f in enumerate(frames):
        out[f"frame{i}"] = f
    dt = np.uint16 if hdr else np.uint8
    S = outS or W
    for f in frames[:3]:
        c.updateFrame(f)
    c.calculateOpticalFlow()
    out["num_passes"] = np.array(c.numPasses())
    for p in range(c.numPasses()):
        info = c.passInfo(p)
        ws = info["windowSize"]
        out[f"pass{p}_info"] = np.array([ws, info["iteration"], info["step"]])
        out[f"pass{p}_sums"] = c.readPassSums(p, R)[:, ::ws, ::ws].copy()
        out[f"pass{p}_layers"] = c.readPassLayers(p)[::ws, ::ws].copy()
        out[f"pass{p}_offsets"] = c.readPassOffsets(p)
    out["offset_array"] = c.readOffsetArray()
    out["flow_first"] = c.readFlow(latest=True)
    out["total_frame_delta_first"] = np.array(c.state().totalFrameDelta, np.uint32)
    c.updateFrame(frames[3])
    c.calculateOpticalFlow()
    out["flow_second"] = c.readFlow(latest=True)
    out["total_frame_delta_second"] = np.array(c.state().totalFrameDelta, np.uint32)
    if with_outputs:
        for t, mode in WARPS:
            if W * H > 30000 and f"warp_m{mode}_t{t:.4f}" not in KEEP_BIG:
                continue
            c.warpFrames(t, mode)
            o = np.zeros(c.outputFrameBytes // dt().itemsize, dt)
            c.downloadFrame(o)
            out[f"warp_m{mode}_t{t:.4f}"] = o.reshape(-1, S)[:, :W].copy()
        c.copyFrame()
        o = np.zeros(c.outputFrameBytes // dt().itemsize, dt)
        c.downloadFrame(o)
        out["copy"] = o.reshape(-1, S)[:, :W].copy()
    st = c.state()
    out["geometry"] = np.array([st.resScalar, st.flowWidth, st.flowHeight])
    c.close()
    return out


def _savez_lzma(path, arrays):
    """np.savez with LZMA members (np.load reads them like any .npz)."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for k, a in arrays.items():
            with z.open(k + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


def save_case(dst, name, res):
    """Writes <name>.npz and <name>.outputs.npz (the output frames): split and LZMA-compressed, every file stays
    below 1 MB.  Returns the bytes written."""
    outputs = {k for k in res if k.startswith("warp_") or k == "copy"}
    paths = [os.path.join(dst, name + ".npz"), os.path.join(dst, name + ".outputs.npz")]
    _savez_lzma(paths[0], {k: v for k, v in res.items() if k not in outputs})
    _savez_lzma(paths[1], {k: v for k, v in res.items() if k in outputs})
    return sum(os.path.getsize(p) for p in paths)


def main():
    from oracle import RefCalc
    dst = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden")
    os.makedirs(dst, exist_ok=True)
    probe = RefCalc(64, 64, 0, 0, 8, 6, 0.0, 255.0, 270, False)
    manifest = {"device": probe.deviceName(), "opencl_library": probe.openclLibrary(), "cases": {}}
    probe.close()
    for name, spec in CASES.items():
        res = run_case(lambda *a: RefCalc(*a), name, spec)
        manifest["cases"][name] = {"bytes": save_case(dst, name, res), "passes": int(res["num_passes"])}
        print(name, manifest["cases"][name], flush=True)
    with open(os.path.join(dst, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print(json.dumps(manifest))


if __name__ == "__main__":
    main()
