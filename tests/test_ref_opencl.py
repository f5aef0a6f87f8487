"""Three-way parity on the GPU: the REFERENCE ITSELF (oracle/_ref = unmodified HopperRender host classes + OpenCL kernel
strings, executed by the NVIDIA OpenCL driver on the B200) vs the CPU oracle vs the CUDA path.

test_reference_opencl_vs_oracle_vs_cuda runs the reference live; it is skipped where oracle/_ref is not built (it needs
the HopperRender sources, see oracle/README.md) or no OpenCL device is reachable.

test_recorded_reference_vs_oracle_vs_cuda needs nothing outside the repository: the reference's side is what it computed
on a B200, recorded in tests/golden by tools/make_golden.py (MANIFEST.json names the device).  Search ladder pass by pass
(window sums, winning layers, offsets), blurred flow and m_totalFrameDelta are bit-exact.  Where the reference's offsets
outgrow the frame (only on the random-noise cases), its single-reflection mirror reads outside the plane (undefined,
SURVEY.md A.9): the windows that stay inside are compared, and the comparison of the search stops at that pass (the states
diverge from there on).  Output frames, all warped with the reference's flow: CUDA == oracle, and both within +-1 LSB of
the reference (8-bit SDR, 10-bit HDR)."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, make_pair, oob_windows, out_array
from test_oracle_golden import CASE_IDS, FILES, load_case

sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden import WARPS  # noqa: E402  (the exact (blendingScalar, mode) pairs the reference was driven with)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref_cls():
    from oracle import RefCalc, ref_available
    if not ref_available():
        pytest.skip("oracle/_ref (reference on OpenCL) not available on this machine")
    return RefCalc


CASES = [
    (False, 64, 48, 270, 0, 5, "scene"),
    (True, 130, 70, 270, 192, 16, "random"),
    (False, 258, 146, 73, 272, 11, "scene"),
    (True, 512, 288, 72, 0, 16, "scene"),
    (False, 640, 360, 360, 0, 16, "scene"),
    (True, 960, 540, 540, 0, 8, "scene"),
]


@pytest.mark.parametrize("hdr,W,H,maxres,inS,R,kind", CASES)
def test_reference_opencl_vs_oracle_vs_cuda(synth, ref_cls, hdr, W, H, maxres, inS, R, kind):
    from test_gpu_parity import frames
    g, o = make_pair(hdr, H, W, inS, 0, maxres=maxres, R=R)
    r = ref_cls(H, W, inS, 0, 8, 6, 0.0, 255.0, maxres, hdr)
    r.setParams(searchRadius=R)
    for c in (o, r):
        c.enableTaps(True)
    g.setTapMode(True)
    fs = frames(synth, W, H, hdr, 4, inS or None, kind)
    for fr in fs[:3]:
        for c in (g, o, r):
            c.updateFrame(fr)
    for c in (g, o, r):
        c.calculateOpticalFlow()
    assert r.numPasses() == o.numPasses() == g.numPasses()
    st = o.state()
    left_frame = False
    for p in range(r.numPasses()):
        info = r.passInfo(p)
        ws = info["windowSize"]
        assert info == o.passInfo(p)
        s_ref = r.readPassSums(p, R)[:, ::ws, ::ws]
        if kind == "random":
            # tiny noise frames: offsets outgrow the frame and the reference reads outside the plane (undefined);
            # compare the windows that stay inside, and stop once one did not (the states diverge from there on)
            before = r.readPassOffsets(p - 1) if p else np.zeros_like(r.readPassOffsets(0))
            bad = oob_windows(before, ws, R, info["step"], W, H, st.resScalar)
            assert np.array_equal(s_ref[~bad], o.readPassSums(p, R)[:, ::ws, ::ws][~bad])
            assert np.array_equal(s_ref[~bad], g.readPassSums(p, R)[~bad])
            if bad.any():
                left_frame = True
                break
        assert np.array_equal(s_ref, o.readPassSums(p, R)[:, ::ws, ::ws]), f"pass {p}: oracle sums != reference"
        assert np.array_equal(s_ref, g.readPassSums(p, R)), f"pass {p}: CUDA sums != reference"
        l_ref = r.readPassLayers(p)[::ws, ::ws]
        assert np.array_equal(l_ref, o.readPassLayers(p)[::ws, ::ws]) and np.array_equal(l_ref, g.readPassLayers(p))
        off = r.readPassOffsets(p)
        assert np.array_equal(off, o.readPassOffsets(p)) and np.array_equal(off, g.readPassOffsets(p))
    if not left_frame:
        fl = r.readFlow(latest=True)
        assert np.array_equal(fl, o.readFlow(latest=True)) and np.array_equal(fl, g.readFlow(latest=True))
    assert r.state().totalFrameDelta == o.state().totalFrameDelta == g.m_totalFrameDelta
    for c in (g, o, r):
        c.updateFrame(fs[3])
        c.calculateOpticalFlow()
    common = o.readFlow()   # warp all three with the same flow even where the searches diverged
    g.writeFlow(common)
    r.writeFlow(common)
    tol = 64 if hdr else 1  # +-1 LSB of 10-bit (HDR samples are 10 bits in the MSBs of 16) / 8-bit
    for t, mode in [(0.0, 2), (1.0 / 6.0, 2), (0.5, 2), (0.4, 0), (0.4, 1), (0.4, 4), (0.4, 5), (0.4, 6), (1.0, 2)]:
        outs = []
        for c in (g, o, r):
            c.warpFrames(t, mode)
            a = out_array(g, hdr)
            c.downloadFrame(a)
            outs.append(a.astype(np.int64))
        assert np.array_equal(outs[0], outs[1]), "CUDA != oracle"
        d = np.abs(outs[1] - outs[2])
        assert d.max() <= tol, f"mode {mode} t {t}: oracle vs reference max diff {d.max()}"
    for c in (g, o, r):
        c.copyFrame()
    outs = []
    for c in (g, o, r):
        a = out_array(g, hdr)
        c.downloadFrame(a)
        outs.append(a.astype(np.int64))
    assert np.array_equal(outs[0], outs[1])
    assert np.abs(outs[1] - outs[2]).max() <= tol


@pytest.mark.parametrize("path", FILES, ids=CASE_IDS)
def test_recorded_reference_vs_oracle_vs_cuda(path):
    rec, (hdr, W, H, maxres, inS, outS, R, ds, ns, black, white, kind) = load_case(path)
    g, o = make_pair(hdr, H, W, inS, outS, ds, ns, black, white, maxres, R)
    o.enableTaps(True)
    g.setTapMode(True)
    for i in range(3):
        for c in (g, o):
            c.updateFrame(rec[f"frame{i}"])
    for c in (g, o):
        c.calculateOpticalFlow()
    n = int(rec["num_passes"])
    assert o.numPasses() == g.numPasses() == n
    rs = int(rec["geometry"][0])
    left_frame = False
    for p in range(n):
        ws, it, st = (int(v) for v in rec[f"pass{p}_info"])
        gi = g.passInfo(p)
        assert o.passInfo(p) == {"windowSize": ws, "iteration": it, "step": st} == {k: gi[k] for k in ("windowSize", "iteration", "step")}
        s_ref = rec[f"pass{p}_sums"]
        before = rec[f"pass{p - 1}_offsets"] if p else np.zeros_like(rec["pass0_offsets"])
        bad = oob_windows(before, ws, R, st, W, H, rs)
        assert np.array_equal(s_ref[~bad], o.readPassSums(p, R)[:, ::ws, ::ws][~bad]), f"pass {p}: oracle sums != reference"
        assert np.array_equal(s_ref[~bad], g.readPassSums(p, R)[~bad]), f"pass {p}: CUDA sums != reference"
        if bad.any():
            # the pass is set by the reference's recorded offsets (which CUDA and oracle matched up to here), not by
            # either calculator under test; as in test_oracle_golden, it may exclude only a sliver of the windows
            assert bad.mean() < 0.02, f"pass {p}: {bad.mean():.3f} of the windows leave the frame"
            left_frame = True
            break
        l_ref = rec[f"pass{p}_layers"]
        assert np.array_equal(l_ref, o.readPassLayers(p)[::ws, ::ws]) and np.array_equal(l_ref, g.readPassLayers(p))
        off = rec[f"pass{p}_offsets"]
        assert np.array_equal(off, o.readPassOffsets(p)) and np.array_equal(off, g.readPassOffsets(p))
    if kind != "random":
        assert not left_frame, "only the random-noise cases may leave the frame"
    else:
        assert p >= 3, f"the search left the frame at pass {p} of {n}: too little of the ladder compared"
    if not left_frame:
        fl = rec["flow_first"]
        assert np.array_equal(fl, o.readFlow(latest=True)) and np.array_equal(fl, g.readFlow(latest=True))
    assert int(rec["total_frame_delta_first"]) == o.state().totalFrameDelta == g.m_totalFrameDelta
    for c in (g, o):
        c.updateFrame(rec["frame3"])
        c.calculateOpticalFlow()
    if not left_frame:
        fl = rec["flow_second"]
        assert np.array_equal(fl, o.readFlow(latest=True)) and np.array_equal(fl, g.readFlow(latest=True))
    assert int(rec["total_frame_delta_second"]) == o.state().totalFrameDelta == g.m_totalFrameDelta
    for c in (g, o):
        c.writeFlow(rec["flow_first"])  # the field the reference's warps read (m_blurredOffsetArray[0])
    So = outS or W
    tol = 64 if hdr else 1  # +-1 LSB of 10-bit (HDR samples are 10 bits in the MSBs of 16) / 8-bit

    def outputs(op):
        """(CUDA, oracle) output frame of op() on both calculators, cropped to the frame width as recorded."""
        res = []
        for c in (g, o):
            op(c)
            a = out_array(g, hdr)
            c.downloadFrame(a)
            res.append(a.reshape(-1, So)[:, :W].astype(np.int64))
        return res

    done = 0
    for t, mode in WARPS:
        key = f"warp_m{mode}_t{t:.4f}"
        if key not in rec:  # the larger cases keep a subset of the outputs (MANIFEST.json)
            continue
        a, b = outputs(lambda c: c.warpFrames(t, mode))
        d_ref = np.abs(b - rec[key].astype(np.int64))
        if mode == 3:
            step = 256 if hdr else 1  # the HSV visualisation is quantised to 8 bits (atan2) before its << 7 / << 8
            d = np.abs(a - b)
            assert d.max() <= step and np.count_nonzero(d) <= max(4, d.size // 500), f"{key}: CUDA vs oracle max diff {d.max()}"
            assert d_ref.max() <= step, f"{key}: oracle vs reference max diff {d_ref.max()}"
        else:
            assert np.array_equal(a, b), f"{key}: CUDA != oracle in {np.count_nonzero(a != b)} samples"
            assert d_ref.max() <= tol, f"{key}: oracle vs reference max diff {d_ref.max()}"
        done += 1
    assert done >= 4
    a, b = outputs(lambda c: c.copyFrame())
    d_ref = np.abs(b - rec["copy"].astype(np.int64))
    assert np.array_equal(a, b) and d_ref.max() <= tol and not d_ref[H:].any(), f"copy: max diff to the reference {d_ref.max()}"
