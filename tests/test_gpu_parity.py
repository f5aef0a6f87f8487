"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Bars (BASELINE.json north_star): delta sums, lowest-layer indices and offset arrays bit-exact; blurred
flow and output pixels within +-1 LSB — we assert exact equality everywhere except the HSV
visualisation (atan2), where one 8-bit step is allowed on a vanishing fraction of samples.
"""
import numpy as np
import pytest

from conftest import make_pair, out_array

pytestmark = pytest.mark.gpu


def frames(synth, W, H, hdr, n, stride=None, kind="scene", seed=0):
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


def rep_view(full, ws):
    """[R][lh][lw] reference-shaped sums -> values at the window representatives [R][nWy][nWx]."""
    return full[..., ::ws, ::ws]


@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("W,H,inS,outS", [(64, 48, 0, 0), (130, 70, 192, 160), (258, 146, 258, 262)])
@pytest.mark.parametrize("black,white", [(0.0, 255.0), (16.0, 235.0), (3.5, 200.25)])
def test_copy_frame(synth, hdr, W, H, inS, outS, black, white):
    g, o = make_pair(hdr, H, W, inS, outS, black=black, white=white)
    f = frames(synth, W, H, hdr, 3, inS or None, "random")
    for i, fr in enumerate(f):
        g.updateFrame(fr)
        o.updateFrame(fr)
        g.copyFrame()
        o.copyFrame()
        a, b = out_array(g, hdr), out_array(o, hdr)
        g.downloadFrame(a)
        o.downloadFrame(b)
        S = outS or W
        a2, b2 = a.reshape(-1, S)[:, :W], b.reshape(-1, S)[:, :W]
        assert np.array_equal(a2, b2), f"frame {i}: {np.count_nonzero(a2 != b2)} samples differ"


def _smooth_flow(lh, lw, rng, amp):
    base = rng.integers(-amp, amp + 1, (2, (lh + 7) // 8 + 1, (lw + 7) // 8 + 1))
    fl = np.repeat(np.repeat(base, 8, 1), 8, 2)[:, :lh, :lw]
    fl = fl + rng.integers(-2, 3, fl.shape)
    return fl.astype(np.int16)


@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("mode,variant", [(0, 0), (1, 0), (2, 0), (0, 1), (1, 1), (2, 1), (3, 0), (4, 0), (5, 0), (6, 0)])
@pytest.mark.parametrize("W,H,maxres,inS,outS", [(64, 48, 270, 0, 0), (130, 70, 35, 136, 144), (256, 144, 36, 0, 320), (320, 176, 22, 0, 0),
                                                 (200, 120, 270, 200, 204),
                                                 # wide enough for interior items (test_warp_shapes.py): the lean form at
                                                 # rs 1 with an odd flow width, at rs 0, and warpItem's INSIDE form (odd outS)
                                                 (1030, 580, 290, 1094, 1062), (1024, 576, 576, 0, 1056), (1280, 720, 360, 1344, 1281)])
def test_warp_modes(synth, hdr, mode, variant, W, H, maxres, inS, outS):
    """All seven output modes over flows from zero to far beyond the rounding tables and blend scalars 0 .. 1.  The warp
    does not read the search variant: the variant-1 rows check that setting it leaves modes 0-2 unchanged."""
    g, o = make_pair(hdr, H, W, inS, outS, black=4.0, white=250.0, maxres=maxres)
    g.setSearchVariant(variant)
    for fr in frames(synth, W, H, hdr, 3, inS or None):
        g.updateFrame(fr)
        o.updateFrame(fr)
    lh, lw = g.m_opticalFlowFrameHeight, g.m_opticalFlowFrameWidth
    rng = np.random.default_rng(W * 7 + mode)
    for amp, t in [(0, 0.5), (9, 0.0), (9, 1.0 / 6.0), (40, 0.4), (300, 0.5), (9, 1.0), (2000, 0.3)]:
        fl = _smooth_flow(lh, lw, rng, amp)
        g.writeFlow(fl)
        o.writeFlow(fl)
        g.warpFrames(t, mode)
        o.warpFrames(t, mode)
        a, b = out_array(g, hdr), out_array(o, hdr)
        g.downloadFrame(a)
        o.downloadFrame(b)
        S = outS or W
        a2, b2 = a.reshape(-1, S)[:, :W].astype(np.int64), b.reshape(-1, S)[:, :W].astype(np.int64)
        if mode == 3:
            step = 256 if hdr else 1  # the visualisation is quantised to 8 bits (<< 8 in HDR chroma, << 7 luma)
            d = np.abs(a2 - b2)
            assert d.max() <= step and np.count_nonzero(d) <= max(4, d.size // 500), (d.max(), np.count_nonzero(d))
        else:
            assert np.array_equal(a2, b2), f"mode {mode} amp {amp} t {t}: {np.count_nonzero(a2 != b2)} differ, max {np.abs(a2 - b2).max()}"


@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_warp_flow_outliers_beyond_the_tables(synth, hdr, mode):
    """A smooth flow with a few outliers of 150-300 pixels on a frame large enough for interior items: the lean warp items
    check their own displacements, items that hold an outlier (directly or through the displaced reverse-flow lookup) take
    the general path, and the batch equals the oracle frame by frame."""
    W, H = 1280, 960
    g, o = make_pair(hdr, H, W, 0, 0, black=2.0, white=252.0, maxres=H)
    for fr in frames(synth, W, H, hdr, 3, None):
        g.updateFrame(fr)
        o.updateFrame(fr)
    lh, lw = g.m_opticalFlowFrameHeight, g.m_opticalFlowFrameWidth
    assert (lh, lw) == (H, W)
    rng = np.random.default_rng(77 + mode)
    fl = _smooth_flow(lh, lw, rng, 12)
    for k in range(40):  # isolated outliers and small patches, both axes, both signs, also near the frame edge
        y, x = int(rng.integers(0, lh - 8)), int(rng.integers(0, lw - 8))
        fl[int(rng.integers(0, 2)), y:y + int(rng.integers(1, 8)), x:x + int(rng.integers(1, 8))] = int(rng.choice([-300, -180, -150, 150, 200, 300]))
    g.writeFlow(fl)
    o.writeFlow(fl)
    ts = [0.0, 1.0 / 6.0, 0.5, 0.83]
    g.warpFramesBatch(ts, mode)
    for t in ts:
        o.warpFrames(t, mode)
        a, b = out_array(g, hdr), out_array(o, hdr)
        g.downloadFrame(a)
        o.downloadFrame(b)
        assert np.array_equal(a, b), f"t {t}: {np.count_nonzero(a != b)} samples differ"


@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 5])
@pytest.mark.parametrize("W,H,maxres,outS", [(256, 144, 270, 0), (130, 70, 35, 144), (320, 176, 88, 0)])
def test_warp_batch_equals_single_calls(synth, hdr, mode, W, H, maxres, outS):
    """hrb_ofc_warp_frames_batch: frame i of a batch is bit for bit the frame of warpFrames(t[i], mode), and both match the oracle."""
    g, o = make_pair(hdr, H, W, 0, outS, black=4.0, white=250.0, maxres=maxres)
    for fr in frames(synth, W, H, hdr, 3):
        g.updateFrame(fr)
        o.updateFrame(fr)
    lh, lw = g.m_opticalFlowFrameHeight, g.m_opticalFlowFrameWidth
    fl = _smooth_flow(lh, lw, np.random.default_rng(W + mode), 30)
    g.writeFlow(fl)
    o.writeFlow(fl)
    ts = [0.0, 1.0 / 6.0, 2.0 / 6.0, 0.5, 4.0 / 6.0, 5.0 / 6.0, 1.0]
    g.warpFramesBatch(ts, mode)
    batch = []
    for _ in ts:
        a = out_array(g, hdr)
        g.downloadFrame(a)
        batch.append(a)
    S = outS or W
    for t, a in zip(ts, batch):
        g.warpFrames(t, mode)
        o.warpFrames(t, mode)
        b, c = out_array(g, hdr), out_array(o, hdr)
        g.downloadFrame(b)
        o.downloadFrame(c)
        a2, b2, c2 = (x.reshape(-1, S)[:, :W].astype(np.int64) for x in (a, b, c))
        assert np.array_equal(a2, b2), f"t {t}: batch and single call differ in {np.count_nonzero(a2 != b2)} samples"
        if mode == 3:
            step = 256 if hdr else 1
            d = np.abs(a2 - c2)
            assert d.max() <= step and np.count_nonzero(d) <= max(4, d.size // 500)
        else:
            assert np.array_equal(a2, c2), f"t {t}: {np.count_nonzero(a2 != c2)} samples differ from the oracle"
    with pytest.raises(RuntimeError):
        g.warpFramesBatch([0.5, 1.5], 2)


def test_warp_rejects_blend_above_one(synth):
    g, o = make_pair(False, 48, 64)
    with pytest.raises(RuntimeError):
        g.warpFrames(1.5, 2)
    with pytest.raises(RuntimeError):
        o.warpFrames(1.5, 2)


SEARCH_CASES = [
    # hdr, W, H, maxres, inS, R, kind
    (False, 64, 48, 270, 0, 5, "scene"),
    (False, 64, 48, 270, 0, 16, "random"),
    (True, 64, 48, 270, 80, 11, "scene"),
    (False, 130, 70, 270, 0, 6, "scene"),
    (True, 130, 70, 270, 0, 16, "random"),
    (False, 258, 146, 73, 272, 16, "scene"),    # rs = 1, odd flow size 129x73
    (True, 512, 288, 72, 0, 16, "scene"),       # rs = 2, flow 128x72
    (False, 320, 200, 270, 0, 16, "identical"),
    (False, 320, 200, 270, 0, 9, "ramp"),
    (True, 384, 224, 270, 0, 16, "scene"),
    (False, 16, 16, 270, 0, 5, "random"),
    (False, 722, 430, 430, 0, 16, "scene"),     # both sizes = 2 (mod 4): no tile kernel; partial tiles on both edges of the small-window and generic kernels, windows 512..2
    (True, 640, 384, 384, 672, 7, "scene"),
    (False, 450, 258, 258, 0, 12, "random"),    # large offsets; both sizes = 2 (mod 4), so the tile kernel is skipped (the 452x260 row reaches it)
    (False, 200, 120, 270, 0, 2, "scene"),      # radii below the filter's minimum of 5 take the generic kernel
    (True, 200, 120, 270, 0, 3, "random"),
    (False, 290, 170, 270, 0, 13, "scene"),
    (True, 290, 170, 270, 300, 15, "random"),
    (False, 272, 160, 270, 0, 4, "ramp"),
    # both sizes multiples of 4: the tile kernel serves windows >= 16 (>= 4 under variants 2 and 3), one row per radius
    (True, 128, 96, 270, 0, 6, "random"),
    (False, 256, 128, 270, 0, 8, "scene"),
    (True, 320, 180, 270, 0, 10, "random"),
    (False, 452, 260, 270, 0, 12, "random"),    # large offsets: mirrored halos of the tile kernel's boxes
    (True, 292, 172, 270, 0, 13, "scene"),
    (False, 384, 216, 270, 416, 14, "random"),
    (True, 288, 168, 270, 0, 15, "scene"),
]


def check_ladder_taps(synth, hdr, W, H, maxres, inS, R, kind, variant, ds=8, ns=6):
    """Every pass of the ladder against the oracle with taps: window sums, arg-min layers and offsets bit-exact, then the
    final offsets, the blurred flow and the frame delta.  Then the same frames without taps, where the ladder runs from a
    CUDA graph: the two blurred-flow buffers alternate, so calculations 1 and 2 capture a graph each and calculation 3
    replays the first; each must give the same offsets, flow and frame delta as the tap run and the oracle."""
    g, o = make_pair(hdr, H, W, inS, 0, ds=ds, ns=ns, maxres=maxres, R=R)
    g.setSearchVariant(variant)
    g.setTapMode(True)
    o.enableTaps(True)
    for fr in frames(synth, W, H, hdr, 3, inS or None, kind):
        g.updateFrame(fr)
        o.updateFrame(fr)
    g.calculateOpticalFlow()
    o.calculateOpticalFlow()
    assert g.numPasses() == o.numPasses() > 0
    for p in range(o.numPasses()):
        gi, oi = g.passInfo(p), o.passInfo(p)
        assert (gi["windowSize"], gi["iteration"], gi["step"]) == (oi["windowSize"], oi["iteration"], oi["step"])
        ws = oi["windowSize"]
        s_ref = rep_view(o.readPassSums(p, R), ws)
        s_gpu = g.readPassSums(p, R)
        assert s_gpu.shape == s_ref.shape
        assert np.array_equal(s_gpu, s_ref), f"pass {p} (ws {ws}): {np.count_nonzero(s_gpu != s_ref)} window sums differ"
        l_ref = o.readPassLayers(p)[::ws, ::ws]
        assert np.array_equal(g.readPassLayers(p), l_ref), f"pass {p}: layers differ"
        assert np.array_equal(g.readPassOffsets(p), o.readPassOffsets(p)), f"pass {p}: offsets differ"
    off, flow, delta = o.readOffsetArray(), o.readFlow(latest=True), o.state().totalFrameDelta
    assert np.array_equal(g.readOffsetArray(), off)
    assert np.array_equal(g.readFlow(latest=True), flow), "blurred flow differs"
    assert g.m_totalFrameDelta == delta
    g.setTapMode(False)
    for k in range(3):
        g.calculateOpticalFlow()
        assert np.array_equal(g.readOffsetArray(), off), f"production calculation {k}: offsets differ"
        assert np.array_equal(g.readFlow(latest=True), flow), f"production calculation {k}: blurred flow differs"
        assert g.m_totalFrameDelta == delta, f"production calculation {k}: frame delta"


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4], ids=["auto", "generic", "notma", "perpixel", "butterfly"])
@pytest.mark.parametrize("hdr,W,H,maxres,inS,R,kind", SEARCH_CASES)
def test_search_ladder_taps(synth, hdr, W, H, maxres, inS, R, kind, variant):
    """Every pass of the ladder: window sums, arg-min layers and offsets are bit-exact — with the automatic kernel
    selection (sliding-window kernels for windows >= 32) and with the generic kernel forced for every pass — and the
    production path (no taps, CUDA graph) gives the same final offsets, flow and frame delta."""
    check_ladder_taps(synth, hdr, W, H, maxres, inS, R, kind, variant)


@pytest.mark.parametrize("ds,ns", [(0, 0), (31, 31), (24, 31), (31, 0)])
@pytest.mark.parametrize("hdr,W,H,maxres,inS,R,kind", [
    (False, 512, 256, 270, 0, 16, "scene"),    # tile kernel for windows >= 16
    (True, 258, 146, 270, 0, 11, "random"),    # sizes = 2 (mod 4): small-window kernel for windows <= 32, generic above
])
def test_search_ladder_scalar_extremes(synth, hdr, W, H, maxres, inS, R, kind, ds, ns):
    """deltaScalar / neighborBiasScalar at the ends of 0..31, where the uint32 window sums wrap: bit-exact pass by pass."""
    check_ladder_taps(synth, hdr, W, H, maxres, inS, R, kind, 0, ds=ds, ns=ns)


def test_flow_graph_cache_beyond_64_keys(synth):
    """More than 64 distinct (radius, scalars, input slots, output buffer) flow-graph keys through one small handle (the
    cache starts over past 64), the flow checked against the oracle after every calculation; then early keys again."""
    W, H = 96, 64
    g, o = make_pair(False, H, W, R=5)
    fs = frames(synth, W, H, False, 6)
    for fr in fs[:3]:
        g.updateFrame(fr)
        o.updateFrame(fr)
    keys = [(R, ds, ns) for ds, ns in [(8, 6), (0, 0), (31, 31), (4, 10), (12, 1)] for R in range(2, 17)]
    assert len(keys) > 64
    for k, (R, ds, ns) in enumerate(keys + keys[:10]):
        if k % 9 == 8:   # rotate the input slots now and then
            fr = fs[3 + (k // 9) % 3]
            g.updateFrame(fr)
            o.updateFrame(fr)
        g.m_opticalFlowSearchRadius = R
        g.m_deltaScalar = ds
        g.m_neighborBiasScalar = ns
        o.setParams(R, ds, ns)
        g.calculateOpticalFlow()
        o.calculateOpticalFlow()
        assert np.array_equal(g.readOffsetArray(), o.readOffsetArray()), f"calculation {k} {(R, ds, ns)}: offsets differ"
        assert np.array_equal(g.readFlow(latest=True), o.readFlow(latest=True)), f"calculation {k} {(R, ds, ns)}: flow differs"
        assert g.m_totalFrameDelta == o.state().totalFrameDelta, f"calculation {k} {(R, ds, ns)}: frame delta"


@pytest.mark.parametrize("hdr,W,H,maxres,R", [(False, 1920, 1080, 270, 16), (False, 1920, 1080, 540, 16), (True, 960, 540, 2160, 5)])
def test_search_final_flow_midsize(synth, hdr, W, H, maxres, R):
    """BASELINE configs 1 and 2 at full size (and a quarter-size full-resolution HDR case): final flow bit-exact."""
    g, o = make_pair(hdr, H, W, maxres=maxres, R=R)
    for fr in frames(synth, W, H, hdr, 3):
        g.updateFrame(fr)
        o.updateFrame(fr)
    g.calculateOpticalFlow()
    o.calculateOpticalFlow()
    assert np.array_equal(g.readOffsetArray(), o.readOffsetArray())
    assert np.array_equal(g.readFlow(latest=True), o.readFlow(latest=True))
    assert g.m_totalFrameDelta == o.state().totalFrameDelta


@pytest.mark.parametrize("hdr", [False, True])
def test_filter_sequence(synth, hdr):
    """The filter's call order (HopperRender.cpp:953-1186) over several source frames: every delivered frame matches."""
    W, H = 192, 112
    g, o = make_pair(hdr, H, W, 0, 200, maxres=270, R=8)
    blend = 0.0
    for t, fr in enumerate(frames(synth, W, H, hdr, 6)):
        g.updateFrame(fr)
        o.updateFrame(fr)
        if g.m_frameCount >= 3:
            g.calculateOpticalFlow()
            o.calculateOpticalFlow()
            assert g.m_totalFrameDelta == o.state().totalFrameDelta
        for _ in range(3):
            if g.m_frameCount >= 3:
                g.warpFrames(blend, 2)
                o.warpFrames(blend, 2)
            else:
                g.copyFrame()
                o.copyFrame()
            a, b = out_array(g, hdr), out_array(o, hdr)
            g.downloadFrame(a)
            o.downloadFrame(b)
            a2, b2 = a.reshape(-1, 200)[:, :W], b.reshape(-1, 200)[:, :W]
            assert np.array_equal(a2, b2), f"source frame {t}, blend {blend}"
            blend += 0.4
            if blend >= 1.0:
                blend -= 1.0
    assert g.m_frameCount == o.state().frameCount == 6
    assert g.m_ofcCalcTime > 0 and g.m_warpCalcTime > 0


def test_live_parameter_updates(synth):
    """Fields the filter writes on a live object take effect at the next call (HopperRender.cpp:1386-1389,1448)."""
    W, H = 128, 96
    g, o = make_pair(False, H, W, R=5)
    fs = frames(synth, W, H, False, 4)
    for fr in fs[:3]:
        g.updateFrame(fr)
        o.updateFrame(fr)
    for R, ds, ns, bl, wh in [(5, 8, 6, 0.0, 255.0), (6, 4, 2, 10.0, 240.0), (16, 10, 0, 0.0, 128.0), (7, 0, 10, 20.0, 255.0)]:
        g.m_opticalFlowSearchRadius = R
        g.m_deltaScalar = ds
        g.m_neighborBiasScalar = ns
        g.m_outputBlackLevel = bl
        g.m_outputWhiteLevel = wh
        o.setParams(R, ds, ns, bl, wh)
        g.calculateOpticalFlow()
        o.calculateOpticalFlow()
        g.calculateOpticalFlow()   # twice, so that the flow warpFrames reads is the one just computed
        o.calculateOpticalFlow()
        assert np.array_equal(g.readFlow(), o.readFlow())
        g.warpFrames(0.5, 2)
        o.warpFrames(0.5, 2)
        a, b = out_array(g, False), out_array(o, False)
        g.downloadFrame(a)
        o.downloadFrame(b)
        assert np.array_equal(a, b)
    g.m_frameCount = 0
    assert g.m_frameCount == 0


def test_device_resident_and_async_paths(synth):
    """update_frame_device / calculate_async / download_async give the same bytes as the blocking calls."""
    import torch
    W, H = 256, 144
    g, o = make_pair(True, H, W, R=16)
    out_pinned = torch.zeros(g.outputFrameBytes // 2, dtype=torch.int16).pin_memory()
    for fr in frames(synth, W, H, True, 4):
        dev = torch.from_numpy(fr.view(np.int16)).cuda()
        torch.cuda.synchronize()
        g.updateFrameDevice(dev)
        o.updateFrame(fr)
        if g.m_frameCount >= 3:
            g.calculateOpticalFlowAsync()
            o.calculateOpticalFlow()
            g.warpFrames(0.25, 2)
            o.warpFrames(0.25, 2)
            g.downloadFrameAsync(out_pinned)
            g.synchronize()
            b = out_array(o, True)
            o.downloadFrame(b)
            assert np.array_equal(out_pinned.numpy().view(np.uint16), b)
            assert g.m_totalFrameDelta == o.state().totalFrameDelta


def test_full_size_4k_p010_properties(synth):
    """BASELINE config 3 (3840x2160 P010, full-resolution flow, R=16): against the oracle at full size, plus
    size-independent properties (identical frames -> zero flow and pass-through blend)."""
    W, H = 3840, 2160
    g, o = make_pair(True, H, W, maxres=2160, R=16)
    fs = frames(synth, W, H, True, 3)
    for fr in fs:
        g.updateFrame(fr)
        o.updateFrame(fr)
    g.calculateOpticalFlow()
    o.calculateOpticalFlow()
    assert g.m_totalFrameDelta == o.state().totalFrameDelta
    fg, fo = g.readFlow(latest=True), o.readFlow(latest=True)
    assert np.array_equal(fg, fo), f"{np.count_nonzero(fg != fo)} flow samples differ"
    # the dominant motion of the synthetic scene is (+6,-3) px/frame => offsets (-6,+3)
    off = g.readOffsetArray()
    assert np.median(off[0]) == -6 and np.median(off[1]) == 3
    g.calculateOpticalFlow()
    o.calculateOpticalFlow()
    g.warpFrames(0.5, 2)
    o.warpFrames(0.5, 2)
    a, b = out_array(g, True), out_array(o, True)
    g.downloadFrame(a)
    o.downloadFrame(b)
    assert np.array_equal(a, b)
    # identical frames: zero flow, and the blend of two identical frames is the level-corrected frame itself
    for _ in range(3):
        g.updateFrame(fs[0])
    g.calculateOpticalFlow()
    assert not g.readOffsetArray().any() and not g.readFlow(latest=True).any()
    g.calculateOpticalFlow()
    g.warpFrames(0.5, 2)
    g.downloadFrame(a)
    # zero flow + identical sources: the blend is the source itself up to the HDR level scale 65535/65280 (SURVEY.md A.5.7)
    src = fs[0][:W * H].reshape(H, W)[1:-1, 1:-1].astype(np.float32)
    exp = np.minimum(src / np.float32(65280.0) * np.float32(65535.0), np.float32(65535.0)).astype(np.uint16)
    assert np.array_equal(a[:W * H].reshape(H, W)[1:-1, 1:-1], exp)


@pytest.mark.parametrize("hdr", [False, True])
def test_cpp_shim_replay_matches_python_replay_over_the_oracle(synth, hdr, tmp_path):
    """tools/replay.cpp drives include/opticalFlowCalc*.h (the header-compatible classes a DirectShow build would
    use) through the filter's delivery loop; the delivered frames must be the ones the oracle produces under
    hopperrender_b200.replay.DeliveryLoop (same loop, python)."""
    import os
    import subprocess
    import zlib

    from conftest import ROOT, OracleAsCalc
    from hopperrender_b200 import replay
    from oracle import OracleCalc
    exe = os.path.join(ROOT, "tools", "replay_cpp.bin")
    if not os.path.exists(exe):
        pytest.skip("tools/replay_cpp.bin not built (python -c 'import __graft_entry__ as g; g.build()')")
    W, H, n = 256, 144, 9
    fs = frames(synth, W, H, hdr, n)
    fs[6] = synth.make_random_frame(W, H, 77, hdr)  # a scene cut in the middle
    raw = tmp_path / "frames.raw"
    with open(raw, "wb") as f:
        for fr in fs:
            f.write(fr.tobytes())
    res = subprocess.run([exe, str(raw), str(W), str(H), "1" if hdr else "0", str(n), str(replay.TARGET_FRAME_TIME_60), "270", "7"],
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    got = [ln.split() for ln in res.stdout.strip().splitlines()]
    o = OracleAsCalc(OracleCalc(H, W, W, W, 8, 6, 0.0, 255.0, 270, hdr))
    o.m_opticalFlowSearchRadius = 7
    loop = replay.DeliveryLoop(o, target_frame_time=replay.TARGET_FRAME_TIME_60, auto_adjust=False)
    exp = []
    out = np.zeros(o.outputFrameBytes, np.uint8)
    for fr in fs:
        loop.deliver(fr, out, sink=lambda buf, info: exp.append((info, zlib.crc32(buf.tobytes()) & 0xFFFFFFFF)))
    assert len(got) == len(exp) > n
    for g_line, (info, crc) in zip(got, exp):
        assert int(g_line[0]) == info["source"] and int(g_line[1]) == info["index"]
        assert abs(float(g_line[2]) - info["blend"]) < 1e-8
        assert int(g_line[3]) == int(info["warped"])
        assert int(g_line[5], 16) == crc, f"delivered frame {g_line[:2]} differs"
    assert any(not i["warped"] and i["source"] >= 3 for i, _ in exp), "the scene cut should have forced a copyFrame"


def lean_sample_masks(W, H):
    """(luma [H][W], chroma pairs [H/2][W/2]): the samples a zero-flow warp of a full frame sends through the lean form."""
    from test_warp_shapes import ITEM, LEAN, warp_item_maps
    maps = warp_item_maps(W, H, W, H, 0, W, None, 0, None, [0.5], 2)
    luma = np.repeat(maps[0][1] == LEAN, ITEM, axis=1)[:, :W]
    pairs = np.repeat(maps[1][1] == LEAN, ITEM // 2, axis=1)[:, :W // 2]
    return luma, pairs


@pytest.mark.parametrize("black,white", [(0.0, 255.0), (16.0, 235.0), (3.5, 200.25), (0.0, 1.0), (100.0, 101.0), (250.0, 5.0)])
def test_levels_exhaustive(black, white):
    """Level correction for every 16-bit (P010 container) and 8-bit input value, luma and chroma, against the oracle's
    IEEE division — pins the hoisted-reciprocal division of the CUDA kernels (copy, warp) to correctly rounded results.
    At 512 wide every warp item takes warpItem; at 2048 wide every value also passes the lean form's division (HDR) and
    its level tables (SDR), in luma items and as both the U and the V sample of chroma pairs."""
    for hdr, W, H in [(True, 512, 128), (False, 512, 16), (True, 2048, 176), (False, 2048, 16)]:
        g, o = make_pair(hdr, H, W, black=black, white=white)
        dt = np.uint16 if hdr else np.uint8
        nvals = 65536 if hdr else 256
        fr = np.zeros((H + H // 2) * W, dt)
        fr[:H * W] = np.arange(H * W) % nvals            # every value in the luma plane ...
        fr[H * W:] = (np.arange(H * W // 2) * 2 + np.arange(H * W // 2) % 2) % nvals  # ... and in both chroma channels
        if hdr and W == 512:
            assert H * W >= nvals and H * W // 2 >= nvals // 2
        if W == 2048:  # at 2048 wide the warp's lean form runs: lay every value out in its luma items and chroma pairs
            lean_luma, lean_pairs = lean_sample_masks(W, H)
            planes = fr.reshape(H + H // 2, W)
            planes[:H][lean_luma] = np.arange(np.count_nonzero(lean_luma)) % nvals
            pairs = planes[H:].reshape(H // 2, W // 2, 2)
            pairs[lean_pairs] = (np.arange(np.count_nonzero(lean_pairs)) % nvals)[:, None]  # the same value as U and as V
            assert np.unique(planes[:H][lean_luma]).size == nvals
            assert np.unique(pairs[lean_pairs][:, 0]).size == np.unique(pairs[lean_pairs][:, 1]).size == nvals
        for _ in range(3):
            g.updateFrame(fr)
            o.updateFrame(fr)
        a, b = out_array(g, hdr), out_array(o, hdr)
        g.copyFrame()
        o.copyFrame()
        g.downloadFrame(a)
        o.downloadFrame(b)
        assert np.array_equal(a, b), f"copyFrame hdr={hdr}: {np.count_nonzero(a != b)} differ"
        # zero flow, identical frames: warp mode 2 blends each sample with itself -> levels applied to every interior value
        g.warpFrames(0.5, 2)
        o.warpFrames(0.5, 2)
        g.downloadFrame(a)
        o.downloadFrame(b)
        assert np.array_equal(a, b), f"warpFrames hdr={hdr}: {np.count_nonzero(a != b)} differ"


@pytest.mark.parametrize("hdr", [False, True])
def test_pipelined_transfers_match_the_oracle(synth, hdr):
    """Asynchronous upload / download entry points (own streams, 4 input slots, ring of 3 output frames, tickets):
    every delivered frame equals the oracle's, whatever the overlap."""
    import torch
    W, H = 320, 176
    g, o = make_pair(hdr, H, W, R=9)
    dt = torch.int16 if hdr else torch.uint8
    n_el = g.outputFrameBytes // (2 if hdr else 1)
    pool = [torch.zeros(n_el, dtype=dt).pin_memory() for _ in range(12)]
    fs = frames(synth, W, H, hdr, 7)
    pins = [torch.from_numpy(f.view(np.int16) if hdr else f).pin_memory() for f in fs]
    expected, tickets = [], []
    k = 0
    for t, fr in enumerate(fs):
        g.updateFrameAsync(pins[t])
        o.updateFrame(fr)
        if t >= 2:
            g.calculateOpticalFlowAsync()
            o.calculateOpticalFlow()
        for j in range(3):
            blend = (0.4 * (3 * t + j)) % 1.0
            if t >= 2:
                g.warpFrames(blend, 2)
                o.warpFrames(blend, 2)
            else:
                g.copyFrame()
                o.copyFrame()
            tickets.append((g.downloadFrameAsync(pool[k % len(pool)]), k % len(pool)))
            b = out_array(o, hdr)
            o.downloadFrame(b)
            expected.append(b)
            k += 1
            if len(tickets) > 9:   # consume in order, a few frames behind
                tk, slot = tickets.pop(0)
                g.waitDownload(tk)
                got = pool[slot].numpy().view(np.uint16 if hdr else np.uint8)
                assert np.array_equal(got, expected.pop(0)), f"delivered frame {k - len(tickets) - 1} differs"
    while tickets:
        tk, slot = tickets.pop(0)
        g.waitDownload(tk)
        got = pool[slot].numpy().view(np.uint16 if hdr else np.uint8)
        assert np.array_equal(got, expected.pop(0))
    g.synchronize()
    assert g.m_frameCount == 7 and g.m_totalFrameDelta == o.state().totalFrameDelta


@pytest.mark.parametrize("hdr,mode", [(False, 2), (True, 2), (True, 3), (False, 6)])
def test_output_stripes_tile_the_full_frame(synth, hdr, mode):
    """hrb_ofc_set_output_stripe: four calculators fed the same frames, each producing one quarter of the rows (what the
    ranks of a spatial split do), together reproduce the single-calculator output — warp, copy and download."""
    from hopperrender_b200.split import merge_stripes, stripe_bounds
    W, H, n = 256, 160, 4
    full, o = make_pair(hdr, H, W, R=8)
    parts = [make_pair(hdr, H, W, R=8)[0] for _ in range(n)]
    for p, (y0, y1) in zip(parts, stripe_bounds(H, n)):
        p.setOutputStripe(y0, y1)
    for t, fr in enumerate(frames(synth, W, H, hdr, 4)):
        for c in [full, o] + parts:
            c.updateFrame(fr)
        if t >= 2:
            for c in [full, o] + parts:
                c.calculateOpticalFlow()
    for op in ("warp", "copy"):
        outs = []
        for c in [full, o] + parts:
            if op == "warp":
                c.warpFrames(0.3, mode)
            else:
                c.copyFrame()
            a = out_array(full, hdr)
            c.downloadFrame(a)
            outs.append(a)
        merged = merge_stripes(outs[2:], H, W)
        if mode != 3:
            assert np.array_equal(outs[0], outs[1])
        assert np.array_equal(merged, outs[0]), f"{op}: stripes do not tile the full frame"
        # a stripe download must leave the rest of the caller's buffer alone
        assert not outs[2][W * (H // n):W * H].any()


@pytest.mark.parametrize("hdr,W,H", [(True, 3840, 2160), (False, 1920, 1080)])
def test_overlapped_flow_equals_the_serial_schedule(synth, hdr, W, H):
    """calculateOpticalFlowAsync runs the search on its own stream beside the warps of the same source frame.  At sizes
    where the kernels really overlap, every output frame, every flow field and every frame delta must equal those of the
    same calls with the overlap switched off (whose small-size equality with the oracle the other tests establish)."""
    import torch
    import hopperrender_b200 as hr
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    dt = torch.int16 if hdr else torch.uint8
    fs = [torch.from_numpy(f.view(np.int16) if hdr else f).cuda() for f in frames(synth, W, H, hdr, 6)]
    results = []
    for overlap in (True, False):
        g = cls(H, W, 0, 0, 8, 6, 16.0, 235.0, 2160)
        g.setFlowOverlap(overlap)
        n_el = g.outputFrameBytes // (2 if hdr else 1)
        outs, deltas, flows = [], [], []
        pool = [torch.zeros(n_el, dtype=dt).pin_memory() for _ in range(12)]
        tickets = []
        for t, fr in enumerate(fs):
            g.updateFrameDevice(fr)
            if t >= 2:
                g.calculateOpticalFlowAsync()
                for j in range(3):
                    g.warpFrames((0.3 * (3 * t + j)) % 1.0, 2)
                    tickets.append(g.downloadFrameAsync(pool[len(tickets)]))
        for tk in tickets:
            g.waitDownload(tk)
        g.synchronize()
        outs = [p.numpy().copy() for p in pool[:len(tickets)]]
        flows = g.readFlow(latest=True).copy()
        results.append((outs, flows, g.m_totalFrameDelta))
        g.close()
    (oa, fa, da), (ob, fb, db) = results
    assert len(oa) == len(ob) == 12
    for i, (x, y) in enumerate(zip(oa, ob)):
        assert np.array_equal(x, y), f"output frame {i} differs between the overlapped and the serial schedule"
    assert np.array_equal(fa, fb) and da == db
    assert np.abs(fa).max() > 0
