"""Flow batch (hrb_flow_batch_*, FlowBatch): the flows of many same-size streams searched together on one GPU, a generic
pass of every member in one launch.  After a batched calculate every member must be in exactly the state its own
calculate leaves a lone handle fed the same frames in: offsets, both blurred flows, flow peaks, frame delta and raw
delta, pass by pass in tap mode, over asynchronous sequences with warps in between.  The members mix SDR and HDR, padded
strides, delta and neighbour scalars, content, and frame history.
"""
import ctypes as C

import numpy as np
import pytest

from test_ladder_shapes import expected_kernel, mosaic_frames


# ---------------------------------------------------------------------------------------------------------------------
# CPU: argument checks that need no device
# ---------------------------------------------------------------------------------------------------------------------
def test_create_rejects_bad_arguments_without_a_device():
    from hopperrender_b200 import _lib
    lib = _lib.load()
    out = C.c_void_p()
    two = (C.c_void_p * 2)(None, None)
    assert lib.hrb_flow_batch_create(None, two, 1) == 1
    assert lib.hrb_flow_batch_create(C.byref(out), None, 1) == 1
    assert lib.hrb_flow_batch_create(C.byref(out), two, 2) == 1 and b"null handle" in lib.hrb_last_error()
    for n in (0, -1, 65):
        assert lib.hrb_flow_batch_create(C.byref(out), two, n) == 1 and b"1..64" in lib.hrb_last_error()
    same = (C.c_void_p * 2)(0x1000, 0x1000)  # never dereferenced: the repeat is found first
    assert lib.hrb_flow_batch_create(C.byref(out), same, 2) == 1 and b"twice" in lib.hrb_last_error()
    assert out.value is None
    assert lib.hrb_flow_batch_calculate_optical_flow(None) == 1
    assert lib.hrb_flow_batch_calculate_optical_flow_async(None) == 1
    lib.hrb_flow_batch_destroy(None)


def ladder_passes(lw, lh, R, rs, variant=0):
    """(generic passes, tile + small-window passes) of one flow's ladder, as planSearchPass plans them."""
    m = max(lw, lh)
    ws = m if m & (m - 1) == 0 else 1 << m.bit_length()
    ws //= 2
    generic = other = 0
    for it in range(ws.bit_length() - 1):
        w = ws >> it
        for lu in (lh, lw):  # step 0 runs along the flow height, step 1 along the width
            if expected_kernel(w, lu, R, rs, variant) == "generic":
                generic += 1
            else:
                other += 1
    return generic, other


def test_ladder_pass_counts():
    """cfg1 (480x270) and cfg2 (960x540) flows run 16 and 18 generic passes; a full-resolution 1024x576 flow none."""
    assert ladder_passes(480, 270, 16, 2) == (16, 0)
    assert ladder_passes(960, 540, 9, 1) == (18, 0)
    assert ladder_passes(1024, 576, 16, 0) == (0, 18)
    assert ladder_passes(1024, 576, 16, 0, variant=1) == (18, 0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _member_spec(k, hdr_all=None):
    """Member k's settings: SDR / HDR alternate, every third member has a padded input stride, the delta and neighbour
    scalars cycle through 0, 8 and 31, odd members see motion-mosaic content, member 2 lags one frame."""
    return dict(hdr=(k % 2 == 1) if hdr_all is None else hdr_all, pad=k % 3 == 1, ds=(8, 0, 31)[k % 3], ns=(6, 31, 0, 8)[k % 4],
                kind="mosaic" if k % 2 else "scene", lag=k == 2)


def _calc(spec, W, H, maxres, R, variant=0, stream=None):
    import hopperrender_b200 as hr
    cls = hr.OpticalFlowCalcHDR if spec["hdr"] else hr.OpticalFlowCalcSDR
    g = cls(H, W, W + 64 if spec["pad"] else 0, 0, spec["ds"], spec["ns"], 0.0, 255.0, maxres, 0, stream)
    g.m_opticalFlowSearchRadius = R
    if variant:
        g.setSearchVariant(variant)
    return g


_FRAMES = {}


def _frames(synth, spec, W, H):
    """The frames member `spec` is fed (one more at the front when it lags): cached per content, format and stride."""
    key = (spec["kind"], spec["hdr"], spec["pad"], W, H)
    if key not in _FRAMES:
        S = W + 64 if spec["pad"] else None
        if spec["kind"] == "mosaic":
            fs = mosaic_frames(synth, W, H, spec["hdr"], seed=W + H + spec["hdr"], stride=S)
        else:
            fs = [synth.make_frame(W, H, t, synth.SEED_BASE + 31 + spec["hdr"], spec["hdr"], S) for t in range(3)]
        _FRAMES.clear() if len(_FRAMES) > 8 else None
        _FRAMES[key] = fs
    fs = _FRAMES[key]
    return [fs[2]] + fs if spec["lag"] else fs


def _result(c):
    return dict(offsets=c.readOffsetArray(), flow=c.readFlow(), latest=c.readFlow(latest=True), peak=c.readFlowPeak(), delta=c.m_totalFrameDelta,
                raw=c.readRawFrameDelta(), count=c.m_ofcCalcCount, frames=c.m_frameCount)


def _assert_same(got, want, label):
    for k in ("offsets", "flow", "latest"):
        assert np.array_equal(got[k], want[k]), f"{label}: {np.count_nonzero(got[k] != want[k])} values of {k} differ"
    for k in ("peak", "delta", "raw", "count", "frames"):
        assert got[k] == want[k], f"{label}: {k} {got[k]} != {want[k]}"


def _lone_results(synth, specs, W, H, maxres, R, variant):
    out = []
    for s in specs:
        c = _calc(s, W, H, maxres, R, variant)
        for f in _frames(synth, s, W, H):
            c.updateFrame(f)
        c.calculateOpticalFlow()
        out.append(_result(c))
        c.close()
    return out


def _batch_equals_lone(synth, W, H, maxres, R, S, variant=0, hdr_all=None, check_launches=True):
    import hopperrender_b200 as hr
    specs = [_member_spec(k, hdr_all) for k in range(S)]
    want = _lone_results(synth, specs, W, H, maxres, R, variant)
    calcs = [_calc(s, W, H, maxres, R, variant) for s in specs]
    for c, s in zip(calcs, specs):
        for f in _frames(synth, s, W, H):
            c.updateFrame(f)
    b = hr.FlowBatch(calcs)
    assert len(b) == S
    before = hr.kernel_launch_count()
    b.calculateOpticalFlow()
    launches = hr.kernel_launch_count() - before
    g = calcs[0]
    lw, lh, rs = g.m_opticalFlowFrameWidth, g.m_opticalFlowFrameHeight, g.m_opticalFlowResScalar
    for k, c in enumerate(calcs):
        _assert_same(_result(c), want[k], f"{W}x{H} rs {rs} R {R} variant {variant} S {S}: member {k} {specs[k]}")
    if check_launches:
        generic, other = ladder_passes(lw, lh, R, rs, variant)
        assert launches == generic + 1 + S * other, f"{launches} launches for {generic} generic and {other} other passes, S {S}"
    b.close()
    for c in calcs:
        c.close()
    return launches


BATCH_CASES = [
    # W, H, maxres, R, S, variant, all HDR
    (1920, 1080, 270, 16, 1, 0, None),     # cfg1: a 480x270 flow, every pass generic
    (1920, 1080, 270, 16, 2, 0, None),
    (1920, 1080, 270, 16, 7, 0, None),
    (1920, 1080, 270, 16, 64, 0, None),
    (1920, 1080, 540, 9, 4, 0, None),      # cfg2-like: a 960x540 flow
    (1030, 580, 290, 16, 3, 0, None),      # a 515x290 flow: odd width
    (1024, 576, 576, 2, 3, 0, None),       # R 2 and 4: the generic kernel below R 5, full resolution
    (1024, 576, 576, 4, 3, 0, None),
    (1024, 576, 576, 16, 3, 1, None),      # variant 1: the generic kernel everywhere, windows beyond a tile, per-member tickets
    (1030, 580, 580, 16, 3, 0, None),      # rs 0: Y passes of windows >= 64 generic, the others tile / small-window per member
    (3840, 2160, 2160, 16, 3, 0, True),    # 4K P010 at full resolution
]


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,maxres,R,S,variant,hdr_all", BATCH_CASES)
def test_batch_equals_lone_handles(synth, W, H, maxres, R, S, variant, hdr_all):
    """Every member holds what a lone handle fed its frames computes, and the batch launches each generic pass once."""
    launches = _batch_equals_lone(synth, W, H, maxres, R, S, variant, hdr_all)
    if maxres in (270, 540):
        assert launches in (17, 19)


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,maxres", [(1920, 1080, 270), (1024, 576, 576)])
def test_taps_pass_by_pass(synth, W, H, maxres):
    """With tap mode on, every member's sums, layers and offsets equal the lone handle's, pass by pass."""
    import hopperrender_b200 as hr
    R, S = 16, 3
    specs = [_member_spec(k) for k in range(S)]
    lone = [_calc(s, W, H, maxres, R) for s in specs]
    calcs = [_calc(s, W, H, maxres, R) for s in specs]
    for c, s in zip(lone + calcs, specs + specs):
        for f in _frames(synth, s, W, H):
            c.updateFrame(f)
        c.setTapMode(True)
    for c in lone:
        c.calculateOpticalFlow()
    b = hr.FlowBatch(calcs)
    b.calculateOpticalFlow()
    for k, (c, l) in enumerate(zip(calcs, lone)):
        n = l.numPasses()
        assert c.numPasses() == n > 0
        for p in range(n):
            where = f"member {k} pass {p} {l.passInfo(p)}"
            assert c.passInfo(p) == l.passInfo(p), where
            assert np.array_equal(c.readPassSums(p, R), l.readPassSums(p, R)), f"{where}: sums differ"
            assert np.array_equal(c.readPassLayers(p), l.readPassLayers(p)), f"{where}: layers differ"
            assert np.array_equal(c.readPassOffsets(p), l.readPassOffsets(p)), f"{where}: offsets differ"
        _assert_same(_result(c), _result(l), f"member {k}")
    b.close()
    for c in lone + calcs:
        c.close()


@pytest.mark.gpu
def test_async_sequence_with_warps(synth):
    """Six frames through the asynchronous batch calculate; member 1 has flow overlap off, member 2 runs on a stream the
    caller supplied.  After every calculate each member warps a batch of frames and downloads them: every output frame
    and both flows equal those of lone handles run the same way."""
    import torch
    import hopperrender_b200 as hr
    W, H, maxres, R, S = 1920, 1080, 270, 16, 3
    specs = [_member_spec(k) for k in range(S)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    lone = [_calc(s, W, H, maxres, R, stream=streams[0].cuda_stream if k == 2 else None) for k, s in enumerate(specs)]
    calcs = [_calc(s, W, H, maxres, R, stream=streams[1].cuda_stream if k == 2 else None) for k, s in enumerate(specs)]
    lone[1].setFlowOverlap(False)
    calcs[1].setFlowOverlap(False)
    seqs = []
    for k, s in enumerate(specs):
        base = _frames(synth, s, W, H)
        extra = [synth.make_frame(W, H, t, synth.SEED_BASE + 40 + k, s["hdr"], W + 64 if s["pad"] else None) for t in range(6)]
        seqs.append((base + extra)[:6])
    b = hr.FlowBatch(calcs)
    ts = [0.25, 0.5, 0.75]
    for t in range(6):
        for k in range(S):
            lone[k].updateFrame(seqs[k][t])
            calcs[k].updateFrame(seqs[k][t])
        if t < 1:
            continue
        for c in lone:
            c.calculateOpticalFlowAsync()
        b.calculateOpticalFlowAsync()
        for k in range(S):
            outs = []
            for c in (lone[k], calcs[k]):
                c.warpFramesBatch(ts, 2)
                frames = []
                for _ in ts:
                    a = np.zeros(c.outputFrameBytes, np.uint8)
                    c.downloadFrame(a)
                    frames.append(a)
                outs.append(frames)
            for j in range(len(ts)):
                assert np.array_equal(outs[1][j], outs[0][j]), f"frame {t}: member {k} output {j} differs"
            assert np.array_equal(calcs[k].readFlow(), lone[k].readFlow()), f"frame {t}: member {k} flow for warp differs"
            assert np.array_equal(calcs[k].readFlow(latest=True), lone[k].readFlow(latest=True)), f"frame {t}: member {k} latest flow differs"
            assert calcs[k].readFlowPeak() == lone[k].readFlowPeak() and calcs[k].m_totalFrameDelta == lone[k].m_totalFrameDelta, f"frame {t}: member {k}"
    b.close()
    for c in lone + calcs:
        c.close()


@pytest.mark.gpu
def test_ingest_is_ordered_behind_an_asynchronous_batch(synth):
    """An asynchronous batch reads the search planes of two input slots of every member; three updateFrameDevice calls
    later the ingest overwrites one of them and must wait for the batch.  synchronize on one member afterwards leaves its
    state equal to the lone handle's."""
    import torch
    import hopperrender_b200 as hr
    W, H, R, S = 1920, 1088, 16, 2
    specs = [dict(_member_spec(k), hdr=True, pad=False, lag=False) for k in range(S)]
    fr = [[synth.make_frame(W, H, t, synth.SEED_BASE + 50 + k, True) for t in range(6)] for k in range(S)]
    want = []
    for k, s in enumerate(specs):
        c = _calc(s, W, H, H, R)
        for t in range(3):
            c.updateFrame(fr[k][t])
        c.calculateOpticalFlow()
        want.append(_result(c))
        c.close()
    calcs = [_calc(s, W, H, H, R) for s in specs]
    dev = [[torch.from_numpy(f.view(np.int16)).cuda() for f in fs] for fs in fr]
    for k, c in enumerate(calcs):
        for t in range(3):
            c.updateFrameDevice(dev[k][t])
    b = hr.FlowBatch(calcs)
    b.calculateOpticalFlowAsync()
    for t in range(3, 6):  # no calculate, no join in between
        for k, c in enumerate(calcs):
            c.updateFrameDevice(dev[k][t])
    for k, c in enumerate(calcs):
        assert np.array_equal(c.readFlow(latest=True), want[k]["latest"]), f"member {k}: the ingest overtook the batch"
    # a fresh batch on the same frames as the lone handles, then synchronize on one member only
    for k, c in enumerate(calcs):
        for t in range(3):
            c.updateFrameDevice(dev[k][t])
    b.calculateOpticalFlowAsync()
    calcs[1].synchronize()
    got = _result(calcs[1])
    assert np.array_equal(got["latest"], want[1]["latest"]) and got["delta"] == want[1]["delta"] and got["raw"] == want[1]["raw"]
    b.close()
    for c in calcs:
        c.close()


@pytest.mark.gpu
def test_argument_checks(synth):
    """Members that disagree are refused at create, or at calculate when a parameter changed since, naming the field;
    the profile and the debug timeline are refused; a member used alone between batch calls still equals a lone handle."""
    import hopperrender_b200 as hr
    W, H, R = 448, 256, 9
    sa, sb = _member_spec(0), _member_spec(1)
    a, b = _calc(sa, W, H, 256, R), _calc(sb, W, H, 256, R)
    for other, field in [(_calc(sa, 512, H, 256, R), "frame_width"), (_calc(sa, W, 288, 288, R), "frame_height"),
                         (_calc(sa, W, H, 128, R), "res_scalar"), (_calc(sa, W, H, 256, 10), "search_radius"),
                         (_calc(sa, W, H, 256, R, variant=1), "search_variant")]:
        with pytest.raises(RuntimeError, match=f"hrb error 1.*{field}"):
            hr.FlowBatch([a, other])
        other.close()
    with pytest.raises(RuntimeError, match="hrb error 1.*twice"):
        hr.FlowBatch([a, a])
    with pytest.raises(RuntimeError, match="hrb error 1.*1..64"):
        hr.FlowBatch([])
    for c, s in ((a, sa), (b, sb)):
        for f in _frames(synth, s, W, H):
            c.updateFrame(f)
    batch = hr.FlowBatch([a, b])
    for change, undo, field in [(lambda c: setattr(c, "m_opticalFlowSearchRadius", 16), lambda c: setattr(c, "m_opticalFlowSearchRadius", R), "search_radius"),
                                (lambda c: c.setSearchVariant(1), lambda c: c.setSearchVariant(0), "search_variant")]:
        change(b)
        with pytest.raises(RuntimeError, match=f"hrb error 1.*{field}"):
            batch.calculateOpticalFlow()
        undo(b)
        batch.calculateOpticalFlow()  # agree again
    for on, off in [(lambda c: c.setProfile(True), lambda c: c.setProfile(False)), (lambda c: c.debugTimeline(1024), lambda c: c.debugTimeline(0))]:
        on(b)
        with pytest.raises(RuntimeError, match="hrb error 5"):
            batch.calculateOpticalFlowAsync()
        off(b)
    # a member used alone between two batch calls
    lone = _calc(sa, W, H, 256, R)
    for f in _frames(synth, sa, W, H):
        lone.updateFrame(f)
    for _ in range(4):  # a's two batch calls above, its own call and the next batch call
        lone.calculateOpticalFlow()
    a.calculateOpticalFlow()
    batch.calculateOpticalFlow()
    _assert_same(_result(a), _result(lone), "member used alone in between")
    batch.close()
    for c in (a, b, lone):
        c.close()


@pytest.mark.gpu
def test_members_on_different_devices_are_refused(synth):
    import torch
    import hopperrender_b200 as hr
    if torch.cuda.device_count() < 2:
        pytest.skip(f"{torch.cuda.device_count()} CUDA device: members on two devices need at least 2")
    a = _calc(_member_spec(0), 448, 256, 256, 9)
    cls = hr.OpticalFlowCalcSDR
    b = cls(256, 448, 0, 0, 8, 6, 0.0, 255.0, 256, 1)
    b.m_opticalFlowSearchRadius = 9
    with pytest.raises(RuntimeError, match="hrb error 1.*device"):
        hr.FlowBatch([a, b])
    a.close()
    b.close()


@pytest.mark.gpu
def test_statistics_per_member(synth):
    """ofc_calc_count counts each member's own calculations, and total_frame_delta uses each member's SDR or HDR divisor."""
    import hopperrender_b200 as hr
    W, H, maxres, R = 1920, 1080, 270, 16
    specs = [dict(_member_spec(k), lag=False) for k in range(2)]
    assert specs[0]["hdr"] != specs[1]["hdr"]
    calcs = [_calc(s, W, H, maxres, R) for s in specs]
    for c, s in zip(calcs, specs):
        for f in _frames(synth, s, W, H):
            c.updateFrame(f)
    calcs[0].calculateOpticalFlow()  # member 0 has one calculation more
    b = hr.FlowBatch(calcs)
    for _ in range(3):
        b.calculateOpticalFlow()
    assert [c.m_ofcCalcCount for c in calcs] == [4, 3]
    lw, lh = calcs[0].m_opticalFlowFrameWidth, calcs[0].m_opticalFlowFrameHeight
    for c, s in zip(calcs, specs):
        raw = c.readRawFrameDelta()
        assert raw > 0
        assert c.m_totalFrameDelta == raw // (lw * lh * (6 if s["hdr"] else 10))
        assert c.m_ofcCalcTime > 0
    b.close()
    for c in calcs:
        c.close()
