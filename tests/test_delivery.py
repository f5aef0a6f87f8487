"""The delivery loop in the library (hrb_delivery_*, include/hrb.h "delivery loop"): DeliverToRenderer's output count,
auto-tuner, flow, frame-delta history, GPU-side scene-change rule and blend advance.  Its frames and decisions are checked
frame for frame against hopperrender_b200.replay.DeliveryLoop(batch=True), over the oracle and over a second CUDA handle
driven with blocking calls."""
import ctypes as C

import numpy as np
import pytest

from conftest import OracleAsCalc, out_array

SRC = 417083                  # 23.976 fps
T144, T60, T240 = 69444, 166667, 41667


# ---- without a device ------------------------------------------------------------------------------------------------
def desc(**kw):
    from hopperrender_b200 import _lib as L
    d = dict(source_frame_time=SRC, target_frame_time=T144, frame_output_mode=2, scene_change_threshold=200, active=1, auto_adjust=0)
    d.update(kw)
    return L.hrb_delivery_desc(**d)


def test_create_checks_its_arguments_without_a_device():
    from hopperrender_b200 import _lib as L
    lib = L.load()
    out = C.c_void_p()
    assert lib.hrb_delivery_create(None, None, C.byref(desc())) == 1
    assert lib.hrb_delivery_create(C.byref(out), None, None) == 1 and b"null" in lib.hrb_last_error()
    assert lib.hrb_delivery_create(C.byref(out), None, C.byref(desc())) == 1 and b"null handle" in lib.hrb_last_error()
    for m in (-1, 7):
        assert lib.hrb_delivery_create(C.byref(out), None, C.byref(desc(frame_output_mode=m))) == 1 and b"0..6" in lib.hrb_last_error()
    for kw in (dict(source_frame_time=0), dict(target_frame_time=-5), dict(source_frame_time=-1)):
        assert lib.hrb_delivery_create(C.byref(out), None, C.byref(desc(**kw))) == 1 and b"positive" in lib.hrb_last_error()
    # 23.976 -> 480 fps needs 21 output frames for the first source frame: more than the output ring holds
    assert lib.hrb_delivery_create(C.byref(out), None, C.byref(desc(target_frame_time=20833))) == 1 and b"more than 16" in lib.hrb_last_error()
    # ... unless interpolation is off: then every step is one copy
    assert lib.hrb_delivery_create(C.byref(out), None, C.byref(desc(target_frame_time=20833, active=0))) == 1 and b"null handle" in lib.hrb_last_error()
    assert out.value is None


def test_null_delivery_is_an_argument_error():
    from hopperrender_b200 import _lib as L
    lib = L.load()
    n = C.c_int()
    fr = (L.hrb_delivery_frame * 16)()
    o = L.hrb_delivery_outcome()
    assert lib.hrb_delivery_next_count(None, C.byref(n)) == 1
    assert lib.hrb_delivery_step(None, fr, 16, C.byref(n)) == 1
    assert lib.hrb_delivery_step_to(None, None, 16, fr, C.byref(n)) == 1
    assert lib.hrb_delivery_outcome_of(None, 0, 1, C.byref(o)) == 1
    assert lib.hrb_delivery_set(None, C.byref(desc())) == 1
    assert lib.hrb_delivery_new_segment(None, 1.0) == 1
    lib.hrb_delivery_destroy(None)


# ---- helpers ---------------------------------------------------------------------------------------------------------
class BatchOracle(OracleAsCalc):
    """OracleAsCalc with warpFramesBatch: frame i of the batch is warped when downloadFrame i fetches it."""

    def __init__(self, o):
        super().__init__(o)
        self._pending, self._mode = [], 0

    def warpFramesBatch(self, ts, mode):
        self._pending, self._mode = list(ts), mode

    def downloadFrame(self, out):
        if self._pending:
            self._o.warpFrames(self._pending.pop(0), self._mode)
        self._o.downloadFrame(out)


def oracle_calc(hdr, H, W, R, maxres=270):
    from oracle import OracleCalc
    o = BatchOracle(OracleCalc(H, W, W, W, 8, 6, 0.0, 255.0, maxres, hdr))
    o.m_opticalFlowSearchRadius = R
    return o


def cuda_calc(hdr, H, W, R, maxres=270):
    import hopperrender_b200 as hr
    c = (hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR)(H, W, 0, 0, 8, 6, 0.0, 255.0, maxres)
    c.m_opticalFlowSearchRadius = R
    return c


def cut_frames(synth, W, H, hdr, n, cut=6, switch=11):
    """A moving synthetic scene with a random frame inserted at `cut` and a different synthetic scene from `switch` on."""
    fs = [synth.make_frame(W, H, t, synth.SEED_BASE + (7 if t >= switch else 0), hdr) for t in range(n)]
    if cut is not None and cut < n:
        fs[cut] = synth.make_random_frame(W, H, 77, hdr)
    return fs


def rule(hist):
    """(d1, d2) of replay.DeliveryLoop._scene_change on a frameDeltaHistory (0, 0 below three entries)."""
    n = len(hist)
    if n < 3:
        return 0, 0
    count = min(n - 2, 10)
    avg = sum(int(hist[n - 2 - i][1]) for i in range(count)) // count
    cur, nxt = int(hist[n - 2][1]), int(hist[n - 1][1])
    return cur - avg, cur - nxt


def apply_loop(loop, op):
    kind, arg = op
    if kind == "segment":
        loop.new_segment(arg)
    elif kind == "reset":
        loop.calc.m_frameCount = 0
    elif kind == "set":
        c = loop.calc
        loop.update_user_settings(arg.get("active", True), arg.get("mode", loop.iFrameOutput), arg.get("fps", 0.0), False,
                                  c.m_deltaScalar, c.m_neighborBiasScalar, c.m_outputBlackLevel, c.m_outputWhiteLevel, loop.iSceneChangeThreshold, 0)


def apply_delivery(d, op):
    kind, arg = op
    if kind == "segment":
        d.new_segment(arg)
    elif kind == "reset":
        d.calc.m_frameCount = 0
    elif kind == "set":
        fps = arg.get("fps")
        d.set_settings(active=arg.get("active", True), frame_output=arg.get("mode"),
                       target_frame_time=int((1.0 / float(fps)) * 1e7) if fps else None)


def run_loop(calc, frames, hdr, kw, ops=None, radii=None):
    """replay.DeliveryLoop(batch=True): per output frame (info, bytes, (d1, d2) of the rule, history length, peaks)."""
    from hopperrender_b200 import replay
    loop = replay.DeliveryLoop(calc, auto_adjust=False, **kw)
    loop.batch = True
    out = out_array(calc, hdr)
    got = []

    def sink(buf, info):
        h = list(loop.frameDeltaHistory)
        got.append((dict(info), buf.copy(), rule(h), len(h), (loop.iPeakSceneChangeDelta, loop.iPeakSceneChangeDelta2)))
    for k, f in enumerate(frames):
        for op in (ops or {}).get(k, []):
            apply_loop(loop, op)
        if radii is not None:
            calc.m_opticalFlowSearchRadius = radii[k]
        loop.deliver(f, out, sink=sink)
    return got


def device_planes(frame, H, W, hdr):
    import torch
    f = torch.from_numpy(frame.view(np.int16) if hdr else frame).cuda().reshape(H + H // 2, W)
    return f[:H], f[H:]


def padded_outs(n, H, W, hdr):
    """n destinations with padded pitches, each in an allocation of its own."""
    import torch
    dt = torch.int16 if hdr else torch.uint8
    outs = []
    for _ in range(n):
        y = torch.zeros((H, W + 64), dtype=dt, device="cuda")[:, :W]
        uv = torch.zeros((H // 2, W + 128), dtype=dt, device="cuda")[:, :W]
        outs.append((y, uv))
    return outs


def run_delivery(calc, frames, hdr, kw, ops=None, to=False):
    """hopperrender_b200.Delivery over a CUDA calculator: per output frame (info, bytes, outcome, radius)."""
    import hopperrender_b200 as hr
    import torch
    H, W = calc.m_frameHeight, calc.m_frameWidth
    d = hr.Delivery(calc, **dict(dict(auto_adjust=False), **kw))  # as run_loop, unless the test turns the tuner on
    got = []
    try:
        out = out_array(calc, hdr)
        for k, f in enumerate(frames):
            for op in (ops or {}).get(k, []):
                apply_delivery(d, op)
            if not to:
                d.deliver(f, out, sink=lambda buf, info: got.append((dict(info), buf.copy(), info["outcome"], info["radius"])))
                continue
            y, uv = device_planes(f, H, W, hdr)
            outs = padded_outs(d.next_count(), H, W, hdr)
            infos = d.deliver_to(y, uv, outs)
            calc.synchronize()
            radius = calc.m_opticalFlowSearchRadius
            for info, (oy, ouv) in zip(infos, outs):
                o = d.outcome(info["step"])
                buf = torch.cat([oy.reshape(-1), ouv.reshape(-1)]).cpu().numpy()
                info.update(warped=o["warped"], scene_change=o["scene_change"])
                got.append((info, buf.view(np.uint16) if hdr else buf, o, radius))
    finally:
        d.close()
    return got


def assert_same(got, exp, src_fps=SRC):
    """Frame for frame: bytes, source, index, blend, warped, scene change, the rule's deltas and the peaks built from them."""
    assert len(got) == len(exp) > 0
    frames_in_1s = int(1.0 * 10000000.0 / src_fps)
    peaks_hist, peaks = [], (0, 0)
    for k, ((gi, gb, o, _), (ei, eb, (d1, d2), n_hist, epeaks)) in enumerate(zip(got, exp)):
        where = f"output {k} (source {ei['source']}, index {ei['index']})"
        for key in ("source", "index", "blend", "warped", "scene_change"):
            assert gi[key] == ei[key], f"{where}: {key} {gi[key]} != {ei[key]}"
        assert (o["delta1"], o["delta2"]) == (d1, d2), f"{where}: deltas {(o['delta1'], o['delta2'])} != {(d1, d2)}"
        assert np.array_equal(gb, eb), f"{where}: delivered bytes differ"
        if ei["index"] == 0 and n_hist == 0:
            peaks_hist, peaks = [], (0, 0)  # history cleared (set / new_segment)
        if n_hist >= 3 and d1 > 0:
            peaks_hist.append((ei["source"], d1, max(d2, 0)))
            while peaks_hist and ei["source"] - peaks_hist[0][0] > frames_in_1s:
                peaks_hist.pop(0)
            best = (0, 0)
            for _, a, b in peaks_hist:
                if a > best[0]:
                    best = (a, b)
            peaks = best
        if n_hist >= 3:
            assert peaks == epeaks, f"{where}: peaks {peaks} != {epeaks}"


# ---- against the oracle ----------------------------------------------------------------------------------------------
ORACLE_CASES = [  # mode, hdr, W, H, target
    (0, False, 256, 144, T144), (1, True, 320, 200, T60), (2, False, 320, 200, T144), (3, True, 256, 144, T144),
    (4, False, 256, 144, T60), (5, True, 320, 200, T144), (6, False, 320, 200, T60), (2, True, 256, 144, T60),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,hdr,W,H,target", ORACLE_CASES)
@pytest.mark.parametrize("to", [False, True], ids=["ring", "to"])
def test_delivery_matches_the_python_loop_over_the_oracle(synth, mode, hdr, W, H, target, to):
    """16 source frames with a random frame and a scene switch: more than 12 history entries, so the average spans 10."""
    frames = cut_frames(synth, W, H, hdr, 16)
    kw = dict(target_frame_time=target, frame_output=mode)
    exp = run_loop(oracle_calc(hdr, H, W, 7), frames, hdr, kw)
    got = run_delivery(cuda_calc(hdr, H, W, 7), frames, hdr, kw, to=to)
    assert_same(got, exp)
    assert any(not i["warped"] and i["source"] >= 3 for i, *_ in exp), "a cut should have forced a copy"
    assert max(n for *_, n, _ in exp) > 12


@pytest.mark.gpu
@pytest.mark.parametrize("to", [False, True], ids=["ring", "to"])
def test_settings_segments_and_resets_match_the_python_loop(synth, to):
    """new_segment at rates 0.5, 1 and 2, activation off and on, a new target rate and a frame-count reset, between steps."""
    W, H, hdr = 256, 144, False
    frames = cut_frames(synth, W, H, hdr, 22, cut=5, switch=15)
    ops = {4: [("segment", 0.5)], 8: [("set", dict(active=False))], 10: [("set", dict(active=True, fps=60.0))], 13: [("segment", 2.0)],
           16: [("reset", None)], 18: [("segment", 1.0), ("set", dict(active=True, fps=144.0, mode=1))]}
    kw = dict(target_frame_time=T144, frame_output=2)
    exp = run_loop(oracle_calc(hdr, H, W, 6), frames, hdr, kw, ops)
    got = run_delivery(cuda_calc(hdr, H, W, 6), frames, hdr, kw, ops, to=to)
    assert_same(got, exp)


# ---- at production sizes, against the blocking calls of a second CUDA handle ------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,maxres,R,cut,switch,thr", [(False, 1920, 1080, 270, 16, 6, 99, 200), (True, 3840, 2160, 2160, 16, None, 5, 1)],
                         ids=["1080p-nv12-random-frame", "4k-p010-full-res-scene-switch"])
@pytest.mark.parametrize("to", [False, True], ids=["ring", "to"])
def test_delivery_matches_blocking_calls_at_production_sizes(synth, hdr, W, H, maxres, R, cut, switch, thr, to):
    """At 4K with a full-resolution flow the frame deltas are a few units (the raw sum over 3840 x 2160 x 6): the cut there
    is a switch to another scene under a threshold of 1."""
    frames = cut_frames(synth, W, H, hdr, 9, cut=cut, switch=switch)
    kw = dict(target_frame_time=T144, frame_output=2, scene_change_threshold=thr)
    exp = run_loop(cuda_calc(hdr, H, W, R, maxres), frames, hdr, kw)
    got = run_delivery(cuda_calc(hdr, H, W, R, maxres), frames, hdr, kw, to=to)
    assert_same(got, exp)
    assert any(not i["warped"] and i["source"] >= 3 for i, *_ in exp)


# ---- ordering ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_decisions_read_the_flow_of_their_step_without_host_waits(synth):
    """48 source frames at 4K issued in runs of 16 steps with no host wait in between (device ingest of frame N+1 beside the
    flow of frame N): every outcome's frame delta is the total_frame_delta that flow has when computed alone."""
    import hopperrender_b200 as hr
    W, H, hdr = 3840, 2160, True
    base = [synth.make_frame(W, H, t, synth.SEED_BASE + 3, hdr) for t in range(7)]
    base[3] = synth.make_random_frame(W, H, 5, hdr)  # steps next to it have large deltas: a stale read would show
    order = [i for _ in range(4) for i in list(range(7)) + list(range(5, 0, -1))][:48]
    a = cuda_calc(hdr, H, W, 12, 2160)
    d = hr.Delivery(a, target_frame_time=T60, frame_output=2, auto_adjust=False)
    planes = [device_planes(f, H, W, hdr) for f in base]
    outs = padded_outs(3, H, W, hdr)
    outcomes = []
    for run in range(3):
        steps = []
        for k in order[16 * run:16 * run + 16]:
            steps += [i["step"] for i in d.deliver_to(*planes[k], outs)][:1]
        outcomes += [d.outcome(s) for s in steps]
    d.close()
    b = cuda_calc(hdr, H, W, 12, 2160)
    deltas = []
    for k in order:
        b.updateFrame(base[k])
        if b.m_frameCount >= 3:
            b.calculateOpticalFlow()
            deltas.append(b.m_totalFrameDelta)
        else:
            deltas.append(0)
    assert [o["frame_delta"] for o in outcomes] == deltas
    assert sum(x != y for x, y in zip(deltas[2:], deltas[3:])) >= 10


# ---- rule edges --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_threshold_flips_exactly_at_greater_or_equal(synth):
    W, H, hdr = 256, 144, False
    frames = cut_frames(synth, W, H, hdr, 10, cut=6, switch=99)
    kw = dict(target_frame_time=T60, frame_output=2)
    base = run_delivery(cuda_calc(hdr, H, W, 7), frames, hdr, dict(kw, scene_change_threshold=200))
    for i, _, o, _ in base[:2]:
        assert o["delta1"] == 0 and o["delta2"] == 0 and not o["scene_change"]  # fewer than 3 history entries
    cut = [o for _, _, o, _ in base if o["scene_change"]]
    assert cut, "the random frame should be detected at the default threshold"
    t = min(cut[0]["delta1"], cut[0]["delta2"])
    at = run_delivery(cuda_calc(hdr, H, W, 7), frames, hdr, dict(kw, scene_change_threshold=t))
    above = run_delivery(cuda_calc(hdr, H, W, 7), frames, hdr, dict(kw, scene_change_threshold=t + 1))
    k = next(j for j, (_, _, o, _) in enumerate(base) if o["scene_change"])
    assert at[k][2]["scene_change"] and not at[k][0]["warped"]
    assert not above[k][2]["scene_change"] and above[k][0]["warped"]


# ---- output counts -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("to", [False, True], ids=["ring", "to"])
def test_steps_of_more_than_eight_frames(synth, to):
    """23.976 -> 240 fps: 10 or 11 output frames per source frame, two warp batches under one decision."""
    W, H, hdr = 640, 360, False
    frames = cut_frames(synth, W, H, hdr, 8, cut=5, switch=99)
    kw = dict(target_frame_time=T240, frame_output=2)
    exp = run_loop(cuda_calc(hdr, H, W, 8), frames, hdr, kw)
    got = run_delivery(cuda_calc(hdr, H, W, 8), frames, hdr, kw, to=to)
    assert_same(got, exp)
    assert max(i["index"] for i, *_ in got) >= 9


@pytest.mark.gpu
def test_settings_needing_more_than_16_frames_are_refused(synth):
    import hopperrender_b200 as hr
    c = cuda_calc(False, 144, 256, 5)
    d = hr.Delivery(c, target_frame_time=T240)
    with pytest.raises(RuntimeError, match="hrb error 1.*more than 16"):
        d.new_segment(0.5)  # playback 834166 / 41667: 21 frames
    with pytest.raises(RuntimeError, match="hrb error 1.*more than 16"):
        d.set_settings(target_frame_time=20833)
    assert d.next_count() == 11  # unchanged
    d.close()


# ---- auto-tuner --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("src,target,start,end", [(10, 2, 16, 5), (10 ** 9, 2 * 10 ** 8, 5, 16)], ids=["down", "up"])
def test_auto_tuner_on_unambiguous_timings(synth, src, target, start, end):
    W, H, hdr = 640, 360, False
    frames = cut_frames(synth, W, H, hdr, 15, cut=None, switch=99)
    kw = dict(source_frame_time=src, target_frame_time=target, frame_output=2)
    got = run_delivery(cuda_calc(hdr, H, W, start), frames, hdr, dict(kw, auto_adjust=True))
    radii = []
    for i, _, _, r in got:
        if i["index"] == 0:
            radii.append(r)
    # the first step has no timing yet (0 < source frame time / 1.6): it steps up, which at 16 leaves the radius alone
    exp_radii = [max(16 - k, 5) for k in range(len(frames))] if end < start else [min(start + k + 1, 16) for k in range(len(frames))]
    assert radii == exp_radii
    from hopperrender_b200 import replay
    exp = run_loop(cuda_calc(hdr, H, W, start), frames, hdr, dict(kw, source_frame_time=src), radii=radii)
    assert replay.num_int_frames(0.0, target, src) == 5
    assert_same(got, exp, src_fps=src)


# ---- exclusive use -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_exclusive_use_while_attached(synth):
    import hopperrender_b200 as hr
    W, H, hdr = 256, 144, False
    c = cuda_calc(hdr, H, W, 5)
    fs = cut_frames(synth, W, H, hdr, 4, cut=None, switch=99)
    d = hr.Delivery(c, target_frame_time=T60)
    with pytest.raises(RuntimeError, match="hrb error 5"):
        hr.Delivery(c)  # one delivery per handle
    with pytest.raises(RuntimeError, match="hrb error 5"):
        hr.FlowBatch([c])
    out = out_array(c, hdr)
    for f in fs:
        d.deliver(f, out)  # ingest and downloads work
    y, uv = padded_outs(1, H, W, hdr)[0]
    for call in (c.calculateOpticalFlow, c.calculateOpticalFlowAsync, lambda: c.warpFrames(0.5, 2), lambda: c.warpFramesBatch([0.5], 2),
                 c.copyFrame, lambda: c.warpFramesTo([0.5], 2, [(y, uv)]), lambda: c.copyFrameTo((y, uv))):
        with pytest.raises(RuntimeError, match="hrb error 5.*delivery attached"):
            call()
    c.updateFrame(fs[0])
    assert c.m_totalFrameDelta >= 0 and c.m_frameCount == 5
    d.close()
    c.calculateOpticalFlow()
    c.warpFrames(0.5, 2)
    c.downloadFrame(out)
    c.copyFrameTo((y, uv))
    hr.FlowBatch([c]).close()
