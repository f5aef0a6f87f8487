"""Split search (hrb_split_*, SplitSearch): a group of handles computes one flow, each shard searching the windows of its
flow-row stripe in the passes with windows of at most 128 rows, with halo rows exchanged between iterations.  Every
handle of the group must end up with exactly the flow a lone handle computes: offsets, blurred flow, flow peak and frame
delta, pass by pass in tap mode, over asynchronous sequences with warps in between, and against the oracle.

All GPU tests run on one device (shards of a group may share a device); the multi-device case runs where there are
several GPUs and skips otherwise.
"""
import numpy as np
import pytest

from test_ladder_shapes import mosaic_frames

ALIGN = 128  # kSplitAlign (hrb_internal.cuh)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the stripe plan
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lh", [256, 270, 540, 576, 1080, 1800, 2160, 4320])
def test_split_plan_bounds(lh):
    """Bounds are multiples of 128 from 0 to lh, strictly increasing, every stripe within 128 rows of lh / n; an n that
    would leave a stripe empty is rejected, and so is n < 1."""
    import hopperrender_b200 as hr
    accepted = 0
    for n in range(1, 9):
        want = [ALIGN * int(np.floor(k * lh / (n * ALIGN) + 0.5)) for k in range(n)] + [lh]
        if any(b1 <= b0 for b0, b1 in zip(want, want[1:])):
            with pytest.raises(RuntimeError, match="hrb error 1"):
                hr.split_plan(lh, n)
            continue
        b = hr.split_plan(lh, n)
        accepted += 1
        assert b == want
        assert b[0] == 0 and b[-1] == lh
        assert all(x % ALIGN == 0 for x in b[:-1])
        assert all(b1 > b0 for b0, b1 in zip(b, b[1:]))
        assert all(abs((b1 - b0) - lh / n) <= ALIGN for b0, b1 in zip(b, b[1:])), b
    assert accepted >= 2  # n = 1 and n = 2 always fit these heights
    for n in (0, -1, 65):
        with pytest.raises(RuntimeError, match="hrb error 1"):
            hr.split_plan(lh, n)
    with pytest.raises(RuntimeError, match="hrb error 1"):
        hr.split_plan(lh, lh // ALIGN + 2)


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _calc(hdr, W, H, inS=0, maxres=None, R=16, ds=8, ns=6, variant=0, device=0):
    import hopperrender_b200 as hr
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    g = cls(H, W, inS, 0, ds, ns, 0.0, 255.0, maxres or H, device)
    g.m_opticalFlowSearchRadius = R
    if variant:
        g.setSearchVariant(variant)
    return g


def _frames(synth, kind, W, H, hdr, inS=0):
    if kind == "mosaic":
        return mosaic_frames(synth, W, H, hdr, seed=W + H, stride=inS or None)
    return [synth.make_frame(W, H, t, synth.SEED_BASE + 5, hdr, inS or None) for t in range(3)]


def _result(c):
    return dict(offsets=c.readOffsetArray(), flow=c.readFlow(latest=True), peak=c.readFlowPeak()[1], delta=c.m_totalFrameDelta)


def _assert_same(got, want, label):
    assert np.array_equal(got["offsets"], want["offsets"]), f"{label}: {np.count_nonzero(got['offsets'] != want['offsets'])} offsets differ"
    assert np.array_equal(got["flow"], want["flow"]), f"{label}: {np.count_nonzero(got['flow'] != want['flow'])} flow values differ"
    assert got["peak"] == want["peak"], f"{label}: flow peak {got['peak']} != {want['peak']}"
    assert got["delta"] == want["delta"], f"{label}: frame delta {got['delta']} != {want['delta']}"


def _group_equals_lone(synth, hdr, W, H, inS, maxres, R, ns, variant, kind, ns_list, devices=None):
    import hopperrender_b200 as hr
    frames = _frames(synth, kind, W, H, hdr, inS)
    lone = _calc(hdr, W, H, inS, maxres, R, ns=ns, variant=variant)
    for f in frames:
        lone.updateFrame(f)
    lone.calculateOpticalFlow()
    want = _result(lone)
    lone.close()
    ndev = devices or 1
    for n in ns_list:
        calcs = [_calc(hdr, W, H, inS, maxres, R, ns=ns, variant=variant, device=k % ndev) for k in range(n)]
        for c in calcs:
            for f in frames:
                c.updateFrame(f)
        grp = hr.SplitSearch(calcs)
        grp.calculateOpticalFlow()
        for k, c in enumerate(calcs):
            _assert_same(_result(c), want, f"{kind} {W}x{H} R {R} n {n}: shard {k} (rows {grp.stripe(k)})")
        grp.close()
        for c in calcs:
            c.close()


GROUP_CASES = [
    # hdr, W, H, inS, maxres, R, neighbour scalar, variant, frames, shard counts
    (False, 1024, 576, 0, 576, 16, 6, 0, "scene", (2, 3, 4)),
    (False, 1024, 576, 0, 576, 16, 6, 0, "mosaic", (2, 3, 4)),
    (False, 2560, 1440, 2688, 1440, 16, 6, 0, "scene", (2, 5)),        # padded stride
    (True, 3200, 1800, 0, 1800, 13, 6, 0, "scene", (3,)),              # lh not a multiple of 128
    (True, 3840, 2160, 0, 2160, 16, 6, 0, "scene", (2, 4, 8)),
    (True, 3840, 2160, 0, 2160, 16, 6, 0, "mosaic", (4,)),
    (True, 7680, 4320, 0, 4320, 16, 6, 0, "scene", (2, 8)),
    (False, 1920, 1080, 0, 540, 9, 6, 0, "mosaic", (2,)),              # reduced-resolution flow: the generic kernel
    (False, 1024, 576, 0, 576, 9, 6, 1, "mosaic", (3,)),               # variant 1: the generic kernel everywhere
    (False, 1024, 576, 0, 576, 5, 6, 2, "mosaic", (2,)),               # variant 2: the tile kernel down to windows of 4
    (False, 1024, 576, 0, 576, 16, 0, 0, "mosaic", (2,)),              # neighbour scalar 0
    (False, 1024, 576, 0, 576, 16, 31, 0, "mosaic", (3,)),             # neighbour scalar 31
]


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,inS,maxres,R,ns,variant,kind,nlist", GROUP_CASES)
def test_group_equals_lone_handle(synth, hdr, W, H, inS, maxres, R, ns, variant, kind, nlist):
    """Every handle of the group holds the lone handle's final offsets, blurred flow, flow peak and frame delta."""
    _group_equals_lone(synth, hdr, W, H, inS, maxres, R, ns, variant, kind, nlist)


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,R,n,kind", [(False, 1024, 576, 16, 3, "mosaic"), (True, 3840, 2160, 16, 4, "scene")])
def test_taps_pass_by_pass(synth, hdr, W, H, R, n, kind):
    """In replicated passes (windows > 128) every shard's taps equal the lone handle's; in sharded passes the owned window
    rows do, and the other rows of the sums and layer taps are still zero (the shard did not compute them)."""
    import hopperrender_b200 as hr
    frames = _frames(synth, kind, W, H, hdr)
    lone = _calc(hdr, W, H, R=R)
    calcs = [_calc(hdr, W, H, R=R) for _ in range(n)]
    for c in [lone] + calcs:
        for f in frames:
            c.updateFrame(f)
        c.setTapMode(True)
    lone.calculateOpticalFlow()
    grp = hr.SplitSearch(calcs)
    grp.calculateOpticalFlow()
    npass = lone.numPasses()
    sharded_nb = 0
    for k, c in enumerate(calcs):
        assert c.numPasses() == npass
        b0, b1 = grp.stripe(k)
        for p in range(npass):
            info = lone.passInfo(p)
            assert c.passInfo(p) == info
            ws = info["windowSize"]
            where = f"shard {k} rows [{b0}, {b1}) pass {p} (ws {ws}, iteration {info['iteration']}, step {info['step']})"
            s, ls = c.readPassSums(p, R), lone.readPassSums(p, R)
            y, ly = c.readPassLayers(p), lone.readPassLayers(p)
            o, lo = c.readPassOffsets(p), lone.readPassOffsets(p)
            if ws > ALIGN:
                assert np.array_equal(s, ls) and np.array_equal(y, ly) and np.array_equal(o, lo), f"{where}: replicated pass differs"
                continue
            w0, w1 = b0 // ws, -(-b1 // ws)
            assert np.array_equal(s[:, w0:w1], ls[:, w0:w1]), f"{where}: owned sums differ"
            assert np.array_equal(y[w0:w1], ly[w0:w1]), f"{where}: owned layers differ"
            assert np.array_equal(o[:, b0:b1], lo[:, b0:b1]), f"{where}: owned offsets differ"
            assert not s[:, :w0].any() and not s[:, w1:].any(), f"{where}: sums outside the stripe were written"
            assert not y[:w0].any() and not y[w1:].any(), f"{where}: layers outside the stripe were written"
            assert ls[:, w0:w1].any(), f"{where}: the lone handle has only zero sums in the stripe (the zero check proves nothing)"
            sharded_nb += info["iteration"] >= 4
        _assert_same(_result(c), _result(lone), f"shard {k}")
    assert sharded_nb > 0, "no sharded pass with the neighbour bias (iteration >= 4)"
    grp.close()
    for c in [lone] + calcs:
        c.close()


@pytest.mark.gpu
def test_async_sequence_with_warps(synth):
    """Six frames through calculateOpticalFlowAsync with flow overlap on and a batch of warps issued after every
    calculate: every flow and every mode-2 output of every shard equals the lone handle's (stale halos or a level-parity
    mix-up between consecutive calculations would show here)."""
    import hopperrender_b200 as hr
    W, H, R, n = 1024, 576, 16, 3
    base = mosaic_frames(synth, W, H, False, seed=11)
    seq = [base[1], base[2]] + [synth.make_frame(W, H, t, synth.SEED_BASE + 9, False) for t in range(4)]
    lone = _calc(False, W, H, R=R)
    calcs = [_calc(False, W, H, R=R) for _ in range(n)]
    grp = hr.SplitSearch(calcs)
    ts = [0.25, 0.5, 0.75]
    for t, f in enumerate(seq):
        for c in [lone] + calcs:
            c.updateFrame(f)
        if t < 1:
            continue
        lone.calculateOpticalFlowAsync()
        grp.calculateOpticalFlowAsync()
        outs = {}
        for i, c in enumerate([lone] + calcs):
            c.warpFramesBatch(ts, 2)
            outs[i] = []
            for _ in ts:
                a = np.zeros(c.outputFrameBytes, np.uint8)
                c.downloadFrame(a)
                outs[i].append(a)
        for k in range(n):
            for j in range(len(ts)):
                assert np.array_equal(outs[k + 1][j], outs[0][j]), f"frame {t}: shard {k} output {j} differs"
        want = dict(forwarp=lone.readFlow(), latest=lone.readFlow(latest=True), peak=lone.readFlowPeak(), delta=lone.m_totalFrameDelta)
        for k, c in enumerate(calcs):
            assert np.array_equal(c.readFlow(), want["forwarp"]), f"frame {t}: shard {k} flow for warp differs"
            assert np.array_equal(c.readFlow(latest=True), want["latest"]), f"frame {t}: shard {k} latest flow differs"
            assert c.readFlowPeak() == want["peak"] and c.m_totalFrameDelta == want["delta"], f"frame {t}: shard {k}"
    grp.close()
    for c in [lone] + calcs:
        c.close()


@pytest.mark.gpu
def test_stripes_warped_by_shards_equal_the_oracle(synth):
    """SDR 448x256, two shards, R 9: each shard warps its own output stripe; the merged frames equal OracleCalc's."""
    import hopperrender_b200 as hr
    from oracle import OracleCalc
    W, H, R = 448, 256, 9
    o = OracleCalc(H, W, 0, 0, 8, 6, 0.0, 255.0, 270, False)
    o.setParams(searchRadius=R)
    calcs = [_calc(False, W, H, maxres=270, R=R) for _ in range(2)]
    grp = hr.SplitSearch(calcs)
    rs = calcs[0].m_opticalFlowResScalar
    for k, c in enumerate(calcs):
        b0, b1 = grp.stripe(k)
        c.setOutputStripe(b0 << rs, min(b1 << rs, H))
    for t in range(4):
        f = synth.make_frame(W, H, t, synth.SEED_BASE + 2, False)
        o.updateFrame(f)
        for c in calcs:
            c.updateFrame(f)
        if t < 2:
            continue
        o.calculateOpticalFlow()
        grp.calculateOpticalFlow()
        for c in calcs:
            assert np.array_equal(c.readOffsetArray(), o.readOffsetArray()) and np.array_equal(c.readFlow(latest=True), o.readFlow(latest=True))
        for mode in (2, 0):
            o.warpFrames(0.5, mode)
            want = np.zeros(calcs[0].outputFrameBytes, np.uint8)
            o.downloadFrame(want)
            got = np.zeros_like(want)
            for c in calcs:
                c.warpFrames(0.5, mode)
                c.downloadFrame(got)
            assert np.array_equal(got, want), f"frame {t} mode {mode}: merged stripes differ from the oracle"
    grp.close()
    o.close()
    for c in calcs:
        c.close()


@pytest.mark.gpu
def test_argument_checks(synth):
    """Handles that disagree are refused (at create, or at calculate when a parameter changed since), naming the field;
    too many shards, a repeated handle and the profile are refused; a group of one equals the lone handle."""
    import hopperrender_b200 as hr
    W, H = 448, 256
    a, b = _calc(False, W, H, R=9), _calc(False, W, H, R=9)
    for other, field in [(_calc(False, 512, H, R=9), "frame_width"), (_calc(True, W, H, R=9), "is_hdr"),
                         (_calc(False, W, H, maxres=128, R=9), "res_scalar"), (_calc(False, W, H, R=9, ds=7), "delta_scalar"),
                         (_calc(False, W, H, R=9, ns=31), "neighbor_bias_scalar"), (_calc(False, W, H, R=10), "search_radius")]:
        with pytest.raises(RuntimeError, match=f"hrb error 1.*{field}"):
            hr.SplitSearch([a, other])
        other.close()
    with pytest.raises(RuntimeError, match="hrb error 1"):
        hr.SplitSearch([a, b, _calc(False, W, H, R=9)])  # 256 flow rows hold two stripes
    with pytest.raises(RuntimeError, match="hrb error 1.*twice"):
        hr.SplitSearch([a, a])
    fs = _frames(synth, "scene", W, H, False)
    for c in (a, b):
        for f in fs:
            c.updateFrame(f)
    grp = hr.SplitSearch([a, b])
    for change, field in [(lambda c: setattr(c, "m_opticalFlowSearchRadius", 16), "search_radius"),
                          (lambda c: setattr(c, "m_neighborBiasScalar", 3), "neighbor_bias_scalar"),
                          (lambda c: c.setSearchVariant(1), "search_variant")]:
        change(b)
        with pytest.raises(RuntimeError, match=f"hrb error 1.*{field}"):
            grp.calculateOpticalFlow()
        change(a)
        grp.calculateOpticalFlow()  # agree again
    b.setProfile(True)
    with pytest.raises(RuntimeError, match="hrb error 5"):
        grp.calculateOpticalFlowAsync()
    b.setProfile(False)
    grp.close()
    one = hr.SplitSearch([a])
    assert one.stripe(0) == (0, 256)
    b.calculateOpticalFlow()
    one.calculateOpticalFlow()
    _assert_same(_result(a), _result(b), "group of one")
    one.close()
    a.close()
    b.close()


@pytest.mark.gpu
def test_group_equals_lone_handle_across_devices(synth):
    """The 3840x2160 case with shard k on device k mod count: copies between devices go peer to peer."""
    import torch
    count = torch.cuda.device_count()
    if count < 2:
        pytest.skip(f"{count} CUDA device: the cross-device exchange needs at least 2")
    _group_equals_lone(synth, True, 3840, 2160, 0, 2160, 16, 6, 0, "scene", (2, 4, 8), devices=count)


def _lag(calc, cycles):
    """Queue a kernel that spins for `cycles` clocks on the calculator's compute stream, so that everything the calculator
    enqueues after it (here: its part of the next grouped calculate) starts late."""
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.stream(torch.cuda.ExternalStream(calc.streamHandle(), device=dev)):
        torch.cuda._sleep(int(cycles))


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,R,n,kind", [(True, 3840, 2160, 16, 8, "scene"), (False, 1024, 576, 16, 4, "mosaic")])
def test_lagging_shard(synth, hdr, W, H, R, n, kind):
    """One shard starts its part of a grouped calculate tens of milliseconds after the others (a long kernel ahead of it
    on its compute stream, as a warp batch or a serial frame upload would put it): the other shards must still wait for
    it wherever they read or write its level arrays, so every shard ends with the lone handle's flow, bit for bit.  The
    lagging shard is the last, the first and a middle one in turn, over consecutive calculations."""
    import hopperrender_b200 as hr
    frames = _frames(synth, kind, W, H, hdr)
    lone = _calc(hdr, W, H, R=R)
    for f in frames:
        lone.updateFrame(f)
    lone.calculateOpticalFlow()
    want = _result(lone)
    lone.close()
    calcs = [_calc(hdr, W, H, R=R) for _ in range(n)]
    for c in calcs:
        for f in frames:
            c.updateFrame(f)
    grp = hr.SplitSearch(calcs)
    for lagging in (n - 1, 0, n // 2):
        _lag(calcs[lagging], 1e8)
        grp.calculateOpticalFlowAsync()
        for k, c in enumerate(calcs):
            _assert_same(_result(c), want, f"{kind} {W}x{H} n {n}, shard {lagging} lagging: shard {k}")
    grp.close()
    for c in calcs:
        c.close()
