"""The search ladder at the tile shapes, radii and round counts production runs, pass by pass against the oracle.

OracleCalc with taps keeps [R][lh][lw] sums of every pass (12 GB per ladder at 4096x2160, R = 14).  OracleLadder runs the
same schedule (hr_oracle.cpp:548-592) one pass at a time through the oracle's kernel entry points and hands out each
pass's results as it goes, so that a 4K ladder is compared pass by pass in the memory of one pass.  The CPU test below
pins it to OracleCalc bit for bit; the GPU tests compare the CUDA path with it:

  * large frames, where the tile kernel runs with 3..6 warps per CTA (NWV; chooseWarps, kernels_search_slide.cu): the NWV
    each pass ran is read back from the per-CTA debug timeline (word 8);
  * motion-mosaic content, whose blocks move independently by up to ~40 px, so that tile CTAs need 2..4 rounds and the
    per-pixel remainder (round 5, timeline word 7), and small-window CTAs fall back to unstaged fetches;
  * the production path of the same frames (no taps, no timeline, CUDA graph captured and replayed);
  * the search variants that force kernels and staging paths: which passes run the tile kernel, read from the timeline;
  * the timeline's own bound: CTAs whose record does not fit the pass's slice leave no trace.
"""
import numpy as np
import pytest

from oracle import OracleCalc
from oracle import kernels as K

SM_COUNT_OF_TABLE = 148   # the NWV table below was derived for this SM count (B200)


# ---------------------------------------------------------------------------------------------------------------------
# A. the oracle's schedule, one pass at a time
# ---------------------------------------------------------------------------------------------------------------------
def ladder_geometry(lw, lh):
    """First window size and iteration count (hr_oracle.cpp:553-562)."""
    m = max(lw, lh)
    if m and not (m & (m - 1)):
        ws = m
    else:
        while m & (m - 1):
            m &= m - 1
        ws = m << 1
    ws //= 2
    return ws, int(np.log2(ws))


class OracleLadder:
    """The flow calculation of OracleCalc on frame 1 = the second-to-last upload, frame 2 = the last one.

    passes() yields one dict per pass: windowSize, iteration, step, sums and layers at the window representatives
    ([R][nWy][nWx], [nWy][nWx]), offsets after the pass and input_offsets before it ([2][lh][lw]); full=True adds the
    whole [R][lh][lw] sums and [lh][lw] layer buffer as OracleCalc's taps hold them.  frame_delta is set once pass 0
    has run; offsets and flow (the blurred offsets) once the generator is exhausted."""

    def __init__(self, frame1, frame2, hdr, W, H, stride, lh, lw, rs, R, ds, ns):
        dt = np.uint16 if hdr else np.uint8
        self.f1 = np.ascontiguousarray(frame1).view(dt)
        self.f2 = np.ascontiguousarray(frame2).view(dt)
        self.hdr, self.W, self.H, self.stride, self.lh, self.lw, self.rs, self.R, self.ds, self.ns = hdr, W, H, stride, lh, lw, rs, R, ds, ns
        self.frame_delta = self.offsets = self.flow = None

    @classmethod
    def of(cls, frames, hdr, W, H, inS, maxres, R, ds=8, ns=6):
        rs = 0
        while (H >> rs) > maxres:
            rs += 1
        lw, lh = -(-W // (1 << rs)), -(-H // (1 << rs))
        return cls(frames[-2], frames[-1], hdr, W, H, inS or W, lh, lw, rs, R, ds, ns)

    def passes(self, full=False):
        R, lh, lw = self.R, self.lh, self.lw
        ws, iterations = ladder_geometry(lw, lh)
        offs = np.zeros((2, lh, lw), np.int16)
        layers = np.zeros((lh, lw), np.uint8)   # one buffer over the ladder, like the oracle's lowestLayer
        for it in range(iterations):
            for step in (0, 1):
                inp = offs.copy()
                sums = K.calc_delta_sums(self.f1, self.f2, offs, self.H, self.W, self.stride, ws, R, self.rs, it, step, self.ds, self.ns, self.hdr)
                if it == 0 and step == 0:   # hr_oracle.cpp:573-576
                    self.frame_delta = int(sums[R // 2 - 1, 0, 0]) // (lh * lw * (6 if self.hdr else 10))
                K.determine_lowest_layer(sums, layers, ws)
                K.adjust_offset_array(offs, layers, ws, R, step)
                p = dict(windowSize=ws, iteration=it, step=step, sums=sums[:, ::ws, ::ws].copy(), layers=layers[::ws, ::ws].copy(),
                         offsets=offs.copy(), input_offsets=inp)
                if full:
                    p["sums_full"], p["layers_full"] = sums, layers.copy()
                del sums
                yield p
            ws = max(ws >> 1, 1)
        self.offsets = offs
        self.flow = K.blur_flow(offs)


def _frames(synth, W, H, hdr, n, stride=None, kind="scene", seed=0):
    if kind == "scene":
        return [synth.make_frame(W, H, t, synth.SEED_BASE + seed, hdr, stride) for t in range(n)]
    return [synth.make_random_frame(W, H, 1000 + seed + t, hdr, stride) for t in range(n)]


@pytest.mark.parametrize("hdr,W,H,maxres,inS,R,kind", [
    (False, 64, 48, 270, 0, 16, "scene"),
    (True, 64, 48, 270, 80, 2, "random"),      # padded stride, smallest radius
    (False, 258, 146, 73, 272, 16, "scene"),   # rs = 1, padded stride
    (True, 200, 120, 270, 0, 7, "scene"),      # non-power-of-two size, odd radius
    (False, 90, 54, 270, 96, 13, "random"),
])
def test_oracle_ladder_equals_oracle_calc(synth, hdr, W, H, maxres, inS, R, kind):
    """The pass-by-pass generator is OracleCalc with taps, bit for bit: every pass (whole sum and layer buffers, offsets),
    the final offsets, the blurred flow and totalFrameDelta."""
    o = OracleCalc(H, W, inS, 0, 8, 6, 0.0, 255.0, maxres, hdr)
    o.setParams(searchRadius=R)
    o.enableTaps(True)
    fs = _frames(synth, W, H, hdr, 3, inS or None, kind)
    for f in fs:
        o.updateFrame(f)
    o.calculateOpticalFlow()
    lad = OracleLadder.of(fs, hdr, W, H, inS, maxres, R)
    n = 0
    for p, q in enumerate(lad.passes(full=True)):
        info = o.passInfo(p)
        assert (q["windowSize"], q["iteration"], q["step"]) == (info["windowSize"], info["iteration"], info["step"])
        assert np.array_equal(q["sums_full"], o.readPassSums(p, R)), f"pass {p}: sums"
        assert np.array_equal(q["layers_full"], o.readPassLayers(p)), f"pass {p}: layers"
        assert np.array_equal(q["offsets"], o.readPassOffsets(p)), f"pass {p}: offsets"
        prev = o.readPassOffsets(p - 1) if p else np.zeros_like(q["offsets"])
        assert np.array_equal(q["input_offsets"], prev), f"pass {p}: input offsets"
        n += 1
    assert n == o.numPasses() > 0
    assert np.array_equal(lad.offsets, o.readOffsetArray())
    assert np.array_equal(lad.flow, o.readFlow(latest=True))
    assert lad.frame_delta == o.state().totalFrameDelta


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the CUDA ladder against OracleLadder, pass by pass, with the per-CTA timeline on
# ---------------------------------------------------------------------------------------------------------------------
def span_of(R):
    """Extra rows the candidates of one window reach along the candidate axis (CandSpan<R>::SPAN)."""
    sq = lambda d: d * abs(d)
    return sq(R - 1 - R // 2) - sq(-(R // 2))


def expected_kernel(ws, lu, R, rs, variant=0):
    """The kernel planSearchPass (kernels_search.cu) picks for a pass: 'tile', 'cand' or 'generic'.  lu: the whole
    field's extent along u (flow width in Y steps, flow height in X steps)."""
    if R >= 5 and rs == 0 and variant != 1:
        if ws >= (4 if variant in (2, 3) else 16) and lu % 4 == 0:
            return "tile"
        if ws <= 32:
            return "cand"
    return "generic"


def timeline_words(lw, lh):
    """Words per pass that hold every tile CTA of a ladder (128 x 32*NWV flow pixels per CTA, NWV >= 2)."""
    return 16 * max(-(-lw // 128) * -(-lh // 64), -(-lh // 128) * -(-lw // 64))


def cand_unstaged_tiles(inp, ws, step, R, lu, lv):
    """[tiles along v][tiles along u]: the small-window kernel's CTA of that 32 (u) x 128 (v) tile stages nothing and
    fetches from global memory (kernels_search_cand.cu:345-348: RU > 48 or RV > 254), from the pass's input offsets."""
    ox, oy = inp[0, ::ws, ::ws].astype(np.int64), inp[1, ::ws, ::ws].astype(np.int64)  # [nWy][nWx]
    ou, ov = (ox, oy) if step == 1 else (oy.T, ox.T)                                  # [windows along v][along u]
    tu, tv = 32 // ws, 128 // ws
    nv, nu = ou.shape
    Tv, Tu = -(-nv // tv), -(-nu // tu)

    def reduce(a, fn, fill):
        p = np.full((Tv * tv, Tu * tu), fill, np.int64)
        p[:nv, :nu] = a
        return fn(p.reshape(Tv, tv, Tu, tu), axis=(1, 3))

    big = 1 << 40
    ru = 32 + reduce(ou, np.max, -big) - reduce(ou, np.min, big)
    rows = np.minimum(128, lv - 128 * np.arange(Tv))[:, None]
    rv = rows + span_of(R) + reduce(ov, np.max, -big) - reduce(ov, np.min, big)
    return (ru > 48) | (rv > 254)


def compare_ladder(g, lad, label, wpp=None, variant=0):
    """Taps (and the timeline, wpp words per pass) on g, whose frames are uploaded; every pass equals lad's, then the
    final offsets, the blurred flow and the frame delta.  Returns per pass: window size, step, kernel, the timeline
    records of its CTAs and, for small-window passes, the number of unstaged CTAs."""
    R, lh, lw, rs = lad.R, lad.lh, lad.lw, lad.rs
    g.setSearchVariant(variant)
    g.setTapMode(True)
    if wpp:
        g.debugTimeline(wpp)   # zeroes the buffer
    g.calculateOpticalFlow()
    tl = g.readDebugTimeline(wpp) if wpp else None
    out = []
    n = 0
    for p, q in enumerate(lad.passes()):
        ws, step = q["windowSize"], q["step"]
        gi = g.passInfo(p)
        where = f"{label}: pass {p} (ws {ws}, iteration {q['iteration']}, step {step})"
        assert (gi["windowSize"], gi["iteration"], gi["step"]) == (ws, q["iteration"], step), where
        s = g.readPassSums(p, R)
        assert s.shape == q["sums"].shape, where
        assert np.array_equal(s, q["sums"]), f"{where}: {np.count_nonzero(s != q['sums'])} window sums differ"
        assert np.array_equal(g.readPassLayers(p), q["layers"]), f"{where}: layers differ"
        o = g.readPassOffsets(p)
        assert np.array_equal(o, q["offsets"]), f"{where}: {np.count_nonzero(o != q['offsets'])} offsets differ"
        lu, lv = (lw, lh) if step == 1 else (lh, lw)
        kind = expected_kernel(ws, lu, R, rs, variant)
        rec = dict(ws=ws, step=step, kind=kind, lu=lu, lv=lv)
        if tl is not None:
            t = tl[p]
            rec["tl"] = t[t[:, 0] > 0]
            if kind != "tile":
                assert not tl[p].any(), f"{where}: the timeline slice of a {kind} pass is not zero"
            else:
                nwv = np.unique(rec["tl"][:, 8])
                assert len(nwv) == 1, f"{where}: CTAs report NWV {nwv}"
                nwv = int(nwv[0])
                ncta = -(-lu // 128) * -(-lv // (32 * nwv))
                assert len(rec["tl"]) == min(ncta, wpp // 16), f"{where}: {len(rec['tl'])} CTA records, grid {ncta}"
                rec["nwv"] = nwv
        if kind == "cand" and ws <= 8:
            rec["unstaged"] = int(cand_unstaged_tiles(q["input_offsets"], ws, step, R, lu, lv).sum())
        out.append(rec)
        n += 1
    assert g.numPasses() == n > 0
    if tl is not None:
        assert not tl[n:].any(), f"{label}: timeline slices past the last pass are not zero"
    assert np.array_equal(g.readOffsetArray(), lad.offsets), f"{label}: final offsets differ"
    assert np.array_equal(g.readFlow(latest=True), lad.flow), f"{label}: blurred flow differs"
    assert g.m_totalFrameDelta == lad.frame_delta, f"{label}: frame delta"
    return out


def check_production(g, offsets, flow, delta, label):
    """The same frames without taps or timeline: the ladder runs from a CUDA graph.  The two blurred-flow buffers alternate,
    so calculations 1 and 2 capture a graph each and calculation 3 replays the first."""
    g.setTapMode(False)
    g.debugTimeline(0)
    for k in range(3):
        g.calculateOpticalFlow()
        assert np.array_equal(g.readOffsetArray(), offsets), f"{label}: production calculation {k}: final offsets differ"
        assert np.array_equal(g.readFlow(latest=True), flow), f"{label}: production calculation {k}: blurred flow differs"
        assert g.m_totalFrameDelta == delta, f"{label}: production calculation {k}: frame delta"


_NWV_SEEN = {}   # case label -> {(window class, NWV)}: filled by the shape and mosaic tests, checked at the end of the module


def _record_nwv(label, recs):
    _NWV_SEEN[label] = {(min(r["ws"], 128), r["nwv"]) for r in recs if "nwv" in r}
    print(f"{label}: (window class, NWV) {sorted(_NWV_SEEN[label])}")


def _calc(hdr, H, W, inS, maxres, R, ds=8, ns=6):
    import hopperrender_b200 as hr
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    g = cls(H, W, inS, 0, ds, ns, 0.0, 255.0, maxres)
    g.m_opticalFlowSearchRadius = R
    return g


# NWV per window class 16 / 32 / 64 from a host mirror of chooseWarps on 148 SMs (kernels_search_slide.cu):
#   2560x1440 R 16: 3 / 3 / 4     3200x1800 R 13: 4 / 4 / 4     3840x2160 R 6: 5 / 5 / 2     4096x2160 R 14: 5 and 6 / 5 and 6 / 4
SHAPE_CASES = [
    # hdr, W, H, inS, R
    (False, 2560, 1440, 2688, 16),
    (True, 3200, 1800, 0, 13),
    (False, 3840, 2160, 0, 6),
    (True, 4096, 2160, 0, 14),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,inS,R", SHAPE_CASES)
def test_large_tile_shapes_pass_by_pass(synth, hdr, W, H, inS, R):
    """Full-resolution frames large enough that the tile kernel runs with 3..6 warps per CTA: every pass, the final
    offsets, the blurred flow and the frame delta equal the oracle; then the production path of the same frames."""
    label = f"{'HDR' if hdr else 'SDR'} {W}x{H} R {R}"
    f = [synth.make_frame(W, H, t, synth.SEED_BASE + 3, hdr, inS or None) for t in (1, 2)]
    fs = [f[0], f[0], f[1]]
    g = _calc(hdr, H, W, inS, H, R)
    for fr in fs:
        g.updateFrame(fr)
    lad = OracleLadder.of(fs, hdr, W, H, inS, H, R)
    recs = compare_ladder(g, lad, label, timeline_words(lad.lw, lad.lh))
    _record_nwv(label, recs)
    check_production(g, lad.offsets, lad.flow, lad.frame_delta, label)
    g.close()


def mosaic_frames(synth, W, H, hdr, seed, amp=40, stride=None):
    """[frame 0, frame 1, frame 2]: frame 1 a textured scene, frame 2 the same scene cut into blocks of 16-64 pixels that
    move by independent seeded vectors of up to +-amp pixels (even components, so the chroma moves with the luma); blocks
    on the frame edges move outwards.  Frame 0 is frame 1."""
    M = amp + 24
    M += M & 1
    Wb, Hb = W + 2 * M, H + 2 * M
    base = synth.make_frame(Wb, Hb, 0, synth.SEED_BASE + 77 + seed, hdr).reshape(Hb + Hb // 2, Wb)
    Y, UV = base[:Hb], base[Hb:]
    rng = np.random.default_rng(seed)
    S = stride or W
    f1 = np.zeros((H + H // 2, S), base.dtype)
    f2 = np.zeros_like(f1)
    f1[:H, :W] = Y[M:M + H, M:M + W]
    f1[H:, :W] = UV[M // 2:M // 2 + H // 2, M:M + W]
    y = 0
    while y < H:
        bh = min(2 * int(rng.integers(8, 33)), H - y)
        x = 0
        while x < W:
            bw = min(2 * int(rng.integers(8, 33)), W - x)
            vx, vy = (2 * int(v) for v in rng.integers(-(amp // 2), amp // 2 + 1, 2))
            if x == 0:
                vx = -abs(vx)
            if x + bw == W:
                vx = abs(vx)
            if y == 0:
                vy = -abs(vy)
            if y + bh == H:
                vy = abs(vy)
            # frame2[y, x] = frame1[y - vy, x - vx]
            f2[y:y + bh, x:x + bw] = Y[M + y - vy:M + y - vy + bh, M + x - vx:M + x - vx + bw]
            f2[H + y // 2:H + (y + bh) // 2, x:x + bw] = UV[(M + y - vy) // 2:(M + y - vy + bh) // 2, M + x - vx:M + x - vx + bw]
            x += bw
        y += bh
    f1, f2 = f1.reshape(-1), f2.reshape(-1)
    return [f1, f1, f2]


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,inS,R", [(False, 1024, 576, 0, 16), (True, 2560, 1440, 0, 16)])
def test_motion_mosaic_rounds_pass_by_pass(synth, hdr, W, H, inS, R):
    """Independently moving blocks: tile CTAs whose windows are displaced too differently for one box take 2-4 rounds, and
    what is left after 4 the per-pixel path (round 5), on interior and on border tiles; small-window CTAs fall back to
    unstaged fetches.  Every pass equals the oracle, and so does the production path."""
    label = f"mosaic {'HDR' if hdr else 'SDR'} {W}x{H} R {R}"
    fs = mosaic_frames(synth, W, H, hdr, seed=W, stride=inS or None)
    g = _calc(hdr, H, W, inS, H, R)
    for fr in fs:
        g.updateFrame(fr)
    lad = OracleLadder.of(fs, hdr, W, H, inS, H, R)
    recs = compare_ladder(g, lad, label, timeline_words(lad.lw, lad.lh))
    _record_nwv(label, recs)
    tile = np.concatenate([r["tl"][:, 7] for r in recs if r["kind"] == "tile"])
    rounds, border = tile % 100, tile >= 100
    unstaged = {ws: sum(r.get("unstaged", 0) for r in recs if r["ws"] == ws and r["kind"] == "cand") for ws in (2, 4, 8)}
    hist = {k: int(np.count_nonzero(rounds == k)) for k in range(1, 6)}
    print(f"{label}: tile CTAs by rounds {hist}, border CTAs with more than one round {int(np.count_nonzero(border & (rounds > 1)))}, "
          f"unstaged small-window CTAs by window size {unstaged}")
    assert np.any((rounds >= 2) & (rounds <= 4)), f"{label}: no tile CTA ran 2-4 rounds"
    assert np.any(rounds == 5), f"{label}: no tile CTA reached the per-pixel remainder"
    assert np.any(border & (rounds > 1)), f"{label}: no border tile CTA ran more than one round"
    for ws, n in unstaged.items():
        assert n > 0, f"{label}: no unstaged small-window CTA at windows of {ws}"
    check_production(g, lad.offsets, lad.flow, lad.frame_delta, label)
    g.close()


@pytest.mark.gpu
def test_timeline_records_only_what_fits_its_slice(synth):
    """hrb_ofc_debug_timeline with fewer words per pass than the largest tile pass needs: the CTAs past the slice's
    capacity record nothing, the records that are there belong to the first CTAs of their own pass, and the slices of
    the passes the tile kernel does not run stay zero.  The slice is sized so that even a timeline without the bound
    would stay inside its buffer (it would overwrite the following passes' slices instead)."""
    W, H, R = 1024, 576, 16
    fs = _frames(synth, W, H, False, 3)
    g = _calc(False, H, W, 0, H, R)
    for fr in fs:
        g.updateFrame(fr)
    full = timeline_words(W, H) // 16
    cap = 40
    wpp = 16 * cap
    lad = OracleLadder.of(fs, False, W, H, 0, H, R)
    recs = compare_ladder(g, lad, "timeline bound", wpp)
    over = []
    for p, r in enumerate(recs):
        if r["kind"] != "tile":
            continue
        t = r["tl"]
        gx = -(-r["lu"] // 128)
        ncta = gx * -(-r["lv"] // (32 * r["nwv"]))
        assert ncta <= full
        assert p * wpp + 16 * ncta <= 32 * wpp, f"pass {p}: an unbounded timeline would write past the buffer"
        if ncta > cap:
            over.append(p)
        assert len(t) == min(ncta, cap), f"pass {p}: {len(t)} records, grid {ncta}, capacity {cap}"
        idx = (t[:, 6] * gx + t[:, 5]).astype(np.int64)
        assert np.array_equal(idx, np.arange(len(t))), f"pass {p}: the records are not CTAs 0..{len(t) - 1} of this pass"
        assert np.all(t[:, 8] == r["nwv"]) and not t[:, 9:].any()
    # the last tile pass overflows into the slice of the first small-window pass, which must stay zero
    last_tile = max(p for p, r in enumerate(recs) if r["kind"] == "tile")
    assert last_tile in over and recs[last_tile + 1]["kind"] == "cand", (over, last_tile)
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(320, 192), (322, 190)])   # flow sides multiples of 4 / 2 (mod 4)
@pytest.mark.parametrize("variant", [2, 3, 4])
def test_search_variant_kernels_pass_by_pass(synth, variant, W, H):
    """Search variants 2 (tile kernel without TMA, from windows of 4), 3 (... per-pixel path forced) and 4 (like 0, with
    the butterfly form at windows of 2 and 4): every pass equals the oracle, and the timeline shows the tile kernel on
    exactly the passes expected_kernel gives it — none when the sides are 2 (mod 4)."""
    R = 11
    label = f"variant {variant} {W}x{H}"
    fs = _frames(synth, W, H, False, 3, seed=variant)
    g = _calc(False, H, W, 0, H, R)
    for fr in fs:
        g.updateFrame(fr)
    lad = OracleLadder.of(fs, False, W, H, 0, H, R)
    recs = compare_ladder(g, lad, label, timeline_words(lad.lw, lad.lh), variant)
    kinds = {r["kind"] for r in recs}
    assert kinds == ({"tile", "cand"} if W % 4 == 0 else {"cand", "generic"}), f"{label}: {kinds}"
    g.close()


@pytest.mark.gpu
def test_nwv_coverage_across_the_module():
    """NWV 2..6 for windows of 16 and 32 and NWV 2 and 4 for windows of 64 are each reached by the tests above (on a
    148-SM B200; on other SM counts the warps per CTA differ and only the comparisons above apply)."""
    import torch
    expected_cases = len(SHAPE_CASES) + 2
    if len(_NWV_SEEN) < expected_cases:
        pytest.skip("needs the shape and mosaic tests of this module in the same session")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    seen = set().union(*_NWV_SEEN.values())
    print("(window class, NWV) reached:", sorted(seen))
    if sms != SM_COUNT_OF_TABLE:
        pytest.skip(f"{sms} SMs: the NWV table is for {SM_COUNT_OF_TABLE}")
    want = {(c, n) for c in (16, 32) for n in (2, 3, 4, 5, 6)} | {(64, 2), (64, 4)}
    missing = sorted(want - seen)
    assert not missing, f"(window class, NWV) pairs no test reached: {missing}"
