"""The warp kernel at the shapes playback runs, against the oracle.

warpKernel (csrc/kernels_frame.cu) sends each 256-sample item of an output row down one of four forms:

  lean       warpItemFast: modes 0-2, every blend scalar in [0, 1], an even output stride, and an item that stays inside
             [1, dim-2] under the flow peak; it falls back to `untabled` when one of its own displacements is >= 128
  inside     warpItem<TAB=1, INSIDE=1>: inside, peak < 128, but the lean form is not allowed (modes 3/4, odd output stride)
  border     warpItem<TAB=1, INSIDE=0>: not inside, peak < 128
  untabled   warpItem<TAB=0, INSIDE=0>: peak >= 128 (items the lean form does not take), lean outliers, t outside [0, 1]

An item can only be inside when x0 >= 1 + peak and x0 + 255 + peak <= W - 2, so frames narrower than 513 pixels never run
the lean form.  `warp_item_forms` restates that choice on the host; every GPU case asserts that the forms it exists for are
reached, so a case that silently stops reaching its path fails.  The GPU cases compare modes 0-2 and 4-6 with the oracle
bit for bit (mode 3 within one 8-bit step on at most 0.2 % of the samples), row by row over the output stripe or the full
frame, at reduced-resolution flows, padded strides, output stripes, batches of 8, the table edge and in-flight flows.
"""
import numpy as np
import pytest

from conftest import make_pair, out_array

ITEM = 256       # samples per warp item
TAB_HALF = 128   # rounding tables cover displacements -128 .. 127
FORMS = ("lean_luma", "lean_chroma", "inside", "border", "untabled")
LEAN, INSIDE, BORDER, UNTABLED = 1, 2, 3, 4  # codes of warp_item_maps

SOURCE_FRAME_TIME_24 = 416667  # 100-ns units, 24 fps


def item_flow_peaks(flow, rs, cys, cz, n_items, W, lw, lh, reverse):
    """[rows][items]: the largest |component| of the flow cells the lean form reads for each item of the given rows
    (forward flow, and for modes 1 and 2 the reverse flow it gathers where the forward flow points back to)."""
    xs = np.minimum(np.arange(n_items * ITEM), W - 1)
    fx = ((xs >> rs) & ~1) if cz else xs >> rs
    out = np.zeros((len(cys), n_items), np.int64)
    fl = flow.astype(np.int64)
    for r0 in range(0, len(cys), 128):  # row blocks keep a 4K frame's intermediates small
        cy = cys[r0:r0 + 128]
        fy = ((cy >> rs) << 1) if cz else cy >> rs
        ox, oy = fl[0][fy[:, None], fx[None, :]], fl[1][fy[:, None], fx[None, :]]
        m = np.maximum(np.abs(ox), np.abs(oy))
        if reverse:
            gy = np.clip(fy[:, None] - (oy >> rs), 0, lh - 1)
            gx = np.clip(fx[None, :] - (ox >> rs), 0, lw - 1)
            m = np.maximum(m, np.maximum(np.abs(fl[0][gy, gx]), np.abs(fl[1][gy, gx])))
        out[r0:r0 + len(cy)] = m.reshape(len(cy), n_items, ITEM).max(axis=2)
    return out


def warp_item_maps(W, H, lw, lh, rs, So, stripe, peak, flow, ts, mode):
    """{cz: (plane rows, codes[rows][items])} for the luma (cz 0) and chroma (cz 1) rows a launch produces: the form
    warpKernel gives each item (kernels_frame.cu, warpKernel and the outlier check of warpItemFast).  stripe: (y0, y1) of
    hrb_ofc_set_output_stripe or None; peak: the flow peak the kernel reads; flow: [2][lh][lw] (None: zero flow).
    The output levels are assumed to give a non-zero range (the kernel's divY.ok / divUV.ok)."""
    y0, y1 = stripe if stripe else (0, H)
    n = y1 - y0
    unit = all(0.0 <= t <= 1.0 for t in ts)
    tab_ok = peak < TAB_HALF and unit
    lean_ok = mode <= 2 and unit and So % 2 == 0
    x0 = np.arange(0, W, ITEM)
    maps = {}
    for cz, cys in ((0, np.arange(y0, y1)), (1, np.arange(y0 // 2, y0 // 2 + n // 2))):
        dim = H >> cz
        inside = ((x0[None, :] - peak >= 1) & (x0[None, :] + ITEM - 1 + peak <= W - 2)
                  & (cys[:, None] - peak >= 1) & (cys[:, None] + peak <= dim - 2) & (mode <= 4))
        code = np.where(inside, INSIDE, BORDER) if tab_ok else np.full(inside.shape, UNTABLED)
        if lean_ok:
            if flow is None:
                m = np.zeros(inside.shape, np.int64)
            else:
                m = item_flow_peaks(flow, rs, cys, cz, len(x0), W, lw, lh, mode != 0)
            code = np.where(inside, np.where(m < TAB_HALF, LEAN, UNTABLED), code)
        maps[cz] = (cys, code)
    return maps


def warp_item_forms(W, H, lw, lh, rs, So, stripe, peak, flow, ts, mode):
    """Items per form of one warp launch (FORMS), the lean form split into luma and chroma items."""
    maps = warp_item_maps(W, H, lw, lh, rs, So, stripe, peak, flow, ts, mode)
    c = dict.fromkeys(FORMS, 0)
    for cz, (_, code) in maps.items():
        c["lean_chroma" if cz else "lean_luma"] += int(np.count_nonzero(code == LEAN))
        c["inside"] += int(np.count_nonzero(code == INSIDE))
        c["border"] += int(np.count_nonzero(code == BORDER))
        c["untabled"] += int(np.count_nonzero(code == UNTABLED))
    return c


# ---- the mirror on hand-checked geometries (no GPU) -----------------------------------------------------------------

def test_mirror_narrow_frames_have_no_lean_items():
    # W = 320: item x0 = 256 needs 256 + 255 <= 318.  W = 512: x0 = 256 needs 511 <= 510.
    for W, H in [(320, 176), (512, 128)]:
        c = warp_item_forms(W, H, W, H, 0, W, None, 0, None, [0.5], 2)
        assert c["lean_luma"] == c["lean_chroma"] == c["inside"] == c["untabled"] == 0
        assert c["border"] == (H + H // 2) * -(-W // ITEM)


def test_mirror_counts_at_1024x576():
    # 4 items per row, 576 luma + 288 chroma rows: 3456 items.  Peak 0: items x0 = 256 and 512 (x0 >= 1, x0 + 255 <= 1022)
    # on luma rows 1..574 (574 rows) and chroma rows 1..286 (286 rows).  Peak 127: the same two items (x0 >= 128,
    # x0 <= 640) on luma rows 128..447 (320 rows) and chroma rows 128..159 (32 rows).
    W, H = 1024, 576
    zero = np.zeros((2, H, W), np.int16)
    c = warp_item_forms(W, H, W, H, 0, W, None, 0, zero, [0.5], 2)
    assert c == {"lean_luma": 1148, "lean_chroma": 572, "inside": 0, "border": 3456 - 1148 - 572, "untabled": 0}
    flat = np.full((2, H, W), -127, np.int16)
    c = warp_item_forms(W, H, W, H, 0, W, None, 127, flat, [0.5], 2)
    assert c == {"lean_luma": 640, "lean_chroma": 64, "inside": 0, "border": 3456 - 704, "untabled": 0}
    # the same geometry: an odd output stride or mode 3 takes warpItem's INSIDE form instead, modes 5/6 are never inside
    assert warp_item_forms(W, H, W, H, 0, W + 1, None, 127, flat, [0.5], 2)["inside"] == 704
    assert warp_item_forms(W, H, W, H, 0, W, None, 127, flat, [0.5], 3)["inside"] == 704
    assert warp_item_forms(W, H, W, H, 0, W, None, 127, flat, [0.5], 5)["border"] == 3456
    # a peak of 128 leaves the tables: every item the lean form does not take is untabled
    assert warp_item_forms(W, H, W, H, 0, W, None, 128, flat, [0.5], 2)["border"] == 0
    # a blend scalar outside [0, 1] turns off the lean form and the tables
    assert warp_item_forms(W, H, W, H, 0, W, None, 0, zero, [-0.5], 2)["untabled"] == 3456


def test_mirror_item_outliers():
    # one cell of 128 in an interior item: that item falls back; under mode 1 the items whose reverse lookup lands on the
    # cell fall back too (here: the item to its right, whose samples point 20 columns back onto it)
    W, H = 1024, 576
    fl = np.zeros((2, H, W), np.int16)
    fl[0, 300, 500] = 128
    fl[0, 300, 512:540] = 20
    m0 = warp_item_maps(W, H, W, H, 0, W, None, 128, fl, [0.5], 0)[0][1]
    m1 = warp_item_maps(W, H, W, H, 0, W, None, 128, fl, [0.5], 1)[0][1]
    assert m0[300, 1] == UNTABLED and m0[300, 2] == LEAN
    assert m1[300, 1] == UNTABLED and m1[300, 2] == UNTABLED
    # the chroma row 150 reads flow row 300, its pair at column 500 holds the outlier
    assert warp_item_maps(W, H, W, H, 0, W, None, 128, fl, [0.5], 0)[1][1][150, 1] == UNTABLED


# ---- GPU cases ------------------------------------------------------------------------------------------------------

_FRAMES = {}


def src_frames(synth, W, H, hdr, inS=0, n=3):
    key = (W, H, hdr, inS, n)
    if key not in _FRAMES:
        _FRAMES.clear()  # one geometry at a time: 4K P010 frames are 25 MB each
        _FRAMES[key] = [synth.make_frame(W, H, t, synth.SEED_BASE + 5, hdr, inS or None) for t in range(n)]
    return _FRAMES[key]


def written_flow(lh, lw, seed, amp):
    """8x8 blocks of -amp..amp plus -3..3 per cell, clipped to +-amp: odd and even displacements of both signs."""
    rng = np.random.default_rng(seed)
    base = rng.integers(-amp, amp + 1, (2, lh // 8 + 2, lw // 8 + 2))
    fl = np.repeat(np.repeat(base, 8, 1), 8, 2)[:, :lh, :lw] + rng.integers(-3, 4, (2, lh, lw))
    return np.clip(fl, -amp, amp).astype(np.int16)


def setup(synth, hdr, W, H, maxres, inS=0, outS=0, R=16):
    """(cuda calculator, oracle) holding the same three source frames."""
    g, o = make_pair(hdr, H, W, inS, outS, black=4.0, white=250.0, maxres=maxres, R=R)
    for fr in src_frames(synth, W, H, hdr, inS):
        g.updateFrame(fr)
        o.updateFrame(fr)
    return g, o


def real_flow(g):
    """Two calculations on the same frames: the flow warpFrames reads is a searched and blurred one, with the flow peak
    the blur kernel computed on the device."""
    g.calculateOpticalFlow()
    g.calculateOpticalFlow()
    return g.readFlow()


def geometry(g):
    return g.m_opticalFlowResScalar, g.m_opticalFlowFrameWidth, g.m_opticalFlowFrameHeight


def forms_of(g, fl, ts, mode, stripe=None):
    rs, lw, lh = geometry(g)
    peak = int(np.abs(fl.astype(np.int64)).max())
    return warp_item_forms(g.m_frameWidth, g.m_frameHeight, lw, lh, rs, g.m_outputStride, stripe, peak, fl, ts, mode)


def report(name, forms):
    print(f"[warp forms] {name}: " + " ".join(f"{k}={v}" for k, v in forms.items()))


def stripe_rows(H, stripe):
    y0, y1 = stripe if stripe else (0, H)
    return np.r_[y0:y1, H + y0 // 2:H + y1 // 2]


def assert_rows_equal(got, want, hdr, W, So, H, mode, stripe=None, what=""):
    rows = stripe_rows(H, stripe)
    a = got.reshape(-1, So)[rows, :W].astype(np.int64)
    b = want.reshape(-1, So)[rows, :W].astype(np.int64)
    if mode == 3:
        d = np.abs(a - b)
        step = 256 if hdr else 1
        assert d.max() <= step and np.count_nonzero(d) <= max(4, d.size // 500), f"{what}: {(d.max(), np.count_nonzero(d))}"
    else:
        assert np.array_equal(a, b), f"{what}: {np.count_nonzero(a != b)} samples differ, first at {np.argwhere(a != b)[:1].tolist()}"


def warp_batch(g, hdr, ts, mode, fill=0):
    """warpFramesBatch and one download per frame (fill: the value the host buffers hold before the download)."""
    g.warpFramesBatch(ts, mode)
    outs = []
    for _ in ts:
        a = out_array(g, hdr)
        a[:] = fill
        g.downloadFrame(a)
        outs.append(a)
    return outs


def oracle_frame(o, hdr, t, mode):
    o.warpFrames(t, mode)
    b = out_array(o, hdr)
    o.downloadFrame(b)
    return b


def check_against_oracle(g, o, hdr, ts, mode, name):
    W, H, So = g.m_frameWidth, g.m_frameHeight, g.m_outputStride
    for t, a in zip(ts, warp_batch(g, hdr, ts, mode)):
        assert_rows_equal(a, oracle_frame(o, hdr, t, mode), hdr, W, So, H, mode, None, f"{name} mode {mode} t {t}")


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["real", "written"])
@pytest.mark.parametrize("hdr,W,H,maxres,rs", [
    (False, 1920, 1080, 270, 2),   # cfg1: 480x270 flow
    (False, 1920, 1080, 540, 1),   # cfg2: 960x540 flow
    (False, 1030, 580, 290, 1),    # odd flow width 515: the scalar fetch at rs 1 with a flow row of odd length
    (True, 1920, 1080, 270, 2),
])
def test_reduced_resolution_flow(synth, hdr, W, H, maxres, rs, source):
    """The lean form's scalar flow fetch (rs > 0 or an odd flow width), luma and chroma rows, modes 0-2."""
    g, o = setup(synth, hdr, W, H, maxres)
    assert g.m_opticalFlowResScalar == rs
    _, lw, lh = geometry(g)
    fl = real_flow(g) if source == "real" else written_flow(lh, lw, W + rs, 45)
    if source == "written":
        g.writeFlow(fl)
    o.writeFlow(fl)
    ts = [0.25, 0.5, 5.0 / 6.0]
    for mode in (0, 1, 2):
        forms = forms_of(g, fl, ts, mode)
        report(f"A {W}x{H} rs{rs} {'P010' if hdr else 'NV12'} {source} mode {mode}", forms)
        assert forms["lean_luma"] > 0 and forms["lean_chroma"] > 0
        check_against_oracle(g, o, hdr, ts, mode, f"{W}x{H} rs {rs} {source}")


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,pad_in,pad_out", [
    (False, 1920, 1080, 64, 32), (False, 1920, 1080, 128, 32), (True, 3840, 2160, 64, 32), (True, 3840, 2160, 128, 32),
    (False, 1920, 1080, 64, 1),    # odd output stride: no lean form, interior items take warpItem<TAB, INSIDE>
])
def test_padded_strides(synth, hdr, W, H, pad_in, pad_out):
    """Input stride != output stride != width: the lean form's base index, y tables and store use the right stride."""
    g, o = setup(synth, hdr, W, H, H, inS=W + pad_in, outS=W + pad_out)
    _, lw, lh = geometry(g)
    fl = written_flow(lh, lw, W + pad_in + pad_out, 50)
    g.writeFlow(fl)
    o.writeFlow(fl)
    ts = [0.2, 0.5, 0.9]
    for mode in (0, 1, 2):
        forms = forms_of(g, fl, ts, mode)
        report(f"B {W}x{H} inS W+{pad_in} outS W+{pad_out} mode {mode}", forms)
        if pad_out % 2:
            assert forms["lean_luma"] == forms["lean_chroma"] == 0 and forms["inside"] > 0
        else:
            assert forms["lean_luma"] > 0 and forms["lean_chroma"] > 0
        check_against_oracle(g, o, hdr, ts, mode, f"{W}x{H} strides {W + pad_in}/{W + pad_out}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4])
@pytest.mark.parametrize("hdr,W,H,maxres,source", [(True, 3840, 2160, 2160, "written"), (False, 1920, 1080, 270, "real")])
def test_output_stripes(synth, hdr, W, H, maxres, source, n):
    """Calculators that each warp one output stripe (split.stripe_bounds): every stripe's rows equal the oracle's full
    frame, and the rest of the caller's buffer is left as it was."""
    from hopperrender_b200.split import stripe_bounds
    g0, o = setup(synth, hdr, W, H, maxres)
    _, lw, lh = geometry(g0)
    fl = real_flow(g0) if source == "real" else written_flow(lh, lw, W + n, 40)
    o.writeFlow(fl)
    g0.close()
    ts = [0.3, 0.6]
    sentinel = 0x5A5A if hdr else 0x5A
    want = {(t, mode): oracle_frame(o, hdr, t, mode) for mode in (2, 0) for t in ts}
    for stripe in stripe_bounds(H, n):
        g, _ = make_pair(hdr, H, W, black=4.0, white=250.0, maxres=maxres)
        g.setOutputStripe(*stripe)
        for fr in src_frames(synth, W, H, hdr):
            g.updateFrame(fr)
        g.writeFlow(fl)
        rows = stripe_rows(H, stripe)
        for mode in (2, 0):
            forms = forms_of(g, fl, ts, mode, stripe)
            report(f"C {W}x{H} {n} stripes {stripe} mode {mode}", forms)
            assert forms["lean_luma"] > 0 and forms["lean_chroma"] > 0
            for t, a in zip(ts, warp_batch(g, hdr, ts, mode, sentinel)):
                assert_rows_equal(a, want[(t, mode)], hdr, W, W, H, mode, stripe, f"stripe {stripe} mode {mode} t {t}")
                rest = np.ones(H + H // 2, bool)
                rest[rows] = False
                assert (a.reshape(-1, W)[rest] == sentinel).all(), f"stripe {stripe}: rows outside the stripe were written"
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("rate", ["23.976->144", "24->60"])
@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("W,H,maxres", [(1024, 576, 576), (1920, 1080, 540)])
def test_batches_of_eight(synth, hdr, W, H, maxres, rate):
    """Batches of 8 and 7 back to back (30 frames: the batch of frames 15-22 wraps the 16-slot output ring of a fresh
    calculator) at the blend scalars the filter produces: frame i equals the single-call frame and the oracle's."""
    from hopperrender_b200 import replay
    target, source = {"23.976->144": (replay.TARGET_FRAME_TIME_144, replay.SOURCE_FRAME_TIME_23976),
                      "24->60": (replay.TARGET_FRAME_TIME_60, SOURCE_FRAME_TIME_24)}[rate]
    ts = [t for row in replay.output_schedule(40, target, source) for t in row][:30]
    assert len(ts) == 30 and len(set(ts)) > 8
    g, o = setup(synth, hdr, W, H, maxres)
    fl = real_flow(g)
    o.writeFlow(fl)
    forms = forms_of(g, fl, ts[:8], 2)
    report(f"D {W}x{H} {'P010' if hdr else 'NV12'} {rate}", forms)
    assert forms["lean_luma"] > 0 and forms["lean_chroma"] > 0
    batched = []
    for b0, b1 in [(0, 8), (8, 15), (15, 23), (23, 30)]:
        batched += warp_batch(g, hdr, ts[b0:b1], 2)
    for i, (t, a) in enumerate(zip(ts, batched)):
        g.warpFrames(t, 2)
        single = out_array(g, hdr)
        g.downloadFrame(single)
        assert np.array_equal(a, single), f"frame {i} (t {t}): batch and single call differ in {np.count_nonzero(a != single)} samples"
        assert_rows_equal(a, oracle_frame(o, hdr, t, 2), hdr, W, W, H, 2, None, f"frame {i} t {t}")


def _edge_flow(lh, lw, seed):
    """-30..30 per cell: at t = 0.5 odd luma displacements and chroma y displacements = 2 (mod 4) are rounding ties, and
    odd x displacements split a chroma pair."""
    return np.random.default_rng(seed).integers(-30, 31, (2, lh, lw)).astype(np.int16)


@pytest.mark.gpu
@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("peak", [126, 127, 128, 129])
def test_frame_peak_at_the_table_edge(synth, hdr, peak):
    """A frame peak just inside and just beyond the rounding tables (1280x720, full-resolution written flow)."""
    W, H = 1280, 720
    g, o = setup(synth, hdr, W, H, H)
    fl = _edge_flow(H, W, peak)
    fl[0, 360, 640], fl[1, 200, 300] = peak, -peak
    g.writeFlow(fl)
    o.writeFlow(fl)
    assert g.readFlowPeak()[0] == peak
    ts = [0.5, 0.25, 1.0, 0.0]
    for mode in (0, 1, 2):
        forms = forms_of(g, fl, ts, mode)
        report(f"E {'P010' if hdr else 'NV12'} frame peak {peak} mode {mode}", forms)
        assert forms["lean_luma"] > 0 and forms["lean_chroma"] > 0
        if peak < TAB_HALF:
            assert forms["untabled"] == 0 and forms["border"] > 0
        else:
            assert forms["border"] == 0 and forms["untabled"] > 0
        check_against_oracle(g, o, hdr, ts, mode, f"frame peak {peak}")


@pytest.mark.gpu
@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("frame_peak", [200, 170])
def test_item_peak_at_the_table_edge(synth, hdr, frame_peak):
    """Single items whose own largest displacement is 127 (lean), 128 or 129 (the item falls back) under a larger frame
    peak, on luma and on chroma rows.  A chroma row of a 720-row frame is inside only under a peak of at most 178, so the
    chroma items are checked under a frame peak of 170."""
    W, H = 1280, 720
    g, o = setup(synth, hdr, W, H, H)
    fl = _edge_flow(H, W, frame_peak)
    fl[0, 2, 2] = frame_peak  # in a border item, out of reach of every interior item's reverse lookup
    # (cz, plane row, column, own peak): each in its own item, more than 30 + 129 samples from the others
    targets = [(0, 250, 300, 127), (0, 350, 600, 128), (0, 450, 900, 129),
               (1, 175, 300, 127), (1, 180, 600, 128), (1, 185, 900, 129)]
    for cz, r, x, v in targets:
        fr = 2 * r if cz else r
        fl[0, fr, x], fl[1, fr, x] = v, -v
    g.writeFlow(fl)
    o.writeFlow(fl)
    assert g.readFlowPeak()[0] == frame_peak
    ts = [0.5, 0.75, 1.0 / 6.0]
    for mode in (0, 1, 2):
        maps = warp_item_maps(W, H, W, H, 0, W, None, frame_peak, fl, ts, mode)
        for cz, r, x, v in targets:
            code = maps[cz][1][r, x // ITEM]
            if cz == 0 or frame_peak == 170:
                assert code == (LEAN if v < TAB_HALF else UNTABLED), (cz, r, x, v, code)
            else:
                assert code == UNTABLED, (cz, r, x, v, code)
        forms = forms_of(g, fl, ts, mode)
        report(f"E {'P010' if hdr else 'NV12'} items under peak {frame_peak} mode {mode}", forms)
        assert forms["lean_luma"] > 0 and (forms["lean_chroma"] > 0) == (frame_peak == 170)
        check_against_oracle(g, o, hdr, ts, mode, f"item peaks under {frame_peak}")


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,maxres,variant", [
    (False, 1920, 1080, 270, 0),   # rs 2, flow 480x270: blurFlowCellKernel
    (False, 1920, 1080, 540, 0),   # rs 1, flow 960x540: blurFlowCellKernel
    (False, 1030, 580, 290, 0),    # rs 1, flow 515x290 (odd width): blurFlowKernel
    (False, 1920, 1080, 540, 1),   # variant 1: blurFlowKernel
    (True, 1024, 576, 576, 1),     # rs 0, variant 1: blurFlowKernel
    (True, 3840, 2160, 2160, 0),   # rs 0, flow 3840x2160: blurFlowCellKernel
])
def test_flow_peak_bounds_the_flow(synth, hdr, W, H, maxres, variant):
    """The device flow peak both blur kernels compute (the bound of the warp's inside test and table range) equals the
    largest absolute value of the flow it belongs to, for both flow buffers, over consecutive calculations."""
    g, _ = make_pair(hdr, H, W, maxres=maxres, R=16)
    g.setSearchVariant(variant)
    fs = [synth.make_frame(W, H, t, synth.SEED_BASE + 5, hdr) for t in range(5)]
    for t, fr in enumerate(fs):
        g.updateFrame(fr)
        if t < 2:
            continue
        g.calculateOpticalFlow()
        warp, latest = g.readFlow(), g.readFlow(latest=True)
        want = (int(np.abs(warp.astype(np.int64)).max()), int(np.abs(latest.astype(np.int64)).max()))
        assert want[1] > 0
        assert g.readFlowPeak() == want, f"calculation {t - 1}: peaks {g.readFlowPeak()}, max |flow| {want}"


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,maxres", [(False, 1920, 1080, 540), (True, 3840, 2160, 2160)])
def test_warps_beside_a_flow_in_flight(synth, hdr, W, H, maxres):
    """calculateOpticalFlowAsync and batched warps while the search runs (the warp's short-CTA grid), six source frames:
    every delivered frame equals the oracle's warp of the flow a serial calculator computes on the same frames."""
    import torch
    import hopperrender_b200 as hr
    cls = hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR
    g = cls(H, W, 0, 0, 8, 6, 4.0, 250.0, maxres)
    s, o = make_pair(hdr, H, W, black=4.0, white=250.0, maxres=maxres)
    for c in (g, s):
        c.m_opticalFlowSearchRadius = 16
    o.setParams(searchRadius=16)
    dt = torch.int16 if hdr else torch.uint8
    n_el = g.outputFrameBytes // (2 if hdr else 1)
    pool = [torch.zeros(n_el, dtype=dt).pin_memory() for _ in range(12)]
    tickets, expected = [], []
    for t in range(6):
        fr = synth.make_frame(W, H, t, synth.SEED_BASE + 6, hdr)
        g.updateFrameDevice(torch.from_numpy(fr.view(np.int16) if hdr else fr).cuda())
        s.updateFrame(fr)
        o.updateFrame(fr)
        if t < 2:
            continue
        g.calculateOpticalFlowAsync()
        ts = [(0.3 * (3 * t + j)) % 1.0 for j in range(3)]
        g.warpFramesBatch(ts, 2)
        for _ in ts:
            tickets.append(g.downloadFrameAsync(pool[len(tickets)]))
        s.calculateOpticalFlow()
        fl = s.readFlow()
        o.writeFlow(fl)
        forms = forms_of(s, fl, ts, 2)
        report(f"G {W}x{H} source frame {t}", forms)
        assert forms["lean_luma"] > 0 and forms["lean_chroma"] > 0
        expected += [oracle_frame(o, hdr, b, 2) for b in ts]
    for tk in tickets:
        g.waitDownload(tk)
    g.synchronize()
    assert len(tickets) == len(expected) == 12
    for i, (p, want) in enumerate(zip(pool, expected)):
        got = p.numpy().view(np.uint16 if hdr else np.uint8)
        assert np.array_equal(got, want), f"delivered frame {i}: {np.count_nonzero(got != want)} samples differ from the oracle"
    assert np.array_equal(g.readFlow(latest=True), s.readFlow(latest=True))
    g.close()
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("hdr", [False, True])
@pytest.mark.parametrize("mode", [3, 4, 5, 6])
def test_other_modes_at_production_size(synth, hdr, mode):
    """Modes 3-6 at 1920x1080 with padded strides: warpItem's INSIDE form (modes 3, 4) and the side-by-side modes."""
    W, H = 1920, 1080
    g, o = setup(synth, hdr, W, H, H, inS=W + 64, outS=W + 32)
    fl = written_flow(H, W, 11 + mode, 40)
    g.writeFlow(fl)
    o.writeFlow(fl)
    ts = [0.3, 0.7]
    forms = forms_of(g, fl, ts, mode)
    report(f"H {'P010' if hdr else 'NV12'} mode {mode}", forms)
    assert forms["lean_luma"] == forms["lean_chroma"] == 0
    if mode <= 4:
        assert forms["inside"] > 0 and forms["border"] > 0
    else:
        assert forms["inside"] == 0 and forms["border"] > 0
    check_against_oracle(g, o, hdr, ts, mode, f"mode {mode}")
