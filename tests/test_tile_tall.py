"""Tall tiles of the tile search kernel (sadTileKernel, kernels_search_slide.cu): 256-row CTAs (NWV 8) for windows of 64,
and for windows of 256 and more, at the frame sizes where chooseWarps picks them.  Every pass equals the oracle, pass by
pass, and each tile pass launches the grid of the NWV its CTAs report.  3200x1800 has a u-extent that is not a multiple
of 16 in X steps (1800), so the last tile column is partial; the mosaic pair moves blocks independently, so CTAs of
windows of 64 need more than one round inside a 256-row tile."""
import numpy as np
import pytest

from test_ladder_shapes import OracleLadder, _calc, check_production, compare_ladder, mosaic_frames, timeline_words

SM_COUNT_OF_TABLE = 148   # the NWV expectations below hold for this SM count (B200)


def _tile_passes(recs):
    return [r for r in recs if r["kind"] == "tile"]


def _check_heights(label, recs):
    """Class 128: NWV 8 exactly where a 256-row tile lies inside one window, else 4.  Returns {(class, NWV)}."""
    seen = set()
    for r in _tile_passes(recs):
        cls = min(r["ws"], 128)
        seen.add((cls, r["nwv"]))
        if cls == 128:
            assert r["nwv"] in ((4, 8) if r["ws"] % 256 == 0 else (4,)), f"{label}: ws {r['ws']} ran NWV {r['nwv']}"
        if cls == 64:
            assert r["nwv"] in (2, 4, 6, 8), f"{label}: ws 64 ran NWV {r['nwv']}"
    print(f"{label}: (window class, NWV) {sorted(seen)}")
    return seen


_SEEN = {}


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,R,kind", [
    (3840, 2160, 16, "scene"),
    (3840, 2160, 11, "scene"),
    (3200, 1800, 16, "scene"),
    (3200, 1800, 11, "scene"),
    (3840, 2160, 16, "mosaic"),
])
def test_tall_tiles_pass_by_pass(synth, W, H, R, kind):
    """HDR at full flow resolution: every pass, the final offsets, the blurred flow and the frame delta equal the oracle,
    and every tile pass's CTA count is the grid of its NWV; then the production path (CUDA graph) of the same frames."""
    label = f"{kind} {W}x{H} R {R}"
    if kind == "scene":
        f = [synth.make_frame(W, H, t, synth.SEED_BASE + 5, True) for t in (1, 2)]
        fs = [f[0], f[0], f[1]]
    else:
        fs = mosaic_frames(synth, W, H, True, seed=7)
    g = _calc(True, H, W, 0, H, R)
    for fr in fs:
        g.updateFrame(fr)
    lad = OracleLadder.of(fs, True, W, H, 0, H, R)
    recs = compare_ladder(g, lad, label, timeline_words(lad.lw, lad.lh))
    _SEEN[label] = _check_heights(label, recs)
    if kind == "mosaic":
        tall64 = [r for r in _tile_passes(recs) if r["ws"] == 64 and r["nwv"] == 8]
        if tall64:
            rounds = np.concatenate([r["tl"][:, 7] % 100 for r in tall64])
            assert np.any(rounds >= 2), f"{label}: no 256-row CTA of windows of 64 ran more than one round"
    check_production(g, lad.offsets, lad.flow, lad.frame_delta, label)
    g.close()


@pytest.mark.gpu
def test_tall_tiles_are_reached():
    """On a 148-SM B200 the model picks 256-row tiles for windows of 64 at 3840x2160 R 16 and for windows of 256 and
    more at 3840x2160."""
    import torch
    if len(_SEEN) < 5:
        pytest.skip("needs the pass-by-pass tests of this module in the same session")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != SM_COUNT_OF_TABLE:
        pytest.skip(f"{sms} SMs: the expectations are for {SM_COUNT_OF_TABLE}")
    assert (64, 8) in _SEEN["scene 3840x2160 R 16"]
    assert (128, 8) in _SEEN["scene 3840x2160 R 16"]
    assert (64, 8) in _SEEN["mosaic 3840x2160 R 16"]
