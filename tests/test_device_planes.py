"""Device frame planes (include/hrb.h, "device frame planes"): ingest from and warp into caller-owned pitched NV12 / P010
surfaces on the GPU.  Pitched torch allocations stand in for decoder and encoder surfaces.

Every GPU case compares the new entry points with the existing ones on the same seeded frames, bit for bit:
update_frame_planes with update_frame_device, warp_frames_to with warp_frames_batch + download_frame, copy_frame_to with
copy_frame; one case goes straight against the oracle.  Destinations are filled with a sentinel first, and every byte
outside the planes' rows (pitch padding, the gap between the planes, rows outside the output stripe) must keep it."""
import ctypes as C

import numpy as np
import pytest

from conftest import make_pair, out_array
from test_ladder_shapes import mosaic_frames

SENTINEL = 0xA5


# ---- CPU: argument checks without a device ------------------------------------------------------------------------
def test_new_symbols_are_declared_exported_and_prototyped():
    from test_abi import declared_symbols

    from hopperrender_b200 import _lib
    lib = C.CDLL(_lib.LIB_PATH)
    for n in ("hrb_ofc_update_frame_planes", "hrb_ofc_warp_frames_to", "hrb_ofc_copy_frame_to"):
        assert n in declared_symbols() and n in _lib.PROTOTYPES and hasattr(lib, n)


def test_null_handle_or_planes_are_argument_errors():
    from hopperrender_b200 import _lib as L
    lib = L.load()
    n0 = lib.hrb_kernel_launch_count()
    p = L.hrb_frame_planes(0x1000, 2048, 0x100000, 2048)
    ts = (C.c_float * 1)(0.5)
    assert lib.hrb_ofc_update_frame_planes(None, None) == L.HRB_ERR_INVALID_ARG
    assert lib.hrb_ofc_update_frame_planes(None, C.byref(p)) == L.HRB_ERR_INVALID_ARG
    assert lib.hrb_ofc_warp_frames_to(None, 1, ts, 2, None) == L.HRB_ERR_INVALID_ARG
    assert lib.hrb_ofc_warp_frames_to(None, 1, ts, 2, C.byref(p)) == L.HRB_ERR_INVALID_ARG
    assert lib.hrb_ofc_copy_frame_to(None, None) == L.HRB_ERR_INVALID_ARG
    assert lib.hrb_ofc_copy_frame_to(None, C.byref(p)) == L.HRB_ERR_INVALID_ARG
    assert b"null" in lib.hrb_last_error()
    assert lib.hrb_kernel_launch_count() == n0


@pytest.mark.parametrize("hdr", [False, True])
def test_python_wrappers_refuse_bad_planes_without_a_device(hdr):
    import torch

    from hopperrender_b200.ofc import frame_planes
    H, W = 48, 64
    dt = torch.int16 if hdr else torch.uint8
    y, uv = torch.zeros(H, W, dtype=dt), torch.zeros(H // 2, W, dtype=dt)
    with pytest.raises(TypeError, match="plane y: a torch tensor"):
        frame_planes(np.zeros((H, W), np.uint8), uv, H, W, hdr)
    with pytest.raises(ValueError, match=r"plane y: shape \(48, 62\)"):
        frame_planes(y[:, :62], uv, H, W, hdr)
    with pytest.raises(ValueError, match=r"plane uv: shape \(48, 64\)"):
        frame_planes(y, torch.zeros(H, W, dtype=dt), H, W, hdr)
    with pytest.raises(ValueError, match="plane y: dtype"):
        frame_planes(y.to(torch.int32), uv, H, W, hdr)
    with pytest.raises(ValueError, match="plane uv: dtype"):
        frame_planes(y, uv.to(torch.int16 if not hdr else torch.uint8), H, W, hdr)
    with pytest.raises(ValueError, match="plane uv: inner stride 2"):
        frame_planes(y, torch.zeros(H // 2, 2 * W, dtype=dt)[:, ::2], H, W, hdr)
    with pytest.raises(ValueError, match="plane y: a CUDA tensor"):
        frame_planes(y, uv, H, W, hdr)
    if hdr:  # both 16-bit types are accepted up to the device check
        with pytest.raises(ValueError, match="plane y: a CUDA tensor"):
            frame_planes(y.view(torch.uint16), uv.view(torch.uint16), H, W, hdr)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------
def tdt(hdr):
    import torch
    return torch.int16 if hdr else torch.uint8


def sentinel(hdr):
    return int(np.array([SENTINEL << 8 | SENTINEL], np.uint16).view(np.int16)[0]) if hdr else SENTINEL


def surface(hdr, H, W, y_pitch, uv_pitch, layout, offset=0):
    """(y, uv, backings) on cuda: y (H, W) with row pitch y_pitch samples, uv (H/2, W) with uv_pitch samples.
    layout "decoder": one allocation, chroma at y_pitch * align16(H) (NV12 / P010 as decoders lay it out);
    "separate": one allocation per plane.  offset: samples before the luma plane.  Every sample starts as the sentinel."""
    import torch

    def buf(n):
        return torch.full((n,), sentinel(hdr), dtype=tdt(hdr), device="cuda")
    if layout == "decoder":
        Ha = (H + 15) // 16 * 16
        b = buf(offset + y_pitch * Ha + uv_pitch * (H // 2) + 64)
        y = b.as_strided((H, W), (y_pitch, 1), offset)
        uv = b.as_strided((H // 2, W), (uv_pitch, 1), offset + y_pitch * Ha)
        return y, uv, [b]
    by, bu = buf(offset + y_pitch * H + 32), buf(uv_pitch * (H // 2) + 32)
    return by.as_strided((H, W), (y_pitch, 1), offset), bu.as_strided((H // 2, W), (uv_pitch, 1), 0), [by, bu]


def fill_planes(y, uv, frame, H, W, hdr):
    import torch
    f = torch.from_numpy(frame.view(np.int16) if hdr else frame).cuda().reshape(H + H // 2, -1)
    y.copy_(f[:H, :W])
    uv.copy_(f[H:, :W])


def host(t):
    return t.cpu().numpy()


def calc(hdr, H, W, maxres, R=16, inS=0, outS=0):
    import hopperrender_b200 as hr
    c = (hr.OpticalFlowCalcHDR if hdr else hr.OpticalFlowCalcSDR)(H, W, inS, outS, 8, 6, 4.0, 250.0, maxres)
    c.m_opticalFlowSearchRadius = R
    return c


def state_of(c):
    return dict(offsets=c.readOffsetArray(), flow=c.readFlow(), latest=c.readFlow(latest=True), peaks=c.readFlowPeak(),
                raw=c.readRawFrameDelta(), total=c.m_totalFrameDelta, count=c.m_frameCount)


def ring_frames(c, hdr, ts, mode):
    c.warpFramesBatch(ts, mode)
    outs = []
    for _ in ts:
        a = out_array(c, hdr)
        c.downloadFrame(a)
        outs.append(a)
    return outs


def assert_same_state(a, b, what):
    sa, sb = state_of(a), state_of(b)
    for k in sa:
        assert np.array_equal(np.asarray(sa[k]), np.asarray(sb[k])), f"{what}: {k} differs"


def scene(synth, W, H, hdr, n, seed=0):
    return [synth.make_frame(W, H, t, synth.SEED_BASE + seed, hdr) for t in range(n)]


# ---- ingest -----------------------------------------------------------------------------------------------------------
INGEST = [
    # hdr, W, H, maxres, y pitch (samples), uv pitch, layout, base offset (samples), content, entry
    pytest.param(False, 1920, 1080, 270, 2048, 2048, "decoder", 0, "scene", "planes", id="1080p-nv12-decoder-512B-pitch"),
    pytest.param(True, 3840, 2160, 2160, 3840 + 128, 3840 + 192, "separate", 0, "mosaic", "planes", id="4k-p010-separate-padded"),
    pytest.param(False, 1030, 580, 290, 1030, 1030, "separate", 0, "mosaic", "planes", id="1030x580-unaligned"),
    pytest.param(False, 1920, 1080, 540, 1920 + 64, 1920 + 64, "decoder", 2, "scene", "planes", id="sdr-base-plus-2-bytes"),
    pytest.param(True, 1920, 1080, 270, 2048, 2048, "decoder", 0, "mosaic", "alternate", id="alternating-entry-points"),
    pytest.param(False, 1920, 1080, 270, 2048, 2048, "separate", 0, "scene", "overwrite", id="source-overwritten-after-call"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,maxres,yp,up,layout,offset,content,entry", INGEST)
def test_update_frame_planes_equals_update_frame_device(synth, hdr, W, H, maxres, yp, up, layout, offset, content, entry):
    import torch
    frames = scene(synth, W, H, hdr, 6) if content == "scene" else (mosaic_frames(synth, W, H, hdr, 3) + mosaic_frames(synth, W, H, hdr, 4))
    a, b = calc(hdr, H, W, maxres), calc(hdr, H, W, maxres)
    stream_b = torch.cuda.ExternalStream(b.streamHandle())
    y, uv, _ = surface(hdr, H, W, yp, up, layout, offset)
    ts = [0.25, 0.5, 0.75]
    for t, fr in enumerate(frames):
        dev = torch.from_numpy(fr.view(np.int16) if hdr else fr).cuda()
        torch.cuda.synchronize()
        a.updateFrameDevice(dev)
        if entry == "alternate" and t % 2:
            b.updateFrameDevice(dev)
        else:
            fill_planes(y, uv, fr, H, W, hdr)
            torch.cuda.synchronize()
            b.updateFramePlanes(y, uv)
            if entry == "overwrite":  # the caller's next frame lands behind the ingest on the handle's stream
                with torch.cuda.stream(stream_b):
                    y.fill_(7)
                    uv.fill_(9)
        if t >= 1:
            a.calculateOpticalFlow()
            b.calculateOpticalFlow()
            assert_same_state(a, b, f"frame {t}")
            for i, (p, q) in enumerate(zip(ring_frames(a, hdr, ts, 2), ring_frames(b, hdr, ts, 2))):
                assert np.array_equal(p, q), f"frame {t}: warped output {i} differs"
    a.close()
    b.close()


# ---- egress -----------------------------------------------------------------------------------------------------------
def expected_backing(back, y, uv, ring, H, W, So, stripe):
    """back's contents after a correct warp into (y, uv): the sentinel everywhere except the stripe's rows of each plane
    that lies in back, which hold the ring frame's rows."""
    exp = np.full(back.numel(), sentinel(y.element_size() == 2), host(back).dtype)
    r = ring.reshape(-1, So)
    y0, y1 = stripe
    for plane, first, (r0, r1) in ((y, 0, (y0, y1)), (uv, H, (y0 // 2, y1 // 2))):
        off = (plane.data_ptr() - back.data_ptr()) // plane.element_size()
        if not 0 <= off < back.numel():
            continue
        pitch, rows = plane.stride(0), plane.shape[0]
        exp[off:off + rows * pitch].reshape(rows, pitch)[r0:r1, :W] = r[first + r0:first + r1, :W]
    return exp


def check_to(c, ts, mode, outs, ring, stripe):
    """outs: [(y, uv, backings)] a _to call wrote; ring: the ring frames of the same call."""
    import torch
    torch.cuda.synchronize()
    H, W, So = c.m_frameHeight, c.m_frameWidth, c.m_outputStride
    for i, ((y, uv, backs), r) in enumerate(zip(outs, ring)):
        for b in backs:
            got, exp = host(b), expected_backing(b, y, uv, r, H, W, So, stripe)
            diff = np.flatnonzero(got != exp)
            assert diff.size == 0, f"mode {mode} output {i}: {diff.size} samples differ, first at backing index {diff[:3].tolist()}"


EGRESS = [
    # hdr, W, H, maxres, y pitch, uv pitch, layout, stripe of 3
    pytest.param(False, 1920, 1080, 270, 2048, 1920 + 96, "separate", None, id="1080p-nv12"),
    pytest.param(True, 3840, 2160, 2160, 3840 + 64, 4096, "separate", None, id="4k-p010"),
    pytest.param(False, 1920, 1080, 270, 2048, 2048, "decoder", 1, id="1080p-nv12-decoder-stripe"),
    pytest.param(True, 3840, 2160, 2160, 4096, 4096, "decoder", 2, id="4k-p010-decoder-stripe"),
    pytest.param(False, 1920, 1080, 540, 1920 + 33, 1920 + 33, "separate", None, id="1080p-nv12-odd-pitch"),
    pytest.param(True, 1920, 1080, 270, 1920 + 33, 1920 + 65, "decoder", 0, id="1080p-p010-odd-pitch-stripe"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hdr,W,H,maxres,yp,up,layout,stripe", EGRESS)
def test_warp_frames_to_equals_the_ring(synth, hdr, W, H, maxres, yp, up, layout, stripe):
    c = calc(hdr, H, W, maxres)
    for fr in mosaic_frames(synth, W, H, hdr, 5):
        c.updateFrame(fr)
    c.calculateOpticalFlow()
    c.calculateOpticalFlow()
    rows = (0, H)
    if stripe is not None:
        b = [0, (H // 3) & ~1, (2 * H // 3) & ~1, H]
        rows = (b[stripe], b[stripe + 1])
        c.setOutputStripe(*rows)
    pool = [surface(hdr, H, W, yp, up, layout) for _ in range(8)]
    batches = {1: [0.5], 6: [i / 6 for i in range(1, 7)], 8: [0.0, 0.125, 0.25, 0.4, 0.5, 0.6, 0.875, 1.0]}
    for mode in range(7):
        for n, ts in batches.items():
            outs = pool[:n]
            for y, uv, backs in outs:
                for bb in backs:
                    bb.fill_(sentinel(hdr))
            c.warpFramesTo(ts, mode, [(y, uv) for y, uv, _ in outs])
            ring = ring_frames(c, hdr, ts, mode)
            check_to(c, ts, mode, outs, ring, rows)
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("hdr", [False, True])
def test_warp_frames_to_beside_a_flow_in_flight_and_copy_frame_to(synth, hdr):
    import torch
    W, H, maxres = (1920, 1080, 270)
    c = calc(hdr, H, W, maxres)
    frames = mosaic_frames(synth, W, H, hdr, 6)
    for fr in frames:
        c.updateFrame(fr)
    c.calculateOpticalFlow()
    c.updateFrame(frames[1])
    c.calculateOpticalFlowAsync()  # the warps below read the previous flow while this one runs
    ts = [1 / 6, 0.5, 5 / 6]
    outs = [surface(hdr, H, W, 2048, 2048, "decoder") for _ in ts]
    c.warpFramesTo(ts, 2, [(y, uv) for y, uv, _ in outs])
    ring = ring_frames(c, hdr, ts, 2)
    check_to(c, ts, 2, outs, ring, (0, H))
    c.synchronize()
    # copy_frame_to against copy_frame
    dst = surface(hdr, H, W, 1920 + 128, 1920 + 128, "separate")
    c.copyFrameTo(dst[:2])
    c.copyFrame()
    a = out_array(c, hdr)
    c.downloadFrame(a)
    torch.cuda.synchronize()
    check_to(c, [0], "copy", [dst], [a], (0, H))
    c.close()


@pytest.mark.gpu
def test_to_calls_leave_the_ring_alone(synth):
    """A ring warp, then a _to warp, then download_frame: the download returns the ring frame, output_device_ptr still
    points at it, and warp_calc_time is the one the ring's download set."""
    import torch
    hdr, W, H = False, 1920, 1080
    c = calc(hdr, H, W, 270)
    for fr in mosaic_frames(synth, W, H, hdr, 7):
        c.updateFrame(fr)
    c.calculateOpticalFlow()
    c.calculateOpticalFlow()
    want = ring_frames(c, hdr, [0.25], 2)[0]
    c.warpFrames(0.25, 2)
    ptr = c.outputDevicePtr()
    y, uv, _ = surface(hdr, H, W, 2048, 2048, "decoder")
    c.warpFramesTo([0.75], 2, [(y, uv)])
    c.copyFrameTo((y, uv))
    assert c.outputDevicePtr() == ptr
    got = out_array(c, hdr)
    c.downloadFrame(got)
    assert np.array_equal(got, want)
    t_ring = c.m_warpCalcTime
    c.warpFramesTo([0.5], 2, [(y, uv)])
    torch.cuda.synchronize()
    assert c.m_warpCalcTime == t_ring
    c.close()


@pytest.mark.gpu
def test_warp_frames_to_against_the_oracle_at_the_playback_shape(synth):
    """1080p NV12 with the flow at 480x270 (rs 2), a padded decoder-layout destination: pinned to the oracle, not only to
    the ring."""
    import torch
    hdr, W, H = False, 1920, 1080
    g, o = make_pair(hdr, H, W, black=4.0, white=250.0, maxres=270, R=16)
    for fr in mosaic_frames(synth, W, H, hdr, 8):
        g.updateFrame(fr)
        o.updateFrame(fr)
    g.calculateOpticalFlow()
    o.writeFlow(g.readFlow())
    ts = [0.25, 0.5, 5 / 6]
    outs = [surface(hdr, H, W, 2048, 2048, "decoder") for _ in ts]
    g.warpFramesTo(ts, 2, [(y, uv) for y, uv, _ in outs])
    torch.cuda.synchronize()
    for t, (y, uv, _) in zip(ts, outs):
        o.warpFrames(t, 2)
        b = out_array(o, hdr)
        o.downloadFrame(b)
        b = b.reshape(-1, W)
        assert np.array_equal(host(y), b[:H]), f"luma at t {t}"
        assert np.array_equal(host(uv), b[H:]), f"chroma at t {t}"
    g.close()
    o.close()


# ---- refusals -------------------------------------------------------------------------------------------------------
def _refused(c, fn, *args, code=1, needle=None):
    from hopperrender_b200 import _lib as L
    lib = L.load()
    n0 = lib.hrb_kernel_launch_count()
    rc = getattr(lib, fn)(c._h, *args)
    msg = L.last_error()
    assert rc == code, (rc, msg)
    assert lib.hrb_kernel_launch_count() == n0
    if needle:
        assert needle in msg, msg
    return msg


def _planes(y, yp, uv, up):
    from hopperrender_b200 import _lib as L
    return L.hrb_frame_planes(y, yp, uv, up)


@pytest.mark.gpu
@pytest.mark.parametrize("hdr", [False, True])
def test_refusals_launch_nothing(synth, hdr):
    import torch

    from hopperrender_b200 import _lib as L
    W, H = 1920, 1080
    es = 2 if hdr else 1
    c = calc(hdr, H, W, 270)
    for fr in scene(synth, W, H, hdr, 3):
        c.updateFrame(fr)
    c.calculateOpticalFlow()
    P = 2048 * es  # byte pitch
    good = [torch.empty(P * H, dtype=torch.uint8, device="cuda") for _ in range(4)]
    gy, guv = good[0].data_ptr(), good[1].data_ptr()
    ts1 = (C.c_float * 1)(0.5)

    def all_three(p, needle):
        _refused(c, "hrb_ofc_update_frame_planes", C.byref(p), needle=needle)
        _refused(c, "hrb_ofc_warp_frames_to", 1, ts1, 2, C.byref(p), needle=needle)
        _refused(c, "hrb_ofc_copy_frame_to", C.byref(p), needle=needle)

    # host memory, pageable and pinned
    pageable = np.zeros(P * H, np.uint8)
    all_three(_planes(pageable.ctypes.data, P, guv, P), "y plane is host memory")
    pinned = torch.zeros(P * H, dtype=torch.uint8).pin_memory()
    all_three(_planes(gy, P, pinned.data_ptr(), P), "uv plane is host memory")
    # a buffer too small for the plane's extent: a fresh allocation of its own (the caching allocator gives a request
    # above 10 MB a segment of exactly its size once the cache is empty)
    torch.cuda.empty_cache()
    big = torch.empty(12 << 20, dtype=torch.uint8, device="cuda")
    end = big.data_ptr() + big.numel()
    all_three(_planes(end - P * (H - 1), P, guv, P), "runs past the end of its allocation")
    all_three(_planes(gy, P, end - P * (H // 2 - 1) - 2 * es, P), "runs past the end of its allocation")
    # short pitch
    all_three(_planes(gy, W * es - es, guv, P), "pitch is below")
    all_three(_planes(gy, P, guv, W * es - 2 * es), "pitch is below")
    if hdr:  # odd byte pitch or pointer
        all_three(_planes(gy, P + 1, guv, P), "multiples of the sample size")
        all_three(_planes(gy + 1, P, guv, P), "multiples of the sample size")
        all_three(_planes(gy, P, guv + 1, P), "multiples of the sample size")
    # overlapping Y / UV planes
    all_three(_planes(gy, P, gy + P * (H // 2), P), "Y and UV planes of frame 0 overlap")
    # destinations: overlapping, differing pitches
    d = (L.hrb_frame_planes * 2)(_planes(gy, P, guv, P), _planes(gy + P * 10, P, good[2].data_ptr(), P))
    ts2 = (C.c_float * 2)(0.25, 0.75)
    _refused(c, "hrb_ofc_warp_frames_to", 2, ts2, 2, d, needle="dst[0] and dst[1] overlap")
    d = (L.hrb_frame_planes * 2)(_planes(gy, P, guv, P), _planes(good[2].data_ptr(), P - 2 * es, good[3].data_ptr(), P))
    _refused(c, "hrb_ofc_warp_frames_to", 2, ts2, 2, d, needle="share one (y_pitch_bytes, uv_pitch_bytes)")
    # n of 0 or 9, a blend scalar above 1
    d9 = (L.hrb_frame_planes * 9)(*[_planes(gy, P, guv, P)] * 9)
    ts9 = (C.c_float * 9)(*[0.5] * 9)
    _refused(c, "hrb_ofc_warp_frames_to", 0, ts9, 2, d9, needle="batch size")
    _refused(c, "hrb_ofc_warp_frames_to", 9, ts9, 2, d9, needle="batch size")
    _refused(c, "hrb_ofc_warp_frames_to", 1, (C.c_float * 1)(1.5), 2, d9, code=L.HRB_ERR_BLEND_RANGE, needle="greater than 1.0")
    _refused(c, "hrb_ofc_warp_frames_to", 1, ts1, 7, d9, needle="frame_output_mode")
    # the same planes are accepted: the refusals above were for their stated reason
    n0 = L.load().hrb_kernel_launch_count()
    assert L.load().hrb_ofc_warp_frames_to(c._h, 1, ts1, 2, C.byref(_planes(gy, P, guv, P))) == 0
    assert L.load().hrb_ofc_update_frame_planes(c._h, C.byref(_planes(gy, P, guv, P))) == 0
    assert L.load().hrb_kernel_launch_count() == n0 + 2
    c.synchronize()
    c.close()


@pytest.mark.gpu
def test_memory_of_another_gpu_is_refused(synth):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    from hopperrender_b200 import _lib as L
    W, H = 640, 360
    c = calc(False, H, W, 360)
    y = torch.zeros(H, W, dtype=torch.uint8, device="cuda:1")
    uv = torch.zeros(H // 2, W, dtype=torch.uint8, device="cuda:1")
    n0 = L.load().hrb_kernel_launch_count()
    with pytest.raises(RuntimeError, match="hrb error 1.*another device"):
        c.updateFramePlanes(y, uv)
    with pytest.raises(RuntimeError, match="hrb error 1.*another device"):
        c.warpFramesTo([0.5], 2, [(y, uv)])
    assert L.load().hrb_kernel_launch_count() == n0
    c.close()
