"""Host-side mirror of the reference's calculator classes over the C ABI.

Same names, constructor arguments, methods and public fields as `OpticalFlowCalc`,
`OpticalFlowCalcSDR`, `OpticalFlowCalcHDR` (HopperRender/opticalFlowCalc.h:24-138,
opticalFlowCalcSDR.h:13-56, opticalFlowCalcHDR.h:13-56).  The C++ counterpart of this file is
include/opticalFlowCalc.h; this Python one exists so that tests and bench.py read like the
reference's call sequence (HopperRender/HopperRender.cpp:918-957, 1179-1186).

Errors: the reference throws std::runtime_error (opticalFlowCalc.h:15-22, opticalFlowCalcSDR.cpp:143-146);
here every non-zero C-ABI return raises RuntimeError carrying hrb_last_error().
"""
import ctypes as C

import numpy as np

from . import _lib as L

# frameOutputMode values, HopperRender/HopperRender.h:10-18
WarpedFrame12, WarpedFrame21, BlendedFrame, HSVFlow, GreyFlow, SideBySide1, SideBySide2 = range(7)


def _ptr(a):
    """Raw address of a numpy array / torch tensor / int."""
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("frame buffers must be C-contiguous")
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(f"unsupported buffer type {type(a)}")


def _nbytes(a):
    if isinstance(a, np.ndarray):
        return a.nbytes
    if hasattr(a, "element_size"):
        return a.numel() * a.element_size()
    return None


def frame_planes(y, uv, height, width, hdr):
    """hrb_frame_planes of a frame held as two CUDA tensors: y of shape (height, width), uv of shape (height / 2, width)
    (interleaved U, V), uint8 for SDR, int16 or uint16 for HDR, unit inner stride; the row pitch is stride(0) times the
    element size.  Raises before any device is touched; the library checks the memory itself."""
    dtypes = ("torch.int16", "torch.uint16") if hdr else ("torch.uint8",)
    for name, t, rows in (("y", y, height), ("uv", uv, height // 2)):
        if not all(hasattr(t, a) for a in ("dtype", "is_cuda", "stride", "data_ptr")):
            raise TypeError(f"plane {name}: a torch tensor is required, got {type(t).__name__}")
        if tuple(t.shape) != (rows, width):
            raise ValueError(f"plane {name}: shape {tuple(t.shape)}, ({rows}, {width}) needed")
        if str(t.dtype) not in dtypes:
            raise ValueError(f"plane {name}: dtype {t.dtype}, {' or '.join(dtypes)} needed for {'HDR' if hdr else 'SDR'}")
        if t.stride(1) != 1:
            raise ValueError(f"plane {name}: inner stride {t.stride(1)}, 1 needed")
    for name, t in (("y", y), ("uv", uv)):
        if not t.is_cuda:
            raise ValueError(f"plane {name}: a CUDA tensor is required, got one on {t.device}")
    es = 2 if hdr else 1
    return L.hrb_frame_planes(y.data_ptr(), y.stride(0) * es, uv.data_ptr(), uv.stride(0) * es)


class OpticalFlowCalc:
    """Abstract base (HopperRender/opticalFlowCalc.h:24-138).  Instantiate OpticalFlowCalcSDR / HDR."""

    _is_hdr = None

    def __init__(self, frameHeight, frameWidth, inputStride, outputStride, deltaScalar, neighborScalar, blackLevel,
                 whiteLevel, maxCalcRes, device=0, stream=None):
        if self._is_hdr is None:
            raise TypeError("OpticalFlowCalc is abstract; use OpticalFlowCalcSDR or OpticalFlowCalcHDR")
        self._lib = L.load()
        self._h = C.c_void_p()
        d = L.hrb_ofc_desc(frameHeight, frameWidth, inputStride, outputStride, deltaScalar, neighborScalar, blackLevel,
                           whiteLevel, maxCalcRes, 1 if self._is_hdr else 0, device, stream)
        self._check(self._lib.hrb_ofc_create(C.byref(self._h), C.byref(d)))
        s = self._state()
        self._geom = s  # geometry never changes on a live object: read it once (every later field access would be a round trip)
        self._in_bytes = (s.frame_height * s.input_stride + (s.frame_height // 2) * s.input_stride) * (2 if self._is_hdr else 1)
        self._out_bytes = (s.frame_height * s.output_stride + (s.frame_height // 2) * s.output_stride) * (2 if self._is_hdr else 1)

    # ---- plumbing ---------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != L.HRB_OK:
            raise RuntimeError(f"hrb error {rc}: {L.last_error()}")

    def _state(self):
        s = L.hrb_ofc_state()
        self._check(self._lib.hrb_ofc_get_state(self._h, C.byref(s)))
        return s

    def _peek(self):
        """Public fields without waiting for flow calculations still in flight (hrb_ofc_peek_state)."""
        s = L.hrb_ofc_state()
        self._check(self._lib.hrb_ofc_peek_state(self._h, C.byref(s)))
        return s

    def _set(self, **kw):
        s = self._peek()  # the live parameters are host-side values: no need to wait for the GPU
        p = L.hrb_ofc_params(s.search_radius, s.delta_scalar, s.neighbor_bias_scalar, s.output_black_level, s.output_white_level)
        for k, v in kw.items():
            setattr(p, k, v)
        self._check(self._lib.hrb_ofc_set_params(self._h, C.byref(p)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.hrb_ofc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- the five virtuals (opticalFlowCalc.h:100-132) ---------------------------------------------
    def updateFrame(self, inputPlanes):
        n = _nbytes(inputPlanes)
        if n is not None and n < self._in_bytes:
            raise ValueError(f"inputPlanes holds {n} bytes, {self._in_bytes} needed")
        self._check(self._lib.hrb_ofc_update_frame(self._h, _ptr(inputPlanes)))

    def downloadFrame(self, outputPlanes):
        n = _nbytes(outputPlanes)
        if n is not None and n < self._out_bytes:
            raise ValueError(f"outputPlanes holds {n} bytes, {self._out_bytes} needed")
        self._check(self._lib.hrb_ofc_download_frame(self._h, _ptr(outputPlanes)))

    def calculateOpticalFlow(self):
        self._check(self._lib.hrb_ofc_calculate_optical_flow(self._h))

    def warpFrames(self, blendingScalar, frameOutputMode):
        self._check(self._lib.hrb_ofc_warp_frames(self._h, float(blendingScalar), int(frameOutputMode)))

    def warpFramesBatch(self, blendingScalars, frameOutputMode):
        """The output frames of one source pair in one pass (hrb_ofc_warp_frames_batch): fetch them with len(blendingScalars)
        downloadFrame / downloadFrameAsync calls."""
        import ctypes as C
        arr = (C.c_float * len(blendingScalars))(*[float(b) for b in blendingScalars])
        self._check(self._lib.hrb_ofc_warp_frames_batch(self._h, len(blendingScalars), arr, int(frameOutputMode)))

    def copyFrame(self):
        self._check(self._lib.hrb_ofc_copy_frame(self._h))

    # ---- device-resident / asynchronous variants ---------------------------------------------------
    def updateFrameDevice(self, devicePlanes):
        self._check(self._lib.hrb_ofc_update_frame_device(self._h, _ptr(devicePlanes)))

    def calculateOpticalFlowAsync(self):
        self._check(self._lib.hrb_ofc_calculate_optical_flow_async(self._h))

    def _planes(self, y, uv):
        return frame_planes(y, uv, self._geom.frame_height, self._geom.frame_width, self._is_hdr)

    def updateFramePlanes(self, y, uv):
        """updateFrameDevice from two CUDA tensors, luma (H, W) and interleaved chroma (H/2, W), each with its own row pitch
        (hrb_ofc_update_frame_planes).  They are read on streamHandle()."""
        self._check(self._lib.hrb_ofc_update_frame_planes(self._h, C.byref(self._planes(y, uv))))

    def warpFramesTo(self, blendingScalars, frameOutputMode, outs):
        """warpFramesBatch into caller tensors: output frame i goes to outs[i] = (y, uv) (hrb_ofc_warp_frames_to); the
        output ring is not touched.  The frames are ready for work ordered behind streamHandle()."""
        if len(outs) != len(blendingScalars):
            raise ValueError(f"{len(blendingScalars)} blending scalars but {len(outs)} destinations")
        dst = (L.hrb_frame_planes * max(len(outs), 1))(*[self._planes(y, uv) for y, uv in outs])
        arr = (C.c_float * max(len(blendingScalars), 1))(*[float(b) for b in blendingScalars])
        self._check(self._lib.hrb_ofc_warp_frames_to(self._h, len(outs), arr, int(frameOutputMode), dst))

    def copyFrameTo(self, out):
        """copyFrame into a caller tensor pair (y, uv) (hrb_ofc_copy_frame_to)."""
        y, uv = out
        self._check(self._lib.hrb_ofc_copy_frame_to(self._h, C.byref(self._planes(y, uv))))

    def updateFrameAsync(self, pinnedInputPlanes):
        self._check(self._lib.hrb_ofc_update_frame_async(self._h, _ptr(pinnedInputPlanes)))

    def waitUpload(self):
        self._check(self._lib.hrb_ofc_wait_upload(self._h))

    def downloadFrameAsync(self, pinnedOutputPlanes):
        """Enqueue the download; returns the ticket for waitDownload()."""
        t = C.c_ulonglong()
        self._check(self._lib.hrb_ofc_download_frame_async(self._h, _ptr(pinnedOutputPlanes), C.byref(t)))
        return t.value

    def waitDownload(self, ticket):
        self._check(self._lib.hrb_ofc_wait_download(self._h, ticket))

    def synchronize(self):
        self._check(self._lib.hrb_ofc_synchronize(self._h))

    def setOutputStripe(self, rowBegin, rowEnd):
        self._check(self._lib.hrb_ofc_set_output_stripe(self._h, int(rowBegin), int(rowEnd)))

    def outputDevicePtr(self):
        p = C.c_void_p()
        self._check(self._lib.hrb_ofc_output_device_ptr(self._h, C.byref(p)))
        return p.value

    def streamHandle(self):
        p = C.c_void_p()
        self._check(self._lib.hrb_ofc_stream(self._h, C.byref(p)))
        return p.value or 0

    # ---- public fields (opticalFlowCalc.h:26-50) ---------------------------------------------------
    m_frameWidth = property(lambda s: getattr(s._geom, 'frame_width'))
    m_frameHeight = property(lambda s: getattr(s._geom, 'frame_height'))
    m_inputStride = property(lambda s: getattr(s._geom, 'input_stride'))
    m_outputStride = property(lambda s: getattr(s._geom, 'output_stride'))
    m_opticalFlowResScalar = property(lambda s: getattr(s._geom, 'res_scalar'))
    m_opticalFlowFrameWidth = property(lambda s: getattr(s._geom, 'flow_width'))
    m_opticalFlowFrameHeight = property(lambda s: getattr(s._geom, 'flow_height'))
    m_ofcCalcTime = property(lambda s: s._state().ofc_calc_time)
    m_ofcAvgCalcTime = property(lambda s: s._state().ofc_avg_calc_time)
    m_ofcPeakCalcTime = property(lambda s: s._state().ofc_peak_calc_time)
    m_ofcCalcCount = property(lambda s: s._state().ofc_calc_count)
    m_ofcCalcTimeSum = property(lambda s: s._state().ofc_calc_time_sum)
    m_warpCalcTime = property(lambda s: s._state().warp_calc_time)
    m_totalFrameDelta = property(lambda s: s._state().total_frame_delta)

    @property
    def m_frameCount(self):
        return self._peek().frame_count

    @m_frameCount.setter
    def m_frameCount(self, v):  # the filter writes 0 on seek, HopperRender.cpp:840
        self._check(self._lib.hrb_ofc_set_frame_count(self._h, int(v)))

    @property
    def m_opticalFlowSearchRadius(self):
        return self._peek().search_radius

    @m_opticalFlowSearchRadius.setter
    def m_opticalFlowSearchRadius(self, v):  # HopperRender.cpp:1448,1457
        self._set(search_radius=int(v))

    @property
    def m_deltaScalar(self):
        return self._peek().delta_scalar

    @m_deltaScalar.setter
    def m_deltaScalar(self, v):  # HopperRender.cpp:1386
        self._set(delta_scalar=int(v))

    @property
    def m_neighborBiasScalar(self):
        return self._peek().neighbor_bias_scalar

    @m_neighborBiasScalar.setter
    def m_neighborBiasScalar(self, v):  # HopperRender.cpp:1387
        self._set(neighbor_bias_scalar=int(v))

    @property
    def m_outputBlackLevel(self):
        return self._peek().output_black_level

    @m_outputBlackLevel.setter
    def m_outputBlackLevel(self, v):  # HopperRender.cpp:1388
        self._set(black_level=float(v))

    @property
    def m_outputWhiteLevel(self):
        return self._peek().output_white_level

    @m_outputWhiteLevel.setter
    def m_outputWhiteLevel(self, v):  # HopperRender.cpp:1389
        self._set(white_level=float(v))

    # ---- sizes --------------------------------------------------------------------------------------
    @property
    def inputFrameBytes(self):
        return self._in_bytes

    @property
    def outputFrameBytes(self):
        return self._out_bytes

    # ---- test taps ----------------------------------------------------------------------------------
    def setTapMode(self, on):
        self._check(self._lib.hrb_ofc_set_tap_mode(self._h, 1 if on else 0))

    def numPasses(self):
        n = C.c_int()
        self._check(self._lib.hrb_ofc_num_passes(self._h, C.byref(n)))
        return n.value

    def passInfo(self, p):
        v = [C.c_int() for _ in range(5)]
        self._check(self._lib.hrb_ofc_pass_info(self._h, p, *[C.byref(x) for x in v]))
        return dict(zip(("windowSize", "iteration", "step", "windowsX", "windowsY"), (x.value for x in v)))

    def readPassSums(self, p, R):
        i = self.passInfo(p)
        a = np.empty((R, i["windowsY"], i["windowsX"]), np.uint32)
        self._check(self._lib.hrb_ofc_read_pass_tap(self._h, p, L.TAP_WINDOW_SUMS, _ptr(a), a.nbytes))
        return a

    def readPassLayers(self, p):
        i = self.passInfo(p)
        a = np.empty((i["windowsY"], i["windowsX"]), np.uint8)
        self._check(self._lib.hrb_ofc_read_pass_tap(self._h, p, L.TAP_WINDOW_LAYER, _ptr(a), a.nbytes))
        return a

    def _flowShape(self):
        s = self._state()
        return (2, s.flow_height, s.flow_width)

    def readPassOffsets(self, p):
        a = np.empty(self._flowShape(), np.int16)
        self._check(self._lib.hrb_ofc_read_pass_tap(self._h, p, L.TAP_OFFSETS, _ptr(a), a.nbytes))
        return a

    def readOffsetArray(self):
        a = np.empty(self._flowShape(), np.int16)
        self._check(self._lib.hrb_ofc_read_buffer(self._h, L.BUF_OFFSET_ARRAY, _ptr(a), a.nbytes))
        return a

    def readFlow(self, latest=False):
        a = np.empty(self._flowShape(), np.int16)
        self._check(self._lib.hrb_ofc_read_buffer(self._h, L.BUF_FLOW_LATEST if latest else L.BUF_FLOW_FOR_WARP, _ptr(a), a.nbytes))
        return a

    def readFlowPeak(self):
        """(peak |flow| of the field warpFrames reads, of the latest field): the bound the warp kernel uses to skip the mirror."""
        a = np.zeros(2, np.uint32)
        self._check(self._lib.hrb_ofc_read_buffer(self._h, L.BUF_FLOW_PEAK, _ptr(a), a.nbytes))
        return int(a[0]), int(a[1])

    def writeFlow(self, flow, latest=False):
        flow = np.ascontiguousarray(flow, np.int16)
        self._check(self._lib.hrb_ofc_write_flow(self._h, L.BUF_FLOW_LATEST if latest else L.BUF_FLOW_FOR_WARP, _ptr(flow), flow.size))

    def readRawFrameDelta(self):
        a = np.zeros(1, np.uint32)
        self._check(self._lib.hrb_ofc_read_buffer(self._h, L.BUF_RAW_FRAME_DELTA, _ptr(a), 4))
        return int(a[0])

    # ---- measurement ----------------------------------------------------------------------------------
    def setSearchVariant(self, variant):
        self._check(self._lib.hrb_ofc_set_search_variant(self._h, int(variant)))

    def setSideData(self, blobs):
        """Attach the IMediaSideData blobs {guid (16 bytes): bytes} of the frame given to the last updateFrame (hrb_ofc_set_side_data)."""
        items = (L.hrb_side_data * max(len(blobs), 1))()
        keep = []
        for i, (guid, data) in enumerate(blobs.items()):
            assert len(guid) == 16
            items[i].guid[:] = list(guid)
            buf = C.create_string_buffer(bytes(data), len(data))
            keep.append(buf)
            items[i].data = C.cast(buf, C.c_void_p)
            items[i].bytes = len(data)
        self._check(self._lib.hrb_ofc_set_side_data(self._h, items, len(blobs)))

    def getSideData(self):
        """The blobs that belong to the output frames being delivered (hrb_ofc_get_side_data), as {guid: bytes}."""
        n = C.c_int(0)
        self._check(self._lib.hrb_ofc_get_side_data(self._h, None, 0, C.byref(n)))
        items = (L.hrb_side_data * max(n.value, 1))()
        self._check(self._lib.hrb_ofc_get_side_data(self._h, items, n.value, C.byref(n)))
        return {bytes(items[i].guid): C.string_at(items[i].data, items[i].bytes) if items[i].bytes else b"" for i in range(n.value)}

    def debugTimeline(self, words_per_pass):
        """Debug aid: per-CTA timelines of the tile search kernels of the following flow calculations (0 = off)."""
        self._check(self._lib.hrb_ofc_debug_timeline(self._h, int(words_per_pass)))

    def readDebugTimeline(self, words_per_pass, passes=32):
        import numpy as np
        buf = np.zeros(words_per_pass * passes, np.uint64)
        self._check(self._lib.hrb_ofc_debug_timeline_read(self._h, buf.ctypes.data, buf.nbytes))
        return buf.reshape(passes, words_per_pass // 16, 16)

    def setFlowOverlap(self, on):
        """calculateOpticalFlowAsync on its own stream beside the following warps (default) or on the compute stream."""
        self._check(self._lib.hrb_ofc_set_flow_overlap(self._h, 1 if on else 0))

    def joinFlow(self):
        """Order the compute stream behind the flow calculation still in flight (no host wait)."""
        self._check(self._lib.hrb_ofc_join_flow(self._h))

    def setProfile(self, on):
        self._check(self._lib.hrb_ofc_set_profile(self._h, 1 if on else 0))

    def profileReset(self):
        self._check(self._lib.hrb_ofc_profile_reset(self._h))

    def profileRead(self):
        p = L.hrb_ofc_profile()
        self._check(self._lib.hrb_ofc_profile_read(self._h, C.byref(p)))
        return {k: getattr(p, k) for k, _ in p._fields_}


class OpticalFlowCalcSDR(OpticalFlowCalc):
    """NV12 8-bit (HopperRender/opticalFlowCalcSDR.h:13-56)."""
    _is_hdr = False


class OpticalFlowCalcHDR(OpticalFlowCalc):
    """P010 10-bit-in-16 (HopperRender/opticalFlowCalcHDR.h:13-56)."""
    _is_hdr = True


def split_plan(flowHeight, n):
    """Flow-row bounds [b_0 .. b_n] of n shards of a split search (hrb_split_plan); needs no device."""
    b = (C.c_int * (max(int(n), 0) + 1))()
    rc = L.load().hrb_split_plan(int(flowHeight), int(n), b)
    if rc != L.HRB_OK:
        raise RuntimeError(f"hrb error {rc}: {L.last_error()}")
    return list(b)


class SplitSearch:
    """A group of calculators (one per shard, usually one per GPU) that compute ONE flow together (hrb_split_*): shard k
    searches the windows of its flow-row stripe, and afterwards every calculator holds exactly the flow a lone
    calculateOpticalFlow would have computed, so warpFrames / setOutputStripe / downloadFrame work on each unchanged.
    Every calculator must already hold both source frames (updateFrame / updateFrameDevice on each).  The group owns
    nothing: close it before its calculators."""

    def __init__(self, calcs):
        self._lib = L.load()
        self._calcs = list(calcs)  # keeps the handles alive as long as the group
        self._s = C.c_void_p()
        arr = (C.c_void_p * len(self._calcs))(*[c._h.value for c in self._calcs])
        self._check(self._lib.hrb_split_create(C.byref(self._s), arr, len(self._calcs)))

    def _check(self, rc):
        if rc != L.HRB_OK:
            raise RuntimeError(f"hrb error {rc}: {L.last_error()}")

    def calculateOpticalFlow(self):
        self._check(self._lib.hrb_split_calculate_optical_flow(self._s))

    def calculateOpticalFlowAsync(self):
        self._check(self._lib.hrb_split_calculate_optical_flow_async(self._s))

    def stripe(self, k):
        """(first flow row, end flow row) shard k owns."""
        b, e = C.c_int(), C.c_int()
        self._check(self._lib.hrb_split_stripe(self._s, int(k), C.byref(b), C.byref(e)))
        return b.value, e.value

    def __len__(self):
        return len(self._calcs)

    def close(self):
        if getattr(self, "_s", None) is not None and self._s.value:
            self._lib.hrb_split_destroy(self._s)
            self._s = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FlowBatch:
    """The flows of many same-size streams, searched together on one GPU (hrb_flow_batch_*): every generic-kernel pass of
    the ladder, and the blur, is one launch over all calculators.  Afterwards each calculator is in exactly the state its
    own calculateOpticalFlow(Async) would have left it in.  The calculators must agree on frame size, res_scalar, search
    radius, search variant and device; each must already hold its own two source frames.  The batch owns no frame or
    flow memory: close it before its calculators."""

    def __init__(self, calcs):
        self._lib = L.load()
        self._calcs = list(calcs)  # keeps the handles alive as long as the batch
        self._b = C.c_void_p()
        arr = (C.c_void_p * max(len(self._calcs), 1))(*[c._h.value for c in self._calcs])
        self._check(self._lib.hrb_flow_batch_create(C.byref(self._b), arr, len(self._calcs)))

    def _check(self, rc):
        if rc != L.HRB_OK:
            raise RuntimeError(f"hrb error {rc}: {L.last_error()}")

    def calculateOpticalFlow(self):
        self._check(self._lib.hrb_flow_batch_calculate_optical_flow(self._b))

    def calculateOpticalFlowAsync(self):
        self._check(self._lib.hrb_flow_batch_calculate_optical_flow_async(self._b))

    def __len__(self):
        return len(self._calcs)

    def close(self):
        if getattr(self, "_b", None) is not None and self._b.value:
            self._lib.hrb_flow_batch_destroy(self._b)
            self._b = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Delivery:
    """The filter's delivery loop (DeliverToRenderer, HopperRender.cpp:944-1211) over one calculator (hrb_delivery_*):
    output count, auto-tuner, flow, frame-delta history, scene-change rule and blending scalar, with the scene-change
    decision taken on the GPU.  While it is open, calculateOpticalFlow(Async), warpFrames* and copyFrame* on the
    calculator raise; ingest and downloads stay available.  Close it before the calculator.

    deliver() has the signature and the info dicts of hopperrender_b200.replay.DeliveryLoop.deliver; deliver_to() writes
    into caller tensors and leaves the decision in flight (outcome() fetches it)."""

    def __init__(self, calc, source_frame_time=417083, target_frame_time=69444, frame_output=2, scene_change_threshold=200,
                 active=True, auto_adjust=True):
        self._lib = L.load()
        self.calc = calc  # keeps the handle alive as long as the delivery
        self._d = C.c_void_p()
        self._desc = L.hrb_delivery_desc(int(source_frame_time), int(target_frame_time), int(frame_output), int(scene_change_threshold),
                                         1 if active else 0, 1 if auto_adjust else 0)
        self._check(self._lib.hrb_delivery_create(C.byref(self._d), calc._h, C.byref(self._desc)))
        self._frames = (L.hrb_delivery_frame * L.DELIVERY_MAX_FRAMES)()

    def _check(self, rc):
        if rc != L.HRB_OK:
            raise RuntimeError(f"hrb error {rc}: {L.last_error()}")

    def next_count(self):
        n = C.c_int()
        self._check(self._lib.hrb_delivery_next_count(self._d, C.byref(n)))
        return n.value

    def _infos(self, n):
        return [{"source": f.source, "index": f.index, "blend": f.blend, "step": f.step} for f in self._frames[:n]]

    def step(self):
        """One step into the output ring: fetch its frames with len(result) downloads."""
        n = C.c_int()
        self._check(self._lib.hrb_delivery_step(self._d, self._frames, L.DELIVERY_MAX_FRAMES, C.byref(n)))
        return self._infos(n.value)

    def outcome(self, step, wait=True):
        """{warped, scene_change, delta1, delta2, frame_delta} of a step; None while in flight when wait is False."""
        o = L.hrb_delivery_outcome()
        rc = self._lib.hrb_delivery_outcome_of(self._d, int(step), 1 if wait else 0, C.byref(o))
        if rc == L.HRB_ERR_STATE and not wait:
            return None
        self._check(rc)
        return {"warped": bool(o.warped), "scene_change": bool(o.scene_change), "delta1": o.delta1, "delta2": o.delta2,
                "frame_delta": o.frame_delta}

    def deliver(self, in_buffer, out_buffer, sink=None, side_data=None):
        """updateFrame, one step into the ring, one downloadFrame per output frame; sink(out_buffer, info) as in
        replay.DeliveryLoop.deliver.  Returns the number of frames delivered."""
        c = self.calc
        c.updateFrame(in_buffer)
        frames = self.step()
        radius = c.m_opticalFlowSearchRadius
        for info in frames:
            c.downloadFrame(out_buffer)
            o = self.outcome(info["step"])
            info.update(warped=o["warped"], scene_change=o["scene_change"], radius=radius, side_data=side_data, outcome=o)
            if sink is not None:
                sink(out_buffer, info)
        return len(frames)

    def deliver_to(self, y, uv, outs):
        """updateFramePlanes(y, uv), then one step into outs[i] = (y, uv) tensors (at least next_count() of them).  The
        frames are ready for work ordered behind calc.streamHandle(); returns their infos (outcome(info["step"]) gives
        the decision)."""
        c = self.calc
        c.updateFramePlanes(y, uv)
        dst = (L.hrb_frame_planes * max(len(outs), 1))(*[c._planes(a, b) for a, b in outs])
        n = C.c_int()
        self._check(self._lib.hrb_delivery_step_to(self._d, dst, len(outs), self._frames, C.byref(n)))
        return self._infos(n.value)

    def set_settings(self, frame_output=None, scene_change_threshold=None, active=None, auto_adjust=None, target_frame_time=None):
        """UpdateUserSettings (HopperRender.cpp:1355-1390) for the delivery's own settings; clears the delta history."""
        d = L.hrb_delivery_desc.from_buffer_copy(self._desc)
        for k, v in (("frame_output_mode", frame_output), ("scene_change_threshold", scene_change_threshold), ("target_frame_time", target_frame_time)):
            if v is not None:
                setattr(d, k, int(v))
        for k, v in (("active", active), ("auto_adjust", auto_adjust)):
            if v is not None:
                setattr(d, k, 1 if v else 0)
        self._check(self._lib.hrb_delivery_set(self._d, C.byref(d)))
        self._desc = d

    def new_segment(self, rate=1.0):
        """NewSegment (HopperRender.cpp:834-844): seek or playback-speed change."""
        self._check(self._lib.hrb_delivery_new_segment(self._d, float(rate)))

    def close(self):
        if getattr(self, "_d", None) is not None and self._d.value:
            self._lib.hrb_delivery_destroy(self._d)
            self._d = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def kernel_launch_count():
    return int(L.load().hrb_kernel_launch_count())


def microbench_sad_peak(device=0):
    v = C.c_double()
    rc = L.load().hrb_microbench_sad_peak(device, C.byref(v))
    if rc != L.HRB_OK:
        raise RuntimeError(f"hrb error {rc}: {L.last_error()}")
    return v.value
