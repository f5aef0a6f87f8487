// hrb_internal.cuh — shared declarations of the hopperrender_b200 CUDA library (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>
#include <type_traits>
#include <vector>

#include "hrb.h"

namespace hrb {

// ------------------------------------------------------------------------------------------------
// error plumbing (replaces CHECK_ERROR, HopperRender/opticalFlowCalc.h:15-22: no exceptions here,
// the C++ shim in include/opticalFlowCalc.h re-throws)
// ------------------------------------------------------------------------------------------------
void setLastError(const char* fmt, ...);
extern std::atomic<unsigned long long> g_launchCount;  // kernels launched by this process (handles may live on several threads)
extern thread_local unsigned long long t_launchCount;     // ... by this thread: lets a graph capture count its own nodes
constexpr int HRB_MAX_DEVICES = 64;  // per-device launch configuration caches (power of two)

#define HRB_CUDA(call)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (call);                                                                         \
        if (_e != cudaSuccess) {                                                                         \
            ::hrb::setLastError("[hopperrender_b200] CUDA error %d (%s) in %s at %s:%d", (int)_e,        \
                                cudaGetErrorString(_e), __func__, __FILE__, __LINE__);                   \
            return HRB_ERR_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

#define HRB_LAUNCH_CHECK()                                                                               \
    do {                                                                                                 \
        ::hrb::g_launchCount.fetch_add(1, std::memory_order_relaxed);                                     \
        ::hrb::t_launchCount++;                                                                          \
        HRB_CUDA(cudaGetLastError());                                                                    \
    } while (0)

// f(std::integral_constant<int, v>()) for a run-time v in [LO, HI]: picks the template instance of a launcher.  Any other
// v: HRB_ERR_STATE, with a message naming what and v.
template <int LO, int HI, class F> int withConstant(const char* what, int v, const F& f) {
    if (v == LO) return f(std::integral_constant<int, LO>());
    if constexpr (LO < HI) {
        return withConstant<LO + 1, HI>(what, v, f);
    } else {
        setLastError("[hopperrender_b200] %s %d: no such kernel instance", what, v);
        return HRB_ERR_STATE;
    }
}

// Raises Kernel's dynamic shared memory limit on the device to bytes, unless it already allows that much.
template <auto Kernel> int allowDynamicSmem(int device, int bytes) {
    static std::atomic<int> allowed[HRB_MAX_DEVICES];  // per device; handles may be created on several host threads
    std::atomic<int>& cur = allowed[device & (HRB_MAX_DEVICES - 1)];
    if (cur.load(std::memory_order_acquire) >= bytes) return HRB_OK;
    HRB_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    cur.store(bytes, std::memory_order_release);
    return HRB_OK;
}

// ------------------------------------------------------------------------------------------------
// geometry of one search pass (one (iteration, step) of HopperRender/opticalFlowCalcSDR.cpp:72-107)
// ------------------------------------------------------------------------------------------------
struct PassGeom {
    int windowSize;  // ws (power of two >= 2)
    int wsLog2;
    int iteration;
    int step;
    int nWx, nWy;        // windows of this level: ceil(lw/ws), ceil(lh/ws)
    int prevNWx, prevNWy;  // windows of the parent level (ws*2); 0 at iteration 0
};

// Arguments of the search kernels.  Window-level offset arrays replace the per-pixel offsetArray of the
// reference (offsets are constant inside each window, SURVEY.md A.3).
struct SearchArgs {
    // 8-bit search planes (HDR samples >> 8, calcDeltaSumsKernelHDR.h:98-100) of frame N-1 (m_inputFrameArray[1], "1")
    // and frame N (m_inputFrameArray[2], "2"): luma [H][pitch] and the interleaved U,V plane [H/2][pitch] in the
    // NV12 layout; the T planes are the same data transposed, luma [W][pitchT] and chroma [W/2][pitchT] with
    // byte 2*(y>>1)+ch of row x>>1 = channel ch of chroma sample (y>>1, x>>1).  X steps read the T planes.
    const uint8_t *y1, *c1, *y2, *c2;
    const uint8_t *yT1, *cT1, *yT2, *cT2;
    int pitch;               // bytes per row of y / c (multiple of 128)
    int pitchT;              // bytes per row of yT / cT (multiple of 128)
    int W, H;                // frame size
    int lw, lh;              // flow size
    int rs;                  // resolution scalar
    int ws, wsLog2, iteration;
    int deltaScalar, neighborBiasScalar;
    int nWx, nWy, prevNWx;
    // The pass computes (and writes sums, layers, offsets and taps of) only the windows whose flow rows lie in
    // [rowBegin, rowEnd): [0, lh) for a lone handle, a shard's row stripe in the sharded passes of a split search
    // (hrb_split).  Both bounds are multiples of kSplitAlign or lh, so no window straddles them.
    int rowBegin, rowEnd;
    const int16_t* prevX;  // level i-1 offsets (nullptr at iteration 0: all zero)
    const int16_t* prevY;
    int16_t* curX;         // level i offsets: written by step 0, read by step 1
    int16_t* curY;         // level i offsets: written by step 1
    uint32_t* winSums;     // [nW][16] scratch for windows larger than one CTA tile
    unsigned* winTicket;   // [nW] arrival counters of the sliding kernels' fused finalize (zero between passes)
    uint32_t* rawDelta;    // non-null in pass 0: receives sums[R/2-1][window 0]
    uint32_t* tapSums;     // optional [R][nWy][nWx]
    uint8_t* tapLayer;     // optional [nWy][nWx]
    unsigned long long* dbg;  // optional per-CTA timeline of this pass (hrb_ofc_debug_timeline): 16 words per CTA ...
    size_t dbgWords;          // ... in a slice of this many words; CTAs whose record does not fit it record nothing
    bool winLanes;         // small-window kernel: SearchPlan::winLanes, set by its launcher
};

// How one search pass runs.  planSearchPass (kernels_search.cu) is the one place that decides it, from the search variant
// (hrb_ofc_set_search_variant) and the pass; the launchers launch what it says.
struct SearchPlan {
    enum Kernel { Generic, Cand, Tile } kernel;  // sadPassKernel, sadCandKernel, sadTileKernel
    bool useTma;     // tile kernel: the chroma box by TMA (off: variant 2, cp.async only)
    bool forceSlow;  // tile kernel: the per-pixel path for every window (variant 3)
    bool winLanes;   // small-window kernel: one lane per window of 2 and 4 (off: variant 4, the butterfly form)
};
SearchPlan planSearchPass(int variant, const SearchArgs& a, int R, int step);

// Row stripes of a split search start at multiples of this many flow rows: the u-extent of the tile kernel's CTA tile
// (kernels_search_slide.cu).  X steps run on the transposed planes (u = y), so an X-step tile never straddles a stripe,
// and a window of up to kSplitAlign rows lies inside one stripe.
constexpr int kSplitAlign = 128;

// The (u, v) range a pass covers, in the orientation of View (search_common.cuh): u in [u0, lu), v in [v0, lv).  The
// flow rows [rowBegin, rowEnd) lie along v in Y steps (step 1) and along u in X steps (step 0, transposed planes).
struct PassRange {
    int u0, lu, v0, lv;
};
__host__ __device__ inline PassRange passRange(const SearchArgs& a, int step) {
    return step == 1 ? PassRange{0, a.lw, a.rowBegin, a.rowEnd} : PassRange{a.rowBegin, a.rowEnd, 0, a.lw};
}

// The arguments of one generic pass over the members of a flow batch (hrb_flow_batch): member k's are the ones its lone
// pass would get.  Passed by value in kernel parameter space (__grid_constant__), so a pass needs no device table that
// could be overwritten while an earlier batch is still in flight.
struct SearchBatch {
    SearchArgs m[HRB_FLOW_BATCH_MAX];
};
static_assert(sizeof(SearchBatch) <= 32764, "a full flow batch must fit the kernel parameter space of sm_100a (CUDA 12.1 and later)");

// The flow blur of one member of a flow batch: the final level arrays, the blurred flow and its peak
struct BlurMember {
    const int16_t* lvlX;
    const int16_t* lvlY;
    int16_t* out;
    uint32_t* flowMax;
};
struct BlurBatch {
    BlurMember m[HRB_FLOW_BATCH_MAX];
};

// The search representation of one input slot: 8-bit planes in both orientations, one allocation.
struct SearchPlanes {
    uint8_t* base = nullptr;   // the allocation
    uint8_t *y = nullptr, *c = nullptr, *yT = nullptr, *cT = nullptr;
};

struct TmaCache;

struct PassTapDev {
    PassGeom g;
    uint32_t* sums = nullptr;
    uint8_t* layer = nullptr;
    int16_t* offX = nullptr;  // snapshot of the X offsets after the pass
    int16_t* offY = nullptr;
    int wsX = 0, nWxX = 0, nWyX = 0;  // level geometry of the X snapshot
    int wsY = 0, nWxY = 0, nWyY = 0;  // level geometry of the Y snapshot (0 = all zero)
};

struct Profile {
    bool on = false;
    struct Pending {
        cudaEvent_t a, b;
        int cls;
    };
    std::vector<Pending> pending;
    std::vector<cudaEvent_t> pool;
    double ms[5] = {0, 0, 0, 0, 0};
    unsigned long long n[5] = {0, 0, 0, 0, 0};
};
enum { CLS_INGEST = 0, CLS_SEARCH = 1, CLS_BLUR = 2, CLS_WARP = 3, CLS_COPY = 4 };

}  // namespace hrb

// The handle.  Field names mirror HopperRender/opticalFlowCalc.h:26-78 where a counterpart exists.
struct hrb_ofc {
    // video properties
    int frameWidth, frameHeight, inputStride, outputStride;
    float outputBlackLevel, outputWhiteLevel;
    int hdr, bpp;
    // optical flow calculation
    int resScalar, flowWidth, flowHeight, searchRadius;
    double ofcCalcTime, ofcAvgCalcTime, ofcPeakCalcTime;
    int ofcCalcCount;
    double ofcCalcTimeSum, warpCalcTime;
    int deltaScalar, neighborBiasScalar;
    unsigned int totalFrameDelta, frameCount;

    // CUDA
    int device;
    cudaStream_t stream;
    bool ownStream;
    // one record per calculateOpticalFlow in flight: m_ofcStartedEvent / ofcEndEvent of the reference plus the
    // pinned word that receives the raw frame delta; a small ring lets the asynchronous path run ahead of the GPU
    struct FlowRecord {
        cudaEvent_t start, end;
        uint32_t* rawDeltaHost;
        bool startValid, pending;
    };
    static constexpr int kFlowRecords = 4;
    FlowRecord flowRec[kFlowRecords];
    int curRec;
    cudaEvent_t warpStartedEvent, warpEndEvent, uploadDoneEvent;
    bool warpStartedValid;
    // transfers run on their own streams so that the upload of frame N+1 and the downloads of the outputs of frame N
    // overlap the kernels: input slot [3] is the upload target (rotated in by updateFrame), the output is a ring of 3
    cudaStream_t upStream, downStream;
    cudaStream_t flowStream;             // asynchronous flow calculations run here, beside the warps of the same source frame
    cudaEvent_t flowForkEvent, flowJoinEvent;
    bool flowJoinPending, flowOverlap;
    int updatesSinceFlow = 0;      // update_frame calls since the flow in flight was enqueued (see finishUpdate)
    cudaEvent_t spareFreeEvent;          // compute stream: last readers of the buffer that became input slot [3] are enqueued
    static constexpr int kOutRing = 2 * HRB_WARP_BATCH_MAX;  // the batch being written plus the previous one still being downloaded
    cudaEvent_t outReady[kOutRing];      // compute stream: warp/copy into ring slot i finished
    cudaEvent_t outFree[kOutRing];       // download stream: D2H of ring slot i finished
    int outCur;                          // ring slot warpFrames / copyFrame write next (advances on download)
    int outView;                         // ring slot written most recently
    static constexpr int kTickets = 16;
    cudaEvent_t ticketEvent[kTickets];
    unsigned long long downloadSeq;      // downloads enqueued so far (ticket = sequence number, 1-based)

    // device arrays
    size_t inFrameBytes, outFrameBytes;
    uint8_t* inputFrameArray[4];   // raw NV12 / P010 frames, [0..2] rotated like m_inputFrameArray, [3] = upload target
    hrb::SearchPlanes searchPlane[4];  // 8-bit planar search representation of the same slot (row-major + transposed)
    int planePitch;                // bytes per row of the row-major planes
    int planePitchT;               // bytes per row of the transposed planes
    int stripeY0, stripeY1;        // output stripe (luma rows) warpFrames / copyFrame / downloadFrame work on; default the whole frame
    uint8_t* outputRing[kOutRing]; // m_outputFrameArray, as a ring so that downloads overlap the next warps
    int16_t* levelOffsets[2][2];   // [iteration parity][axis] window-level offsets
    size_t levelCapacity;          // entries per level array
    uint32_t* winSums;
    unsigned* winTicket;
    int16_t* offsetArrayScratch;   // [2][lh][lw], materialised on demand for taps
    int16_t* blurredOffsetArray[2];
    uint32_t* flowMaxDev[2];       // max |value| of blurredOffsetArray[i] (rotates with it): lets warpFrames skip the mirror in the interior
    uint32_t* rawDeltaDev;
    // final level geometry after the last calculate (input of blur / offset tap)
    int lastIterParity, lastNWx, lastNWy, lastWs;
    bool haveFlowLevels;

    // taps / profiling
    int searchVariant;  // hrb_ofc_set_search_variant: the search kernels it selects are planned by planSearchPass
    int smCount;
    bool tapMode;
    // instantiated CUDA graphs of the flow calculation (search ladder + blur), one per combination of buffers and
    // parameters it was captured with: the input slots rotate with period 4, so a handful of graphs serve a stream
    struct FlowGraph {
        const void* plane1;
        const void* plane2;
        const void* blurOut;
        int R, deltaScalar, neighborBiasScalar, variant;
        cudaEvent_t pass0;  // pass0Event the graph records (an external event node), or null
        cudaGraphExec_t exec;
        unsigned launches;
    };
    std::vector<FlowGraph> flowGraphs;
    bool flowGraphsOn;
    std::vector<hrb::PassTapDev> taps;
    hrb::Profile prof;
    hrb::TmaCache* tmaCache = nullptr;  // TMA descriptors of the search planes, encoded on first use
    struct TileResidency {
        const void* kernel;
        int nwv, ctasPerSm;
    };
    std::vector<TileResidency> tileResidency;  // CTAs per SM the runtime places, per tile kernel instance and height
    struct SideBlob {
        uint8_t guid[16];
        std::vector<uint8_t> bytes;
    };
    std::vector<SideBlob> sideData;        // IMediaSideData blobs of the newest source frame (opaque, host memory)
    unsigned long long* dbgDev = nullptr;  // per-CTA timelines of the search passes (debug aid, off by default)
    size_t dbgStride = 0;                  // words per pass
    // delivery loop (hrb_delivery): the attached delivery, and the event a flow records right after its pass 0, when
    // rawDeltaDev holds the flow's raw frame delta (null without a delivery)
    hrb_delivery* delivery = nullptr;
    cudaEvent_t pass0Event = nullptr;
    int groups = 0;  // split groups and flow batches the handle belongs to
};

namespace hrb {

// kernels_frame.cu
// Ingest into input slot `slot`: src null packs the slot itself (filled by an upload); otherwise the pack reads the planes
// of src and also writes their samples into the slot.
int launchPackFrame(hrb_ofc* h, int slot, const hrb_frame_planes* src);
// copyFrame / warpFrames into destination planes: ring slots or a caller's surfaces (dst[i] share dst[0]'s pitches).
// gate: null, or a device word; then every CTA returns at once unless *gate == gateWhen (the delivery loop's decision).
// The copy writes the same frame into each of its n destinations (n <= kCopyDstMax).
constexpr int kCopyDstMax = 16;
int launchCopyFrame(hrb_ofc* h, int slot, const hrb_frame_planes* dst, int n = 1, const uint32_t* gate = nullptr, uint32_t gateWhen = 0);
int launchWarpFrames(hrb_ofc* h, int n, const float* t, const hrb_frame_planes* dst, int mode, const uint32_t* gate = nullptr, uint32_t gateWhen = 0);
// kernels_delivery.cu: the delivery loop's scene-change decision (see hrb_api.cu, hrb_delivery)
struct DeliveryRecord {  // mirrors hrb_delivery_outcome
    int warped, sceneChange;
    long long d1, d2;
    unsigned frameDelta;
};
struct DeliveryDecision {
    const uint32_t* rawDelta;  // the flow's raw frame delta (valid when append)
    unsigned divisor;          // lh * lw * (hdr ? 6 : 10)
    uint32_t* ring;            // [16] frame deltas: history entry k sits at ring[(seq of k) % 16]
    int append;                // the step computed a flow: ring[slot] = rawDelta / divisor
    int slot;                  // ring index of the newest history entry (nxt)
    int n;                     // history entries after the append
    int count;                 // min(n - 2, 10): the entries averaged
    long long threshold;
    int copy;                  // the host knows the outputs are copies (inactive, frame_count < 3)
    uint32_t* gate;            // receives sceneChange (read by the gated warps and copy)
    DeliveryRecord* out;
};
int launchDeliveryDecision(hrb_ofc* h, const DeliveryDecision& d);
// kernels_search.cu
int launchSearchPass(hrb_ofc* h, const SearchArgs& a, int R, int step);
// One pass of the n members of a flow batch, on h[0]->stream: a generic pass is one launch over all of them, a tile or
// small-window pass one launch per member.
int launchSearchBatch(hrb_ofc* const* h, const SearchBatch& b, int n, int R, int step);
// The tile and small-window kernels exist for radii 5..16.  Each family is compiled as kSearchParts objects of four
// consecutive radii (-DHRB_SEARCH_PART, Makefile), so that they build in parallel; radius R lives in part searchPart(R).
constexpr int kSearchParts = 3;
constexpr int searchPart(int R) { return (R - 5) / 4; }
constexpr int firstRadiusOf(int part) { return 5 + 4 * part; }
// A pass the plan sends to the tile kernel (kernels_search_slide.cu) / small-window kernel (kernels_search_cand.cu),
// whose radius lies in PART.
template <int PART> int launchTilePart(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p, int R, int step);
template <int PART> int launchCandPart(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p, int R, int step);
void freeTmaCache(hrb_ofc* h);  // tensor maps of the handle's search planes (kernels_search_slide.cu)
int launchBlurFlow(hrb_ofc* h, const int16_t* lvlX, const int16_t* lvlY, int nWx, int wsLog2, int16_t* out, uint32_t* flowMax);
// the blur of the n members of a flow batch in one launch on h[0]->stream (zeroes each member's flowMax first)
int launchBlurFlowBatch(hrb_ofc* const* h, const BlurBatch& b, int n, int nWx, int wsLog2);
int launchExpandOffsets(hrb_ofc* h, const int16_t* lvlX, int nWxX, int wsLog2X, const int16_t* lvlY, int nWxY, int wsLog2Y,
                        int16_t* out);
int microbenchSad(int device, double* gigaAbsdiffPerSec);

// profiling helpers (hrb_api.cu)
void profBegin(hrb_ofc* h, int cls);
void profEnd(hrb_ofc* h, int cls, unsigned launches);

}  // namespace hrb
