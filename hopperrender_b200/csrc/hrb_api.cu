// hrb_api.cu — handle management, the per-frame host schedule and the C ABI (include/hrb.h).
// The schedule restates HopperRender/opticalFlowCalcSDR.cpp / opticalFlowCalcHDR.cpp on one CUDA stream.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <deque>
#include <mutex>
#include <new>

#include <cuda.h>

#include "hrb_internal.cuh"

namespace hrb {

static thread_local std::string t_lastError;
std::atomic<unsigned long long> g_launchCount{0};
thread_local unsigned long long t_launchCount = 0;

void setLastError(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_lastError = buf;
    // the reference also reports on stderr (opticalFlowCalc.h:19-20)
    fputs(buf, stderr);
    fputc('\n', stderr);
}

// ---- profiling -----------------------------------------------------------------------------------
static cudaEvent_t profEvent(hrb_ofc* h) {
    if (!h->prof.pool.empty()) {
        cudaEvent_t e = h->prof.pool.back();
        h->prof.pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

void profBegin(hrb_ofc* h, int cls) {
    if (!h->prof.on) return;
    Profile::Pending p;
    p.a = profEvent(h);
    p.b = nullptr;
    p.cls = cls;
    cudaEventRecord(p.a, h->stream);
    h->prof.pending.push_back(p);
}

void profEnd(hrb_ofc* h, int cls, unsigned launches) {
    h->prof.n[cls] += launches;
    if (!h->prof.on || h->prof.pending.empty()) return;
    Profile::Pending& p = h->prof.pending.back();
    p.b = profEvent(h);
    cudaEventRecord(p.b, h->stream);
}

static int profResolve(hrb_ofc* h) {
    if (h->prof.pending.empty()) return HRB_OK;
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    for (auto& p : h->prof.pending) {
        if (p.a && p.b) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) h->prof.ms[p.cls] += ms;
        }
        if (p.a) h->prof.pool.push_back(p.a);
        if (p.b) h->prof.pool.push_back(p.b);
    }
    h->prof.pending.clear();
    return HRB_OK;
}

// ---- taps ----------------------------------------------------------------------------------------
static void freeTaps(hrb_ofc* h) {
    for (auto& t : h->taps) {
        cudaFree(t.sums);
        cudaFree(t.layer);
        cudaFree(t.offX);
        cudaFree(t.offY);
    }
    h->taps.clear();
}

static int ilog2(int v) {
    int l = 0;
    while ((1 << (l + 1)) <= v) ++l;
    return l;
}

// First window size and iteration count — opticalFlowCalcSDR.cpp:49-65 (NUM_ITERATIONS == 0)
static void ladder(int lw, int lh, int* ws0, int* iterations) {
    int windowSize = 1;
    int maxDim = lw > lh ? lw : lh;
    if (maxDim && !(maxDim & (maxDim - 1))) {
        windowSize = maxDim;
    } else {
        while (maxDim & (maxDim - 1)) maxDim &= (maxDim - 1);
        windowSize = maxDim << 1;
    }
    windowSize /= 2;
    *ws0 = windowSize;
    *iterations = ilog2(windowSize);
}

// The stats block at the end of calculateOpticalFlow — opticalFlowCalcSDR.cpp:119-138
static int resolveRecord(hrb_ofc* h, hrb_ofc::FlowRecord& r) {
    if (!r.pending) return HRB_OK;
    HRB_CUDA(cudaEventSynchronize(r.end));
    r.pending = false;
    // m_totalFrameDelta — opticalFlowCalcSDR.cpp:92-93 (divisor 10) / opticalFlowCalcHDR.cpp:92-93 (divisor 6)
    h->totalFrameDelta = *r.rawDeltaHost;
    h->totalFrameDelta /= (unsigned)(h->flowHeight * h->flowWidth * (h->hdr ? 6 : 10));
    float ms = 0;
    HRB_CUDA(cudaEventElapsedTime(&ms, r.start, r.end));
    h->ofcCalcTime = (double)ms / 1e3;
    if (h->ofcCalcCount >= 240) {  // CALC_TIME_INTERVAL, config.h:17
        h->ofcAvgCalcTime = h->ofcCalcTimeSum / h->ofcCalcCount;
        h->ofcCalcCount = 0;
        h->ofcCalcTimeSum = 0.0;
        h->ofcPeakCalcTime = h->ofcCalcTime;
    }
    h->ofcCalcCount++;
    h->ofcCalcTimeSum += h->ofcCalcTime;
    if (h->ofcCalcTime > h->ofcPeakCalcTime) h->ofcPeakCalcTime = h->ofcCalcTime;
    return HRB_OK;
}

// resolve every flow in flight, oldest first
static int resolveFlow(hrb_ofc* h) {
    for (int i = 1; i <= hrb_ofc::kFlowRecords; ++i) {
        const int rc = resolveRecord(h, h->flowRec[(h->curRec + i) % hrb_ofc::kFlowRecords]);
        if (rc) return rc;
    }
    return HRB_OK;
}

// The arguments of pass (iter, step) of one handle, which computes the windows of flow rows [rowBegin, rowEnd), and the
// pass's tap buffers when tap mode is on.
static int beginPass(hrb_ofc* h, int R, int ws, int iter, int step, int prevNWx, int prevNWy, int rowBegin, int rowEnd, SearchArgs& a) {
    const int par = iter & 1;
    memset(&a, 0, sizeof(a));
    const SearchPlanes& f1 = h->searchPlane[1];  // frame1 = m_inputFrameArray[1], opticalFlowCalcSDR.cpp:79
    const SearchPlanes& f2 = h->searchPlane[2];  // frame2 = m_inputFrameArray[2], opticalFlowCalcSDR.cpp:80
    a.y1 = f1.y; a.c1 = f1.c; a.yT1 = f1.yT; a.cT1 = f1.cT;
    a.y2 = f2.y; a.c2 = f2.c; a.yT2 = f2.yT; a.cT2 = f2.cT;
    a.pitch = h->planePitch;
    a.pitchT = h->planePitchT;
    a.W = h->frameWidth;
    a.H = h->frameHeight;
    a.lw = h->flowWidth;
    a.lh = h->flowHeight;
    a.rs = h->resScalar;
    a.deltaScalar = h->deltaScalar;
    a.neighborBiasScalar = h->neighborBiasScalar;
    a.winSums = h->winSums;
    a.winTicket = h->winTicket;
    a.ws = ws;
    a.wsLog2 = ilog2(ws);
    a.iteration = iter;
    a.nWx = (a.lw + ws - 1) / ws;
    a.nWy = (a.lh + ws - 1) / ws;
    a.rowBegin = rowBegin;
    a.rowEnd = rowEnd;
    a.prevNWx = prevNWx;
    a.prevX = iter ? h->levelOffsets[par ^ 1][0] : nullptr;
    a.prevY = iter ? h->levelOffsets[par ^ 1][1] : nullptr;
    a.curX = h->levelOffsets[par][0];
    a.curY = h->levelOffsets[par][1];
    a.rawDelta = (iter == 0 && step == 0) ? h->rawDeltaDev : nullptr;
    const bool dbgPass = h->dbgDev && iter * 2 + step < 32;
    a.dbg = dbgPass ? h->dbgDev + (size_t)(iter * 2 + step) * h->dbgStride : nullptr;
    a.dbgWords = dbgPass ? h->dbgStride : 0;
    if (h->tapMode) {
        PassTapDev t;
        t.g.windowSize = ws;
        t.g.wsLog2 = a.wsLog2;
        t.g.iteration = iter;
        t.g.step = step;
        t.g.nWx = a.nWx;
        t.g.nWy = a.nWy;
        t.g.prevNWx = prevNWx;
        t.g.prevNWy = prevNWy;
        const size_t nW = (size_t)a.nWx * a.nWy;
        HRB_CUDA(cudaMalloc(&t.sums, nW * R * sizeof(uint32_t)));
        HRB_CUDA(cudaMalloc(&t.layer, nW));
        HRB_CUDA(cudaMalloc(&t.offX, nW * sizeof(int16_t)));
        HRB_CUDA(cudaMalloc(&t.offY, nW * sizeof(int16_t)));
        // zeroed, so that the windows a sharded pass does not compute read back as zero
        HRB_CUDA(cudaMemsetAsync(t.sums, 0, nW * R * sizeof(uint32_t), h->stream));
        HRB_CUDA(cudaMemsetAsync(t.layer, 0, nW, h->stream));
        a.tapSums = t.sums;
        a.tapLayer = t.layer;
        h->taps.push_back(t);
    }
    return HRB_OK;
}

// After the pass: the tap snapshots of the offsets, and the geometry of the handle's newest level.
static int endPass(hrb_ofc* h, const SearchArgs& a, int step, int prevNWx, int prevNWy) {
    if (h->tapMode) {
        PassTapDev& t = h->taps.back();
        const size_t nW = (size_t)a.nWx * a.nWy;
        HRB_CUDA(cudaMemcpyAsync(t.offX, a.curX, nW * sizeof(int16_t), cudaMemcpyDeviceToDevice, h->stream));
        t.wsX = a.ws;
        t.nWxX = a.nWx;
        t.nWyX = a.nWy;
        if (step == 1) {
            HRB_CUDA(cudaMemcpyAsync(t.offY, a.curY, nW * sizeof(int16_t), cudaMemcpyDeviceToDevice, h->stream));
            t.wsY = a.ws;
            t.nWxY = a.nWx;
            t.nWyY = a.nWy;
        } else if (a.iteration > 0) {
            HRB_CUDA(cudaMemcpyAsync(t.offY, a.prevY, (size_t)prevNWx * prevNWy * sizeof(int16_t), cudaMemcpyDeviceToDevice, h->stream));
            t.wsY = a.ws * 2;
            t.nWxY = prevNWx;
            t.nWyY = prevNWy;
        } else {
            t.wsY = 0;  // all zero
        }
    }
    h->lastIterParity = a.iteration & 1;
    h->lastNWx = a.nWx;
    h->lastNWy = a.nWy;
    h->lastWs = a.ws;
    return HRB_OK;
}

// After pass 0 of a handle with a delivery: rawDeltaDev holds the flow's raw frame delta.  Inside a graph capture the record
// becomes an external event-record node, so that the delivery's decision kernel, on the compute stream, waits for pass 0
// of the launched graph and not for the whole ladder.
static int recordPass0(hrb_ofc* h) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    HRB_CUDA(cudaStreamIsCapturing(h->stream, &st));
    if (st == cudaStreamCaptureStatusActive)
        HRB_CUDA(cudaEventRecordWithFlags(h->pass0Event, h->stream, cudaEventRecordExternal));
    else
        HRB_CUDA(cudaEventRecord(h->pass0Event, h->stream));
    return HRB_OK;
}

// One iteration (two passes) of the ladder on one handle; the passes compute the windows of flow rows [rowBegin, rowEnd).
static int issueIteration(hrb_ofc* h, int R, int ws, int iter, int prevNWx, int prevNWy, int rowBegin, int rowEnd, bool issue) {
    for (int step = 0; step < 2; ++step) {
        SearchArgs a;
        int rc = beginPass(h, R, ws, iter, step, prevNWx, prevNWy, rowBegin, rowEnd, a);
        if (!rc && issue) rc = launchSearchPass(h, a, R, step);
        if (!rc && issue && a.rawDelta && h->pass0Event) rc = recordPass0(h);
        if (!rc) rc = endPass(h, a, step, prevNWx, prevNWy);
        if (rc) return rc;
    }
    return HRB_OK;
}

}  // namespace hrb

// A group of handles that compute one flow together (include/hrb.h, split search).  It owns no device memory: the level
// arrays exchanged are the handles' own.
struct hrb_split {
    std::vector<hrb_ofc*> shard;
    std::vector<int> bounds;          // shard k owns the flow rows [bounds[k], bounds[k + 1])
    std::vector<cudaEvent_t> done;    // per shard, created on its device: its part of an iteration / its pushes are enqueued
};

// The members of a flow batch (include/hrb.h): independent handles on one device whose passes are launched together.  It
// owns no frame or flow memory, only the stream the ladder runs on, an event that marks the end of a batch on it, and
// the launch arguments (kernel parameters, copied at each launch).
struct hrb_flow_batch {
    std::vector<hrb_ofc*> member;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    hrb::SearchBatch pass;
    hrb::BlurBatch blur;
};

namespace hrb {

constexpr int kMaxShards = 64;

// The handles one ladder runs on: a lone handle (one shard that owns every flow row), the shards of a group, or the
// members of a flow batch (each computes its own flow over every row; their passes are launched together).
struct Shards {
    hrb_ofc* const* h;
    const int* bounds;   // n + 1 flow-row bounds (split group and lone handle)
    int n;
    cudaEvent_t* done;   // split group only
    hrb_flow_batch* batch;  // flow batch only: every h[k]->stream is its stream while the ladder is enqueued
    explicit Shards(hrb_ofc* lone) : h(&one), bounds(rows), n(1), done(nullptr), batch(nullptr), one(lone), rows{0, lone->flowHeight} {}
    explicit Shards(hrb_split* s)
        : h(s->shard.data()), bounds(s->bounds.data()), n((int)s->shard.size()), done(s->done.data()), batch(nullptr), one(nullptr), rows{0, 0} {}
    explicit Shards(hrb_flow_batch* b) : h(b->member.data()), bounds(nullptr), n((int)b->member.size()), done(nullptr), batch(b), one(nullptr), rows{0, 0} {}
    Shards(const Shards&) = delete;
    Shards& operator=(const Shards&) = delete;

   private:
    hrb_ofc* one;
    int rows[2];
};

// `bytes` from device memory of shard `from` to device memory of shard `to`, on `st`
static int copyShard(const hrb_ofc* to, void* dst, const hrb_ofc* from, const void* src, size_t bytes, cudaStream_t st) {
    if (to->device == from->device)
        HRB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st));
    else
        HRB_CUDA(cudaMemcpyPeerAsync(dst, to->device, src, from->device, bytes, st));
    return HRB_OK;
}

// Between two sharded iterations: the neighbour bias of a window of the next level reads parent windows w/2 +- 1
// (SURVEY.md A.1), so every shard pulls the parent-level window row just above and just below its stripe, both axes,
// from the shards that own them.  Each shard waits for its neighbours' part of the iteration first.  The neighbour
// overwrites these rows two iterations later, after it has waited for this shard's next iteration, which follows the
// copies on this shard's stream.
static int exchangeHalo(const Shards& s, int par, int ws, int nWx, int nWy) {
    for (int k = 0; k < s.n; ++k) {
        HRB_CUDA(cudaSetDevice(s.h[k]->device));
        HRB_CUDA(cudaEventRecord(s.done[k], s.h[k]->stream));
    }
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        HRB_CUDA(cudaSetDevice(h->device));
        const int nb[2] = {k - 1, k + 1};
        const int row[2] = {s.bounds[k] / ws - 1, s.bounds[k + 1] / ws};  // bounds are multiples of ws (or lh, which has no shard below)
        for (int i = 0; i < 2; ++i) {
            if (nb[i] < 0 || nb[i] >= s.n || row[i] < 0 || row[i] >= nWy) continue;
            const hrb_ofc* from = s.h[nb[i]];
            HRB_CUDA(cudaStreamWaitEvent(h->stream, s.done[nb[i]], 0));
            for (int ax = 0; ax < 2; ++ax) {
                const size_t off = (size_t)row[i] * nWx;
                const int rc = copyShard(h, h->levelOffsets[par][ax] + off, from, from->levelOffsets[par][ax] + off, (size_t)nWx * sizeof(int16_t), h->stream);
                if (rc) return rc;
            }
        }
    }
    return HRB_OK;
}

// After the last iteration: every shard pushes the window rows it owns of the final level (and shard 0 the raw frame
// delta, when pass 0 was sharded) to every other shard, then each waits for all pushes into it.
// The pushes start only once EVERY shard has finished its last iteration (an all-to-all barrier, not the neighbour
// ordering of exchangeHalo): the receiver's array of the final level's parity is also the array of levels L-2, L-4, ...,
// which it read and wrote in earlier iterations at a coarser geometry whose offsets overlap the pushed rows, and a
// shard n - 1 hops away is ordered behind the receiver's iteration L - (n - 1) only.  The tap copies of the last
// iteration are enqueued before the barrier too, so they never see a push.
static int gatherLevel(const Shards& s, int par, int ws, int nWx, int nWy, bool rawDelta) {
    for (int k = 0; k < s.n; ++k) {
        HRB_CUDA(cudaSetDevice(s.h[k]->device));
        HRB_CUDA(cudaEventRecord(s.done[k], s.h[k]->stream));
    }
    for (int j = 0; j < s.n; ++j) {
        hrb_ofc* from = s.h[j];
        HRB_CUDA(cudaSetDevice(from->device));
        for (int k = 0; k < s.n; ++k)
            if (k != j) HRB_CUDA(cudaStreamWaitEvent(from->stream, s.done[k], 0));  // (the wait takes the record above)
    }
    for (int j = 0; j < s.n; ++j) {
        hrb_ofc* from = s.h[j];
        HRB_CUDA(cudaSetDevice(from->device));
        const int r0 = s.bounds[j] / ws, r1 = std::min((s.bounds[j + 1] + ws - 1) / ws, nWy);
        for (int k = 0; k < s.n; ++k) {
            if (k == j) continue;
            hrb_ofc* to = s.h[k];
            for (int ax = 0; ax < 2; ++ax) {
                const size_t off = (size_t)r0 * nWx;
                const int rc = copyShard(to, to->levelOffsets[par][ax] + off, from, from->levelOffsets[par][ax] + off, (size_t)(r1 - r0) * nWx * sizeof(int16_t),
                                         from->stream);
                if (rc) return rc;
            }
            if (rawDelta && j == 0) {
                const int rc = copyShard(to, to->rawDeltaDev, from, from->rawDeltaDev, sizeof(uint32_t), from->stream);
                if (rc) return rc;
            }
        }
        HRB_CUDA(cudaEventRecord(s.done[j], from->stream));
    }
    for (int k = 0; k < s.n; ++k) {
        HRB_CUDA(cudaSetDevice(s.h[k]->device));
        for (int j = 0; j < s.n; ++j)
            if (j != k) HRB_CUDA(cudaStreamWaitEvent(s.h[k]->stream, s.done[j], 0));
    }
    return HRB_OK;
}

// One iteration of the ladder on every member of a flow batch: per step, the members' arguments, then one batched pass.
static int issueBatchIteration(const Shards& s, int R, int ws, int iter, int prevNWx, int prevNWy) {
    SearchBatch& b = s.batch->pass;
    for (int step = 0; step < 2; ++step) {
        for (int k = 0; k < s.n; ++k) {
            const int rc = beginPass(s.h[k], R, ws, iter, step, prevNWx, prevNWy, 0, s.h[k]->flowHeight, b.m[k]);
            if (rc) return rc;
        }
        int rc = launchSearchBatch(s.h, b, s.n, R, step);
        for (int k = 0; k < s.n && !rc; ++k) rc = endPass(s.h[k], b.m[k], step, prevNWx, prevNWy);
        if (rc) return rc;
    }
    return HRB_OK;
}

// The search ladder and the blur of one flow calculation, on a lone handle, on the shards of a group or on the members
// of a flow batch.  Passes with
// windows of at most kSplitAlign rows are sharded on a group: shard k computes only the windows of its rows, with
// exchangeHalo between iterations and gatherLevel after the last one.  Passes with taller windows straddle stripes and
// run replicated, on the whole frame, on every shard.  issue = false only replays the host-side bookkeeping (the
// kernels are then launched from a captured graph; lone handles only).
static int issueFlowKernels(const Shards& s, int R, int ws0, int iterations, bool issue) {
    const int lw = s.h[0]->flowWidth, lh = s.h[0]->flowHeight;
    int prevNWx = 0, prevNWy = 0;
    bool prevSharded = false;
    for (int iter = 0; iter < iterations; ++iter) {
        const int ws = ws0 >> iter;
        const int par = iter & 1;
        const bool sharded = !s.batch && s.n > 1 && ws <= kSplitAlign;
        if (sharded && prevSharded) {  // the first sharded iteration reads a parent level every shard computed in full
            const int rc = exchangeHalo(s, par ^ 1, ws * 2, prevNWx, prevNWy);
            if (rc) return rc;
        }
        if (s.batch) {
            const int rc = issueBatchIteration(s, R, ws, iter, prevNWx, prevNWy);
            if (rc) return rc;
        }
        for (int k = 0; k < s.n && !s.batch; ++k) {
            hrb_ofc* h = s.h[k];
            if (s.n > 1) HRB_CUDA(cudaSetDevice(h->device));
            const int rc = issueIteration(h, R, ws, iter, prevNWx, prevNWy, sharded ? s.bounds[k] : 0, sharded ? s.bounds[k + 1] : lh, issue);
            if (rc) return rc;
        }
        prevNWx = (lw + ws - 1) / ws;
        prevNWy = (lh + ws - 1) / ws;
        prevSharded = sharded;
    }
    if (prevSharded) {
        const int rc = gatherLevel(s, (iterations - 1) & 1, ws0 >> (iterations - 1), prevNWx, prevNWy, ws0 <= kSplitAlign);
        if (rc) return rc;
    }

    // blur into m_blurredOffsetArray[0], then swap (opticalFlowCalcSDR.cpp:113-123)
    if (s.batch) {
        BlurBatch& b = s.batch->blur;
        for (int k = 0; k < s.n; ++k) {
            hrb_ofc* h = s.h[k];
            h->haveFlowLevels = true;
            b.m[k] = BlurMember{h->levelOffsets[h->lastIterParity][0], h->levelOffsets[h->lastIterParity][1], h->blurredOffsetArray[0], h->flowMaxDev[0]};
        }
        return launchBlurFlowBatch(s.h, b, s.n, s.h[0]->lastNWx, ilog2(s.h[0]->lastWs));
    }
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        h->haveFlowLevels = true;
        if (issue) {
            if (s.n > 1) HRB_CUDA(cudaSetDevice(h->device));
            const int rc = launchBlurFlow(h, h->levelOffsets[h->lastIterParity][0], h->levelOffsets[h->lastIterParity][1], h->lastNWx, ilog2(h->lastWs),
                                          h->blurredOffsetArray[0], h->flowMaxDev[0]);
            if (rc) return rc;
        }
    }
    return HRB_OK;
}

static void dropFlowGraphs(hrb_ofc* h) {
    for (auto& g : h->flowGraphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    h->flowGraphs.clear();
}

// Launches the flow kernels through a CUDA graph captured on first use for this combination of buffers and parameters
// (24 dependent launches at 4K become one); falls back to plain launches whenever capture is not possible.
static int launchFlowKernels(hrb_ofc* h, int R, int ws0, int iterations) {
    if (!h->flowGraphsOn || h->tapMode || h->prof.on || h->dbgDev) return issueFlowKernels(Shards(h), R, ws0, iterations, true);
    hrb_ofc::FlowGraph key;
    key.plane1 = h->searchPlane[1].base;
    key.plane2 = h->searchPlane[2].base;
    key.blurOut = h->blurredOffsetArray[0];
    key.R = R;
    key.deltaScalar = h->deltaScalar;
    key.neighborBiasScalar = h->neighborBiasScalar;
    key.variant = h->searchVariant;
    key.pass0 = h->pass0Event;
    hrb_ofc::FlowGraph* hit = nullptr;
    for (auto& g : h->flowGraphs)
        if (g.plane1 == key.plane1 && g.plane2 == key.plane2 && g.blurOut == key.blurOut && g.R == key.R && g.deltaScalar == key.deltaScalar &&
            g.neighborBiasScalar == key.neighborBiasScalar && g.variant == key.variant && g.pass0 == key.pass0)
            hit = &g;
    if (!hit) {
        if (h->flowGraphs.size() >= 64) dropFlowGraphs(h);  // 12 radii x 4 slot rotations fit; beyond that parameters keep changing (UI): start over
        const unsigned long long before = t_launchCount;
        if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            h->flowGraphsOn = false;  // e.g. the caller's stream is the legacy default stream
            return issueFlowKernels(Shards(h), R, ws0, iterations, true);
        }
        const int rc = issueFlowKernels(Shards(h), R, ws0, iterations, true);
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
        key.launches = (unsigned)(t_launchCount - before);
        g_launchCount.fetch_sub(key.launches, std::memory_order_relaxed);  // captured, not run yet
        key.exec = nullptr;
        if (rc == HRB_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&key.exec, graph, 0) == cudaSuccess) {
            cudaGraphDestroy(graph);
            h->flowGraphs.push_back(key);
            hit = &h->flowGraphs.back();
        } else {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            h->flowGraphsOn = false;
            if (rc) return rc;
            return issueFlowKernels(Shards(h), R, ws0, iterations, true);
        }
    } else {
        const int rc = issueFlowKernels(Shards(h), R, ws0, iterations, false);
        if (rc) return rc;
    }
    HRB_CUDA(cudaGraphLaunch(hit->exec, h->stream));
    g_launchCount.fetch_add(hit->launches, std::memory_order_relaxed);
    return HRB_OK;
}

// One flow calculation on every shard's current stream (a lone handle is the group of one): the ladder, the blur, the
// raw-delta copy, the flow record and the buffer swap of each handle.
static int enqueueFlow(const Shards& s) {
    hrb_ofc* const h0 = s.h[0];
    const int R = h0->searchRadius;  // m_lowGrid8x8xL[2] = m_opticalFlowSearchRadius, opticalFlowCalcSDR.cpp:46 (equal on every shard)
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        HRB_CUDA(cudaSetDevice(h->device));
        if (h->flowRec[h->curRec].pending) {  // a second calculate on the same upload: its end event is about to be re-recorded
            const int rc = resolveFlow(h);
            if (rc) return rc;
        }
        if (h->searchRadius < 2 || h->searchRadius > 16) {
            setLastError("[hopperrender_b200] search radius %d outside 2..16", h->searchRadius);
            return HRB_ERR_INVALID_ARG;
        }
        if (h->deltaScalar < 0 || h->deltaScalar > 31 || h->neighborBiasScalar < 0 || h->neighborBiasScalar > 31) {
            setLastError("[hopperrender_b200] delta/neighbor scalar outside 0..31");
            return HRB_ERR_INVALID_ARG;
        }
    }
    int ws0, iterations;
    ladder(h0->flowWidth, h0->flowHeight, &ws0, &iterations);
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        hrb_ofc::FlowRecord& rec = h->flowRec[h->curRec];
        if (s.n > 1) HRB_CUDA(cudaSetDevice(h->device));
        if (!rec.startValid) {  // calculate without a preceding updateFrame: time from here
            HRB_CUDA(cudaEventRecord(rec.start, h->stream));
            rec.startValid = true;
        }
        if (h->tapMode) freeTaps(h);
    }

    {
        // a group or a batch runs plain launches: a group's ladder has cross-shard waits and copies between iterations
        const int rc = s.n == 1 && !s.batch ? launchFlowKernels(h0, R, ws0, iterations) : issueFlowKernels(s, R, ws0, iterations, true);
        if (rc) return rc;
    }
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        hrb_ofc::FlowRecord& rec = h->flowRec[h->curRec];
        if (s.n > 1) HRB_CUDA(cudaSetDevice(h->device));
        HRB_CUDA(cudaMemcpyAsync(rec.rawDeltaHost, h->rawDeltaDev, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        HRB_CUDA(cudaEventRecord(rec.end, h->stream));
        int16_t* t0 = h->blurredOffsetArray[0];
        h->blurredOffsetArray[0] = h->blurredOffsetArray[1];
        h->blurredOffsetArray[1] = t0;
        uint32_t* m0 = h->flowMaxDev[0];
        h->flowMaxDev[0] = h->flowMaxDev[1];
        h->flowMaxDev[1] = m0;
        rec.pending = true;
    }
    return HRB_OK;
}

// src: the caller's planes the ingest reads and copies into the new slot; null after an upload into slot [3]
static int finishUpdate(hrb_ofc* h, const hrb_frame_planes* src) {
    // the new frame sits in slot [3]; rotate [0] <- [1] <- [2] <- [3], the old [0] becomes the next upload target
    // (same result as the reference's write-into-[0]-then-rotate, opticalFlowCalcSDR.cpp:20-26)
    auto rot = [](auto** v) {
        auto* f0 = v[0];
        v[0] = v[1];
        v[1] = v[2];
        v[2] = v[3];
        v[3] = f0;
    };
    rot(h->inputFrameArray);
    {
        const SearchPlanes s0 = h->searchPlane[0];
        h->searchPlane[0] = h->searchPlane[1];
        h->searchPlane[1] = h->searchPlane[2];
        h->searchPlane[2] = h->searchPlane[3];
        h->searchPlane[3] = s0;
    }
    h->frameCount++;
    // every reader of the buffer that just became slot [3] (the warps of the previous source frame) is already enqueued
    HRB_CUDA(cudaEventRecord(h->spareFreeEvent, h->stream));
    // an asynchronous flow still in flight reads the search planes of slots [1] and [2] as they were when it was
    // enqueued; the third update after it writes one of them and is ordered behind it.  The first two do not touch
    // them, so in the usual update / calculate alternation the ingest of frame N+1 runs beside the search of frame N.
    if (h->flowJoinPending && ++h->updatesSinceFlow >= 3) HRB_CUDA(cudaStreamWaitEvent(h->stream, h->flowJoinEvent, 0));
    return launchPackFrame(h, 2, src);
}

// `onStream`: the stream the frame copy will be enqueued on; the flow timer starts there (m_ofcStartedEvent is the
// upload event in the reference, opticalFlowCalcSDR.cpp:20)
static int beginUpdate(hrb_ofc* h, cudaStream_t onStream) {
    HRB_CUDA(cudaSetDevice(h->device));
    h->curRec = (h->curRec + 1) % hrb_ofc::kFlowRecords;
    hrb_ofc::FlowRecord& rec = h->flowRec[h->curRec];
    if (rec.pending) {  // the ring is full: wait for the oldest flow before reusing its events
        const int rc = resolveRecord(h, rec);
        if (rc) return rc;
    }
    if (onStream != h->stream) HRB_CUDA(cudaStreamWaitEvent(onStream, h->spareFreeEvent, 0));
    HRB_CUDA(cudaEventRecord(rec.start, onStream));
    rec.startValid = true;
    return HRB_OK;
}

static int uploadFrame(hrb_ofc* h, const uint8_t* input_planes, bool wait) {
    int rc = beginUpdate(h, h->upStream);
    if (rc) return rc;
    // write into the upload slot on the upload stream (opticalFlowCalcSDR.cpp:20), then hand it to the compute stream
    HRB_CUDA(cudaMemcpyAsync(h->inputFrameArray[3], input_planes, h->inFrameBytes, cudaMemcpyHostToDevice, h->upStream));
    HRB_CUDA(cudaEventRecord(h->uploadDoneEvent, h->upStream));
    HRB_CUDA(cudaStreamWaitEvent(h->stream, h->uploadDoneEvent, 0));
    rc = finishUpdate(h, nullptr);
    if (rc) return rc;
    if (wait) HRB_CUDA(cudaEventSynchronize(h->uploadDoneEvent));  // the caller's buffer is free again; everything else continues asynchronously
    return HRB_OK;
}

static int enqueueDownload(hrb_ofc* h, uint8_t* dst, unsigned long long* ticket) {
    HRB_CUDA(cudaSetDevice(h->device));
    const int slot = h->outCur;
    HRB_CUDA(cudaStreamWaitEvent(h->downStream, h->outReady[slot], 0));
    if (h->stripeY0 == 0 && h->stripeY1 == h->frameHeight) {
        HRB_CUDA(cudaMemcpyAsync(dst, h->outputRing[slot], h->outFrameBytes, cudaMemcpyDeviceToHost, h->downStream));
    } else {
        // only the stripe's luma rows and their chroma rows travel, to the same offsets of the caller's full-frame buffer
        const size_t rowBytes = (size_t)h->outputStride * h->bpp;
        const size_t lumaOff = (size_t)h->stripeY0 * rowBytes, lumaLen = (size_t)(h->stripeY1 - h->stripeY0) * rowBytes;
        const size_t chromaOff = ((size_t)h->frameHeight + (h->stripeY0 >> 1)) * rowBytes, chromaLen = lumaLen / 2;
        HRB_CUDA(cudaMemcpyAsync(dst + lumaOff, h->outputRing[slot] + lumaOff, lumaLen, cudaMemcpyDeviceToHost, h->downStream));
        HRB_CUDA(cudaMemcpyAsync(dst + chromaOff, h->outputRing[slot] + chromaOff, chromaLen, cudaMemcpyDeviceToHost, h->downStream));
    }
    HRB_CUDA(cudaEventRecord(h->outFree[slot], h->downStream));
    const unsigned long long seq = ++h->downloadSeq;
    HRB_CUDA(cudaEventRecord(h->ticketEvent[seq % hrb_ofc::kTickets], h->downStream));
    if (ticket) *ticket = seq;
    h->outCur = (slot + 1) % hrb_ofc::kOutRing;
    return HRB_OK;
}

// warpFrames / copyFrame are about to overwrite ring slot outCur: its previous download must have finished
static int beginOutput(hrb_ofc* h) {
    HRB_CUDA(cudaSetDevice(h->device));
    HRB_CUDA(cudaStreamWaitEvent(h->stream, h->outFree[h->outCur], 0));
    HRB_CUDA(cudaEventRecord(h->warpStartedEvent, h->stream));  // m_warpStartedEvent, opticalFlowCalcSDR.cpp:164
    h->warpStartedValid = true;
    h->outView = h->outCur;
    return HRB_OK;
}

// Ring slot `slot` as two planes: luma rows, then the chroma rows (both pitches output_stride)
static hrb_frame_planes ringPlanes(hrb_ofc* h, int slot) {
    const size_t pitch = (size_t)h->outputStride * h->bpp;
    uint8_t* base = h->outputRing[slot];
    return hrb_frame_planes{base, pitch, base + (size_t)h->frameHeight * pitch, pitch};
}

// ---- checks of caller planes (hrb_frame_planes) ----
typedef CUresult (*MemGetAddressRangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);

static MemGetAddressRangeFn memGetAddressRange() {
    static std::once_flag once;
    static MemGetAddressRangeFn fn = nullptr;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (MemGetAddressRangeFn)p;
        cudaGetLastError();
    });
    return fn;
}

// The bytes [lo, hi) one plane of a frame covers
struct PlaneSpan {
    uintptr_t lo, hi;
};

// Checks one plane of `rows` rows (see include/hrb.h, "device frame planes"); the caller has made h's device current.
// `fn` and `what` name the plane in the message.
static int checkPlane(hrb_ofc* h, const void* ptr, size_t pitch, int rows, const char* fn, const char* what, PlaneSpan* span) {
    auto fail = [&](const char* rule) {
        setLastError("[hopperrender_b200] %s: %s plane %s", fn, what, rule);
        return HRB_ERR_INVALID_ARG;
    };
    if (!ptr) return fail("is null");
    const size_t bpp = (size_t)h->bpp, rowBytes = (size_t)h->frameWidth * bpp;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
        cudaGetLastError();
        return fail("is not device memory (cudaPointerGetAttributes failed)");
    }
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) return fail("is host memory: it must be device or managed memory of the handle's device");
    if (attr.device != h->device) return fail("is memory of another device than the handle's");
    if (pitch < rowBytes) return fail("pitch is below frame_width * bytes per sample");
    if ((reinterpret_cast<uintptr_t>(ptr) % bpp) != 0 || (pitch % bpp) != 0) return fail("pointer and pitch must be multiples of the sample size");
    const size_t extent = (size_t)(rows - 1) * pitch + rowBytes;
    if (extent / bpp >= ((size_t)1 << 31)) return fail("extent exceeds 2^31 samples");
    const MemGetAddressRangeFn range = memGetAddressRange();
    if (!range) {
        setLastError("[hopperrender_b200] %s: cuMemGetAddressRange is not available from the driver", fn);
        return HRB_ERR_CUDA;
    }
    CUdeviceptr base = 0;
    size_t size = 0;
    if (range(&base, &size, (CUdeviceptr)reinterpret_cast<uintptr_t>(ptr)) != CUDA_SUCCESS) return fail("lies in no allocation (cuMemGetAddressRange failed)");
    const uintptr_t lo = reinterpret_cast<uintptr_t>(ptr);
    if (lo + extent > (uintptr_t)base + size) return fail("extent, (rows - 1) * pitch + frame_width * bytes per sample, runs past the end of its allocation");
    *span = PlaneSpan{lo, lo + extent};
    return HRB_OK;
}

// Checks the n frames f[0..n-1] (a source: n = 1, isDst false): each plane, every plane disjoint from every other, and
// one pair of pitches for all.
static int checkFrames(hrb_ofc* h, const hrb_frame_planes* f, int n, bool isDst, const char* fn) {
    HRB_CUDA(cudaSetDevice(h->device));
    PlaneSpan spans[2 * HRB_DELIVERY_MAX_FRAMES];
    for (int i = 0; i < n; ++i) {
        char what[2][32];
        snprintf(what[0], sizeof what[0], n > 1 ? "dst[%d].y" : (isDst ? "dst.y" : "src.y"), i);
        snprintf(what[1], sizeof what[1], n > 1 ? "dst[%d].uv" : (isDst ? "dst.uv" : "src.uv"), i);
        int rc = checkPlane(h, f[i].y, f[i].y_pitch_bytes, h->frameHeight, fn, what[0], &spans[2 * i]);
        if (!rc) rc = checkPlane(h, f[i].uv, f[i].uv_pitch_bytes, h->frameHeight / 2, fn, what[1], &spans[2 * i + 1]);
        if (rc) return rc;
        if (f[i].y_pitch_bytes != f[0].y_pitch_bytes || f[i].uv_pitch_bytes != f[0].uv_pitch_bytes) {
            setLastError("[hopperrender_b200] %s: the destinations of one call must share one (y_pitch_bytes, uv_pitch_bytes); dst[%d] differs from dst[0]", fn, i);
            return HRB_ERR_INVALID_ARG;
        }
    }
    for (int a = 0; a < 2 * n; ++a)
        for (int b = a + 1; b < 2 * n; ++b) {
            if (spans[a].lo < spans[b].hi && spans[b].lo < spans[a].hi) {
                if (a / 2 == b / 2)
                    setLastError("[hopperrender_b200] %s: the Y and UV planes of frame %d overlap", fn, a / 2);
                else
                    setLastError("[hopperrender_b200] %s: the destinations dst[%d] and dst[%d] overlap", fn, a / 2, b / 2);
                return HRB_ERR_INVALID_ARG;
            }
        }
    return HRB_OK;
}

// warp_frames_batch's checks of the blend scalars and the mode
static int checkWarpArgs(int n, const float* blending_scalars, int frame_output_mode, const char* fn) {
    if (n < 1 || n > HRB_WARP_BATCH_MAX) {
        setLastError("[hopperrender_b200] %s: batch size outside 1..HRB_WARP_BATCH_MAX", fn);
        return HRB_ERR_INVALID_ARG;
    }
    for (int i = 0; i < n; ++i)
        if (blending_scalars[i] > 1.0f) {  // opticalFlowCalcSDR.cpp:143-146
            setLastError("[HopperRender] Error in function warpFrames: Blending scalar is greater than 1.0");
            return HRB_ERR_BLEND_RANGE;
        }
    if (frame_output_mode < 0 || frame_output_mode > 6) {
        setLastError("[hopperrender_b200] %s: frame_output_mode outside 0..6", fn);
        return HRB_ERR_INVALID_ARG;
    }
    return HRB_OK;
}

static int updateFramePlanes(hrb_ofc* h, const hrb_frame_planes& src, const char* fn) {
    int rc = checkFrames(h, &src, 1, false, fn);
    if (rc) return rc;
    rc = beginUpdate(h, h->stream);
    if (rc) return rc;
    return finishUpdate(h, &src);
}

}  // namespace hrb

using namespace hrb;

// The calls a delivery takes over (include/hrb.h, "delivery loop") refuse while one is attached.
static bool delivering(hrb_ofc* h, const char* fn) {
    if (!h->delivery) return false;
    setLastError("[hopperrender_b200] %s: the handle has a delivery attached (hrb_delivery_destroy it first)", fn);
    return true;
}

#define HRB_REQUIRE(cond, msg)                                       \
    do {                                                             \
        if (!(cond)) {                                               \
            setLastError("[hopperrender_b200] %s: %s", __func__, msg); \
            return HRB_ERR_INVALID_ARG;                              \
        }                                                            \
    } while (0)

extern "C" {

int hrb_ofc_create(hrb_ofc** out, const hrb_ofc_desc* d) {
    HRB_REQUIRE(out && d, "null argument");
    *out = nullptr;
    HRB_REQUIRE(d->frame_width >= 16 && d->frame_height >= 16, "frame must be at least 16x16");
    HRB_REQUIRE((d->frame_width % 2) == 0 && (d->frame_height % 2) == 0, "NV12/P010 frame dimensions must be even");
    HRB_REQUIRE(d->max_calc_res >= 1, "max_calc_res must be positive");
    HRB_REQUIRE(d->input_stride <= 0 || d->input_stride >= d->frame_width, "stride smaller than the frame width");
    HRB_REQUIRE(d->output_stride <= 0 || d->output_stride >= d->frame_width, "stride smaller than the frame width");
    {
        int rs = 0;
        while ((d->frame_height >> rs) > d->max_calc_res) rs++;
        HRB_REQUIRE((d->frame_width >> rs) >= 4 && (d->frame_height >> rs) >= 4, "flow resolution below 4x4 (raise max_calc_res)");
    }
    HRB_REQUIRE(d->delta_scalar >= 0 && d->delta_scalar <= 31 && d->neighbor_scalar >= 0 && d->neighbor_scalar <= 31, "delta/neighbor scalar outside 0..31");
    int nDev = 0;
    if (cudaGetDeviceCount(&nDev) != cudaSuccess || nDev == 0) {
        setLastError("[hopperrender_b200] no CUDA device (this library has no CPU fallback)");
        return HRB_ERR_NO_DEVICE;
    }
    HRB_REQUIRE(d->device_ordinal >= 0 && d->device_ordinal < nDev, "device_ordinal out of range");
    HRB_CUDA(cudaSetDevice(d->device_ordinal));

    hrb_ofc* h = new (std::nothrow) hrb_ofc();
    HRB_REQUIRE(h, "out of host memory");
    // opticalFlowCalcSDR.cpp:208-232
    h->frameWidth = d->frame_width;
    h->frameHeight = d->frame_height;
    h->inputStride = d->input_stride > 0 ? d->input_stride : d->frame_width;
    h->outputStride = d->output_stride > 0 ? d->output_stride : d->frame_width;
    h->outputBlackLevel = d->black_level;
    h->outputWhiteLevel = d->white_level;
    h->hdr = d->is_hdr ? 1 : 0;
    h->bpp = h->hdr ? 2 : 1;
    h->searchRadius = 5;  // MIN_SEARCH_RADIUS, config.h:8
    h->resScalar = 0;
    while ((d->frame_height >> h->resScalar) > d->max_calc_res) h->resScalar++;
    h->flowWidth = (int)std::ceil(h->frameWidth / std::pow(2, h->resScalar));
    h->flowHeight = (int)std::ceil(h->frameHeight / std::pow(2, h->resScalar));
    h->ofcCalcTime = h->ofcAvgCalcTime = h->ofcPeakCalcTime = 0.0;
    h->ofcCalcCount = 0;
    h->ofcCalcTimeSum = 0.0;
    h->warpCalcTime = 0.0;
    h->deltaScalar = d->delta_scalar;
    h->neighborBiasScalar = d->neighbor_scalar;
    h->totalFrameDelta = 0;
    h->frameCount = 0;
    h->device = d->device_ordinal;
    h->stream = nullptr;
    h->ownStream = false;
    h->warpStartedValid = false;
    h->curRec = 0;
    for (auto& r : h->flowRec) {
        r.start = r.end = nullptr;
        r.rawDeltaHost = nullptr;
        r.startValid = r.pending = false;
    }
    h->haveFlowLevels = false;
    h->tapMode = false;
    h->flowGraphsOn = true;
    h->searchVariant = 0;
    h->smCount = 148;
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d->device_ordinal) == cudaSuccess) h->smCount = prop.multiProcessorCount;
    }
    h->lastIterParity = 0;
    h->lastNWx = h->lastNWy = h->lastWs = 0;
    for (int i = 0; i < 4; ++i) {
        h->inputFrameArray[i] = nullptr;
        h->searchPlane[i] = SearchPlanes();
    }
    for (int i = 0; i < hrb_ofc::kOutRing; ++i) {
        h->outputRing[i] = nullptr;
        h->outReady[i] = h->outFree[i] = nullptr;
    }
    for (auto& e : h->ticketEvent) e = nullptr;
    h->upStream = h->downStream = h->flowStream = nullptr;
    h->flowForkEvent = h->flowJoinEvent = nullptr;
    h->spareFreeEvent = nullptr;
    h->outCur = h->outView = 0;
    h->downloadSeq = 0;
    h->stripeY0 = 0;
    h->stripeY1 = d->frame_height;
    h->levelOffsets[0][0] = h->levelOffsets[0][1] = h->levelOffsets[1][0] = h->levelOffsets[1][1] = nullptr;
    h->winSums = nullptr;
    h->winTicket = nullptr;
    h->offsetArrayScratch = nullptr;
    h->blurredOffsetArray[0] = h->blurredOffsetArray[1] = nullptr;
    h->flowMaxDev[0] = h->flowMaxDev[1] = nullptr;
    h->rawDeltaDev = nullptr;
    h->warpStartedEvent = h->warpEndEvent = h->uploadDoneEvent = nullptr;

    auto fail = [&](int rc) {
        hrb_ofc_destroy(h);
        return rc;
    };
    if (h->inputStride < h->frameWidth || h->outputStride < h->frameWidth) {
        setLastError("[hopperrender_b200] hrb_ofc_create: stride smaller than the frame width");
        return fail(HRB_ERR_INVALID_ARG);
    }
    if (h->flowWidth < 4 || h->flowHeight < 4) {
        setLastError("[hopperrender_b200] hrb_ofc_create: flow resolution %dx%d is below 4x4 (raise max_calc_res)", h->flowWidth, h->flowHeight);
        return fail(HRB_ERR_INVALID_ARG);
    }

    const size_t lw = h->flowWidth, lh = h->flowHeight;
    h->inFrameBytes = ((size_t)h->frameHeight * h->inputStride + (size_t)(h->frameHeight / 2) * h->inputStride) * h->bpp;
    h->outFrameBytes = ((size_t)h->frameHeight * h->outputStride + (size_t)(h->frameHeight / 2) * h->outputStride) * h->bpp;
    // planar 8-bit search planes: luma + NV12-style chroma, row-major and transposed (rows padded to 128 bytes: the
    // TMA row stride must be a multiple of 16 and a warp's 128-byte row segment never leaves the allocation)
    h->planePitch = (h->frameWidth + 127) & ~127;
    h->planePitchT = (h->frameHeight + 127) & ~127;
    const size_t planeYBytes = (size_t)h->planePitch * h->frameHeight, planeCBytes = (size_t)h->planePitch * (h->frameHeight / 2);
    const size_t planeYTBytes = (size_t)h->planePitchT * h->frameWidth, planeCTBytes = (size_t)h->planePitchT * (h->frameWidth / 2);
    const size_t planeBytes = planeYBytes + planeCBytes + 256, planeTBytes = planeYTBytes + planeCTBytes + 256;
    h->levelCapacity = ((lw + 1) / 2) * ((lh + 1) / 2);
    const size_t winSumEntries = ((lw + 63) / 64) * ((lh + 63) / 64) * 16 + 16;
    const size_t need = 4 * (h->inFrameBytes + planeBytes + planeTBytes) + hrb_ofc::kOutRing * h->outFrameBytes + 4 * h->levelCapacity * 2 + winSumEntries * 4 + 3 * 2 * lw * lh * 2;

    // replaces detectDevices' memory check (opticalFlowCalc.cpp:48-51,86-96)
    size_t freeB = 0, totalB = 0;
    if (cudaMemGetInfo(&freeB, &totalB) != cudaSuccess) {
        setLastError("[hopperrender_b200] device %d is not usable: %s", h->device, cudaGetErrorString(cudaGetLastError()));
        return fail(HRB_ERR_CUDA);
    }
    if (freeB < need + (64u << 20)) {
        setLastError("[hopperrender_b200] device %d has %zu MiB free, %zu MiB needed", h->device, freeB >> 20, need >> 20);
        return fail(HRB_ERR_NO_DEVICE);
    }

#define HRB_TRY(call)                                                                                                      \
    do {                                                                                                                   \
        cudaError_t _e = (call);                                                                                           \
        if (_e != cudaSuccess) {                                                                                           \
            setLastError("[hopperrender_b200] CUDA error %d (%s) in hrb_ofc_create at %s:%d", (int)_e, cudaGetErrorString(_e), \
                         __FILE__, __LINE__);                                                                              \
            return fail(HRB_ERR_CUDA);                                                                                     \
        }                                                                                                                  \
    } while (0)

    if (d->cuda_stream) {
        h->stream = (cudaStream_t)d->cuda_stream;
    } else {
        HRB_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->ownStream = true;
    }
    for (auto& r : h->flowRec) {
        HRB_TRY(cudaEventCreate(&r.start));
        HRB_TRY(cudaEventCreate(&r.end));
        HRB_TRY(cudaMallocHost(&r.rawDeltaHost, sizeof(uint32_t)));
        *r.rawDeltaHost = 0;
    }
    HRB_TRY(cudaEventCreate(&h->warpStartedEvent));
    HRB_TRY(cudaEventCreate(&h->warpEndEvent));
    HRB_TRY(cudaEventCreateWithFlags(&h->uploadDoneEvent, cudaEventBlockingSync | cudaEventDisableTiming));
    HRB_TRY(cudaStreamCreateWithFlags(&h->upStream, cudaStreamNonBlocking));
    {
        // the search ladder is the critical path of a source frame: its CTAs go first when warps compete for the SMs
        int prioLow = 0, prioHigh = 0;
        HRB_TRY(cudaDeviceGetStreamPriorityRange(&prioLow, &prioHigh));
        HRB_TRY(cudaStreamCreateWithPriority(&h->flowStream, cudaStreamNonBlocking, prioHigh));
    }
    HRB_TRY(cudaEventCreateWithFlags(&h->flowForkEvent, cudaEventDisableTiming));
    HRB_TRY(cudaEventCreateWithFlags(&h->flowJoinEvent, cudaEventDisableTiming));
    h->flowJoinPending = false;
    h->flowOverlap = true;
    HRB_TRY(cudaStreamCreateWithFlags(&h->downStream, cudaStreamNonBlocking));
    HRB_TRY(cudaEventCreateWithFlags(&h->spareFreeEvent, cudaEventDisableTiming));
    for (int i = 0; i < hrb_ofc::kOutRing; ++i) {
        HRB_TRY(cudaEventCreateWithFlags(&h->outReady[i], cudaEventDisableTiming));
        HRB_TRY(cudaEventCreate(&h->outFree[i]));
        HRB_TRY(cudaMalloc(&h->outputRing[i], h->outFrameBytes));
        HRB_TRY(cudaMemsetAsync(h->outputRing[i], 0, h->outFrameBytes, h->stream));
    }
    for (auto& e : h->ticketEvent) HRB_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) {
        HRB_TRY(cudaMalloc(&h->inputFrameArray[i], h->inFrameBytes));
        HRB_TRY(cudaMemsetAsync(h->inputFrameArray[i], 0, h->inFrameBytes, h->stream));
        SearchPlanes& sp = h->searchPlane[i];
        HRB_TRY(cudaMalloc(&sp.base, planeBytes + planeTBytes));
        HRB_TRY(cudaMemsetAsync(sp.base, 0, planeBytes + planeTBytes, h->stream));
        sp.y = sp.base;                       // cudaMalloc returns 256-byte aligned memory; every plane starts 128-byte aligned
        sp.c = sp.y + planeYBytes;
        sp.yT = sp.c + planeCBytes + 256;       // plane sizes are multiples of 128 (padded pitches)
        sp.cT = sp.yT + planeYTBytes;
    }
    for (int p = 0; p < 2; ++p)
        for (int ax = 0; ax < 2; ++ax) {
            HRB_TRY(cudaMalloc(&h->levelOffsets[p][ax], h->levelCapacity * sizeof(int16_t)));
            HRB_TRY(cudaMemsetAsync(h->levelOffsets[p][ax], 0, h->levelCapacity * sizeof(int16_t), h->stream));
        }
    HRB_TRY(cudaMalloc(&h->winSums, winSumEntries * sizeof(uint32_t)));
    HRB_TRY(cudaMemsetAsync(h->winSums, 0, winSumEntries * sizeof(uint32_t), h->stream));
    HRB_TRY(cudaMalloc(&h->winTicket, (winSumEntries / 16 + 1) * sizeof(unsigned)));
    HRB_TRY(cudaMemsetAsync(h->winTicket, 0, (winSumEntries / 16 + 1) * sizeof(unsigned), h->stream));
    HRB_TRY(cudaMalloc(&h->offsetArrayScratch, 2 * lw * lh * sizeof(int16_t)));
    for (int i = 0; i < 2; ++i) {
        HRB_TRY(cudaMalloc(&h->blurredOffsetArray[i], 2 * lw * lh * sizeof(int16_t)));
        HRB_TRY(cudaMemsetAsync(h->blurredOffsetArray[i], 0, 2 * lw * lh * sizeof(int16_t), h->stream));
        HRB_TRY(cudaMalloc(&h->flowMaxDev[i], sizeof(uint32_t)));
        HRB_TRY(cudaMemsetAsync(h->flowMaxDev[i], 0, sizeof(uint32_t), h->stream));
    }
    HRB_TRY(cudaMalloc(&h->rawDeltaDev, sizeof(uint32_t)));
    HRB_TRY(cudaMemsetAsync(h->rawDeltaDev, 0, sizeof(uint32_t), h->stream));
    HRB_TRY(cudaStreamSynchronize(h->stream));
#undef HRB_TRY
    *out = h;
    return HRB_OK;
}

void hrb_ofc_destroy(hrb_ofc* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);  // clFinish, opticalFlowCalcSDR.cpp:186
    if (h->upStream) cudaStreamSynchronize(h->upStream);
    if (h->flowStream) cudaStreamSynchronize(h->flowStream);
    if (h->downStream) cudaStreamSynchronize(h->downStream);
    freeTaps(h);
    for (auto& p : h->prof.pending) {
        if (p.a) cudaEventDestroy(p.a);
        if (p.b) cudaEventDestroy(p.b);
    }
    for (auto e : h->prof.pool) cudaEventDestroy(e);
    for (int i = 0; i < 4; ++i) {
        cudaFree(h->inputFrameArray[i]);
        cudaFree(h->searchPlane[i].base);
    }
    for (int i = 0; i < hrb_ofc::kOutRing; ++i) {
        cudaFree(h->outputRing[i]);
        if (h->outReady[i]) cudaEventDestroy(h->outReady[i]);
        if (h->outFree[i]) cudaEventDestroy(h->outFree[i]);
    }
    for (auto e : h->ticketEvent)
        if (e) cudaEventDestroy(e);
    if (h->spareFreeEvent) cudaEventDestroy(h->spareFreeEvent);
    dropFlowGraphs(h);
    freeTmaCache(h);
    cudaFree(h->dbgDev);
    if (h->upStream) cudaStreamDestroy(h->upStream);
    if (h->flowStream) cudaStreamDestroy(h->flowStream);
    if (h->flowForkEvent) cudaEventDestroy(h->flowForkEvent);
    if (h->flowJoinEvent) cudaEventDestroy(h->flowJoinEvent);
    if (h->downStream) cudaStreamDestroy(h->downStream);
    for (int p = 0; p < 2; ++p)
        for (int ax = 0; ax < 2; ++ax) cudaFree(h->levelOffsets[p][ax]);
    cudaFree(h->winSums);
    cudaFree(h->winTicket);
    cudaFree(h->offsetArrayScratch);
    cudaFree(h->blurredOffsetArray[0]);
    cudaFree(h->blurredOffsetArray[1]);
    cudaFree(h->flowMaxDev[0]);
    cudaFree(h->flowMaxDev[1]);
    cudaFree(h->rawDeltaDev);
    for (auto& r : h->flowRec) {
        if (r.rawDeltaHost) cudaFreeHost(r.rawDeltaHost);
        if (r.start) cudaEventDestroy(r.start);
        if (r.end) cudaEventDestroy(r.end);
    }
    if (h->warpStartedEvent) cudaEventDestroy(h->warpStartedEvent);
    if (h->warpEndEvent) cudaEventDestroy(h->warpEndEvent);
    if (h->uploadDoneEvent) cudaEventDestroy(h->uploadDoneEvent);
    if (h->ownStream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hrb_ofc_update_frame(hrb_ofc* h, const uint8_t* input_planes) {
    HRB_REQUIRE(h && input_planes, "null argument");
    return uploadFrame(h, input_planes, true);
}

int hrb_ofc_update_frame_async(hrb_ofc* h, const uint8_t* pinned_input_planes) {
    HRB_REQUIRE(h && pinned_input_planes, "null argument");
    return uploadFrame(h, pinned_input_planes, false);
}

int hrb_ofc_wait_upload(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    HRB_CUDA(cudaSetDevice(h->device));
    HRB_CUDA(cudaEventSynchronize(h->uploadDoneEvent));
    return HRB_OK;
}

int hrb_ofc_update_frame_device(hrb_ofc* h, const void* device_planes) {
    HRB_REQUIRE(h && device_planes, "null argument");
    const size_t pitch = (size_t)h->inputStride * h->bpp;
    uint8_t* base = static_cast<uint8_t*>(const_cast<void*>(device_planes));
    return updateFramePlanes(h, hrb_frame_planes{base, pitch, base + (size_t)h->frameHeight * pitch, pitch}, __func__);
}

int hrb_ofc_update_frame_planes(hrb_ofc* h, const hrb_frame_planes* src) {
    HRB_REQUIRE(h && src, "null argument");
    return updateFramePlanes(h, *src, __func__);
}

// Orders the compute stream behind the last flow calculation that was enqueued on the flow stream.
static int joinFlow(hrb_ofc* h) {
    if (h->flowJoinPending) {
        HRB_CUDA(cudaSetDevice(h->device));
        HRB_CUDA(cudaStreamWaitEvent(h->stream, h->flowJoinEvent, 0));
        h->flowJoinPending = false;
    }
    return HRB_OK;
}

// warpFrames reads the flow of the PREVIOUS calculation (m_blurredOffsetArray12[0] after the swap,
// opticalFlowCalcSDR.cpp:113-123,150) and the search touches nothing the warp writes, so the calculation of source
// frame N and the warps issued after it are independent: the asynchronous entry point runs the search ladder on its
// own stream, forked behind everything already enqueued (the ingest of frame N, the last readers of the flow buffer
// it overwrites) and joined before the next calculation — i.e. before any warp that needs its result.  On a group
// every shard makes this choice for itself, exactly as its own calculate_optical_flow_async would.
static int calculateFlow(const Shards& s, bool async) {
    for (int k = 0; k < s.n; ++k) {
        const int rc = joinFlow(s.h[k]);
        if (rc) return rc;
    }
    if (!async) {
        int rc = enqueueFlow(s);
        for (int k = 0; k < s.n && !rc; ++k) rc = resolveFlow(s.h[k]);
        return rc;
    }
    cudaStream_t compute[kMaxShards];
    bool forked[kMaxShards];
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        forked[k] = h->flowOverlap && !h->tapMode && !h->prof.on;
        compute[k] = h->stream;
        if (!forked[k]) continue;
        HRB_CUDA(cudaSetDevice(h->device));
        HRB_CUDA(cudaEventRecord(h->flowForkEvent, h->stream));
        HRB_CUDA(cudaStreamWaitEvent(h->flowStream, h->flowForkEvent, 0));
        h->stream = h->flowStream;
    }
    const int rc = enqueueFlow(s);
    for (int k = 0; k < s.n; ++k) s.h[k]->stream = compute[k];
    if (rc) return rc;
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        if (!forked[k]) continue;
        if (s.n > 1) HRB_CUDA(cudaSetDevice(h->device));
        HRB_CUDA(cudaEventRecord(h->flowJoinEvent, h->flowStream));
        h->flowJoinPending = true;
        h->updatesSinceFlow = 0;
    }
    return HRB_OK;
}

int hrb_ofc_calculate_optical_flow_async(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    return calculateFlow(Shards(h), true);
}

int hrb_ofc_calculate_optical_flow(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    return calculateFlow(Shards(h), false);
}

int hrb_ofc_warp_frames(hrb_ofc* h, float blending_scalar, int frame_output_mode) {
    HRB_REQUIRE(h, "null handle");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    if (blending_scalar > 1.0f) {  // opticalFlowCalcSDR.cpp:143-146
        setLastError("[HopperRender] Error in function warpFrames: Blending scalar is greater than 1.0");
        return HRB_ERR_BLEND_RANGE;
    }
    HRB_REQUIRE(frame_output_mode >= 0 && frame_output_mode <= 6, "frame_output_mode outside 0..6");
    int rc = beginOutput(h);
    if (rc) return rc;
    const hrb_frame_planes out = ringPlanes(h, h->outCur);
    rc = launchWarpFrames(h, 1, &blending_scalar, &out, frame_output_mode);
    if (rc) return rc;
    HRB_CUDA(cudaEventRecord(h->outReady[h->outCur], h->stream));
    return HRB_OK;
}

int hrb_ofc_warp_frames_batch(hrb_ofc* h, int n, const float* blending_scalars, int frame_output_mode) {
    HRB_REQUIRE(h && blending_scalars, "null argument");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    int rc = checkWarpArgs(n, blending_scalars, frame_output_mode, __func__);
    if (rc) return rc;
    rc = beginOutput(h);  // waits for the download of the first slot, starts the warp timer
    if (rc) return rc;
    hrb_frame_planes outs[HRB_WARP_BATCH_MAX];
    for (int i = 0; i < n; ++i) {
        const int slot = (h->outCur + i) % hrb_ofc::kOutRing;
        if (i) HRB_CUDA(cudaStreamWaitEvent(h->stream, h->outFree[slot], 0));
        outs[i] = ringPlanes(h, slot);
    }
    rc = launchWarpFrames(h, n, blending_scalars, outs, frame_output_mode);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) HRB_CUDA(cudaEventRecord(h->outReady[(h->outCur + i) % hrb_ofc::kOutRing], h->stream));
    return HRB_OK;
}

int hrb_ofc_copy_frame(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    const int frameIndex = h->frameCount >= 3 ? 0 : h->frameCount >= 2 ? 1 : 2;  // opticalFlowCalcSDR.cpp:173
    int rc = beginOutput(h);
    if (rc) return rc;
    const hrb_frame_planes out = ringPlanes(h, h->outCur);
    rc = launchCopyFrame(h, frameIndex, &out);
    if (rc) return rc;
    HRB_CUDA(cudaEventRecord(h->outReady[h->outCur], h->stream));
    return HRB_OK;
}

// The _to calls write the caller's planes on the compute stream and leave the ring, its cursor, its events and the warp
// timer (warp_calc_time belongs to the ring's downloads) alone.
int hrb_ofc_warp_frames_to(hrb_ofc* h, int n, const float* blending_scalars, int frame_output_mode, const hrb_frame_planes* dst) {
    HRB_REQUIRE(h && blending_scalars && dst, "null argument");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    int rc = checkWarpArgs(n, blending_scalars, frame_output_mode, __func__);
    if (!rc) rc = checkFrames(h, dst, n, true, __func__);
    if (rc) return rc;
    return launchWarpFrames(h, n, blending_scalars, dst, frame_output_mode);
}

int hrb_ofc_copy_frame_to(hrb_ofc* h, const hrb_frame_planes* dst) {
    HRB_REQUIRE(h && dst, "null argument");
    if (delivering(h, __func__)) return HRB_ERR_STATE;
    const int rc = checkFrames(h, dst, 1, true, __func__);
    if (rc) return rc;
    const int frameIndex = h->frameCount >= 3 ? 0 : h->frameCount >= 2 ? 1 : 2;  // opticalFlowCalcSDR.cpp:173
    return launchCopyFrame(h, frameIndex, dst);
}

int hrb_ofc_download_frame(hrb_ofc* h, uint8_t* output_planes) {
    HRB_REQUIRE(h && output_planes, "null argument");
    const int slot = h->outCur;
    const int rc = enqueueDownload(h, output_planes, nullptr);
    if (rc) return rc;
    HRB_CUDA(cudaEventSynchronize(h->outFree[slot]));  // blocking read, opticalFlowCalcSDR.cpp:33
    if (h->warpStartedValid) {  // opticalFlowCalcSDR.cpp:36-41
        float ms = 0;
        HRB_CUDA(cudaEventElapsedTime(&ms, h->warpStartedEvent, h->outFree[slot]));
        h->warpCalcTime = (double)ms / 1e3;
    }
    return HRB_OK;
}

int hrb_ofc_download_frame_async(hrb_ofc* h, uint8_t* pinned_output_planes, unsigned long long* ticket) {
    HRB_REQUIRE(h && pinned_output_planes, "null argument");
    return enqueueDownload(h, pinned_output_planes, ticket);
}

int hrb_ofc_wait_download(hrb_ofc* h, unsigned long long ticket) {
    HRB_REQUIRE(h, "null handle");
    HRB_REQUIRE(ticket >= 1 && ticket <= h->downloadSeq, "unknown ticket");
    HRB_CUDA(cudaSetDevice(h->device));
    // The slot may have been re-recorded by a later download (tickets wrap every kTickets): the download stream is in
    // order, so waiting for that later record also proves that this ticket's copy has landed.  Never return unwaited.
    HRB_CUDA(cudaEventSynchronize(h->ticketEvent[ticket % hrb_ofc::kTickets]));
    return HRB_OK;
}

int hrb_ofc_synchronize(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    HRB_CUDA(cudaSetDevice(h->device));
    HRB_CUDA(cudaStreamSynchronize(h->upStream));
    HRB_CUDA(cudaStreamSynchronize(h->flowStream));
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    HRB_CUDA(cudaStreamSynchronize(h->downStream));
    if (h->flowJoinPending) HRB_CUDA(cudaEventSynchronize(h->flowJoinEvent));  // a flow batch's stream
    h->flowJoinPending = false;
    return resolveFlow(h);
}

int hrb_ofc_stream(hrb_ofc* h, void** out) {
    HRB_REQUIRE(h && out, "null argument");
    *out = (void*)h->stream;
    return HRB_OK;
}

int hrb_ofc_output_device_ptr(hrb_ofc* h, void** out) {
    HRB_REQUIRE(h && out, "null argument");
    *out = h->outputRing[h->outView];
    return HRB_OK;
}

int hrb_host_register(void* ptr, size_t bytes) {
    HRB_REQUIRE(ptr && bytes, "null argument");
    HRB_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return HRB_OK;
}
int hrb_host_unregister(void* ptr) {
    HRB_REQUIRE(ptr, "null argument");
    HRB_CUDA(cudaHostUnregister(ptr));
    return HRB_OK;
}
int hrb_host_alloc(void** out, size_t bytes) {
    HRB_REQUIRE(out && bytes, "null argument");
    HRB_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    return HRB_OK;
}
int hrb_host_free(void* ptr) {
    HRB_REQUIRE(ptr, "null argument");
    HRB_CUDA(cudaFreeHost(ptr));
    return HRB_OK;
}

// folds in the flow calculations that have FINISHED (oldest first), without waiting for the ones still running
static int resolveFinishedFlows(hrb_ofc* h) {
    for (int i = 1; i <= hrb_ofc::kFlowRecords; ++i) {
        hrb_ofc::FlowRecord& r = h->flowRec[(h->curRec + i) % hrb_ofc::kFlowRecords];
        if (!r.pending) continue;
        const cudaError_t q = cudaEventQuery(r.end);
        if (q == cudaErrorNotReady) {
            cudaGetLastError();
            break;  // later records are younger: still running too
        }
        HRB_CUDA(q);
        const int rc = resolveRecord(h, r);
        if (rc) return rc;
    }
    return HRB_OK;
}

static void fillState(const hrb_ofc* h, hrb_ofc_state* s);

int hrb_ofc_peek_state(hrb_ofc* h, hrb_ofc_state* s) {
    HRB_REQUIRE(h && s, "null argument");
    HRB_CUDA(cudaSetDevice(h->device));
    const int rc = resolveFinishedFlows(h);
    if (rc) return rc;
    fillState(h, s);
    return HRB_OK;
}

int hrb_ofc_get_state(hrb_ofc* h, hrb_ofc_state* s) {
    HRB_REQUIRE(h && s, "null argument");
    const int rc = resolveFlow(h);
    if (rc) return rc;
    fillState(h, s);
    return HRB_OK;
}

static void fillState(const hrb_ofc* h, hrb_ofc_state* s) {
    s->frame_width = h->frameWidth;
    s->frame_height = h->frameHeight;
    s->input_stride = h->inputStride;
    s->output_stride = h->outputStride;
    s->output_black_level = h->outputBlackLevel;
    s->output_white_level = h->outputWhiteLevel;
    s->res_scalar = h->resScalar;
    s->flow_width = h->flowWidth;
    s->flow_height = h->flowHeight;
    s->search_radius = h->searchRadius;
    s->ofc_calc_time = h->ofcCalcTime;
    s->ofc_avg_calc_time = h->ofcAvgCalcTime;
    s->ofc_peak_calc_time = h->ofcPeakCalcTime;
    s->ofc_calc_count = h->ofcCalcCount;
    s->ofc_calc_time_sum = h->ofcCalcTimeSum;
    s->warp_calc_time = h->warpCalcTime;
    s->delta_scalar = h->deltaScalar;
    s->neighbor_bias_scalar = h->neighborBiasScalar;
    s->total_frame_delta = h->totalFrameDelta;
    s->frame_count = h->frameCount;
}

int hrb_ofc_set_params(hrb_ofc* h, const hrb_ofc_params* p) {
    HRB_REQUIRE(h && p, "null argument");
    // the same ranges calculateOpticalFlow accepts (the filter keeps the radius in 5..16, config.h:8-9; 2..4 exist for tests)
    HRB_REQUIRE(p->search_radius >= 2 && p->search_radius <= 16, "search radius outside 2..16");
    HRB_REQUIRE(p->delta_scalar >= 0 && p->delta_scalar <= 31 && p->neighbor_bias_scalar >= 0 && p->neighbor_bias_scalar <= 31, "delta/neighbor scalar outside 0..31");
    HRB_REQUIRE(p->black_level == p->black_level && p->white_level == p->white_level, "levels must be numbers");
    h->searchRadius = p->search_radius;
    h->deltaScalar = p->delta_scalar;
    h->neighborBiasScalar = p->neighbor_bias_scalar;
    h->outputBlackLevel = p->black_level;
    h->outputWhiteLevel = p->white_level;
    return HRB_OK;
}

int hrb_ofc_set_frame_count(hrb_ofc* h, unsigned int n) {
    HRB_REQUIRE(h, "null handle");
    h->frameCount = n;
    return HRB_OK;
}

int hrb_ofc_reset(hrb_ofc* h) { return hrb_ofc_set_frame_count(h, 0); }

// ---- taps ----------------------------------------------------------------------------------------
int hrb_ofc_set_tap_mode(hrb_ofc* h, int on) {
    HRB_REQUIRE(h, "null handle");
    HRB_CUDA(cudaSetDevice(h->device));
    if (joinFlow(h)) return HRB_ERR_CUDA;
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    h->tapMode = on != 0;
    if (!h->tapMode) freeTaps(h);
    return HRB_OK;
}

int hrb_ofc_num_passes(hrb_ofc* h, int* out) {
    HRB_REQUIRE(h && out, "null argument");
    *out = (int)h->taps.size();
    return HRB_OK;
}

int hrb_ofc_pass_info(hrb_ofc* h, int pass, int* window_size, int* iteration, int* step, int* windows_x, int* windows_y) {
    HRB_REQUIRE(h, "null handle");
    HRB_REQUIRE(pass >= 0 && pass < (int)h->taps.size(), "pass out of range (is tap mode on?)");
    const PassGeom& g = h->taps[pass].g;
    if (window_size) *window_size = g.windowSize;
    if (iteration) *iteration = g.iteration;
    if (step) *step = g.step;
    if (windows_x) *windows_x = g.nWx;
    if (windows_y) *windows_y = g.nWy;
    return HRB_OK;
}

int hrb_ofc_read_pass_tap(hrb_ofc* h, int pass, int which, void* dst, size_t bytes) {
    HRB_REQUIRE(h && dst, "null argument");
    if (pass < 0 || pass >= (int)h->taps.size()) {
        setLastError("[hopperrender_b200] hrb_ofc_read_pass_tap: no such pass (tap mode must be on before calculate)");
        return HRB_ERR_STATE;
    }
    HRB_CUDA(cudaSetDevice(h->device));
    const PassTapDev& t = h->taps[pass];
    const size_t nW = (size_t)t.g.nWx * t.g.nWy;
    const size_t lwlh = (size_t)h->flowWidth * h->flowHeight;
    if (which == HRB_TAP_WINDOW_SUMS) {
        HRB_REQUIRE(bytes <= nW * 16 * sizeof(uint32_t) && bytes % (nW * sizeof(uint32_t)) == 0, "size must be R*windows*4");
        HRB_CUDA(cudaMemcpyAsync(dst, t.sums, bytes, cudaMemcpyDeviceToHost, h->stream));
    } else if (which == HRB_TAP_WINDOW_LAYER) {
        HRB_REQUIRE(bytes == nW, "size must be windows");
        HRB_CUDA(cudaMemcpyAsync(dst, t.layer, bytes, cudaMemcpyDeviceToHost, h->stream));
    } else if (which == HRB_TAP_OFFSETS) {
        HRB_REQUIRE(bytes == 2 * lwlh * sizeof(int16_t), "size must be 2*flow_w*flow_h*2");
        const int rc = launchExpandOffsets(h, t.offX, t.nWxX, ilog2(t.wsX), t.wsY ? t.offY : nullptr, t.nWxY, t.wsY ? ilog2(t.wsY) : 0,
                                           h->offsetArrayScratch);
        if (rc) return rc;
        HRB_CUDA(cudaMemcpyAsync(dst, h->offsetArrayScratch, bytes, cudaMemcpyDeviceToHost, h->stream));
    } else {
        HRB_REQUIRE(false, "unknown tap");
    }
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    return HRB_OK;
}

int hrb_ofc_read_buffer(hrb_ofc* h, int which, void* dst, size_t bytes) {
    HRB_REQUIRE(h && dst, "null argument");
    HRB_CUDA(cudaSetDevice(h->device));
    if (joinFlow(h)) return HRB_ERR_CUDA;
    const size_t flowBytes = 2 * (size_t)h->flowWidth * h->flowHeight * sizeof(int16_t);
    if (which == HRB_BUF_OFFSET_ARRAY) {
        HRB_REQUIRE(bytes == flowBytes, "size must be 2*flow_w*flow_h*2");
        if (!h->haveFlowLevels) {
            setLastError("[hopperrender_b200] hrb_ofc_read_buffer: no flow has been calculated yet");
            return HRB_ERR_STATE;
        }
        const int s = ilog2(h->lastWs);
        const int rc = launchExpandOffsets(h, h->levelOffsets[h->lastIterParity][0], h->lastNWx, s, h->levelOffsets[h->lastIterParity][1], h->lastNWx, s,
                                           h->offsetArrayScratch);
        if (rc) return rc;
        HRB_CUDA(cudaMemcpyAsync(dst, h->offsetArrayScratch, bytes, cudaMemcpyDeviceToHost, h->stream));
    } else if (which == HRB_BUF_FLOW_FOR_WARP || which == HRB_BUF_FLOW_LATEST) {
        HRB_REQUIRE(bytes == flowBytes, "size must be 2*flow_w*flow_h*2");
        HRB_CUDA(cudaMemcpyAsync(dst, h->blurredOffsetArray[which == HRB_BUF_FLOW_FOR_WARP ? 0 : 1], bytes, cudaMemcpyDeviceToHost, h->stream));
    } else if (which == HRB_BUF_OUTPUT_FRAME) {
        HRB_REQUIRE(bytes <= h->outFrameBytes, "size larger than the output frame");
        HRB_CUDA(cudaMemcpyAsync(dst, h->outputRing[h->outView], bytes, cudaMemcpyDeviceToHost, h->stream));
    } else if (which == HRB_BUF_RAW_FRAME_DELTA) {
        HRB_REQUIRE(bytes == sizeof(uint32_t), "size must be 4");
        HRB_CUDA(cudaMemcpyAsync(dst, h->rawDeltaDev, bytes, cudaMemcpyDeviceToHost, h->stream));
    } else if (which == HRB_BUF_FLOW_PEAK) {
        HRB_REQUIRE(bytes == 2 * sizeof(uint32_t), "size must be 8");
        for (int i = 0; i < 2; ++i)
            HRB_CUDA(cudaMemcpyAsync(static_cast<uint32_t*>(dst) + i, h->flowMaxDev[i], sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    } else {
        HRB_REQUIRE(false, "unknown buffer");
    }
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    return resolveFlow(h);
}

int hrb_ofc_write_flow(hrb_ofc* h, int which, const int16_t* src, size_t count) {
    HRB_REQUIRE(h && src, "null argument");
    HRB_REQUIRE(which == HRB_BUF_FLOW_FOR_WARP || which == HRB_BUF_FLOW_LATEST, "only the blurred flows are writable");
    HRB_REQUIRE(count == 2 * (size_t)h->flowWidth * h->flowHeight, "count must be 2*flow_w*flow_h");
    HRB_CUDA(cudaSetDevice(h->device));
    if (joinFlow(h)) return HRB_ERR_CUDA;
    const int slot = which == HRB_BUF_FLOW_FOR_WARP ? 0 : 1;
    HRB_CUDA(cudaMemcpyAsync(h->blurredOffsetArray[slot], src, count * sizeof(int16_t), cudaMemcpyHostToDevice, h->stream));
    uint32_t peak = 0;
    for (size_t i = 0; i < count; ++i) {
        const uint32_t v = (uint32_t)(src[i] < 0 ? -(int)src[i] : (int)src[i]);
        if (v > peak) peak = v;
    }
    HRB_CUDA(cudaMemcpyAsync(h->flowMaxDev[slot], &peak, sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    return HRB_OK;
}

// ---- measurement -----------------------------------------------------------------------------------
int hrb_ofc_set_profile(hrb_ofc* h, int on) {
    HRB_REQUIRE(h, "null handle");
    HRB_CUDA(cudaSetDevice(h->device));
    if (joinFlow(h)) return HRB_ERR_CUDA;
    const int rc = profResolve(h);
    if (rc) return rc;
    h->prof.on = on != 0;
    return HRB_OK;
}

int hrb_ofc_profile_read(hrb_ofc* h, hrb_ofc_profile* out) {
    HRB_REQUIRE(h && out, "null argument");
    HRB_CUDA(cudaSetDevice(h->device));
    const int rc = profResolve(h);
    if (rc) return rc;
    out->ms_ingest = h->prof.ms[CLS_INGEST];
    out->ms_search = h->prof.ms[CLS_SEARCH];
    out->ms_blur = h->prof.ms[CLS_BLUR];
    out->ms_warp = h->prof.ms[CLS_WARP];
    out->ms_copy = h->prof.ms[CLS_COPY];
    out->n_ingest = h->prof.n[CLS_INGEST];
    out->n_search = h->prof.n[CLS_SEARCH];
    out->n_blur = h->prof.n[CLS_BLUR];
    out->n_warp = h->prof.n[CLS_WARP];
    out->n_copy = h->prof.n[CLS_COPY];
    return HRB_OK;
}

int hrb_ofc_profile_reset(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    const int rc = profResolve(h);
    if (rc) return rc;
    for (int i = 0; i < 5; ++i) {
        h->prof.ms[i] = 0;
        h->prof.n[i] = 0;
    }
    return HRB_OK;
}

int hrb_ofc_set_side_data(hrb_ofc* h, const hrb_side_data* items, int count) {
    HRB_REQUIRE(h && (items || count == 0), "null argument");
    HRB_REQUIRE(count >= 0 && count <= 64, "side-data count outside 0..64");
    for (int i = 0; i < count; ++i) HRB_REQUIRE(items[i].data || items[i].bytes == 0, "null blob with a size");
    h->sideData.clear();
    h->sideData.resize((size_t)count);
    for (int i = 0; i < count; ++i) {
        memcpy(h->sideData[i].guid, items[i].guid, 16);
        const uint8_t* p = static_cast<const uint8_t*>(items[i].data);
        h->sideData[i].bytes.assign(p, p + items[i].bytes);
    }
    return HRB_OK;
}

int hrb_ofc_get_side_data(hrb_ofc* h, hrb_side_data* items, int capacity, int* count) {
    HRB_REQUIRE(h && count, "null argument");
    HRB_REQUIRE(capacity >= 0 && (items || capacity == 0), "null array with a capacity");
    *count = (int)h->sideData.size();
    for (int i = 0; i < capacity && i < *count; ++i) {
        memcpy(items[i].guid, h->sideData[i].guid, 16);
        items[i].data = h->sideData[i].bytes.data();
        items[i].bytes = h->sideData[i].bytes.size();
    }
    return HRB_OK;
}

int hrb_ofc_set_output_stripe(hrb_ofc* h, int row_begin, int row_end) {
    HRB_REQUIRE(h, "null handle");
    HRB_REQUIRE(row_begin >= 0 && row_end <= h->frameHeight && row_begin < row_end, "stripe outside the frame");
    HRB_REQUIRE((row_begin % 2) == 0 && (row_end % 2) == 0, "stripe bounds must be even (chroma rows are shared by luma row pairs)");
    h->stripeY0 = row_begin;
    h->stripeY1 = row_end;
    return HRB_OK;
}

int hrb_ofc_set_flow_overlap(hrb_ofc* h, int on) {
    HRB_REQUIRE(h, "null handle");
    const int rc = joinFlow(h);
    if (rc) return rc;
    h->flowOverlap = on != 0;
    return HRB_OK;
}

int hrb_ofc_join_flow(hrb_ofc* h) {
    HRB_REQUIRE(h, "null handle");
    return joinFlow(h);
}

int hrb_ofc_set_search_variant(hrb_ofc* h, int variant) {
    HRB_REQUIRE(h, "null handle");
    HRB_REQUIRE(variant >= 0 && variant <= 4, "variant must be 0 (automatic), 1 (generic kernel only), 2 (tile kernel without TMA), 3 (tile kernel, per-pixel path forced) or 4 (butterfly form for windows of 2 and 4)");
    h->searchVariant = variant;
    return HRB_OK;
}

// Debug aid: per-CTA timelines of the tile search kernels (16 words per CTA: start, boxes landed, runs done, end
// [globaltimer ns], SM id, block x, block y, rounds, warps per CTA, 7 spare), `words_per_pass` words for each of up to 32
// passes.  CTA i of a pass records only if its record fits the slice (16 * (i + 1) <= words_per_pass).
int hrb_ofc_debug_timeline(hrb_ofc* h, size_t words_per_pass) {
    HRB_REQUIRE(h, "null handle");
    HRB_CUDA(cudaSetDevice(h->device));
    HRB_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(h->dbgDev);
    h->dbgDev = nullptr;
    h->dbgStride = words_per_pass;
    if (words_per_pass) {
        HRB_CUDA(cudaMalloc(&h->dbgDev, words_per_pass * 32 * sizeof(unsigned long long)));
        HRB_CUDA(cudaMemset(h->dbgDev, 0, words_per_pass * 32 * sizeof(unsigned long long)));
    }
    return HRB_OK;
}
int hrb_ofc_debug_timeline_read(hrb_ofc* h, void* dst, size_t bytes) {
    HRB_REQUIRE(h && dst && h->dbgDev, "no timeline buffer");
    HRB_REQUIRE(bytes <= h->dbgStride * 32 * sizeof(unsigned long long), "size larger than the buffer");
    HRB_CUDA(cudaSetDevice(h->device));
    HRB_CUDA(cudaDeviceSynchronize());
    HRB_CUDA(cudaMemcpy(dst, h->dbgDev, bytes, cudaMemcpyDeviceToHost));
    return HRB_OK;
}

// ---- split search ----------------------------------------------------------------------------------
// b_k = 128 * round(k * lh / (n * 128)), b_0 = 0, b_n = lh; false when a stripe would be empty
static bool planStripes(int lh, int n, int* b) {
    if (n < 1 || n > kMaxShards || lh < 1) return false;
    for (int k = 0; k < n; ++k) b[k] = kSplitAlign * (int)((2LL * k * lh + (long long)n * kSplitAlign) / (2LL * n * kSplitAlign));
    b[n] = lh;
    for (int k = 0; k < n; ++k)
        if (b[k + 1] <= b[k]) return false;
    return true;
}

// every shard must compute the flow shard 0 would: same geometry, format and search parameters
static int checkShards(hrb_ofc* const* sh, int n, const char* fn) {
    const hrb_ofc* a = sh[0];
    for (int k = 1; k < n; ++k) {
        const hrb_ofc* b = sh[k];
        const char* f = a->frameWidth != b->frameWidth               ? "frame_width"
                        : a->frameHeight != b->frameHeight           ? "frame_height"
                        : a->hdr != b->hdr                           ? "is_hdr"
                        : a->resScalar != b->resScalar               ? "res_scalar"
                        : a->searchRadius != b->searchRadius         ? "search_radius"
                        : a->deltaScalar != b->deltaScalar           ? "delta_scalar"
                        : a->neighborBiasScalar != b->neighborBiasScalar ? "neighbor_bias_scalar"
                        : a->searchVariant != b->searchVariant       ? "search_variant"
                                                                     : nullptr;
        if (f) {
            setLastError("[hopperrender_b200] %s: shard %d differs from shard 0 in %s", fn, k, f);
            return HRB_ERR_INVALID_ARG;
        }
    }
    return HRB_OK;
}

int hrb_split_plan(int flow_height, int n, int* bounds) {
    HRB_REQUIRE(bounds, "null argument");
    std::vector<int> b((size_t)std::max(n, 0) + 1);
    if (!planStripes(flow_height, n, b.data())) {
        setLastError("[hopperrender_b200] hrb_split_plan: %d shards do not fit %d flow rows (1..%d shards, every stripe at least one row, bounds at multiples of %d)",
                     n, flow_height, kMaxShards, kSplitAlign);
        return HRB_ERR_INVALID_ARG;
    }
    memcpy(bounds, b.data(), b.size() * sizeof(int));
    return HRB_OK;
}

int hrb_split_create(hrb_split** out, hrb_ofc* const* shards, int n) {
    HRB_REQUIRE(out && shards, "null argument");
    *out = nullptr;
    HRB_REQUIRE(n >= 1 && n <= kMaxShards, "shard count outside 1..64");
    for (int k = 0; k < n; ++k) {
        HRB_REQUIRE(shards[k], "null handle");
        for (int j = 0; j < k; ++j) HRB_REQUIRE(shards[j] != shards[k], "a handle appears twice");
    }
    for (int k = 0; k < n; ++k)
        if (delivering(shards[k], __func__)) return HRB_ERR_STATE;
    int rc = checkShards(shards, n, "hrb_split_create");
    if (rc) return rc;
    std::vector<int> b((size_t)n + 1);
    if (!planStripes(shards[0]->flowHeight, n, b.data())) {
        setLastError("[hopperrender_b200] hrb_split_create: %d shards do not fit %d flow rows", n, shards[0]->flowHeight);
        return HRB_ERR_INVALID_ARG;
    }
    // direct peer copies where the devices allow them (a context attribute; otherwise the copies are staged by the driver)
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            const int di = shards[i]->device, dj = shards[j]->device;
            int can = 0;
            if (di == dj || cudaDeviceCanAccessPeer(&can, di, dj) != cudaSuccess || !can) continue;
            HRB_CUDA(cudaSetDevice(di));
            const cudaError_t e = cudaDeviceEnablePeerAccess(dj, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled)
                cudaGetLastError();
            else
                HRB_CUDA(e);
        }
    hrb_split* s = new (std::nothrow) hrb_split();
    HRB_REQUIRE(s, "out of host memory");
    s->shard.assign(shards, shards + n);
    for (hrb_ofc* h : s->shard) h->groups++;
    s->bounds = b;
    s->done.assign((size_t)n, nullptr);
    for (int k = 0; k < n; ++k) {
        cudaError_t e = cudaSetDevice(shards[k]->device);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->done[k], cudaEventDisableTiming);
        if (e != cudaSuccess) {
            setLastError("[hopperrender_b200] CUDA error %d (%s) in hrb_split_create", (int)e, cudaGetErrorString(e));
            hrb_split_destroy(s);
            return HRB_ERR_CUDA;
        }
    }
    *out = s;
    return HRB_OK;
}

void hrb_split_destroy(hrb_split* s) {
    if (!s) return;
    for (hrb_ofc* h : s->shard) h->groups--;
    for (auto e : s->done)
        if (e) cudaEventDestroy(e);
    delete s;
}

int hrb_split_stripe(hrb_split* s, int shard, int* flow_row_begin, int* flow_row_end) {
    HRB_REQUIRE(s && flow_row_begin && flow_row_end, "null argument");
    HRB_REQUIRE(shard >= 0 && shard < (int)s->shard.size(), "shard out of range");
    *flow_row_begin = s->bounds[shard];
    *flow_row_end = s->bounds[shard + 1];
    return HRB_OK;
}

static int splitCalculate(hrb_split* s, bool async, const char* fn) {
    const int rc = checkShards(s->shard.data(), (int)s->shard.size(), fn);
    if (rc) return rc;
    for (hrb_ofc* h : s->shard)
        if (h->prof.on || h->dbgDev) {
            setLastError("[hopperrender_b200] %s: the profile and the debug timeline are not available on a grouped calculate (switch them off on every shard)", fn);
            return HRB_ERR_STATE;
        }
    return calculateFlow(Shards(s), async);
}

int hrb_split_calculate_optical_flow(hrb_split* s) {
    HRB_REQUIRE(s, "null handle");
    return splitCalculate(s, false, "hrb_split_calculate_optical_flow");
}

int hrb_split_calculate_optical_flow_async(hrb_split* s) {
    HRB_REQUIRE(s, "null handle");
    return splitCalculate(s, true, "hrb_split_calculate_optical_flow_async");
}

// ---- flow batch ------------------------------------------------------------------------------------
// the members' passes must be the same launches: same flow geometry, radius and kernel plan, on one device
static int checkMembers(hrb_ofc* const* m, int n, const char* fn) {
    const hrb_ofc* a = m[0];
    for (int k = 1; k < n; ++k) {
        const hrb_ofc* b = m[k];
        const char* f = a->frameWidth != b->frameWidth           ? "frame_width"
                        : a->frameHeight != b->frameHeight       ? "frame_height"
                        : a->resScalar != b->resScalar           ? "res_scalar"
                        : a->searchRadius != b->searchRadius     ? "search_radius"
                        : a->searchVariant != b->searchVariant   ? "search_variant"
                        : a->device != b->device                 ? "device"
                                                                 : nullptr;
        if (f) {
            setLastError("[hopperrender_b200] %s: member %d differs from member 0 in %s", fn, k, f);
            return HRB_ERR_INVALID_ARG;
        }
    }
    return HRB_OK;
}

int hrb_flow_batch_create(hrb_flow_batch** out, hrb_ofc* const* members, int n) {
    HRB_REQUIRE(out && members, "null argument");
    *out = nullptr;
    HRB_REQUIRE(n >= 1 && n <= HRB_FLOW_BATCH_MAX, "member count outside 1..64");
    for (int k = 0; k < n; ++k) {
        HRB_REQUIRE(members[k], "null handle");
        for (int j = 0; j < k; ++j) HRB_REQUIRE(members[j] != members[k], "a handle appears twice");
    }
    for (int k = 0; k < n; ++k)
        if (delivering(members[k], __func__)) return HRB_ERR_STATE;
    const int rc = checkMembers(members, n, "hrb_flow_batch_create");
    if (rc) return rc;
    hrb_flow_batch* b = new (std::nothrow) hrb_flow_batch();
    HRB_REQUIRE(b, "out of host memory");
    b->member.assign(members, members + n);
    for (hrb_ofc* h : b->member) h->groups++;
    b->device = members[0]->device;
    int prioLow = 0, prioHigh = 0;
    cudaError_t e = cudaSetDevice(b->device);
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prioLow, &prioHigh);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&b->stream, cudaStreamNonBlocking, prioHigh);  // as the members' flow streams
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->done, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        setLastError("[hopperrender_b200] CUDA error %d (%s) in hrb_flow_batch_create", (int)e, cudaGetErrorString(e));
        hrb_flow_batch_destroy(b);
        return HRB_ERR_CUDA;
    }
    *out = b;
    return HRB_OK;
}

void hrb_flow_batch_destroy(hrb_flow_batch* b) {
    if (!b) return;
    for (hrb_ofc* h : b->member) h->groups--;
    cudaSetDevice(b->device);
    if (b->stream) {
        cudaStreamSynchronize(b->stream);
        cudaStreamDestroy(b->stream);
    }
    if (b->done) cudaEventDestroy(b->done);
    delete b;
}

// The ladder of every member on the batch's stream, forked behind each member's compute stream.  A member that would
// have forked on its own (asynchronous, flow overlap on, no taps) is joined through its flowJoinEvent like after its own
// calculate_optical_flow_async; every other member's compute stream waits for the batch at once.
static int batchCalculate(hrb_flow_batch* b, bool async, const char* fn) {
    Shards s(b);
    int rc = checkMembers(s.h, s.n, fn);
    if (rc) return rc;
    for (int k = 0; k < s.n; ++k)
        if (s.h[k]->prof.on || s.h[k]->dbgDev) {
            setLastError("[hopperrender_b200] %s: the profile and the debug timeline are not available on a batched calculate (switch them off on every member)", fn);
            return HRB_ERR_STATE;
        }
    HRB_CUDA(cudaSetDevice(b->device));
    cudaStream_t compute[HRB_FLOW_BATCH_MAX];
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        rc = joinFlow(h);
        if (rc) return rc;
        // the ingest of the member's newest frame and the last readers of the flow buffer it overwrites
        HRB_CUDA(cudaEventRecord(h->flowForkEvent, h->stream));
        HRB_CUDA(cudaStreamWaitEvent(b->stream, h->flowForkEvent, 0));
    }
    for (int k = 0; k < s.n; ++k) {
        compute[k] = s.h[k]->stream;
        s.h[k]->stream = b->stream;
    }
    rc = enqueueFlow(s);
    for (int k = 0; k < s.n; ++k) s.h[k]->stream = compute[k];
    if (rc) return rc;
    HRB_CUDA(cudaEventRecord(b->done, b->stream));
    for (int k = 0; k < s.n; ++k) {
        hrb_ofc* h = s.h[k];
        if (async && h->flowOverlap && !h->tapMode) {
            HRB_CUDA(cudaEventRecord(h->flowJoinEvent, b->stream));
            h->flowJoinPending = true;
            h->updatesSinceFlow = 0;
        } else {
            HRB_CUDA(cudaStreamWaitEvent(h->stream, b->done, 0));
        }
    }
    for (int k = 0; k < s.n && !async && !rc; ++k) rc = resolveFlow(s.h[k]);
    return rc;
}

int hrb_flow_batch_calculate_optical_flow(hrb_flow_batch* b) {
    HRB_REQUIRE(b, "null handle");
    return batchCalculate(b, false, "hrb_flow_batch_calculate_optical_flow");
}

int hrb_flow_batch_calculate_optical_flow_async(hrb_flow_batch* b) {
    HRB_REQUIRE(b, "null handle");
    return batchCalculate(b, true, "hrb_flow_batch_calculate_optical_flow_async");
}

// ---- delivery loop ---------------------------------------------------------------------------------
}  // extern "C"

// DeliverToRenderer's state (CHopperRender, HopperRender.cpp:944-1211) over one handle.  The host keeps everything that
// needs no delta value: the blending scalar, the interpolation state, and the frame numbers of the delta history with
// their pruning; the deltas themselves live in a device ring, appended and read by the decision kernel.
struct hrb_delivery {
    enum { Deactivated = 0, NotNeeded = 1, Active = 2 };  // ActiveState, HopperRender.h:20-25
    static constexpr int kRing = 16;  // device delta ring and kept outcomes; the rule reads at most 12 entries
    hrb_ofc* h = nullptr;
    hrb_delivery_desc desc{};
    int state = Deactivated;          // m_iIntActiveState
    long long playback = 0;           // m_rtCurrPlaybackFrameTime
    double blend = 0.0;               // m_dBlendingScalar
    std::deque<long long> history;    // frame numbers of frameDeltaHistory; entry k's delta is ring[(appends - size + k) % 16]
    unsigned long long appends = 0;   // deltas appended to the ring so far
    unsigned long long steps = 0;
    double warpTime = 0.0;            // GPU time of the warps / copy of the newest finished step (auto-tuner)
    bool timing = false;              // tBegin / tEnd hold a step not yet read
    uint32_t* ringDev = nullptr;
    uint32_t* gateDev = nullptr;
    DeliveryRecord* recDev = nullptr;   // [kRing], step s in s % kRing
    DeliveryRecord* recHost = nullptr;  // pinned copy of recDev
    cudaEvent_t recEvent[kRing] = {};
    cudaEvent_t pass0 = nullptr, tBegin = nullptr, tEnd = nullptr;
};

namespace hrb {

// m_iNumIntFrames, HopperRender.cpp:945
static int numIntFrames(double blend, long long target, long long playback) {
    return (int)std::max(std::ceil((1.0 - blend) / ((double)target / (double)playback)), 1.0);
}

// HopperRender.cpp:1192-1197
static double advanceBlend(double blend, long long target, long long playback) {
    blend += (double)target / (double)playback;
    if (blend >= 1.0) blend -= 1.0;
    return blend;
}

// The largest step the settings can produce (the blending scalar is >= 0, and the count falls as it grows).
static int checkCount(int state, long long target, long long playback, const char* fn) {
    if (state == hrb_delivery::Active && numIntFrames(0.0, target, playback) > HRB_DELIVERY_MAX_FRAMES) {
        setLastError("[hopperrender_b200] %s: a frame-time ratio of %lld / %lld needs more than %d output frames per source frame", fn, target, playback,
                     HRB_DELIVERY_MAX_FRAMES);
        return HRB_ERR_INVALID_ARG;
    }
    return HRB_OK;
}

static int checkDesc(const hrb_delivery_desc* d, const char* fn) {
    if (d->frame_output_mode < 0 || d->frame_output_mode > 6) {
        setLastError("[hopperrender_b200] %s: frame_output_mode outside 0..6", fn);
        return HRB_ERR_INVALID_ARG;
    }
    if (d->source_frame_time <= 0 || d->target_frame_time <= 0) {
        setLastError("[hopperrender_b200] %s: frame times must be positive", fn);
        return HRB_ERR_INVALID_ARG;
    }
    return HRB_OK;
}

// UpdateInterpolationStatus, HopperRender.cpp:819-831
static void updateInterpolationStatus(hrb_delivery* d) {
    if (d->state && d->playback > d->desc.target_frame_time)
        d->state = hrb_delivery::Active;
    else if (d->state)
        d->state = hrb_delivery::NotNeeded;
    d->history.clear();
}

static int deliveryCount(const hrb_delivery* d) {
    return d->state == hrb_delivery::Active ? numIntFrames(d->blend, d->desc.target_frame_time, d->playback) : 1;
}

// autoAdjustSettings, HopperRender.cpp:1438-1463, on the newest finished flow and the newest finished step's outputs
static int autoAdjust(hrb_delivery* d) {
    hrb_ofc* h = d->h;
    int rc = resolveFinishedFlows(h);
    if (rc) return rc;
    if (d->timing) {
        const cudaError_t q = cudaEventQuery(d->tEnd);
        if (q == cudaSuccess) {
            float ms = 0;
            HRB_CUDA(cudaEventElapsedTime(&ms, d->tBegin, d->tEnd));
            d->warpTime = (double)ms / 1e3;
            d->timing = false;
        } else if (q == cudaErrorNotReady) {
            cudaGetLastError();  // still running: the previous measurement stands
        } else {
            HRB_CUDA(q);
        }
    }
    const double sourceFrameTime = (double)d->playback / 10000000.0;
    const double currMax = h->ofcCalcTime + d->warpTime;
    if (currMax * 1.4 > sourceFrameTime) {  // UPPER_PERF_BUFFER, config.h:14
        if (h->searchRadius > 5) h->searchRadius--;
    } else if (currMax * 1.6 < sourceFrameTime) {  // LOWER_PERF_BUFFER, config.h:15
        if (h->searchRadius < 16) h->searchRadius++;
    }
    return HRB_OK;
}

// One DeliverToRenderer call: into ring slots outCur .. outCur+n-1 (dst null) or into dst[0..n-1].
static int deliveryStep(hrb_delivery* d, const hrb_frame_planes* dst, int capacity, hrb_delivery_frame* frames, int* nOut, const char* fn) {
    hrb_ofc* h = d->h;
    const int n = deliveryCount(d);
    if (capacity < n) {
        setLastError("[hopperrender_b200] %s: the step produces %d frames, capacity is %d", fn, n, capacity);
        return HRB_ERR_INVALID_ARG;
    }
    const bool active = d->state == hrb_delivery::Active;
    double blends[HRB_DELIVERY_MAX_FRAMES];
    float ts[HRB_DELIVERY_MAX_FRAMES];
    for (int i = 0; i < n; ++i) {
        blends[i] = i == 0 ? d->blend : active ? advanceBlend(blends[i - 1], d->desc.target_frame_time, d->playback) : d->blend;
        ts[i] = (float)blends[i];
        if (ts[i] > 1.0f) {  // opticalFlowCalcSDR.cpp:143-146
            setLastError("[HopperRender] Error in function warpFrames: Blending scalar is greater than 1.0");
            return HRB_ERR_BLEND_RANGE;
        }
    }
    if (dst) {
        const int rc = checkFrames(h, dst, n, true, fn);
        if (rc) return rc;
    }
    HRB_CUDA(cudaSetDevice(h->device));
    if (d->desc.auto_adjust) {
        const int rc = autoAdjust(d);
        if (rc) return rc;
    }
    const unsigned fc = h->frameCount;
    const bool flow = active && fc >= 3;
    if (flow) {
        const int rc = calculateFlow(Shards(h), true);
        if (rc) return rc;
        // The decision reads rawDeltaDev once pass 0 has written it.  The next flow is forked behind the compute stream,
        // i.e. behind the decision kernel enqueued below, so it cannot overwrite rawDeltaDev before the kernel has read it.
        HRB_CUDA(cudaStreamWaitEvent(h->stream, d->pass0, 0));
        d->appends++;
        // frameDeltaHistory, HopperRender.cpp:959-973: entries older than 3 s of source frames leave
        const long long framesIn3s = (long long)(3.0 * 10000000.0 / (double)d->desc.source_frame_time);
        d->history.push_back(fc);
        while (!d->history.empty() && (long long)fc - d->history.front() > framesIn3s) d->history.pop_front();
    }
    const unsigned long long step = d->steps;
    const int rec = (int)(step % hrb_delivery::kRing);
    DeliveryDecision dd;
    dd.rawDelta = h->rawDeltaDev;
    dd.divisor = (unsigned)(h->flowHeight * h->flowWidth * (h->hdr ? 6 : 10));
    dd.ring = d->ringDev;
    dd.append = flow ? 1 : 0;
    dd.slot = (int)((d->appends + hrb_delivery::kRing - 1) % hrb_delivery::kRing);
    dd.n = (int)d->history.size();
    dd.count = dd.n >= 3 ? std::min(dd.n - 2, 10) : 0;
    dd.threshold = d->desc.scene_change_threshold;
    dd.copy = flow ? 0 : 1;
    dd.gate = d->gateDev;
    dd.out = d->recDev + rec;
    int rc = launchDeliveryDecision(h, dd);
    if (rc) return rc;
    HRB_CUDA(cudaMemcpyAsync(d->recHost + rec, d->recDev + rec, sizeof(DeliveryRecord), cudaMemcpyDeviceToHost, h->stream));
    HRB_CUDA(cudaEventRecord(d->recEvent[rec], h->stream));

    // the outputs: warps under "no scene change" and copies under "scene change", or copies the host already knows of
    hrb_frame_planes outs[HRB_DELIVERY_MAX_FRAMES];
    if (!dst) {
        rc = beginOutput(h);  // waits for the download of the first slot, starts the warp timer
        if (rc) return rc;
        for (int i = 0; i < n; ++i) {
            const int slot = (h->outCur + i) % hrb_ofc::kOutRing;
            if (i) HRB_CUDA(cudaStreamWaitEvent(h->stream, h->outFree[slot], 0));
            outs[i] = ringPlanes(h, slot);
        }
        dst = outs;
    }
    HRB_CUDA(cudaEventRecord(d->tBegin, h->stream));
    const int copyIndex = fc >= 3 ? 0 : fc >= 2 ? 1 : 2;  // opticalFlowCalcSDR.cpp:173
    if (flow) {
        for (int i0 = 0; i0 < n && !rc; i0 += HRB_WARP_BATCH_MAX)
            rc = launchWarpFrames(h, std::min(n - i0, HRB_WARP_BATCH_MAX), ts + i0, dst + i0, d->desc.frame_output_mode, d->gateDev, 0);
        if (!rc) rc = launchCopyFrame(h, copyIndex, dst, n, d->gateDev, 1);
    } else {
        rc = launchCopyFrame(h, copyIndex, dst, n);
    }
    if (rc) return rc;
    HRB_CUDA(cudaEventRecord(d->tEnd, h->stream));
    d->timing = true;
    if (dst == outs)
        for (int i = 0; i < n; ++i) HRB_CUDA(cudaEventRecord(h->outReady[(h->outCur + i) % hrb_ofc::kOutRing], h->stream));

    for (int i = 0; i < n; ++i) frames[i] = hrb_delivery_frame{fc, i, blends[i], step};
    if (active) d->blend = advanceBlend(blends[n - 1], d->desc.target_frame_time, d->playback);
    d->steps++;
    *nOut = n;
    return HRB_OK;
}

}  // namespace hrb

extern "C" {

void hrb_delivery_destroy(hrb_delivery* d) {
    if (!d) return;
    hrb_ofc* h = d->h;
    if (h) {
        cudaSetDevice(h->device);
        cudaStreamSynchronize(h->flowStream);
        cudaStreamSynchronize(h->stream);
        // the graphs that record this delivery's pass-0 event go with it
        for (auto& g : h->flowGraphs)
            if (g.pass0 == d->pass0 && g.exec) {
                cudaGraphExecDestroy(g.exec);
                g.exec = nullptr;
            }
        h->flowGraphs.erase(std::remove_if(h->flowGraphs.begin(), h->flowGraphs.end(), [](const hrb_ofc::FlowGraph& g) { return !g.exec; }), h->flowGraphs.end());
        if (h->delivery == d) {
            h->delivery = nullptr;
            h->pass0Event = nullptr;
        }
    }
    cudaFree(d->ringDev);
    cudaFree(d->gateDev);
    cudaFree(d->recDev);
    if (d->recHost) cudaFreeHost(d->recHost);
    for (auto e : d->recEvent)
        if (e) cudaEventDestroy(e);
    if (d->pass0) cudaEventDestroy(d->pass0);
    if (d->tBegin) cudaEventDestroy(d->tBegin);
    if (d->tEnd) cudaEventDestroy(d->tEnd);
    delete d;
}

int hrb_delivery_create(hrb_delivery** out, hrb_ofc* h, const hrb_delivery_desc* desc) {
    HRB_REQUIRE(out && desc, "null argument");
    *out = nullptr;
    int rc = checkDesc(desc, __func__);
    if (!rc) rc = checkCount(desc->active ? hrb_delivery::Active : hrb_delivery::Deactivated, desc->target_frame_time, desc->source_frame_time, __func__);
    if (rc) return rc;
    HRB_REQUIRE(h, "null handle");
    if (h->delivery || h->groups) {
        setLastError("[hopperrender_b200] %s: the handle already has a delivery, or belongs to a split group or a flow batch", __func__);
        return HRB_ERR_STATE;
    }
    HRB_CUDA(cudaSetDevice(h->device));
    hrb_delivery* d = new (std::nothrow) hrb_delivery();
    HRB_REQUIRE(d, "out of host memory");
    d->desc = *desc;
    d->state = desc->active ? hrb_delivery::Active : hrb_delivery::Deactivated;  // as the filter starts: no status update yet
    d->playback = desc->source_frame_time;
    cudaError_t e = cudaMalloc(&d->ringDev, hrb_delivery::kRing * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemsetAsync(d->ringDev, 0, hrb_delivery::kRing * sizeof(uint32_t), h->stream);
    if (e == cudaSuccess) e = cudaMalloc(&d->gateDev, sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&d->recDev, hrb_delivery::kRing * sizeof(DeliveryRecord));
    if (e == cudaSuccess) e = cudaMallocHost(&d->recHost, hrb_delivery::kRing * sizeof(DeliveryRecord));
    for (auto& ev : d->recEvent)
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d->pass0, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&d->tBegin);
    if (e == cudaSuccess) e = cudaEventCreate(&d->tEnd);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) {
        setLastError("[hopperrender_b200] CUDA error %d (%s) in hrb_delivery_create", (int)e, cudaGetErrorString(e));
        hrb_delivery_destroy(d);
        return HRB_ERR_CUDA;
    }
    d->h = h;
    h->delivery = d;
    h->pass0Event = d->pass0;
    *out = d;
    return HRB_OK;
}

int hrb_delivery_next_count(hrb_delivery* d, int* n) {
    HRB_REQUIRE(d && n, "null argument");
    *n = deliveryCount(d);
    return HRB_OK;
}

int hrb_delivery_step(hrb_delivery* d, hrb_delivery_frame* frames, int capacity, int* n) {
    HRB_REQUIRE(d && frames && n, "null argument");
    return deliveryStep(d, nullptr, capacity, frames, n, __func__);
}

int hrb_delivery_step_to(hrb_delivery* d, const hrb_frame_planes* dst, int capacity, hrb_delivery_frame* frames, int* n) {
    HRB_REQUIRE(d && dst && frames && n, "null argument");
    return deliveryStep(d, dst, capacity, frames, n, __func__);
}

int hrb_delivery_outcome_of(hrb_delivery* d, unsigned long long step, int wait, hrb_delivery_outcome* out) {
    HRB_REQUIRE(d && out, "null argument");
    HRB_REQUIRE(step < d->steps && step + hrb_delivery::kRing >= d->steps, "step not among the last 16 steps");
    HRB_CUDA(cudaSetDevice(d->h->device));
    const int rec = (int)(step % hrb_delivery::kRing);
    if (wait) {
        HRB_CUDA(cudaEventSynchronize(d->recEvent[rec]));
    } else {
        const cudaError_t q = cudaEventQuery(d->recEvent[rec]);
        if (q == cudaErrorNotReady) {
            cudaGetLastError();
            setLastError("[hopperrender_b200] %s: the decision of step %llu is still in flight", __func__, step);
            return HRB_ERR_STATE;
        }
        HRB_CUDA(q);
    }
    const DeliveryRecord& r = d->recHost[rec];
    out->warped = r.warped;
    out->scene_change = r.sceneChange;
    out->delta1 = r.d1;
    out->delta2 = r.d2;
    out->frame_delta = r.frameDelta;
    return HRB_OK;
}

int hrb_delivery_set(hrb_delivery* d, const hrb_delivery_desc* desc) {
    HRB_REQUIRE(d && desc, "null argument");
    int rc = checkDesc(desc, __func__);
    if (rc) return rc;
    HRB_REQUIRE(desc->source_frame_time == d->desc.source_frame_time, "source_frame_time differs from the delivery's (a new source rate is a new delivery)");
    // UpdateUserSettings, HopperRender.cpp:1355-1390, then UpdateInterpolationStatus
    const int state = !desc->active ? (int)hrb_delivery::Deactivated : d->state ? d->state : (int)hrb_delivery::Active;
    const int after = state && d->playback > desc->target_frame_time ? (int)hrb_delivery::Active : state ? (int)hrb_delivery::NotNeeded : state;
    rc = checkCount(after, desc->target_frame_time, d->playback, __func__);
    if (rc) return rc;
    d->desc = *desc;
    d->state = state;
    updateInterpolationStatus(d);
    return HRB_OK;
}

int hrb_delivery_new_segment(hrb_delivery* d, double rate) {
    HRB_REQUIRE(d, "null argument");
    HRB_REQUIRE(rate > 0.0 && std::isfinite(rate), "rate must be a positive number");
    // NewSegment, HopperRender.cpp:834-844
    const long long playback = (long long)((double)d->desc.source_frame_time * (1.0 / rate));
    HRB_REQUIRE(playback > 0, "rate too high for the source frame time");
    const int after = d->state && playback > d->desc.target_frame_time ? (int)hrb_delivery::Active : d->state ? (int)hrb_delivery::NotNeeded : d->state;
    const int rc = checkCount(after, d->desc.target_frame_time, playback, __func__);
    if (rc) return rc;
    d->playback = playback;
    updateInterpolationStatus(d);
    d->h->frameCount = 0;
    return HRB_OK;
}

uint64_t hrb_kernel_launch_count(void) { return g_launchCount.load(std::memory_order_relaxed); }

int hrb_microbench_sad_peak(int device_ordinal, double* giga_absdiff_per_s) {
    HRB_REQUIRE(giga_absdiff_per_s, "null argument");
    return microbenchSad(device_ordinal, giga_absdiff_per_s);
}

const char* hrb_last_error(void) { return t_lastError.c_str(); }
const char* hrb_version(void) { return "hopperrender_b200 0.1 (sm_100a)"; }

}  // extern "C"
