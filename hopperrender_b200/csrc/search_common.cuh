// search_common.cuh — device helpers shared by the search kernels (kernels_search.cu, kernels_search_big.cu).
#pragma once
#include "hrb_internal.cuh"

namespace hrb {
namespace {

constexpr int TILE = 32;  // flow pixels per CTA tile edge

// sq(d) = d*d*sign(d) — calcDeltaSumsKernelSDR.h:70-71 / adjustOffsetArrayKernelSDR.h:18
__host__ __device__ constexpr int signedSquare(int d) { return d * d * (d > 0 ? 1 : -1); }
template <int R> __host__ __device__ constexpr int candOffset(int z) { return signedSquare(z - R / 2); }

// single reflection + clamp — calcDeltaSumsKernelSDR.h:86-95
__device__ __forceinline__ int mirrorSearch(int n, int dim) {
    if (n >= dim) {
        n = dim - (n - dim + 1);
    } else if (n < 0) {
        n = -n - 1;
    }
    return min(max(n, 0), dim - 1);
}

// d = sum_i |a.b[i] - b.b[i]| + c : one VABSDIFF4.U8.ACC
__device__ __forceinline__ uint32_t sad4(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// A pass seen along its candidate axis: v is the axis the candidates move along and the row index of the planes in
// use, u the contiguous axis.  Y steps read the row-major planes (u = x, v = y); X steps read the TRANSPOSED planes
// (u = y, v = x).  Both steps therefore run the same code and every warp access is a contiguous row segment.  In
// either orientation the chroma bytes that belong to luma sample (v, u) are c[(v >> 1) * pitch + (u & ~1)] and + 1
// (hrb_internal.cuh, SearchArgs).  Window bookkeeping (offset arrays, biases) stays in (x, y).
//
// The pass covers u in [u0, lu) and v in [v0, lv) (passRange): the whole flow field, or on a shard of a split search the
// flow rows [rowBegin, rowEnd) — along v in Y steps, along u in X steps.  Grids start at (u0, v0) (the small-window
// kernel's at 0: its CTAs before the stripe return at once); lu / lv bound the pixels and windows a CTA computes, so a
// tile that runs past the stripe end is masked like one at the field's end.
// Everything else stays frame-relative: dimU / dimV are the frame, a stripe edge inside the frame is NOT a mirror edge,
// and staging reads the rows beyond a stripe edge from the frame like any other rows.
template <int STEP> struct View {
    const uint8_t* __restrict__ y1;
    const uint8_t* __restrict__ c1;
    const uint8_t* __restrict__ y2;
    const uint8_t* __restrict__ c2;
    int pitch, dimU, dimV, u0, lu, v0, lv;
    __device__ __forceinline__ explicit View(const SearchArgs& a) {
        if (STEP == 1) {
            y1 = a.y1; c1 = a.c1; y2 = a.y2; c2 = a.c2; pitch = a.pitch; dimU = a.W; dimV = a.H;
        } else {
            y1 = a.yT1; c1 = a.cT1; y2 = a.yT2; c2 = a.cT2; pitch = a.pitchT; dimU = a.H; dimV = a.W;
        }
        const PassRange r = passRange(a, STEP);
        u0 = r.u0; lu = r.lu; v0 = r.v0; lv = r.lv;
    }
    static __device__ __forceinline__ int wx(int wu, int wv) { return STEP == 1 ? wu : wv; }
    static __device__ __forceinline__ int wy(int wu, int wv) { return STEP == 1 ? wv : wu; }
    static __device__ __forceinline__ int ou(int ox, int oy) { return STEP == 1 ? ox : oy; }
    static __device__ __forceinline__ int ov(int ox, int oy) { return STEP == 1 ? oy : ox; }
};

// base + rows * pitch (bytes) as ONE IMAD.WIDE on the FMA pipe: keeps the per-fetch address arithmetic off the
// ALU pipe, which the VABSDIFF4 stream saturates (nvcc otherwise emits 4-5 ALU instructions per row-strided fetch).
__device__ __forceinline__ const uint8_t* rowPtr(const uint8_t* base, int pitchBytes, int rows) {
    unsigned long long r;
    asm("mad.wide.s32 %0, %1, %2, %3;" : "=l"(r) : "r"(pitchBytes), "r"(rows), "l"((unsigned long long)base));
    return reinterpret_cast<const uint8_t*>(r);
}

// The reference's three samples of one pixel as a word {Y, U, V, 0}: one VABSDIFF4 on two such words is its 3-term
// delta (calcDeltaSumsKernelSDR.h:98-100).  (v, u) must be inside the frame.
__device__ __forceinline__ uint32_t fetchPixel(const uint8_t* __restrict__ y, const uint8_t* __restrict__ c, int pitch, int v, int u) {
    const uint32_t l = __ldg(rowPtr(y, pitch, v) + u);
    const uint32_t uv = __ldg(reinterpret_cast<const uint16_t*>(rowPtr(c, pitch, v >> 1) + (u & ~1)));
    return l | (uv << 8);
}

// Four horizontally adjacent pixels (u0 a multiple of 4) as four {Y, U, V, 0} words, from one luma word and one
// chroma word: 6 PRMT.
__device__ __forceinline__ void expand4(uint32_t yw, uint32_t cw, uint32_t (&w)[4]) {
    const uint32_t cA = __byte_perm(cw, 0u, 0x4104);  // {0, U0, V0, 0}
    const uint32_t cB = __byte_perm(cw, 0u, 0x4324);  // {0, U1, V1, 0}
    w[0] = __byte_perm(yw, cA, 0x7650);
    w[1] = __byte_perm(yw, cA, 0x7651);
    w[2] = __byte_perm(yw, cB, 0x7652);
    w[3] = __byte_perm(yw, cB, 0x7653);
}

// 16-byte asynchronous copy global -> shared (LDGSTS): no register staging, so a thread keeps all its copies in
// flight at once; completed by cpAsyncWaitAll() + a barrier.
__device__ __forceinline__ void cpAsync16(void* smemDst, const void* gmemSrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smemDst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmemSrc) : "memory");
}
__device__ __forceinline__ void cpAsyncWaitAll() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

struct WindowCtx {
    int o;          // current offset of the window along the axis of this step
    uint32_t nw;    // in-range flow pixels of the window
    int nb[4];      // neighbour offsets along the axis (down, right, left, up)
    bool useNb;
};

template <int STEP> __device__ __forceinline__ void loadWindowOffsets(const SearchArgs& a, int wx, int wy, int& ox, int& oy) {
    const int pidx = (wy >> 1) * a.prevNWx + (wx >> 1);
    if (STEP == 0) {
        ox = a.prevX ? a.prevX[pidx] : 0;
    } else {
        ox = a.curX[wy * a.nWx + wx];
    }
    oy = a.prevY ? a.prevY[pidx] : 0;
}

template <int STEP> __device__ __forceinline__ WindowCtx loadWindowCtx(const SearchArgs& a, int wx, int wy, int ox, int oy) {
    WindowCtx c;
    c.o = STEP == 0 ? ox : oy;
    const int x0 = wx << a.wsLog2, y0 = wy << a.wsLog2;
    c.nw = (uint32_t)((min(x0 + a.ws, a.lw) - x0) * (min(y0 + a.ws, a.lh) - y0));
    c.useNb = a.iteration >= 4;  // FIRST_NEIGHBOR_ITERATION, calcDeltaSumsKernelSDR.h:3,112
    if (c.useNb) {
        // neighbours at +-2*ws flow pixels, clamped to the array (calcDeltaSumsKernelSDR.h:6-9,114-131) = window
        // index +-2 clamped; their offsets still have parent-level granularity.
        const int16_t* __restrict__ p = STEP == 0 ? a.prevX : a.prevY;
        const int wyD = min(wy + 2, a.nWy - 1), wyU = max(wy - 2, 0);
        const int wxR = min(wx + 2, a.nWx - 1), wxL = max(wx - 2, 0);
        c.nb[0] = p[(wyD >> 1) * a.prevNWx + (wx >> 1)];
        c.nb[1] = p[(wy >> 1) * a.prevNWx + (wxR >> 1)];
        c.nb[2] = p[(wy >> 1) * a.prevNWx + (wxL >> 1)];
        c.nb[3] = p[(wyU >> 1) * a.prevNWx + (wx >> 1)];
    } else {
        c.nb[0] = c.nb[1] = c.nb[2] = c.nb[3] = 0;
    }
    return c;
}

// Window sum of layer z in the reference's terms: sum over the window's pixels of
// (delta << deltaScalar) + offsetBias + (neighborBias << neighborBiasScalar)   (calcDeltaSumsKernelSDR.h:101-151)
template <int R> __device__ __forceinline__ uint32_t windowTotal(const SearchArgs& a, const WindowCtx& c, uint32_t sad, int z) {
    const int cand = (int)(short)(c.o + signedSquare(z - R / 2));
    uint32_t bias = (uint32_t)abs(cand);
    if (c.useNb) {
        const uint32_t nbs = (uint32_t)abs(c.nb[0] - cand) + (uint32_t)abs(c.nb[1] - cand) + (uint32_t)abs(c.nb[2] - cand) + (uint32_t)abs(c.nb[3] - cand);
        bias += nbs << a.neighborBiasScalar;
    }
    return (sad << a.deltaScalar) + c.nw * bias;
}

// determineLowestLayerKernelSDR.h:17-25 ordering: lowest sum, ties -> lowest layer
__device__ __forceinline__ unsigned long long layerKey(uint32_t total, int z) { return ((unsigned long long)total << 32) | (unsigned)z; }

// adjustOffsetArrayKernelSDR.h:14-18 applied to the window, plus the taps
template <int R, int STEP> __device__ __forceinline__ void commitWindow(const SearchArgs& a, int wx, int wy, int o, int bestLayer) {
    const int16_t n = (int16_t)(o + signedSquare(bestLayer - R / 2));
    const int widx = wy * a.nWx + wx;
    if (STEP == 0)
        a.curX[widx] = n;
    else
        a.curY[widx] = n;
    if (a.tapLayer) a.tapLayer[widx] = (uint8_t)bestLayer;
}

template <int R> __device__ __forceinline__ void tapTotal(const SearchArgs& a, int wx, int wy, int z, uint32_t total) {
    if (a.tapSums) a.tapSums[((size_t)z * a.nWy + wy) * a.nWx + wx] = total;
    // m_totalFrameDelta's raw value: layer R/2-1 of the first window of the first pass (opticalFlowCalcSDR.cpp:92)
    if (a.rawDelta && wx == 0 && wy == 0 && z == R / 2 - 1) *a.rawDelta = total;
}

// Sequential finalize of one window whose R sums are in memory.
template <int R, int STEP> __device__ __forceinline__ void finalizeWindow(const SearchArgs& a, int wx, int wy, const uint32_t* sums) {
    int ox, oy;
    loadWindowOffsets<STEP>(a, wx, wy, ox, oy);
    const WindowCtx c = loadWindowCtx<STEP>(a, wx, wy, ox, oy);
    unsigned long long best = ~0ull;
#pragma unroll
    for (int z = 0; z < R; ++z) {
        const uint32_t total = windowTotal<R>(a, c, sums[z], z);
        tapTotal<R>(a, wx, wy, z, total);
        best = min(best, layerKey(total, z));
    }
    commitWindow<R, STEP>(a, wx, wy, c.o, (int)(best & 0xff));
}

// Butterfly stage of a recursive-halving reduction: lanes whose `upper` bit is clear keep the lower
// half of their N values, the others the upper half; each receives the partner's copy of what it keeps.
template <int N> __device__ __forceinline__ void bfly(uint32_t (&acc)[16], int mask, bool upper) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        const uint32_t send = upper ? acc[i] : acc[i + N / 2];
        const uint32_t keep = upper ? acc[i + N / 2] : acc[i];
        acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
    }
}

__device__ __forceinline__ unsigned long long shflXor64(unsigned long long v, int mask) {
    const unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, mask);
    const unsigned hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), mask);
    return ((unsigned long long)hi << 32) | lo;
}

}  // namespace
}  // namespace hrb
