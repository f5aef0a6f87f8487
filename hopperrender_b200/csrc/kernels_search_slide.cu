// kernels_search_slide.cu — the tile kernel: search passes for windows of 16 flow pixels and larger at full flow
// resolution (16 of the 22 passes at 4K; down to windows of 4 under search variant 2).  Same arithmetic as sadPassKernel
// (kernels_search.cu), different data movement.
//
// Data: the 8-bit planar search planes (luma + NV12-style chroma, see SearchArgs), so one VABSDIFF4 covers FOUR
// luma pixels, or the U,V samples of four pixels, instead of one pixel, and the two frames of a pass are 25 MB —
// they stay in the 126 MB L2 over the whole ladder.
//
// Work split (u = contiguous axis, v = candidate axis, see View): a CTA owns a tile of 128 (u) x 32*NWV (v) flow
// pixels; a warp owns 128 x 32 of it, a lane a column of 4 pixels (one word), which it walks in runs of
// RUN = min(ws, 32) rows (one window row per run).
//   * frame 1: one luma box and one chroma box per tile hold every sample any candidate of any window of the tile can
//     touch: tile + candidate span + the spread of the tile's window displacements (motion fields are smooth: a few
//     pixels).  The chroma box is one TMA copy (cp.async.bulk.tensor.2d issued by one elected thread, completion by
//     transaction count on an mbarrier); the luma rows are 144-160 bytes wide, where 16-byte cp.async copies issued by
//     all threads (arriving on a second mbarrier, cp.async.mbarrier.arrive.noinc) measured faster than a TMA box.  Boxes
//     start at the 16-byte boundary below the smallest displaced column (TMA needs that alignment); each lane re-aligns
//     its words with one funnel shift per sample.  Tiles whose boxes leave the frame are staged by cp.async through the
//     reference's mirror (calcDeltaSumsKernelSDR.h:86-95): mirrored ROW indices for the top / bottom edge, byte-reversed
//     16-byte chunks for the left / right edge (stageIssue / stageFixup).
//   * windows of a tile whose displacements differ by more than the box allows are handled in up to MAX_ROUNDS rounds
//     (each round stages the box of one group of windows); what is still left takes a per-pixel path.
//   * along v every lane slides over its staged column: each frame-1 sample is fetched ONCE and feeds every
//     (row, candidate) pair it belongs to (up to R of them), all register indices being compile-time.
//   * chroma: the U,V pair of luma (v, u) is c[v >> 1][u & ~1].  Along v, luma rows 2k and 2k+1 with displacement s
//     read chroma rows k + ((e + s) >> 1), e = 0, 1: the same row when s is even (one SAD, weight 2), two rows when
//     it is odd.  Along u, a displacement ou maps a pixel pair onto one chroma pair when ou is even (weight 2) and
//     onto two neighbouring pairs when it is odd (two passes over the staged rows, 2 bytes apart, weight 1 each).
//   * windows up to 32 pixels are reduced and finalized inside the warp (butterfly over the window's lanes), 64-pixel
//     windows inside the CTA, larger ones through R atomics per CTA into the per-window scratch: the last CTA of a
//     window (arrival ticket) finalizes it.  No fills, no extra launch.
//   * row stripes (split search, hrb_split): a sharded pass computes only the windows of flow rows [rowBegin, rowEnd).
//     The grid starts at the stripe's first row (v in Y steps, u in X steps) and tiles that run past the stripe end are
//     masked like tiles at the end of the field.  Borders stay frame-relative: a stripe edge inside the frame is not a
//     mirror edge, the `border` test and the staging are unchanged there, and boxes read the rows beyond the stripe from
//     the frame like any other rows.
#include <cuda.h>

#include <climits>
#include <cstring>
#include <mutex>

#include "search_common.cuh"

namespace hrb {

namespace {

template <int R> struct CandSpan {
    static constexpr int LO = candOffset<R>(0);
    static constexpr int HI = candOffset<R>(R - 1);
    static constexpr int SPAN = HI - LO;  // extra samples along the candidate axis
};

__host__ __device__ constexpr int floorHalf(int v) { return v >= 0 ? (v >> 1) : -((1 - v) >> 1); }
__host__ __device__ constexpr int align128(int v) { return (v + 127) & ~127; }
__host__ __device__ constexpr int ilog2c(int v) { return v <= 1 ? 0 : 1 + ilog2c(v >> 1); }

// window-size class WSC: 4, 8, 16, 32, 64 or 128 (= every window of 128 pixels and more)
template <int WSC> struct Cls {
    static constexpr int RUN = WSC < 32 ? WSC : 32;          // rows of one run (one window row)
    static constexpr int NRUN = 32 / RUN;                    // runs of a warp
    static constexpr int SEG = (WSC < 128 ? WSC : 128) / 4;  // lanes per window
    static constexpr bool SPREAD = WSC < 128;                // the windows of a tile may be displaced differently
    static constexpr int SU = SPREAD ? 12 : 0;               // displacement spread the boxes cover, along u ...
    static constexpr int SV = SPREAD ? 15 : 0;               // ... and along v
    static constexpr int BW = SPREAD ? 160 : 144;            // box width in bytes: 128 + 16-byte alignment slack + spread
    static constexpr int BWW = BW / 4;
};

// Launch-time geometry (host and device agree through this struct).
struct TileParams {
    int nwv;          // warps of a CTA = tile rows / 32
    int rowsY;        // luma rows of the staged box (cp.async, 16 bytes per copy)
    int boxHC;        // chroma rows of the staged box (one TMA box)
    int lumaBytes;    // shared-memory bytes of the luma rows (multiple of 128)
    int chromaBytes;
    int useTma;       // 0: stage with plain loads (A/B, and when no tensor map could be encoded)
    int forceSlow;    // 1: every tile takes the per-pixel path (A/B and parity coverage of that path)
};

// ---- mbarrier / TMA -------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbarInit(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarExpectTx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarWait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tmaLoad2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(dst)),
                 "l"(map), "r"(x), "r"(y), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}

// ---- the sliding loops ---------------------------------------------------------------------------------------------
// luma: acc[z] += sum over the run's rows p of SAD4(frame1 row p + d_z, frame2 row p); fetch(j) returns the lane's
// frame-1 word of staged row j = p + d_z - LO.  Samples no (row, candidate) pair uses are never fetched.
template <int R, int RUN, typename Fetch> __device__ __forceinline__ void slideLuma(uint32_t (&acc)[16], const uint32_t (&f2)[RUN], Fetch fetch) {
    constexpr int LO = CandSpan<R>::LO;
#pragma unroll
    for (int j = 0; j < RUN + CandSpan<R>::SPAN; ++j) {
        bool used = false;
#pragma unroll
        for (int z = 0; z < R; ++z) {
            const int p = j - (candOffset<R>(z) - LO);
            used = used || (p >= 0 && p < RUN);
        }
        if (!used) continue;
        const uint32_t f1 = fetch(j);
#pragma unroll
        for (int z = 0; z < R; ++z) {
            const int p = j - (candOffset<R>(z) - LO);
            if (p >= 0 && p < RUN) acc[z] = sad4(f1, f2[p], acc[z]);
        }
    }
}

// chroma: PI = parity of the window's displacement along v.  Luma rows 2k + e of the run with candidate z read
// staged chroma row k + floorHalf(e + PI + d_z) - AMIN; e = 0 and e = 1 coincide when PI + d_z is even (one SAD,
// the caller doubles the sum, chromaShift).
template <int R, int RUN, int PI, typename Fetch> __device__ __forceinline__ void slideChroma(uint32_t (&acc)[16], const uint32_t (&f2c)[RUN / 2], Fetch fetch) {
    constexpr int LO = CandSpan<R>::LO, HI = CandSpan<R>::HI;
    constexpr int AMIN = floorHalf(PI + LO);
    constexpr int CLEN = RUN / 2 + floorHalf(1 + PI + HI) - AMIN;
#pragma unroll
    for (int jc = 0; jc < CLEN; ++jc) {
        bool used = false;
#pragma unroll
        for (int z = 0; z < R; ++z) {
            const int k0 = jc - (floorHalf(PI + candOffset<R>(z)) - AMIN), k1 = jc - (floorHalf(1 + PI + candOffset<R>(z)) - AMIN);
            used = used || (k0 >= 0 && k0 < RUN / 2) || (k1 >= 0 && k1 < RUN / 2);
        }
        if (!used) continue;
        const uint32_t c1 = fetch(jc);
#pragma unroll
        for (int z = 0; z < R; ++z) {
            const int a0 = floorHalf(PI + candOffset<R>(z)) - AMIN;
            const int a1 = floorHalf(1 + PI + candOffset<R>(z)) - AMIN;
            const int k0 = jc - a0, k1 = jc - a1;
            if (k0 >= 0 && k0 < RUN / 2) acc[z] = sad4(c1, f2c[k0], acc[z]);
            if (a1 != a0 && k1 >= 0 && k1 < RUN / 2) acc[z] = sad4(c1, f2c[k1], acc[z]);
        }
    }
}
template <int R> __device__ __forceinline__ int chromaShift(int pi, int z) { return ((pi + candOffset<R>(z)) & 1) ? 0 : 1; }

// Staging of a box with cp.async, through the reference's mirror (calcDeltaSumsKernelSDR.h:86-95): rows [r0, r1) x
// the 16-byte chunks [kLo, kLo + nK) of the box; box row r / byte c <-> plane row rb + r / byte ca + c (ca a multiple
// of 16).  Every chunk is one copy — all copies of a thread in flight at once, and no dependent global load, which
// would queue behind the staging traffic of the whole grid: rows go through the mirrored row index, chunks left / right
// of the plane come from their mirror chunk, which arrives in forward order and is reversed in shared memory afterwards
// (stageFixup, after the copies have landed).  Chunks that have no mirror chunk (plane width not a multiple of 16,
// displacements beyond the frame size) are filled byte by byte in stageFixup.  One function for the luma box of every
// tile and for the chroma box wherever TMA does not apply, so that the rarely taken paths run instructions that are
// already in the instruction cache (a cold path fetches its code through the same congested memory system).
struct BoxGeom {
    uint8_t* buf;
    const uint8_t* plane;
    int bw, pitch, dimU, dimV, rb, r0, r1, kLo, nK, nCh, pc0;
    bool whole;
    __device__ __forceinline__ BoxGeom(uint8_t* buf_, int bw_, const uint8_t* plane_, int pitch_, int dimU_, int dimV_, int rb_, int ca, int r0_, int r1_, int c0, int c1)
        : buf(buf_), plane(plane_), bw(bw_), pitch(pitch_), dimU(dimU_), dimV(dimV_), rb(rb_), r0(r0_), r1(r1_) {
        kLo = c0 >> 4;
        nK = max(((c1 + 15) >> 4) - kLo, 0);
        nCh = dimU >> 4;           // whole chunks of a plane row
        pc0 = (ca >> 4) + kLo;     // plane chunk of box chunk kLo
        whole = (dimU & 15) == 0;
    }
    __device__ __forceinline__ int srcChunk(int pc) const { return pc < 0 ? -pc - 1 : (pc >= nCh ? 2 * nCh - pc - 1 : pc); }
    __device__ __forceinline__ bool direct(int pc) const {  // the chunk is a (possibly reversed) copy of a plane chunk
        const int sc = srcChunk(pc);
        return whole ? (sc >= 0 && sc < nCh) : (pc >= 0 && pc < nCh);
    }
    __device__ __forceinline__ bool outsideChunks() const { return pc0 < 0 || pc0 + nK > nCh; }
    // the box reaches the last, partial chunk of a row (plane width not a multiple of 16): stageIssue leaves it to
    // stageFixup even where the tile reads only in-plane bytes of it
    __device__ __forceinline__ bool partialTail() const { return !whole && pc0 + nK > nCh; }
};

__device__ __noinline__ void stageIssue(const BoxGeom g, int tid, int nThreads) {
    const int n = (g.r1 - g.r0) * g.nK;
#pragma unroll 1
    for (int i = tid; i < n; i += nThreads) {
        const int rr = i / g.nK, k = i - rr * g.nK;
        const int r = g.r0 + rr, pc = g.pc0 + k;
        if (g.direct(pc)) cpAsync16(g.buf + r * g.bw + 16 * (g.kLo + k), rowPtr(g.plane, g.pitch, mirrorSearch(g.rb + r, g.dimV)) + 16 * g.srcChunk(pc));
    }
}

// pairs: chroma plane — columns are mirrored as (U,V) pairs
__device__ __noinline__ void stageFixup(const BoxGeom g, bool pairs, int tid, int nThreads) {
    const int nLeft = min(max(-g.pc0, 0), g.nK);               // box chunks [0, nLeft) lie left of the plane
    const int rightStart = min(max(g.nCh - g.pc0, 0), g.nK);   // box chunks [rightStart, nK) lie right of it (or straddle its last column)
    const int nOut = nLeft + (g.nK - rightStart);
    const int n = (g.r1 - g.r0) * nOut;
#pragma unroll 1
    for (int i = tid; i < n; i += nThreads) {
        const int rr = i / nOut;
        int k = i - rr * nOut;
        if (k >= nLeft) k += rightStart - nLeft;
        const int r = g.r0 + rr, pc = g.pc0 + k;
        uint8_t* __restrict__ d = g.buf + r * g.bw + 16 * (g.kLo + k);
        if (g.direct(pc)) {
            const uint4 w = *reinterpret_cast<const uint4*>(d);
            const unsigned sel = pairs ? 0x1032u : 0x0123u;  // reverse the (U,V) pairs / the bytes of a word
            *reinterpret_cast<uint4*>(d) = make_uint4(__byte_perm(w.w, 0u, sel), __byte_perm(w.z, 0u, sel), __byte_perm(w.y, 0u, sel), __byte_perm(w.x, 0u, sel));
        } else {
            const uint8_t* __restrict__ srcRow = rowPtr(g.plane, g.pitch, mirrorSearch(g.rb + r, g.dimV));
#pragma unroll 1
            for (int j = 0; j < 16; ++j) {
                const int vc = 16 * pc + j;
                d[j] = __ldg(srcRow + (pairs ? 2 * mirrorSearch(vc >> 1, g.dimU >> 1) + (vc & 1) : mirrorSearch(vc, g.dimU)));
            }
        }
    }
}

// lean per-layer total: same arithmetic as windowTotal (search_common.cuh), candidate offset given
__device__ __forceinline__ uint32_t layerTotalOf(const SearchArgs& a, const WindowCtx& c, uint32_t sad, int sq) {
    const int cand = (int)(short)(c.o + sq);
    uint32_t bias = (uint32_t)abs(cand);
    if (c.useNb) bias += __sad(c.nb[0], cand, __sad(c.nb[1], cand, __sad(c.nb[2], cand, __sad(c.nb[3], cand, 0u)))) << a.neighborBiasScalar;
    return (sad << a.deltaScalar) + c.nw * bias;
}

// ---- the kernel ------------------------------------------------------------------------------------------------------
// Windows of a tile whose displacements do not fit one pair of boxes are handled in ROUNDS: each round picks the
// pending windows around the smallest pending displacement, stages their boxes and runs them; a smooth field needs
// one round, a tile on a motion boundary two or three.  What is left after MAX_ROUNDS takes the per-pixel path.
constexpr int MAX_ROUNDS = 4;

template <int R, int STEP, int WSC>
__global__ void __maxnreg__(128)
    sadTileKernel(const SearchArgs a, const __grid_constant__ CUtensorMap mapC, const TileParams tp) {
    using C = Cls<WSC>;
    constexpr int LO = CandSpan<R>::LO, SPAN = CandSpan<R>::SPAN;
    constexpr int RUN = C::RUN, BW = C::BW, BWW = C::BWW;
    constexpr int WSL = WSC < 128 ? ilog2c(WSC) : 0;  // log2 of the window size for the classes below 128
    extern __shared__ uint8_t smemRaw[];
    __shared__ uint64_t barY, barC, barC2;
    __shared__ int s_rng[4];           // min ou, max ou, min ov, max ov over the windows of the current round
    __shared__ int s_bb[4];            // bounding box of the round's windows inside the tile: min / max window column, min / max window row
    __shared__ uint32_t s_red[8][16];  // CTA-level sums: [window of the tile][layer] (classes 64 and 128)
    uint8_t* const smem = smemRaw + ((128u - ((unsigned)__cvta_generic_to_shared(smemRaw) & 127u)) & 127u);
    uint8_t* const bufY = smem;
    uint8_t* const bufC = smem + tp.lumaBytes;
    int* const s_off = reinterpret_cast<int*>(smem + tp.lumaBytes + tp.chromaBytes);  // per window of the tile: (ou & 0xffff) | (ov << 16)
    const int TV = 32 * tp.nwv;
    const int nwu = C::SPREAD ? (128 >> WSL) : 1;        // windows of the tile along u, v
    const int nwv = C::SPREAD ? (TV >> WSL) : 1;
    uint8_t* const s_state = reinterpret_cast<uint8_t*>(s_off + nwu * nwv);  // 0 pending, 1 in this round, 2 done / not there

    const View<STEP> vw(a);
    const int lane = threadIdx.x, warp = threadIdx.y;
    const int NT = 32 * tp.nwv;
    const int tid = warp * 32 + lane;
    const int U0 = vw.u0 + blockIdx.x * 128, V0 = vw.v0 + blockIdx.y * TV;  // (u0, v0): multiples of kSplitAlign
    const int wsLog2 = WSC < 128 ? WSL : a.wsLog2;
    const int tileRows = min(TV, vw.lv - V0);            // flow rows of the tile that exist (> 0 by the grid)
    const int tileCols = min(128, vw.lu - U0);           // ... columns (a multiple of 4)

    auto now = [] {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        return t;
    };
    // 16 words per CTA; a CTA whose record does not fit the pass's slice records nothing (CTA-uniform)
    const size_t cta = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    unsigned long long* const dbg = a.dbg && 16 * (cta + 1) <= a.dbgWords ? a.dbg + 16 * cta : nullptr;
    if (tid == 0) {
        mbarInit(&barY, NT);  // every thread arrives once its own cp.async copies of the luma box have landed
        mbarInit(&barC, 1);   // the elected thread arrives with the byte count of the chroma TMA box
        mbarInit(&barC2, NT); // ... or every thread, where the chroma box is staged by cp.async too
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (dbg) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            dbg[0] = now();
            dbg[4] = smid;
            dbg[5] = blockIdx.x;
            dbg[6] = blockIdx.y;
            dbg[8] = blockDim.y;  // warps of the CTA (NWV)
        }
    }
    for (int i = tid; i < 128; i += NT) s_red[i >> 4][i & 15] = 0;

    // ---- A. displacements of the tile's windows -----------------------------------------------------------------------
    int uniOu = 0, uniOv = 0;  // class 128: the one window of the tile
    if (C::SPREAD) {
        for (int i = tid; i < nwu * nwv; i += NT) {
            const int lwu = i % nwu, lwv = i / nwu;
            const int wu = (U0 >> WSL) + lwu, wv = (V0 >> WSL) + lwv;
            int packed = 0;
            uint8_t st = 2;
            if ((wu << WSL) < vw.lu && (wv << WSL) < vw.lv) {
                int ox, oy;
                loadWindowOffsets<STEP>(a, View<STEP>::wx(wu, wv), View<STEP>::wy(wu, wv), ox, oy);
                packed = (View<STEP>::ou(ox, oy) & 0xffff) | (View<STEP>::ov(ox, oy) << 16);
                st = 0;
            }
            s_off[i] = packed;
            s_state[i] = st;
        }
    } else {
        int ox, oy;
        const int wu = U0 >> wsLog2, wv = V0 >> wsLog2;
        loadWindowOffsets<STEP>(a, View<STEP>::wx(wu, wv), View<STEP>::wy(wu, wv), ox, oy);
        uniOu = View<STEP>::ou(ox, oy);
        uniOv = View<STEP>::ov(ox, oy);
    }
    const bool manual = !tp.useTma;
    const int cu = U0 + 4 * lane;
    const bool colOk = cu < vw.lu;   // (lu is a multiple of 4: words are never partial)

#pragma unroll 1
    for (int round = 0; round <= MAX_ROUNDS; ++round) {
        // ---- B. the windows of this round and the range of their displacements --------------------------------------
        const bool slow = tp.forceSlow || round == MAX_ROUNDS;   // per-pixel path for everything still pending
        int minOu = uniOu, maxOu = uniOu, minOv = uniOv, maxOv = uniOv;
        if (C::SPREAD) {
            __syncthreads();  // s_off / s_state of the previous step are visible; nobody reads s_rng or the boxes any more
            if (tid < 4) {
                s_rng[tid] = (tid & 1) ? INT_MIN : INT_MAX;
                s_bb[tid] = (tid & 1) ? INT_MIN : INT_MAX;
            }
            __syncthreads();
            {
                int mn = INT_MAX;
                for (int i = tid; i < nwu * nwv; i += NT)
                    if (s_state[i] == 0) mn = min(mn, (int)(short)(s_off[i] & 0xffff));
                mn = __reduce_min_sync(0xffffffffu, mn);
                if (lane == 0 && mn != INT_MAX) atomicMin(&s_rng[0], mn);
            }
            __syncthreads();
            minOu = s_rng[0];
            if (minOu == INT_MAX) break;  // nothing pending (CTA-uniform)
            const int limU = slow ? INT_MAX : minOu + C::SU;
            {
                int mn = INT_MAX;
                for (int i = tid; i < nwu * nwv; i += NT)
                    if (s_state[i] == 0 && (int)(short)(s_off[i] & 0xffff) <= limU) mn = min(mn, s_off[i] >> 16);
                mn = __reduce_min_sync(0xffffffffu, mn);
                if (lane == 0 && mn != INT_MAX) atomicMin(&s_rng[2], mn);
            }
            __syncthreads();
            minOv = s_rng[2];
            const int limV = slow ? INT_MAX : minOv + C::SV;
            {
                int mxU = INT_MIN, mxV = INT_MIN, bu0 = INT_MAX, bu1 = INT_MIN, bv0 = INT_MAX, bv1 = INT_MIN;
                for (int i = tid; i < nwu * nwv; i += NT) {
                    const int ou = (int)(short)(s_off[i] & 0xffff), ov = s_off[i] >> 16;
                    if (s_state[i] == 0 && ou <= limU && ov >= minOv && ov <= limV) {
                        s_state[i] = 1;
                        mxU = max(mxU, ou);
                        mxV = max(mxV, ov);
                        const int lwu = i % nwu, lwv = i / nwu;
                        bu0 = min(bu0, lwu); bu1 = max(bu1, lwu); bv0 = min(bv0, lwv); bv1 = max(bv1, lwv);
                    }
                }
                mxU = __reduce_max_sync(0xffffffffu, mxU);
                mxV = __reduce_max_sync(0xffffffffu, mxV);
                bu0 = __reduce_min_sync(0xffffffffu, bu0); bu1 = __reduce_max_sync(0xffffffffu, bu1);
                bv0 = __reduce_min_sync(0xffffffffu, bv0); bv1 = __reduce_max_sync(0xffffffffu, bv1);
                if (lane == 0 && mxU != INT_MIN) {
                    atomicMax(&s_rng[1], mxU);
                    atomicMax(&s_rng[3], mxV);
                    atomicMin(&s_bb[0], bu0); atomicMax(&s_bb[1], bu1); atomicMin(&s_bb[2], bv0); atomicMax(&s_bb[3], bv1);
                }
            }
            __syncthreads();
            maxOu = s_rng[1];
            maxOv = s_rng[3];
        } else {
            if (round > 0) break;
            __syncthreads();  // barriers and s_red are initialised
        }
        const bool staged = !slow;

        // ---- C. stage the frame-1 boxes of the round ------------------------------------------------------------------
        // luma box: plane rows rb .., bytes ca ..; chroma box: chroma rows rbc .., bytes caC ..
        const int cbMin = U0 + minOu;
        const int ca = cbMin & ~15;
        const int rb = V0 + minOv + LO;
        const int cbMinC = U0 + (minOu & ~1);
        const int caC = cbMinC & ~15;
        const int rbc = rb >> 1;
        const int rowsNeeded = tileRows + SPAN + (maxOv - minOv);               // luma rows of the box that are ever read
        const int rowsNeededC = ((rb + rowsNeeded - 1) >> 1) - rbc + 1;
        const int colEnd = cbMin - ca + tileCols + (maxOu - minOu) + 4;         // bytes [cbMin - ca, colEnd) of a luma row are read
        const int colEndC = cbMinC - caC + tileCols + ((maxOu & ~1) - (minOu & ~1)) + 2 + 4;
        const bool border = cbMin < 0 || cbMin + tileCols + (maxOu - minOu) + 2 > vw.dimU || rb < 0 || rb + rowsNeeded > vw.dimV;
        // rounds after the first stage only the rows and columns their windows can touch (s_bb: bounding box of the round's
        // windows, in windows of the tile)
        int subR0 = 0, subR1 = rowsNeeded, subC0 = cbMin - ca, subC1 = min(colEnd, BW), subC0C = cbMinC - caC, subC1C = min(colEndC, BW);
        if (C::SPREAD && round > 0) {
            const int t0 = s_bb[2] << WSL, t1 = min((s_bb[3] + 1) << WSL, tileRows);   // tile rows of the round's windows
            const int u0 = s_bb[0] << WSL, u1 = min((s_bb[1] + 1) << WSL, tileCols);   // tile columns
            subR0 = t0;
            subR1 = min(rowsNeeded, t1 + SPAN + (maxOv - minOv));
            subC0 = cbMin - ca + u0;
            subC1 = min(cbMin - ca + u1 + (maxOu - minOu) + 4, BW);
            subC0C = cbMinC - caC + u0;
            subC1C = min(cbMinC - caC + u1 + ((maxOu & ~1) - (minOu & ~1)) + 2 + 4, BW);
        }
        const int subR0C = ((rb + subR0) >> 1) - rbc, subR1C = ((rb + subR1 - 1) >> 1) - rbc + 1;
        const BoxGeom gy(bufY, BW, vw.y1, vw.pitch, vw.dimU, vw.dimV, rb, ca, subR0, subR1, subC0, subC1);
        const BoxGeom gc(bufC, BW, vw.c1, vw.pitch, vw.dimU, vw.dimV >> 1, rbc, caC, subR0C, subR1C, subC0C, subC1C);
        const bool needFix = gc.outsideChunks() || gy.outsideChunks();                  // chunks left / right of the plane: reversed after landing
        // CTA-uniform, like the two below.  The TMA branch runs no fix-up: a luma box that reaches the partial last chunk
        // of a row is staged like a border tile
        const bool tmaStage = staged && !manual && !border && round == 0 && !gy.partialTail();
        const bool pipeStage = staged && round == 0 && !tmaStage && !needFix;
        const bool asyncStage = tmaStage || pipeStage;
        if (tmaStage) {
            // interior tile: the chroma box through the TMA engine (one elected thread), the luma box through the LSU path as
            // 16-byte cp.async copies of all threads — both in flight at once, each completing on its own mbarrier
            if (tid == 0) {
                mbarExpectTx(&barC, (unsigned)(tp.boxHC * BW));
                tmaLoad2d(bufC, &mapC, caC, rbc, &barC);
            }
            stageIssue(gy, tid, NT);
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"((unsigned)__cvta_generic_to_shared(&barY)) : "memory");
        } else if (pipeStage) {
            // tile at the top / bottom border (rows come through the mirrored row index) or no TMA: both boxes by cp.async, each on
            // its own mbarrier, so that the chroma of a run is worked on while the luma box is still landing
            stageIssue(gc, tid, NT);
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"((unsigned)__cvta_generic_to_shared(&barC2)) : "memory");
            stageIssue(gy, tid, NT);
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"((unsigned)__cvta_generic_to_shared(&barY)) : "memory");
        } else if (staged) {
            // left / right border or a later round: both boxes by cp.async, then the mirror fix-up of the chunks outside the plane
            stageIssue(gc, tid, NT);
            stageIssue(gy, tid, NT);
            cpAsyncWaitAll();
            __syncthreads();
            if (needFix) {
                stageFixup(gc, true, tid, NT);
                stageFixup(gy, false, tid, NT);
                __syncthreads();
            }
        }
        const bool waitTma = asyncStage;
        uint64_t* const barChroma = tmaStage ? &barC : &barC2;
        const unsigned parity = 0;   // the barriers are used once, by the first round
        bool waitedC = false, waitedY = false;
        if (dbg && tid == 0) {
            if (waitTma) {
                mbarWait(barChroma, parity);
                mbarWait(&barY, parity);
                waitedC = waitedY = true;
            }
            dbg[1] = now();
            dbg[7] = round + 1 + (border ? 100 : 0);
        }

        // ---- D. the runs of this lane -----------------------------------------------------------------------------------
#pragma unroll 1
        for (int run = 0; run < C::NRUN; ++run) {
            const int v0 = V0 + 32 * warp + run * RUN;
            const bool rowOk = v0 < vw.lv;           // warp-uniform
            const int np = min(RUN, vw.lv - v0);     // rows of the run (even)
            // the window of this lane in this run, its state and its displacement
            const int wu = cu >> wsLog2, wv = v0 >> wsLog2;
            const bool winThere = rowOk && (wu << wsLog2) < vw.lu;   // the lane's window exists (its own column may not)
            int ou = uniOu, ov = uniOv;
            bool active = winThere;
            if (C::SPREAD && winThere) {
                const int li = (wv - (V0 >> WSL)) * nwu + (wu - (U0 >> WSL));
                active = s_state[li] == 1;
                const int packed = s_off[li];
                ou = (int)(short)(packed & 0xffff);
                ov = packed >> 16;
            }
            if (C::SPREAD && !__any_sync(0xffffffffu, active)) continue;  // nothing of this warp's run belongs to the round
            const bool runOk = active && colOk;
            const int pi = ov & 1;
            const bool odd = (ou & 1) != 0;
            uint32_t acc[16];
#pragma unroll
            for (int z = 0; z < 16; ++z) acc[z] = 0;

            if (runOk && staged && np == RUN) {
                // frame 2 of the run first: these loads are in flight while the TMA boxes land
                uint32_t f2c[RUN / 2], f2[RUN];
                {
                    const uint8_t* __restrict__ pc = rowPtr(vw.c2 + cu, vw.pitch, v0 >> 1);
#pragma unroll
                    for (int k = 0; k < RUN / 2; ++k) f2c[k] = __ldg(reinterpret_cast<const uint32_t*>(rowPtr(pc, vw.pitch, k)));
                    const uint8_t* __restrict__ py = rowPtr(vw.y2 + cu, vw.pitch, v0);
#pragma unroll
                    for (int p = 0; p < RUN; ++p) f2[p] = __ldg(reinterpret_cast<const uint32_t*>(rowPtr(py, vw.pitch, p)));
                }
                uint32_t accC[16];
#pragma unroll
                for (int z = 0; z < 16; ++z) accC[z] = 0;
                // chroma: one pass (ou even) or two passes 2 bytes apart (ou odd)
                if (waitTma && !waitedC) {
                    mbarWait(barChroma, parity);
                    waitedC = true;
                }
                {
                    const int offC = cu + (ou & ~1) - caC;
                    const int rowC0 = ((v0 + ov + LO) >> 1) - rbc;
                    const uint32_t* __restrict__ q0 = reinterpret_cast<const uint32_t*>(bufC + rowC0 * BW + (offC & ~3));
                    const int sh0 = (offC & 3) * 8;
                    const uint32_t* __restrict__ q1 = reinterpret_cast<const uint32_t*>(bufC + rowC0 * BW + ((offC + 2) & ~3));
                    const int sh1 = ((offC + 2) & 3) * 8;
                    if (pi) {
                        slideChroma<R, RUN, 1>(accC, f2c, [&](int j) { return __funnelshift_r(q0[j * BWW], q0[j * BWW + 1], sh0); });
                        if (odd) slideChroma<R, RUN, 1>(accC, f2c, [&](int j) { return __funnelshift_r(q1[j * BWW], q1[j * BWW + 1], sh1); });
                    } else {
                        slideChroma<R, RUN, 0>(accC, f2c, [&](int j) { return __funnelshift_r(q0[j * BWW], q0[j * BWW + 1], sh0); });
                        if (odd) slideChroma<R, RUN, 0>(accC, f2c, [&](int j) { return __funnelshift_r(q1[j * BWW], q1[j * BWW + 1], sh1); });
                    }
                }
                // luma
                if (waitTma && !waitedY) {
                    mbarWait(&barY, parity);
                    waitedY = true;
                }
                {
                    const int offY = cu + ou - ca;
                    const int rowY0 = v0 + ov + LO - rb;
                    const uint32_t* __restrict__ q = reinterpret_cast<const uint32_t*>(bufY + rowY0 * BW + (offY & ~3));
                    const int sh = (offY & 3) * 8;
                    slideLuma<R, RUN>(acc, f2, [&](int j) { return __funnelshift_r(q[j * BWW], q[j * BWW + 1], sh); });
                }
                // chroma weight = (rows coincide ? 2 : 1) * (columns coincide ? 2 : 1)
                const int evenU = odd ? 0 : 1;
#pragma unroll
                for (int z = 0; z < R; ++z) acc[z] += accC[z] << (chromaShift<R>(pi, z) + evenU);
            } else if (runOk && staged) {
                // partial run at the last rows of the flow field: compact loops, one (row, candidate) at a time
                if (waitTma && !waitedC) {
                    mbarWait(barChroma, parity);
                    waitedC = true;
                }
                if (waitTma && !waitedY) {
                    mbarWait(&barY, parity);
                    waitedY = true;
                }
                const int offC = cu + (ou & ~1) - caC;
                const int rowC0 = ((v0 + ov + LO) >> 1) - rbc;
                const int amin = (pi + LO) >> 1;
                const int evenU = odd ? 0 : 1;
                for (int pass = 0; pass < (odd ? 2 : 1); ++pass) {
                    const uint32_t* __restrict__ q = reinterpret_cast<const uint32_t*>(bufC + rowC0 * BW + ((offC + 2 * pass) & ~3));
                    const int sh = ((offC + 2 * pass) & 3) * 8;
                    for (int k = 0; k < (np >> 1); ++k) {
                        const uint32_t f2 = __ldg(reinterpret_cast<const uint32_t*>(rowPtr(vw.c2 + cu, vw.pitch, (v0 >> 1) + k)));
#pragma unroll
                        for (int z = 0; z < R; ++z) {
                            const int d = pi + candOffset<R>(z);
                            const int j = k + (d >> 1) - amin;
                            uint32_t sd = sad4(__funnelshift_r(q[j * BWW], q[j * BWW + 1], sh), f2, 0u);
                            if (d & 1) sd = sad4(__funnelshift_r(q[(j + 1) * BWW], q[(j + 1) * BWW + 1], sh), f2, sd);
                            acc[z] += sd << (((d & 1) ? 0 : 1) + evenU);
                        }
                    }
                }
                const int offY = cu + ou - ca;
                const int rowY0 = v0 + ov + LO - rb;
                const uint32_t* __restrict__ q = reinterpret_cast<const uint32_t*>(bufY + rowY0 * BW + (offY & ~3));
                const int sh = (offY & 3) * 8;
                for (int p = 0; p < np; ++p) {
                    const uint32_t f2 = __ldg(reinterpret_cast<const uint32_t*>(rowPtr(vw.y2 + cu, vw.pitch, v0 + p)));
#pragma unroll
                    for (int z = 0; z < R; ++z) {
                        const int j = p + candOffset<R>(z) - LO;
                        acc[z] = sad4(__funnelshift_r(q[j * BWW], q[j * BWW + 1], sh), f2, acc[z]);
                    }
                }
            } else if (runOk) {
                // per-pixel path straight from the planes
                for (int i = 0; i < 4; ++i) {
                    const int fu = mirrorSearch(cu + i + ou, vw.dimU);
                    for (int p = 0; p < np; ++p) {
                        const uint32_t f2 = fetchPixel(vw.y2, vw.c2, vw.pitch, v0 + p, cu + i);
                        const int bv = v0 + p + ov;
#pragma unroll
                        for (int z = 0; z < R; ++z) acc[z] = sad4(fetchPixel(vw.y1, vw.c1, vw.pitch, mirrorSearch(bv + candOffset<R>(z), vw.dimV), fu), f2, acc[z]);
                    }
                }
            }

            // ---- E. reduce over the window's lanes and finalize ----------------------------------------------------------
            const bool b0 = lane & 1, b1 = lane & 2, b2 = lane & 4, b3 = lane & 8;
            if (WSC <= 32) {
                // the window lives in SEG lanes of this warp: butterfly over them, every lane then owns NZ layers
                constexpr int NZ = 16 / C::SEG;
                if (C::SEG >= 2) bfly<16>(acc, 1, b0);
                if (C::SEG >= 4) bfly<8>(acc, 2, b1);
                if (C::SEG >= 8) bfly<4>(acc, 4, b2);
                const int zbase = (C::SEG >= 2 && b0 ? 8 : 0) + (C::SEG >= 4 && b1 ? 4 : 0) + (C::SEG >= 8 && b2 ? 2 : 0);
                const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
                uint32_t bestT = 0xffffffffu;
                int bestZ = zbase < R ? zbase : 0xff;  // no layer beats a sum of 2^32-1: the lane's first layer stands, as with strict <
                WindowCtx c;
                c.o = 0;
                if (active) {
                    // (lanes of a window past the last column still finalize their layers)
                    c = loadWindowCtx<STEP>(a, wx, wy, STEP == 1 ? ou : ov, STEP == 1 ? ov : ou);
#pragma unroll
                    for (int i = 0; i < NZ; ++i) {
                        const int z = zbase + i;
                        if (z < R) {
                            const uint32_t total = layerTotalOf(a, c, acc[i], signedSquare(z - R / 2));
                            tapTotal<R>(a, wx, wy, z, total);
                            if (total < bestT) {  // z ascends inside a lane: strict < keeps the lowest layer of a tie
                                bestT = total;
                                bestZ = z;
                            }
                        }
                    }
                }
                unsigned long long best = layerKey(bestT, bestZ);
                if (C::SEG >= 2) best = min(best, shflXor64(best, 1));
                if (C::SEG >= 4) best = min(best, shflXor64(best, 2));
                if (C::SEG >= 8) best = min(best, shflXor64(best, 4));
                if (active && (lane & (C::SEG - 1)) == 0) commitWindow<R, STEP>(a, wx, wy, c.o, (int)(best & 0xff));
            } else {
                // windows of 64 pixels and more: sums of the CTA in shared memory first
                bfly<16>(acc, 1, b0);
                bfly<8>(acc, 2, b1);
                bfly<4>(acc, 4, b2);
                bfly<2>(acc, 8, b3);
                uint32_t sm = acc[0];
                const int z = (b0 ? 8 : 0) + (b1 ? 4 : 0) + (b2 ? 2 : 0) + (b3 ? 1 : 0);  // the layer this lane ended up with
                int lwin = 0;
                if (WSC == 64) {
                    lwin = (lane >> 4) + 2 * ((32 * warp) >> 6);  // window of the tile: 2 across, TV / 64 down
                } else {
                    sm += __shfl_xor_sync(0xffffffffu, sm, 16);
                }
                if (active && z < R && (WSC == 64 || lane < 16)) atomicAdd(&s_red[lwin][z], sm);
            }
        }

        if (C::SPREAD) {
            __syncthreads();  // every lane is done with the round's boxes and states
            for (int i = tid; i < nwu * nwv; i += NT)
                if (s_state[i] == 1) s_state[i] = 2;
        }
    }

    if (dbg) {
        __syncthreads();
        if (tid == 0) dbg[2] = now();
    }
    if (WSC >= 64) {
        __syncthreads();
        if (WSC == 64) {
            // every window of the tile is complete inside the CTA: one thread per window finalizes it
            const int nWin = 2 * (TV >> 6);
            if (tid < nWin) {
                const int wu = (U0 >> 6) + (tid & 1), wv = (V0 >> 6) + (tid >> 1);
                const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
                if ((wu << 6) < vw.lu && (wv << 6) < vw.lv) finalizeWindow<R, STEP>(a, wx, wy, s_red[tid]);
            }
        } else {
            // add the CTA's sums to the window's scratch; the LAST CTA to arrive (ticket) finds them complete, finalizes the
            // window and leaves scratch and ticket zeroed for the next pass — no finalize kernel, no memset between passes.
            // A tile lies inside one window (chooseWarps), so the window's CTAs are its tiles.  A sharded pass (split
            // search) has windows of at most 128 rows here, hence 128-row tiles, and every CTA covering an owned window
            // lies inside the stripe (stripes start at multiples of 128): the count is unchanged.
            const int wu = U0 >> wsLog2, wv = V0 >> wsLog2;
            const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
            const size_t widx = (size_t)(wy * a.nWx + wx);
            if (warp == 0) {
                if (lane < R) atomicAdd(&a.winSums[widx * 16 + lane], s_red[0][lane]);
                __threadfence();
                __syncwarp();
                int last = 0;
                if (lane == 0) {
                    const int uext = min(a.ws, vw.lu - (wu << wsLog2)), vext = min(a.ws, vw.lv - (wv << wsLog2));
                    const unsigned need = (unsigned)(((uext + 127) >> 7) * ((vext + TV - 1) / TV));
                    last = atomicAdd(&a.winTicket[widx], 1u) == need - 1;
                }
                last = __shfl_sync(0xffffffffu, last, 0);
                if (last) {
                    __threadfence();
                    uint32_t sum = 0;
                    if (lane < R) {
                        sum = __ldcg(&a.winSums[widx * 16 + lane]);
                        a.winSums[widx * 16 + lane] = 0;
                    }
                    if (lane == 0) a.winTicket[widx] = 0;
                    int ox, oy;
                    loadWindowOffsets<STEP>(a, wx, wy, ox, oy);
                    const WindowCtx c = loadWindowCtx<STEP>(a, wx, wy, ox, oy);
                    unsigned long long key = ~0ull;
                    if (lane < R) {
                        const uint32_t total = windowTotal<R>(a, c, sum, lane);
                        tapTotal<R>(a, wx, wy, lane, total);
                        key = layerKey(total, lane);
                    }
                    key = min(key, shflXor64(key, 1));
                    key = min(key, shflXor64(key, 2));
                    key = min(key, shflXor64(key, 4));
                    key = min(key, shflXor64(key, 8));
                    if (lane == 0) commitWindow<R, STEP>(a, wx, wy, c.o, (int)(key & 0xff));
                }
            }
        }
    }
    if (dbg) {
        __syncthreads();
        if (tid == 0) dbg[3] = now();
    }
}

// ---- tensor maps ------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encodeTiled() {
    static std::once_flag once;
    static EncodeTiledFn fn = nullptr;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
        cudaGetLastError();
    });
    return fn;
}

}  // namespace

struct TmaCache {
    struct alignas(64) Entry {
        CUtensorMap map;
        const void* base;
        int dimU, dimV, pitch, boxW, boxH;
    };
    std::vector<Entry*> entries;
};

#if HRB_SEARCH_PART == 0
void freeTmaCache(hrb_ofc* h) {
    if (!h->tmaCache) return;
    for (auto* e : h->tmaCache->entries) delete e;
    delete h->tmaCache;
    h->tmaCache = nullptr;
}
#endif

namespace {

// u8 plane [dimV][pitch] seen as a 2-D tensor of dimU x dimV bytes; boxes of boxW x boxH.  nullptr: not encodable.
const CUtensorMap* tensorMapFor(hrb_ofc* h, const uint8_t* base, int dimU, int dimV, int pitch, int boxW, int boxH) {
    if (!h->tmaCache) h->tmaCache = new TmaCache();
    for (auto* e : h->tmaCache->entries)
        if (e->base == base && e->dimU == dimU && e->dimV == dimV && e->pitch == pitch && e->boxW == boxW && e->boxH == boxH) return &e->map;
    EncodeTiledFn enc = encodeTiled();
    if (!enc || boxH > 256 || boxW > 256) return nullptr;
    auto* e = new TmaCache::Entry();
    const cuuint64_t dims[2] = {(cuuint64_t)dimU, (cuuint64_t)dimV};
    const cuuint64_t strides[1] = {(cuuint64_t)pitch};
    const cuuint32_t box[2] = {(cuuint32_t)boxW, (cuuint32_t)boxH};
    const cuuint32_t es[2] = {1, 1};
    if (enc(&e->map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
        delete e;
        return nullptr;
    }
    e->base = base; e->dimU = dimU; e->dimV = dimV; e->pitch = pitch; e->boxW = boxW; e->boxH = boxH;
    if (h->tmaCache->entries.size() >= 512) {  // geometry and slots are fixed per handle: this never grows in practice
        for (auto* o : h->tmaCache->entries) delete o;
        h->tmaCache->entries.clear();
    }
    h->tmaCache->entries.push_back(e);
    return &e->map;
}

// shared memory of a CTA with nwv warps: the two boxes (each staged as two TMA boxes) + the per-window displacements
template <int R, int WSC> TileParams tileParams(int nwv) {
    using C = Cls<WSC>;
    TileParams tp;
    tp.nwv = nwv;
    const int rowsY = 32 * nwv + CandSpan<R>::SPAN + C::SV;
    tp.rowsY = rowsY;
    tp.boxHC = rowsY / 2 + 2;
    tp.lumaBytes = align128(rowsY * C::BW);
    tp.chromaBytes = align128(tp.boxHC * C::BW);
    tp.useTma = 1;
    tp.forceSlow = 0;
    return tp;
}
template <int WSC> int tileSmem(const TileParams& tp) {
    const int nWin = Cls<WSC>::SPREAD ? (128 / WSC) * ((32 * tp.nwv) / WSC) : 0;
    return tp.lumaBytes + tp.chromaBytes + nWin * 4 + ((nWin + 15) & ~15) + 128;  // boxes, window displacements, window states, alignment slack
}

// CTAs of sadTileKernel<R, STEP, WSC> with nwv warps the runtime places on one SM, asked once per handle.  The kernel's
// dynamic shared-memory limit is raised first (the runtime counts 0 CTAs for a kernel not allowed that much), and the
// carve-out is set to the maximum, so that the driver does not pick a smaller one that drops a CTA.
template <int R, int STEP, int WSC> int residentTiles(hrb_ofc* h, int nwv, int smem, int& perSm) {
    const void* fn = reinterpret_cast<const void*>(sadTileKernel<R, STEP, WSC>);
    for (const auto& e : h->tileResidency)
        if (e.kernel == fn && e.nwv == nwv) {
            perSm = e.ctasPerSm;
            return HRB_OK;
        }
    const int rc = allowDynamicSmem<sadTileKernel<R, STEP, WSC>>(h->device, smem);
    if (rc) return rc;
    HRB_CUDA(cudaFuncSetAttribute(sadTileKernel<R, STEP, WSC>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    HRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, sadTileKernel<R, STEP, WSC>, 32 * nwv, smem));
    h->tileResidency.push_back({fn, nwv, perSm});
    return HRB_OK;
}

// Warps per CTA (tile rows / 32): the choice that needs the fewest rounds of resident CTAs, then the smallest halo share.
// Classes 64 and 128 count rounds from the CTAs per SM the runtime places.  A tile of class 128 lies inside one window
// (32 * nwv divides ws: the window's CTAs are counted by its arrival ticket), and a tile of class 64 holds whole window
// rows, at most 8 windows (s_red).  Classes 16 and 32 keep the fixed residency estimate their shapes were tuned with.
template <int R, int STEP, int WSC> int chooseWarps(hrb_ofc* h, int lu, int lv, int ws, int& nwvOut) {
    nwvOut = 4;
    double bestCost = 1e30;
    for (int nwv = 2; nwv <= 8; ++nwv) {
        if (WSC >= 128 ? (nwv != 4 && nwv != 8) || ws % (32 * nwv) : WSC == 64 ? (nwv & 1) != 0 : nwv > 6) continue;
        const TileParams tp = tileParams<R, WSC>(nwv);
        if (tp.boxHC > 256) continue;  // the chroma box is one TMA box
        const int smem = tileSmem<WSC>(tp);
        int perSm = min(min((233472) / (smem + 1040), 3), 2048 / (32 * nwv));
        if (WSC >= 64) {
            const int rc = residentTiles<R, STEP, WSC>(h, nwv, smem, perSm);
            if (rc) return rc;
        }
        if (perSm < 1) continue;
        const long tiles = (long)((lu + 127) / 128) * ((lv + 32 * nwv - 1) / (32 * nwv));
        const long slots = (long)h->smCount * perSm;
        const long rounds = (tiles + slots - 1) / slots;
        // a round costs the tile's rows plus the candidate span; few resident warps hide latency badly.  Class 128 counts
        // the tiles of the busiest SM instead of rounds: its grids are one round at either height, and the rows that SM
        // stages (the span once per tile) are what a taller tile saves
        const long perBusiest = WSC >= 128 ? (tiles + h->smCount - 1) / h->smCount : rounds;
        const long resident = WSC >= 128 ? min((long)perSm, perBusiest) : perSm;
        const double cost = (double)perBusiest * (32 * nwv + CandSpan<R>::SPAN) * (1.0 + 2.0 / (resident * nwv));
        if (cost < bestCost) {
            bestCost = cost;
            nwvOut = nwv;
        }
    }
    return HRB_OK;
}

template <int R, int STEP, int WSC> int launchTile(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p) {
    using C = Cls<WSC>;
    const PassRange r = passRange(a, STEP);  // the pass's rows: a stripe on a shard of a split search
    const int lu = r.lu - r.u0, lv = r.lv - r.v0;
    const int dimU = STEP == 1 ? a.W : a.H, dimV = STEP == 1 ? a.H : a.W;
    const uint8_t* c1 = STEP == 1 ? a.c1 : a.cT1;
    const int pitch = STEP == 1 ? a.pitch : a.pitchT;
    int nwv;
    int rc = chooseWarps<R, STEP, WSC>(h, lu, lv, a.ws, nwv);
    if (rc) return rc;
    TileParams tp = tileParams<R, WSC>(nwv);
    tp.useTma = p.useTma;
    tp.forceSlow = p.forceSlow;
    const int smem = tileSmem<WSC>(tp);
    rc = allowDynamicSmem<sadTileKernel<R, STEP, WSC>>(h->device, smem);
    if (rc) return rc;
    const CUtensorMap* mC = tp.useTma ? tensorMapFor(h, c1, dimU, dimV / 2, pitch, C::BW, tp.boxHC) : nullptr;
    CUtensorMap dummy;
    memset(&dummy, 0, sizeof(dummy));
    if (!mC) {
        tp.useTma = 0;
        mC = &dummy;
    }
    const dim3 grid((lu + 127) / 128, (lv + 32 * tp.nwv - 1) / (32 * tp.nwv), 1);
    sadTileKernel<R, STEP, WSC><<<grid, dim3(32, tp.nwv, 1), smem, h->stream>>>(a, *mC, tp);
    HRB_LAUNCH_CHECK();
    return HRB_OK;
}

template <int R, int STEP> int launchTileStep(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p) {
    switch (a.ws) {
        case 4: return launchTile<R, STEP, 4>(h, a, p);
        case 8: return launchTile<R, STEP, 8>(h, a, p);
        case 16: return launchTile<R, STEP, 16>(h, a, p);
        case 32: return launchTile<R, STEP, 32>(h, a, p);
        case 64: return launchTile<R, STEP, 64>(h, a, p);
    }
    if (a.ws >= 128) return launchTile<R, STEP, 128>(h, a, p);
    setLastError("[hopperrender_b200] tile kernel, window size %d: no such kernel instance", a.ws);
    return HRB_ERR_STATE;
}

}  // namespace

// One whole pass for ws >= 4 at full flow resolution, for the radii of part PART (hrb_internal.cuh).
template <int PART> int launchTilePart(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p, int R, int step) {
    return withConstant<firstRadiusOf(PART), firstRadiusOf(PART) + 3>("tile kernel, search radius", R, [&](auto r) {
        constexpr int RC = decltype(r)::value;
        return step == 1 ? launchTileStep<RC, 1>(h, a, p) : launchTileStep<RC, 0>(h, a, p);
    });
}
template int launchTilePart<HRB_SEARCH_PART>(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p, int R, int step);

}  // namespace hrb
