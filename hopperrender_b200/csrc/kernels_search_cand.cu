// kernels_search_cand.cu — search passes for the small windows (2, 4, 8 flow pixels; up to 32 when the tile kernel does
// not apply) at full flow resolution: the last 3 of the 11 iterations at 4K, where every window has its own offset.
//
// The generic kernel fetches frame 1 once per pixel-candidate from global memory: one 64-bit address computation and
// one L1 transaction per VABSDIFF4.  Here a CTA owns a 32 x 128 tile (u x v, see View) and first looks at the offsets
// of all windows in the tile.  Motion fields are smooth, so they almost always span a few pixels only; the CTA then
// stages the frame-1 region every candidate of every window of the tile can touch —
//     (128 + (HI-LO) + spread_v) rows  x  (32 + spread_u) columns  (<= 254 x 48 pixels) —
// in shared memory, expanded from the planar planes to one {Y, U, V, 0} word per pixel (expand4), so that ANY displaced
// pixel is one aligned LDS with an IMMEDIATE offset (the candidate displacement is a compile-time multiple of the row
// pitch) followed by one VABSDIFF4.  Regions that leave the frame are staged through the reference's mirror without
// leaving the fast path: mirrored row indices, and words beyond the left / right edge read from the reflected position
// with their pixels reversed.  Tiles whose offsets spread too far for the buffer fall back to global fetches.
//   * windows of 2 and 4: one lane owns one window (winGroups): sums, context and arg-min stay in the lane;
//   * windows of 8 and more: lanes own pixel columns, butterfly reduction, per-window sums in shared memory (candGroups).
#include <climits>

#include "search_common.cuh"

namespace hrb {

namespace {

constexpr int CT_U = 32, CT_V = 128;  // tile
constexpr int SP = 52;                 // staged row pitch in words (48 + alignment slack, 13 x 16 B)
constexpr int RV_MAX = 254;            // staged rows: 128 + (HI-LO <= 113) + spread_v (<= 13); sized so that four CTAs fit an SM
constexpr int RU_MAX = 48;             // staged columns actually addressed
// dynamic shared memory of one CTA: staged region + (ws >= 8) per-window sums + per-window offsets + 4 range words
template <int WS> __host__ __device__ constexpr int candWindows() { return (CT_U / WS) * (CT_V / WS); }
template <int WS> __host__ __device__ constexpr int candSumWords() { return WS >= 8 ? candWindows<WS>() * 16 : 0; }
template <int WS> __host__ __device__ constexpr size_t candSmem() { return ((size_t)RV_MAX * SP + candSumWords<WS>() + candWindows<WS>() + 4) * 4; }
static_assert(candSmem<2>() + 1024 <= 232448 / 4, "four CTAs per SM");

// lean per-layer total for the in-register finalize: same arithmetic as windowTotal, candidate offset given
__device__ __forceinline__ uint32_t layerTotal(const SearchArgs& a, const WindowCtx& c, uint32_t sad, int sq) {
    const int cand = (int)(short)(c.o + sq);
    uint32_t bias = (uint32_t)abs(cand);
    if (c.useNb) bias += __sad(c.nb[0], cand, __sad(c.nb[1], cand, __sad(c.nb[2], cand, __sad(c.nb[3], cand, 0u)))) << a.neighborBiasScalar;
    return (sad << a.deltaScalar) + c.nw * bias;
}

struct CandTile {
    const uint32_t* s_f1;
    uint32_t (*s_sums)[16];
    const int* s_off;
    int U0, V0, minOu, minOv, sh;
    bool staged;
};

// SADs and per-window reduction of one warp's 16 rows.  A warp accumulates groups of min(WS, 16) rows (one window row
// each) before the lanes are reduced, so the reduction is paid once per window row.  FULL: the tile lies inside the
// flow field and is staged, so no pixel needs a range check.
template <int R, int STEP, bool TAPS, int WS, bool FULL>
__device__ __forceinline__ void candGroups(const SearchArgs& a, const View<STEP>& vw, const CandTile& t, int lane, int warp) {
    constexpr int LO = candOffset<R>(0);
    constexpr int L2 = WS == 2 ? 1 : WS == 4 ? 2 : WS == 8 ? 3 : WS == 16 ? 4 : 5;
    constexpr int GH = WS < 16 ? WS : 16;
    constexpr int NWU = CT_U >> L2;
    const int cu = t.U0 + lane;
    const bool b0 = lane & 1, b1 = lane & 2, b2 = lane & 4, b3 = lane & 8;

    // layers a lane finalizes for WS <= 4 (what the butterfly leaves it with) and their displacements
    constexpr int NZ = WS == 2 ? 8 : 4;
    const int zbase = WS == 2 ? (b0 ? 8 : 0) : (b0 ? 8 : 0) + (b1 ? 4 : 0);
    int sqv[NZ];
    if (WS <= 4) {
#pragma unroll
        for (int i = 0; i < NZ; ++i) {
            if (WS == 2)
                sqv[i] = b0 ? signedSquare(8 + i - R / 2) : signedSquare(i - R / 2);
            else
                sqv[i] = b0 ? (b1 ? signedSquare(12 + i - R / 2) : signedSquare(8 + i - R / 2)) : (b1 ? signedSquare(4 + i - R / 2) : signedSquare(i - R / 2));
        }
    }

#pragma unroll 1
    for (int g = 0; g < 16; g += GH) {
        const int cv0 = t.V0 + warp * 16 + g;
        const int wu = cu >> L2, wv = cv0 >> L2;
        const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
        const bool pixOk = FULL || (cu < vw.lu && cv0 < vw.lv);
        const bool winOk = FULL || ((wu << L2) < vw.lu && cv0 < vw.lv);
        const int packed = t.s_off[(wv - (t.V0 >> L2)) * NWU + (wu - (t.U0 >> L2))];
        const int ou = (int)(short)(packed & 0xffff), ov = packed >> 16;
        const int ox = STEP == 1 ? ou : ov, oy = STEP == 1 ? ov : ou;
        uint32_t acc[16];
#pragma unroll
        for (int z = 0; z < 16; ++z) acc[z] = 0;
        if (pixOk) {
            if (FULL || t.staged) {
                // word index of (row cv0 + ov + LO, column cu + ou) inside the staged region
                const uint32_t* __restrict__ q = &t.s_f1[(cv0 - t.V0 + ov - t.minOv) * SP + (lane + ou - t.minOu + t.sh)];
                constexpr int RB = GH < 8 ? GH : 8;  // frame-2 rows loaded before the first one is consumed
#pragma unroll
                for (int r0 = 0; r0 < GH; r0 += RB) {
                    uint32_t f2r[RB];
#pragma unroll
                    for (int r = 0; r < RB; ++r) f2r[r] = (FULL || cv0 + r0 + r < vw.lv) ? fetchPixel(vw.y2, vw.c2, vw.pitch, cv0 + r0 + r, cu) : 0u;
#pragma unroll
                    for (int r = 0; r < RB; ++r) {
                        if (FULL || cv0 + r0 + r < vw.lv) {
#pragma unroll
                            for (int z = 0; z < R; ++z) acc[z] = sad4(q[(r0 + r + candOffset<R>(z) - LO) * SP], f2r[r], acc[z]);
                        }
                    }
                }
            } else {
                const int fu = mirrorSearch(cu + ou, vw.dimU);
                for (int r = 0; r < GH; ++r) {
                    if (cv0 + r >= vw.lv) break;
                    const uint32_t f2 = fetchPixel(vw.y2, vw.c2, vw.pitch, cv0 + r, cu);
                    const int bv = cv0 + r + ov;
#pragma unroll
                    for (int z = 0; z < R; ++z) acc[z] = sad4(fetchPixel(vw.y1, vw.c1, vw.pitch, mirrorSearch(bv + candOffset<R>(z), vw.dimV), fu), f2, acc[z]);
                }
            }
        }

        if (WS <= 4) {
            // windows of 2 or 4 lanes: reduce inside the segment; every lane then finalizes a slice of the layers
            bfly<16>(acc, 1, b0);
            if (WS == 4) bfly<8>(acc, 2, b1);
            WindowCtx c;
            c.o = 0;
            uint32_t bestT = 0xffffffffu;
            int bestZ = zbase < R ? zbase : 0xff;  // no layer beats a sum of 2^32-1: the lane's first layer stands, as with strict <
            if (winOk) {
                c = loadWindowCtx<STEP>(a, wx, wy, ox, oy);
#pragma unroll
                for (int i = 0; i < NZ; ++i) {
                    const int z = zbase + i;
                    if (R == 16 || z < R) {
                        const uint32_t total = layerTotal(a, c, acc[i], sqv[i]);
                        if (TAPS) tapTotal<R>(a, wx, wy, z, total);
                        if (total < bestT) {  // z ascends inside a lane: strict < keeps the lowest layer of a tie
                            bestT = total;
                            bestZ = z;
                        }
                    }
                }
            }
            unsigned long long best = layerKey(bestT, bestZ);
            best = min(best, shflXor64(best, 1));
            if (WS == 4) best = min(best, shflXor64(best, 2));
            if (winOk && (lane & (WS - 1)) == 0) {
                const int bestLayer = (int)(best & 0xff);
                const int16_t nOff = (int16_t)(c.o + signedSquare(bestLayer - R / 2));
                if (STEP == 0)
                    a.curX[wy * a.nWx + wx] = nOff;
                else
                    a.curY[wy * a.nWx + wx] = nOff;
                if (TAPS && a.tapLayer) a.tapLayer[wy * a.nWx + wx] = (uint8_t)bestLayer;
            }
        } else {
            bfly<16>(acc, 1, b0);
            bfly<8>(acc, 2, b1);
            bfly<4>(acc, 4, b2);
            int z0 = (b0 ? 8 : 0) + (b1 ? 4 : 0) + (b2 ? 2 : 0);
            const int lwin = ((cv0 - t.V0) >> L2) * NWU + (lane >> L2);
            if (WS == 8) {
                atomicAdd(&t.s_sums[lwin][z0], acc[0]);
                atomicAdd(&t.s_sums[lwin][z0 + 1], acc[1]);
            } else {  // WS == 16, 32
                bfly<2>(acc, 8, b3);
                z0 += b3 ? 1 : 0;
                if (WS == 32) {
                    acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 16);
                    if (lane < 16) atomicAdd(&t.s_sums[lwin][z0], acc[0]);
                } else
                    atomicAdd(&t.s_sums[lwin][z0], acc[0]);
            }
        }
    }
}

// Frame-2 samples of one window of 2 or 4 as they lie in the planes: WS luma rows (2 or 4 bytes each) and the WS/2 chroma
// rows under them.  Loaded one window ahead of the arithmetic (the first one before the tile is staged).
template <int WS> struct RawWindow {
    uint32_t y[WS], c[WS / 2];
};
template <int STEP, int WS> __device__ __forceinline__ RawWindow<WS> loadRawWindow(const View<STEP>& vw, int cu, int cv) {
    RawWindow<WS> w;
#pragma unroll
    for (int r = 0; r < WS; ++r) {
        const uint8_t* p = rowPtr(vw.y2, vw.pitch, cv + r) + cu;
        w.y[r] = WS == 2 ? (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(p)) : __ldg(reinterpret_cast<const uint32_t*>(p));
    }
#pragma unroll
    for (int r = 0; r < WS / 2; ++r) {
        const uint8_t* p = rowPtr(vw.c2, vw.pitch, (cv >> 1) + r) + cu;
        w.c[r] = WS == 2 ? (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(p)) : __ldg(reinterpret_cast<const uint32_t*>(p));
    }
    return w;
}
// window (column wl, row k of the warp's group `it`) of lane `lane` in warp `warp`: first pixel inside the tile
template <int WS> __device__ __forceinline__ void winOfLane(int lane, int warp, int it, int& wl, int& lwv) {
    constexpr int NWU = CT_U / WS, ROWS = 32 / NWU;
    wl = lane & (NWU - 1);
    lwv = (warp * 16) / WS + it * ROWS + lane / NWU;
}

// Windows of 2 or 4 flow pixels on a tile that needs no range checks: ONE LANE OWNS ONE WINDOW.  Its R sums stay in the
// lane's registers from the first SAD to the arg-min — no butterfly between lanes, the window's context (offsets of the
// four neighbours) is loaded once, and the arg-min needs no shuffle.  A warp covers 16 x 2 (ws = 2) or 8 x 4 (ws = 4)
// windows of its 16 tile rows.  Lanes of window row k visit the window's columns rotated by k, which spreads the 32
// lanes of one LDS over 32 banks (the window rows lie a multiple of 8 words apart).
template <int R, int STEP, bool TAPS, int WS>
__device__ __forceinline__ void winGroups(const SearchArgs& a, const View<STEP>& vw, const CandTile& t, int lane, int warp, RawWindow<WS> ahead) {
    constexpr int LO = candOffset<R>(0);
    constexpr int L2 = WS == 2 ? 1 : 2;
    constexpr int NWU = CT_U >> L2;          // windows across the tile: 16 / 8
    constexpr int ROWS = 32 / NWU;           // window rows a warp covers at once: 2 / 4
    constexpr int NIT = 16 / (ROWS * WS);    // iterations over the warp's 16 tile rows: 4 / 1
    const int k = lane / NWU;
#pragma unroll 1
    for (int it = 0; it < NIT; ++it) {
        int wl, lwv;  // window column / row inside the tile
        winOfLane<WS>(lane, warp, it, wl, lwv);
        const int cu = t.U0 + wl * WS, cv = t.V0 + lwv * WS;
        const RawWindow<WS> raw = ahead;
        if (it + 1 < NIT && cu < vw.lu && cv + ROWS * WS < vw.lv) ahead = loadRawWindow<STEP, WS>(vw, cu, cv + ROWS * WS);
        if (cu >= vw.lu || cv >= vw.lv) continue;  // tile at the end of the field: the window does not exist (windows are whole here)
        const int wu = cu >> L2, wv = cv >> L2;
        const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
        const int packed = t.s_off[lwv * NWU + wl];
        const int ou = (int)(short)(packed & 0xffff), ov = packed >> 16;
        const int ox = STEP == 1 ? ou : ov, oy = STEP == 1 ? ov : ou;
        const uint32_t* __restrict__ q = &t.s_f1[(cv - t.V0 + ov - t.minOv) * SP + (wl * WS + ou - t.minOu + t.sh)];

        // frame-2 pixels of the window as {Y, U, V, 0} words, columns in this lane's rotated order
        uint32_t f2[WS][WS];
        const uint32_t* qc[WS];
        if (WS == 2) {
            const uint32_t y0 = raw.y[0], y1 = raw.y[1], uv = raw.c[0];
            const uint32_t selA = k ? 0x7541u : 0x7540u, selB = k ? 0x7540u : 0x7541u;  // {Y_c, U, V, 0}
            f2[0][0] = __byte_perm(y0, uv, selA); f2[0][1] = __byte_perm(y0, uv, selB);
            f2[1][0] = __byte_perm(y1, uv, selA); f2[1][1] = __byte_perm(y1, uv, selB);
            qc[0] = q + k; qc[1] = q + (k ^ 1);
        } else {
            const uint32_t rot = k == 0 ? 0x3210u : k == 1 ? 0x0321u : k == 2 ? 0x1032u : 0x2103u;  // bytes rotated right by k
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                const uint32_t cw = raw.c[rr];
                const uint32_t cA = __byte_perm(cw, 0u, 0x4104), cB = __byte_perm(cw, 0u, 0x4324);  // {0, U, V, 0} of columns 0-1 / 2-3
#pragma unroll
                for (int r = 2 * rr; r < 2 * rr + 2; ++r) {
                    const uint32_t yw = __byte_perm(raw.y[r], 0u, rot);
#pragma unroll
                    for (int j = 0; j < 4; ++j) f2[r][j] = __byte_perm(yw, (((j + k) & 3) >> 1) ? cB : cA, 0x7650 + j);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) qc[j] = q + ((j + k) & 3);
        }

        uint32_t acc[16];
#pragma unroll
        for (int z = 0; z < 16; ++z) acc[z] = 0;
#pragma unroll
        for (int r = 0; r < WS; ++r)
#pragma unroll
            for (int z = 0; z < R; ++z)
#pragma unroll
                for (int j = 0; j < WS; ++j) acc[z] = sad4(qc[j][(r + candOffset<R>(z) - LO) * SP], f2[r][j], acc[z]);

        const WindowCtx c = loadWindowCtx<STEP>(a, wx, wy, ox, oy);
        uint32_t bestT = 0xffffffffu;
        int bestZ = 0;  // no layer beats a sum of 2^32-1: layer 0 stands, as with the reference's strict <
#pragma unroll
        for (int z = 0; z < R; ++z) {
            const uint32_t total = layerTotal(a, c, acc[z], candOffset<R>(z));
            if (TAPS) tapTotal<R>(a, wx, wy, z, total);
            if (total < bestT) {
                bestT = total;
                bestZ = z;
            }
        }
        const int16_t nOff = (int16_t)(c.o + signedSquare(bestZ - R / 2));
        if (STEP == 0)
            a.curX[wy * a.nWx + wx] = nOff;
        else
            a.curY[wy * a.nWx + wx] = nOff;
        if (TAPS && a.tapLayer) a.tapLayer[wy * a.nWx + wx] = (uint8_t)bestZ;
    }
}

template <int R, int STEP, bool TAPS, int WS> __global__ void __launch_bounds__(256, 4) sadCandKernel(const SearchArgs a) {
    constexpr int LO = candOffset<R>(0), HI = candOffset<R>(R - 1), SPAN = HI - LO;
    constexpr int wsLog2 = WS == 2 ? 1 : WS == 4 ? 2 : WS == 8 ? 3 : WS == 16 ? 4 : 5;
    constexpr int nwu = CT_U >> wsLog2, nwv = CT_V >> wsLog2;  // windows of the tile along u, v
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* __restrict__ s_f1 = smem;                                        // [RV_MAX][SP]
    uint32_t (*s_sums)[16] = reinterpret_cast<uint32_t (*)[16]>(smem + RV_MAX * SP);  // [window inside the tile][layer] (ws >= 8)
    int* __restrict__ s_off = reinterpret_cast<int*>(smem + RV_MAX * SP + candSumWords<WS>());  // per window: (ou & 0xffff) | (ov << 16)
    int* __restrict__ s_rng = s_off + candWindows<WS>();                       // min ou, max ou, min ov, max ov

    const View<STEP> vw(a);
    const int lane = threadIdx.x, warp = threadIdx.y;
    const int tid = warp * 32 + lane;
    const int U0 = blockIdx.x * CT_U, V0 = blockIdx.y * CT_V;
    // A sharded pass (split search) launches its grid from flow row 0 and the CTAs above the stripe return here: the tile
    // origin stays plain blockIdx arithmetic, which this kernel (64 registers) cannot afford to keep an offset for.
    // (u0, v0) is a multiple of 128, so the remaining tiles are exactly those of a grid started at the stripe.
    if ((STEP == 1 ? V0 : U0) < a.rowBegin) return;  // CTA-uniform, before any barrier

    // windows of 2 and 4 on a full tile: frame-2 samples of the lane's first window, in flight while the tile is staged
    constexpr int WSW = WS <= 4 ? WS : 2;
    const bool fullTile = U0 + CT_U <= vw.lu && V0 + CT_V <= vw.lv;
    // one lane per window wherever the tile holds whole windows only
    const bool winTile = WS <= 4 && a.winLanes && (fullTile || (vw.lu % WSW == 0 && vw.lv % WSW == 0));
    RawWindow<WSW> ahead = {};
    if (winTile) {
        int wl, lwv;
        winOfLane<WSW>(lane, warp, 0, wl, lwv);
        if (U0 + wl * WSW < vw.lu && V0 + lwv * WSW < vw.lv) ahead = loadRawWindow<STEP, WSW>(vw, U0 + wl * WSW, V0 + lwv * WSW);
    }

    // ---- A. offsets of the tile's windows, and their range ------------------------------------------------------
    if (tid < 4) s_rng[tid] = (tid & 1) ? INT_MIN : INT_MAX;
    if (WS >= 8)
        for (int i = tid; i < nwu * nwv * 16; i += 256) s_sums[0][i] = 0;
    __syncthreads();
    {
        int mnU = INT_MAX, mxU = INT_MIN, mnV = INT_MAX, mxV = INT_MIN;
#pragma unroll
        for (int i0 = 0; i0 < nwu * nwv; i0 += 256) {
            const int i = i0 + tid;
            if (nwu * nwv >= 256 || i < nwu * nwv) {
                const int lwu = i % nwu, lwv = i / nwu;
                const int wu = (U0 >> wsLog2) + lwu, wv = (V0 >> wsLog2) + lwv;
                int packed = 0;
                if ((wu << wsLog2) < vw.lu && (wv << wsLog2) < vw.lv) {
                    int ox, oy;
                    loadWindowOffsets<STEP>(a, View<STEP>::wx(wu, wv), View<STEP>::wy(wu, wv), ox, oy);
                    const int ou = View<STEP>::ou(ox, oy), ov = View<STEP>::ov(ox, oy);
                    packed = (ou & 0xffff) | (ov << 16);
                    mnU = min(mnU, ou); mxU = max(mxU, ou); mnV = min(mnV, ov); mxV = max(mxV, ov);
                }
                s_off[i] = packed;
            }
        }
        mnU = __reduce_min_sync(0xffffffffu, mnU); mxU = __reduce_max_sync(0xffffffffu, mxU);
        mnV = __reduce_min_sync(0xffffffffu, mnV); mxV = __reduce_max_sync(0xffffffffu, mxV);
        if (lane == 0) {
            atomicMin(&s_rng[0], mnU); atomicMax(&s_rng[1], mxU); atomicMin(&s_rng[2], mnV); atomicMax(&s_rng[3], mxV);
        }
    }
    __syncthreads();
    const int minOu = s_rng[0], minOv = s_rng[2];
    const int tileRows = min(CT_V, vw.lv - V0);  // flow rows of this tile that exist
    const int RU = CT_U + (s_rng[1] - minOu), RV = tileRows + SPAN + (s_rng[3] - minOv);
    const bool staged = RU <= RU_MAX && RV <= RV_MAX;  // CTA-uniform

    // ---- B. stage the frame-1 region ------------------------------------------------------------------------------
    const int cb = U0 + minOu;            // first column any candidate reads
    const int ca = cb & ~3;               // 16-byte aligned start of the staged rows
    const int sh = cb - ca;
    const int rb = V0 + minOv + LO;       // first row any candidate reads
    if (staged) {
        // Whole rows are copied word by word (4 pixels), through the reference's mirror where the region leaves the frame
        // (calcDeltaSumsKernelSDR.h:86-95 reflects each coordinate on its own): rows by a mirrored row index; a word of four
        // columns beyond the left / right edge is the aligned word at the reflected position with its pixels reversed —
        // luma bytes reversed, the two chroma pairs swapped (frame widths that are multiples of 4 keep words from
        // straddling the edge).
        const bool colsFast = (vw.dimU & 3) == 0 && ca >= -vw.dimU && ca + SP <= 2 * vw.dimU;
        if (colsFast) {
            // the region is assembled from the planes: one luma word and one chroma word give four {Y,U,V,0} words
            // (expand4); four rows per iteration keep eight loads of a thread in flight
            const int c4 = tid & 15;
            if (c4 < SP / 4) {
                const int cc = ca + c4 * 4;
                const bool rev = cc < 0 || cc >= vw.dimU;
                const int src = cc < 0 ? -cc - 4 : cc >= vw.dimU ? 2 * vw.dimU - cc - 4 : cc;
                const uint32_t selY = rev ? 0x0123u : 0x3210u, selC = rev ? 0x1032u : 0x3210u;
                const uint8_t* __restrict__ ysrc = vw.y1 + src;
                const uint8_t* __restrict__ csrc = vw.c1 + src;
                for (int r = tid >> 4; r < RV; r += 64) {
                    uint32_t yw[4], cw[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int mr = mirrorSearch(rb + min(r + 16 * i, RV - 1), vw.dimV);
                        yw[i] = __ldg(reinterpret_cast<const uint32_t*>(rowPtr(ysrc, vw.pitch, mr)));
                        cw[i] = __ldg(reinterpret_cast<const uint32_t*>(rowPtr(csrc, vw.pitch, mr >> 1)));
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int rr = r + 16 * i;
                        if (rr < RV) {
                            uint32_t w[4];
                            expand4(__byte_perm(yw[i], 0u, selY), __byte_perm(cw[i], 0u, selC), w);
                            *reinterpret_cast<uint4*>(&s_f1[rr * SP + c4 * 4]) = make_uint4(w[0], w[1], w[2], w[3]);
                        }
                    }
                }
            }
        } else {
            for (int idx = tid; idx < RV * SP; idx += 256) {
                const int r = idx / SP, c = idx - r * SP;
                s_f1[idx] = fetchPixel(vw.y1, vw.c1, vw.pitch, mirrorSearch(rb + r, vw.dimV), mirrorSearch(ca + c, vw.dimU));
            }
        }
    }
    __syncthreads();

    // ---- C. SADs, reduction per window ----------------------------------------------------------------------------
    CandTile t;
    t.s_f1 = s_f1; t.s_sums = s_sums; t.s_off = s_off;
    t.U0 = U0; t.V0 = V0; t.minOu = minOu; t.minOv = minOv; t.sh = sh; t.staged = staged;
    if (staged && winTile)
        winGroups<R, STEP, TAPS, WSW>(a, vw, t, lane, warp, ahead);
    else if (staged && fullTile)
        candGroups<R, STEP, TAPS, WS, true>(a, vw, t, lane, warp);
    else
        candGroups<R, STEP, TAPS, WS, false>(a, vw, t, lane, warp);

    if (WS >= 8) {
        __syncthreads();
        if (tid < nwu * nwv) {
            const int wu = (U0 >> wsLog2) + (tid % nwu), wv = (V0 >> wsLog2) + (tid / nwu);
            const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
            // (tiles start at multiples of 32 / 128 from a stripe origin, a multiple of 128: a tile never crosses an
            // interior stripe end, so the field bound is the stripe bound)
            if (wx < a.nWx && wy < a.nWy) finalizeWindow<R, STEP>(a, wx, wy, s_sums[tid]);
        }
    }
}

template <int R, int STEP, bool TAPS, int WS> int launchCandOne(hrb_ofc* h, const SearchArgs& a) {
    const int rc = allowDynamicSmem<sadCandKernel<R, STEP, TAPS, WS>>(h->device, (int)candSmem<WS>());
    if (rc) return rc;
    const PassRange r = passRange(a, STEP);  // up to the end of the pass's rows: a stripe on a shard of a split search
    const dim3 grid((r.lu + CT_U - 1) / CT_U, (r.lv + CT_V - 1) / CT_V, 1);
    sadCandKernel<R, STEP, TAPS, WS><<<grid, dim3(32, 8, 1), candSmem<WS>(), h->stream>>>(a);
    HRB_LAUNCH_CHECK();
    return HRB_OK;
}

template <int R, int STEP, bool TAPS> int launchCandWs(hrb_ofc* h, const SearchArgs& a) {
    switch (a.ws) {
        case 2: return launchCandOne<R, STEP, TAPS, 2>(h, a);
        case 4: return launchCandOne<R, STEP, TAPS, 4>(h, a);
        case 8: return launchCandOne<R, STEP, TAPS, 8>(h, a);
        case 16: return launchCandOne<R, STEP, TAPS, 16>(h, a);
        case 32: return launchCandOne<R, STEP, TAPS, 32>(h, a);
    }
    setLastError("[hopperrender_b200] small-window kernel, window size %d: no such kernel instance", a.ws);
    return HRB_ERR_STATE;
}

}  // namespace

// One whole pass (SAD + arg-min + offset update) for 2 <= ws <= 32 at full flow resolution, for the radii of part PART
// (hrb_internal.cuh): the 12 search radii x 2 steps x 2 (taps) x 5 window sizes are 240 kernels.
template <int PART> int launchCandPart(hrb_ofc* h, const SearchArgs& pass, const SearchPlan& p, int R, int step) {
    SearchArgs a = pass;
    a.winLanes = p.winLanes;
    const bool taps = a.tapSums || a.tapLayer || a.rawDelta;
    return withConstant<firstRadiusOf(PART), firstRadiusOf(PART) + 3>("small-window kernel, search radius", R, [&](auto r) {
        constexpr int RC = decltype(r)::value;
        if (step == 1) return taps ? launchCandWs<RC, 1, true>(h, a) : launchCandWs<RC, 1, false>(h, a);
        return taps ? launchCandWs<RC, 0, true>(h, a) : launchCandWs<RC, 0, false>(h, a);
    });
}
template int launchCandPart<HRB_SEARCH_PART>(hrb_ofc* h, const SearchArgs& pass, const SearchPlan& p, int R, int step);

}  // namespace hrb
