// kernels_search.cu — the pyramidal block-matching search and the flow blur.
//
// One search pass = calcDeltaSumsKernel + determineLowestLayerKernel + adjustOffsetArrayKernel of the
// reference (HopperRender/opticalFlowCalcSDR.cpp:72-107) for one (iteration, step).  The design uses
// three facts (SURVEY.md A.1, A.3):
//   * the search only looks at 8-bit data, so both frames are kept as 8-bit planes (luma + NV12-style chroma, in both
//     orientations); the generic kernel below assembles {Y,U,V,0} words, so that one VABSDIFF4.U8.ACC evaluates the
//     reference's 3-term delta for one pixel-candidate, the specialised kernels work on the planes directly;
//   * offsets are constant inside each aligned window, so they live in per-window arrays and the
//     offset / neighbour bias of a window is (pixel count) x (a per-window constant);
//   * sums are uint32 modulo 2^32, so any summation order is bit-exact.
// Nothing is zero-filled or materialised per flow pixel: windows that fit a CTA tile are reduced and
// arg-min'ed inside the SAD kernel; larger windows go through R atomics per tile, the last tile of a window finalizes it.
#include "search_common.cuh"

namespace hrb {

namespace {

// ------------------------------------------------------------------------------------------------
// The generic SAD pass (any window size, any resolution scalar).  CTA = 8 warps over a TILE x TILE block of
// flow pixels in (u, v) coordinates (see View); a warp owns 4 consecutive v, a lane one u.  R is compile-time
// so the candidate displacements fold into the address arithmetic.
// ------------------------------------------------------------------------------------------------
// The arguments of the pass a CTA computes: a lone pass's, or those of member blockIdx.z of a flow batch (hrb_flow_batch)
__device__ __forceinline__ const SearchArgs& passArgs(const SearchArgs& a) { return a; }
__device__ __forceinline__ const SearchArgs& passArgs(const SearchBatch& b) { return b.m[blockIdx.z]; }

template <int R, int STEP, bool WIDE, class P> __global__ void __launch_bounds__(256) sadPassKernel(const __grid_constant__ P p) {
    const SearchArgs a = passArgs(p);  // a copy: the lone instances compile exactly as when a was the parameter itself
    __shared__ uint32_t s_sums[16][16];  // [window inside the tile][layer]
    const View<STEP> vw(a);
    const int lane = threadIdx.x, warp = threadIdx.y;
    const int tid = warp * 32 + lane;
    const int ws = a.ws;
    const bool small = ws <= 4;
    if (!small) {
        s_sums[tid >> 4][tid & 15] = 0;
        __syncthreads();
    }
    const int U0 = vw.u0 + blockIdx.x * TILE, V0 = vw.v0 + blockIdx.y * TILE;  // (u0, v0): multiples of kSplitAlign
    const int cu = U0 + lane;
    const int rowBase = V0 + warp * 4;
    const int gh = ws < 4 ? ws : 4;  // rows of one accumulation group (inside one window row)
    constexpr int LO = candOffset<R>(0), HI = candOffset<R>(R - 1);

    for (int g = 0; g < 4; g += gh) {
        const int cv0 = rowBase + g;
        const int wu = cu >> a.wsLog2, wv = cv0 >> a.wsLog2;
        const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
        const bool pixOk = cu < vw.lu && cv0 < vw.lv;                 // this lane has pixels to accumulate
        const bool winOk = (wu << a.wsLog2) < vw.lu && cv0 < vw.lv;   // this lane's window exists (it may finalize a slice of it)
        uint32_t acc[16];
#pragma unroll
        for (int z = 0; z < 16; ++z) acc[z] = 0;
        int ox = 0, oy = 0;
        if (winOk) loadWindowOffsets<STEP>(a, wx, wy, ox, oy);
        if (pixOk) {
            const int su = cu << a.rs;
            const int ou = View<STEP>::ou(ox, oy), ov = View<STEP>::ov(ox, oy);
            const int fu = mirrorSearch(su + ou, vw.dimU);  // frame-1 column of this lane
            // WIDE (flow fields of a few hundred tiles at most): the rows of the group are independent; unrolled, the loads of all
            // of them are in flight together — a pass over so few tiles is bound by the latency of its dependent loads, not by
            // their number.  Larger fields keep the rolled loop (fewer registers, more resident warps).
#pragma unroll(WIDE ? 4 : 1)
            for (int r = 0; r < 4; ++r) {
                const int cv = min(cv0 + r, vw.lv - 1);
                const bool rowOk = r < gh && cv0 + r < vw.lv;
                const int sv = cv << a.rs;
                const uint32_t f2 = fetchPixel(vw.y2, vw.c2, vw.pitch, sv, su);
                const int bv = sv + ov;
                if (bv + LO >= 0 && bv + HI < vw.dimV) {
#pragma unroll
                    for (int z = 0; z < R; ++z) {
                        const uint32_t s = sad4(fetchPixel(vw.y1, vw.c1, vw.pitch, bv + candOffset<R>(z), fu), f2, 0u);
                        if (rowOk) acc[z] += s;
                    }
                } else {
#pragma unroll
                    for (int z = 0; z < R; ++z) {
                        const uint32_t s = sad4(fetchPixel(vw.y1, vw.c1, vw.pitch, mirrorSearch(bv + candOffset<R>(z), vw.dimV), fu), f2, 0u);
                        if (rowOk) acc[z] += s;
                    }
                }
            }
        }

        const bool b0 = lane & 1, b1 = lane & 2, b2 = lane & 4, b3 = lane & 8;
        if (small) {
            // windows of 2 or 4 lanes x gh rows: reduce inside the segment, every lane finalizes a slice of the layers
            bfly<16>(acc, 1, b0);
            int n = 8, zbase = b0 ? 8 : 0;
            if (ws == 4) {
                bfly<8>(acc, 2, b1);
                n = 4;
                zbase += b1 ? 4 : 0;
            }
            WindowCtx c;
            c.o = 0;
            if (winOk) c = loadWindowCtx<STEP>(a, wx, wy, ox, oy);
            unsigned long long best = ~0ull;
            if (winOk) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int z = zbase + i;
                    if (i < n && z < R) {
                        const uint32_t total = windowTotal<R>(a, c, acc[i], z);
                        tapTotal<R>(a, wx, wy, z, total);
                        best = min(best, layerKey(total, z));
                    }
                }
            }
            best = min(best, shflXor64(best, 1));
            if (ws == 4) best = min(best, shflXor64(best, 2));
            if (winOk && (lane & (ws - 1)) == 0) commitWindow<R, STEP>(a, wx, wy, c.o, (int)(best & 0xff));
        } else {
            // windows of >= 8 lanes: reduce over min(ws, 32) lanes, then accumulate in shared memory
            bfly<16>(acc, 1, b0);
            bfly<8>(acc, 2, b1);
            bfly<4>(acc, 4, b2);
            int z0 = (b0 ? 8 : 0) + (b1 ? 4 : 0) + (b2 ? 2 : 0);
            int lwin = 0;
            if (ws <= TILE) lwin = ((cv0 - V0) >> a.wsLog2) * (TILE >> a.wsLog2) + (lane >> a.wsLog2);
            if (ws == 8) {
                atomicAdd(&s_sums[lwin][z0], acc[0]);
                atomicAdd(&s_sums[lwin][z0 + 1], acc[1]);
            } else {
                bfly<2>(acc, 8, b3);
                z0 += b3 ? 1 : 0;
                if (ws == 16) {
                    atomicAdd(&s_sums[lwin][z0], acc[0]);
                } else {
                    acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 16);
                    if (lane < 16) atomicAdd(&s_sums[lwin][z0], acc[0]);
                }
            }
        }
    }

    if (!small) {
        __syncthreads();
        if (ws <= TILE) {
            const int perEdge = TILE >> a.wsLog2;
            if (tid < perEdge * perEdge) {
                const int wu = (U0 >> a.wsLog2) + (tid % perEdge);
                const int wv = (V0 >> a.wsLog2) + (tid / perEdge);
                const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
                if ((wu << a.wsLog2) < vw.lu && (wv << a.wsLog2) < vw.lv) finalizeWindow<R, STEP>(a, wx, wy, s_sums[tid]);
            }
        } else {
            // the tile lies inside one window larger than the tile: add to the window's global sums; the CTA that
            // arrives last (ticket) finds them complete, does the arg-min and leaves sums and ticket zeroed for the next pass.
            // In a sharded pass every tile of an owned window lies inside the stripe, so the ticket count is unchanged.
            __shared__ bool s_last;
            const int wu = U0 >> a.wsLog2, wv = V0 >> a.wsLog2;
            const int wx = View<STEP>::wx(wu, wv), wy = View<STEP>::wy(wu, wv);
            const size_t w = (size_t)(wy * a.nWx + wx);
            if (tid < R) {
                atomicAdd(&a.winSums[w * 16 + tid], s_sums[0][tid]);
                __threadfence();
            }
            __syncthreads();
            if (tid == 0) {
                const int x0 = wx << a.wsLog2, y0 = wy << a.wsLog2;
                const unsigned tiles = (unsigned)(((min(ws, a.lw - x0) + TILE - 1) / TILE) * ((min(ws, a.lh - y0) + TILE - 1) / TILE));
                s_last = atomicAdd(&a.winTicket[w], 1u) == tiles - 1;
            }
            __syncthreads();
            if (s_last && tid == 0) {
                __threadfence();
                uint32_t sums[16];
#pragma unroll
                for (int z = 0; z < 16; ++z) {
                    sums[z] = z < R ? __ldcg(&a.winSums[w * 16 + z]) : 0u;
                    if (z < R) a.winSums[w * 16 + z] = 0;
                }
                a.winTicket[w] = 0;
                finalizeWindow<R, STEP>(a, wx, wy, sums);
            }
        }
    }
}

// the generic kernel; windows larger than its tile are finalized by the last CTA of each window
template <int R> int launchGeneric(hrb_ofc* h, const SearchArgs& a, int step) {
    const dim3 block(32, 8, 1);
    const PassRange r = passRange(a, step);  // X steps run on the transposed planes (View)
    const dim3 grid((r.lu - r.u0 + TILE - 1) / TILE, (r.lv - r.v0 + TILE - 1) / TILE, 1);
    const bool wide = grid.x * grid.y <= 2u * (unsigned)h->smCount;
    if (step == 0) {
        if (wide)
            sadPassKernel<R, 0, true, SearchArgs><<<grid, block, 0, h->stream>>>(a);
        else
            sadPassKernel<R, 0, false, SearchArgs><<<grid, block, 0, h->stream>>>(a);
    } else {
        if (wide)
            sadPassKernel<R, 1, true, SearchArgs><<<grid, block, 0, h->stream>>>(a);
        else
            sadPassKernel<R, 1, false, SearchArgs><<<grid, block, 0, h->stream>>>(a);
    }
    HRB_LAUNCH_CHECK();
    return HRB_OK;
}

// one generic pass over the members of a flow batch: one launch, grid z = member
template <int R> int launchGenericBatch(cudaStream_t st, int smCount, const SearchBatch& b, int n, int step) {
    const dim3 block(32, 8, 1);
    const PassRange r = passRange(b.m[0], step);
    const dim3 grid((r.lu - r.u0 + TILE - 1) / TILE, (r.lv - r.v0 + TILE - 1) / TILE, (unsigned)n);
    const bool wide = grid.x * grid.y * grid.z <= 2u * (unsigned)smCount;
    if (step == 0) {
        if (wide)
            sadPassKernel<R, 0, true, SearchBatch><<<grid, block, 0, st>>>(b);
        else
            sadPassKernel<R, 0, false, SearchBatch><<<grid, block, 0, st>>>(b);
    } else {
        if (wide)
            sadPassKernel<R, 1, true, SearchBatch><<<grid, block, 0, st>>>(b);
        else
            sadPassKernel<R, 1, false, SearchBatch><<<grid, block, 0, st>>>(b);
    }
    HRB_LAUNCH_CHECK();
    return HRB_OK;
}

// ------------------------------------------------------------------------------------------------
// blurFlowKernel — blurFlowKernelSDR.h:17-92: 8x8 box (taps -4..+3), mirrored borders, int sum / 64.
// Reads the window-level offsets of the last pass directly (value of flow pixel (x,y) = level[y>>s][x>>s]).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int mirrorBlur(int pos, int dim) {  // blurFlowKernelSDR.h:7-14
    if (pos >= dim) return dim - (pos - dim + 1);
    if (pos < 0) return -pos - 1;
    return pos;
}

constexpr int BT = 32;          // outputs per tile edge
constexpr int BIN = BT + 7;     // input rows / columns a tile needs

// axis 0 blurs lvl into the X plane of out, axis 1 into the Y plane
__device__ __forceinline__ void blurFlow(const int16_t* __restrict__ lvl, int axis, int nWx, int wsLog2, int16_t* __restrict__ out, int lw, int lh,
                                         uint32_t* __restrict__ flowMax) {
    __shared__ int16_t s_in[BIN][BIN + 1];
    __shared__ int s_h[BIN][BT];
    const int X0 = blockIdx.x * BT, Y0 = blockIdx.y * BT;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    for (int i = tid; i < BIN * BIN; i += 256) {
        const int r = i / BIN, c = i % BIN;
        const int y = min(max(mirrorBlur(Y0 - 4 + r, lh), 0), lh - 1);
        const int x = min(max(mirrorBlur(X0 - 4 + c, lw), 0), lw - 1);
        s_in[r][c] = lvl[(y >> wsLog2) * nWx + (x >> wsLog2)];
    }
    __syncthreads();
    for (int i = tid; i < BIN * BT; i += 256) {
        const int r = i / BT, c = i % BT;
        int s = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += s_in[r][c + k];
        s_h[r][c] = s;
    }
    __syncthreads();
    const int x = X0 + threadIdx.x;
    int peak = 0;  // largest |flow| this thread wrote: bounds every displacement warpFrames can apply
    if (x < lw) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ly = threadIdx.y * 4 + j;
            const int y = Y0 + ly;
            if (y >= lh) break;
            int s = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) s += s_h[ly + k][threadIdx.x];
            const int v = s / 64;
            out[(size_t)axis * lw * lh + (size_t)y * lw + x] = (int16_t)v;
            peak = max(peak, abs(v));
        }
    }
    peak = __reduce_max_sync(0xffffffffu, peak);
    if (threadIdx.x == 0 && (uint32_t)peak > *reinterpret_cast<volatile uint32_t*>(flowMax)) atomicMax(flowMax, (uint32_t)peak);
}

__global__ void __launch_bounds__(256) blurFlowKernel(const int16_t* __restrict__ lvlX, const int16_t* __restrict__ lvlY, int nWx, int wsLog2,
                                                     int16_t* __restrict__ out, int lw, int lh, uint32_t* __restrict__ flowMax) {
    blurFlow(blockIdx.z == 0 ? lvlX : lvlY, blockIdx.z, nWx, wsLog2, out, lw, lh, flowMax);
}

// over the members of a flow batch: blockIdx.z = 2 * member + axis
__global__ void __launch_bounds__(256) blurFlowBatchKernel(const __grid_constant__ BlurBatch b, int nWx, int wsLog2, int lw, int lh) {
    const BlurMember& m = b.m[blockIdx.z >> 1];
    const int axis = blockIdx.z & 1;
    blurFlow(axis ? m.lvlY : m.lvlX, axis, nWx, wsLog2, m.out, lw, lh, m.flowMax);
}

// Fast path for the usual case — last pass at 2x2 windows, even flow dimensions.  The field is constant on aligned 2x2
// cells, so the 8 taps of an even output coordinate 2c cover cells c-2..c+1 twice each, and those of an odd coordinate
// 2c+1 cover c-2 and c+2 once and c-1..c+1 twice; the mirror rule maps to cells unchanged (column -1-p <-> cell -1-c).
// Both passes therefore run on the cell grid: 5 loads give the two horizontal sums of a cell, 5 more per sum give the
// four outputs of the cell.  Same integer sums as blurFlowKernel, a sixth of the instructions.
constexpr int BC_W = 32, BC_H = 16;  // cells per tile -> 64 x 32 outputs

__device__ __forceinline__ int mirrorCell(int c, int n) { return c < 0 ? -c - 1 : (c >= n ? 2 * n - c - 1 : c); }
__device__ __forceinline__ int div64(int s) { return (s + ((s >> 31) & 63)) >> 6; }  // C division: truncates toward zero

__device__ __forceinline__ void blurFlowCell(const int16_t* __restrict__ lvl, int axis, int nCx, int nCy, int16_t* __restrict__ out, int lw, int lh,
                                             uint32_t* __restrict__ flowMax) {
    __shared__ int16_t s_in[BC_H + 4][BC_W + 4 + 2];
    __shared__ int s_he[BC_H + 4][BC_W], s_ho[BC_H + 4][BC_W];
    const int C0 = blockIdx.x * BC_W, R0 = blockIdx.y * BC_H;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    for (int i = tid; i < (BC_H + 4) * (BC_W + 4); i += 256) {
        const int r = i / (BC_W + 4), c = i - r * (BC_W + 4);
        const int cy = min(mirrorCell(R0 - 2 + r, nCy), nCy - 1), cx = min(mirrorCell(C0 - 2 + c, nCx), nCx - 1);
        s_in[r][c] = lvl[cy * nCx + cx];
    }
    __syncthreads();
    for (int i = tid; i < (BC_H + 4) * BC_W; i += 256) {
        const int r = i >> 5, c = i & 31;
        const int l0 = s_in[r][c], l4 = s_in[r][c + 4];
        const int mid = s_in[r][c + 1] + s_in[r][c + 2] + s_in[r][c + 3];
        s_he[r][c] = 2 * (mid + l0);
        s_ho[r][c] = 2 * mid + l0 + l4;
    }
    __syncthreads();
    int peak = 0;  // largest |flow| this thread wrote: bounds every displacement warpFrames can apply
    const int cx = C0 + threadIdx.x;
    if (cx < nCx) {
        int16_t* __restrict__ o = out + (size_t)axis * lw * lh;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int r = threadIdx.y * 2 + j;
            const int cy = R0 + r;
            if (cy >= nCy) break;
            const int e0 = s_he[r][threadIdx.x], e4 = s_he[r + 4][threadIdx.x];
            const int em = s_he[r + 1][threadIdx.x] + s_he[r + 2][threadIdx.x] + s_he[r + 3][threadIdx.x];
            const int o0 = s_ho[r][threadIdx.x], o4 = s_ho[r + 4][threadIdx.x];
            const int om = s_ho[r + 1][threadIdx.x] + s_ho[r + 2][threadIdx.x] + s_ho[r + 3][threadIdx.x];
            const int v00 = div64(2 * (em + e0)), v01 = div64(2 * (om + o0));        // row 2cy:   columns 2cx, 2cx+1
            const int v10 = div64(2 * em + e0 + e4), v11 = div64(2 * om + o0 + o4);  // row 2cy+1
            *reinterpret_cast<uint32_t*>(o + (size_t)(2 * cy) * lw + 2 * cx) = (uint32_t)(uint16_t)v00 | ((uint32_t)(uint16_t)v01 << 16);
            *reinterpret_cast<uint32_t*>(o + (size_t)(2 * cy + 1) * lw + 2 * cx) = (uint32_t)(uint16_t)v10 | ((uint32_t)(uint16_t)v11 << 16);
            peak = max(max(peak, max(abs(v00), abs(v01))), max(abs(v10), abs(v11)));
        }
    }
    peak = __reduce_max_sync(0xffffffffu, peak);
    if (threadIdx.x == 0 && (uint32_t)peak > *reinterpret_cast<volatile uint32_t*>(flowMax)) atomicMax(flowMax, (uint32_t)peak);
}

__global__ void __launch_bounds__(256) blurFlowCellKernel(const int16_t* __restrict__ lvlX, const int16_t* __restrict__ lvlY, int nCx, int nCy,
                                                         int16_t* __restrict__ out, int lw, int lh, uint32_t* __restrict__ flowMax) {
    blurFlowCell(blockIdx.z == 0 ? lvlX : lvlY, blockIdx.z, nCx, nCy, out, lw, lh, flowMax);
}

__global__ void __launch_bounds__(256) blurFlowCellBatchKernel(const __grid_constant__ BlurBatch b, int nCx, int nCy, int lw, int lh) {
    const BlurMember& m = b.m[blockIdx.z >> 1];
    const int axis = blockIdx.z & 1;
    blurFlowCell(axis ? m.lvlY : m.lvlX, axis, nCx, nCy, m.out, lw, lh, m.flowMax);
}

// per-pixel offsetArray [2][lh][lw] from window-level arrays (test taps only)
__global__ void expandOffsetsKernel(const int16_t* __restrict__ lvlX, int nWxX, int sX, const int16_t* __restrict__ lvlY, int nWxY, int sY,
                                    int16_t* __restrict__ out, int lw, int lh) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= lw || y >= lh) return;
    out[(size_t)y * lw + x] = lvlX ? lvlX[(y >> sX) * nWxX + (x >> sX)] : (int16_t)0;
    out[(size_t)lw * lh + (size_t)y * lw + x] = lvlY ? lvlY[(y >> sY) * nWxY + (x >> sY)] : (int16_t)0;
}

// peak-issue microbenchmark of the packed SAD instruction: 8 independent accumulator chains per thread
__global__ void __launch_bounds__(256) sadPeakKernel(uint32_t* out, uint32_t seed, int iters) {
    uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3u, a2 = a0 * 5u, a3 = a0 * 7u, a4 = a0 * 11u, a5 = a0 * 13u, a6 = a0 * 17u, a7 = a0 * 19u;
    const uint32_t b = seed * 0x9e3779b9u + blockIdx.x;
    uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0, c5 = 0, c6 = 0, c7 = 0;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            c0 = sad4(a0, b, c0); c1 = sad4(a1, b, c1); c2 = sad4(a2, b, c2); c3 = sad4(a3, b, c3);
            c4 = sad4(a4, b, c4); c5 = sad4(a5, b, c5); c6 = sad4(a6, b, c6); c7 = sad4(a7, b, c7);
        }
        a0 ^= c7;  // keeps the loop from being hoisted; 1 extra op per 64 SADs
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = c0 + c1 + c2 + c3 + c4 + c5 + c6 + c7;
}

}  // namespace

SearchPlan planSearchPass(int variant, const SearchArgs& a, int R, int step) {
    // The tile and small-window kernels run radii of 5 and more on full-resolution flows, on the planar planes; variant 1
    // runs the generic kernel everywhere.  The tile kernel needs whole 4-pixel columns along u, over the whole field
    // (also on a shard of a split search).  It covers windows of 4 and 8 too (variants 2 and 3 run it there, which is how
    // the parity tests reach those classes), but the small-window kernel is faster on them and is the default.
    const bool planar = R >= 5 && a.rs == 0 && variant != 1;
    const int minWs = variant == 2 || variant == 3 ? 4 : 16;
    const int lu = step == 1 ? a.lw : a.lh;
    SearchPlan p;
    p.kernel = planar && a.ws >= minWs && lu % 4 == 0 ? SearchPlan::Tile : planar && a.ws <= 32 ? SearchPlan::Cand : SearchPlan::Generic;
    p.useTma = variant != 2;
    p.forceSlow = variant == 3;
    p.winLanes = variant != 4;
    return p;
}

static int checkRadius(int R) {
    if (R < 2 || R > 16) {
        setLastError("[hopperrender_b200] search radius %d outside 2..16", R);
        return HRB_ERR_INVALID_ARG;
    }
    return HRB_OK;
}

static int launchPlannedPass(hrb_ofc* h, const SearchArgs& a, const SearchPlan& p, int R, int step) {
    profBegin(h, CLS_SEARCH);
    int rc;
    if (p.kernel == SearchPlan::Tile)
        rc = withConstant<0, kSearchParts - 1>("tile kernel, search part", searchPart(R),
                                               [&](auto part) { return launchTilePart<decltype(part)::value>(h, a, p, R, step); });
    else if (p.kernel == SearchPlan::Cand)
        rc = withConstant<0, kSearchParts - 1>("small-window kernel, search part", searchPart(R),
                                               [&](auto part) { return launchCandPart<decltype(part)::value>(h, a, p, R, step); });
    else
        rc = withConstant<2, 16>("generic kernel, search radius", R, [&](auto r) { return launchGeneric<decltype(r)::value>(h, a, step); });
    profEnd(h, CLS_SEARCH, rc == HRB_OK ? 1 : 0);
    return rc;
}

int launchSearchPass(hrb_ofc* h, const SearchArgs& a, int R, int step) {
    const int rc = checkRadius(R);
    if (rc) return rc;
    return launchPlannedPass(h, a, planSearchPass(h->searchVariant, a, R, step), R, step);
}

int launchSearchBatch(hrb_ofc* const* h, const SearchBatch& b, int n, int R, int step) {
    int rc = checkRadius(R);
    if (rc) return rc;
    // the plan depends only on the variant, the geometry, R and the step, on which the members agree
    const SearchPlan p = planSearchPass(h[0]->searchVariant, b.m[0], R, step);
    if (p.kernel != SearchPlan::Generic) {
        for (int k = 0; k < n && !rc; ++k) rc = launchPlannedPass(h[k], b.m[k], p, R, step);
        return rc;
    }
    rc = withConstant<2, 16>("generic kernel, search radius", R,
                             [&](auto r) { return launchGenericBatch<decltype(r)::value>(h[0]->stream, h[0]->smCount, b, n, step); });
    for (int k = 0; k < n && !rc; ++k) profEnd(h[k], CLS_SEARCH, 1);  // each member's pass ran in one launch
    return rc;
}

int launchBlurFlow(hrb_ofc* h, const int16_t* lvlX, const int16_t* lvlY, int nWx, int wsLog2, int16_t* out, uint32_t* flowMax) {
    const dim3 block(32, 8, 1);
    const dim3 grid((h->flowWidth + BT - 1) / BT, (h->flowHeight + BT - 1) / BT, 2);
    HRB_CUDA(cudaMemsetAsync(flowMax, 0, sizeof(uint32_t), h->stream));
    profBegin(h, CLS_BLUR);
    const int lw = h->flowWidth, lh = h->flowHeight;
    if (wsLog2 == 1 && !(lw & 1) && !(lh & 1) && lw >= 8 && lh >= 8 && nWx == lw / 2 && h->searchVariant != 1) {
        const dim3 cgrid((lw / 2 + BC_W - 1) / BC_W, (lh / 2 + BC_H - 1) / BC_H, 2);
        blurFlowCellKernel<<<cgrid, block, 0, h->stream>>>(lvlX, lvlY, lw / 2, lh / 2, out, lw, lh, flowMax);
    } else
        blurFlowKernel<<<grid, block, 0, h->stream>>>(lvlX, lvlY, nWx, wsLog2, out, h->flowWidth, h->flowHeight, flowMax);
    HRB_LAUNCH_CHECK();
    profEnd(h, CLS_BLUR, 1);
    return HRB_OK;
}

int launchBlurFlowBatch(hrb_ofc* const* h, const BlurBatch& b, int n, int nWx, int wsLog2) {
    const dim3 block(32, 8, 1);
    const hrb_ofc* h0 = h[0];
    const int lw = h0->flowWidth, lh = h0->flowHeight;
    for (int k = 0; k < n; ++k) HRB_CUDA(cudaMemsetAsync(b.m[k].flowMax, 0, sizeof(uint32_t), h0->stream));
    if (wsLog2 == 1 && !(lw & 1) && !(lh & 1) && lw >= 8 && lh >= 8 && nWx == lw / 2 && h0->searchVariant != 1) {
        const dim3 cgrid((lw / 2 + BC_W - 1) / BC_W, (lh / 2 + BC_H - 1) / BC_H, 2 * n);
        blurFlowCellBatchKernel<<<cgrid, block, 0, h0->stream>>>(b, lw / 2, lh / 2, lw, lh);
    } else {
        const dim3 grid((lw + BT - 1) / BT, (lh + BT - 1) / BT, 2 * n);
        blurFlowBatchKernel<<<grid, block, 0, h0->stream>>>(b, nWx, wsLog2, lw, lh);
    }
    HRB_LAUNCH_CHECK();
    for (int k = 0; k < n; ++k) profEnd(h[k], CLS_BLUR, 1);
    return HRB_OK;
}

int launchExpandOffsets(hrb_ofc* h, const int16_t* lvlX, int nWxX, int wsLog2X, const int16_t* lvlY, int nWxY, int wsLog2Y, int16_t* out) {
    const dim3 block(32, 8, 1);
    const dim3 grid((h->flowWidth + 31) / 32, (h->flowHeight + 7) / 8, 1);
    expandOffsetsKernel<<<grid, block, 0, h->stream>>>(lvlX, nWxX, wsLog2X, lvlY, nWxY, wsLog2Y, out, h->flowWidth, h->flowHeight);
    HRB_LAUNCH_CHECK();
    return HRB_OK;
}

int microbenchSad(int device, double* gigaAbsdiffPerSec) {
    HRB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    HRB_CUDA(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    uint32_t* d = nullptr;
    HRB_CUDA(cudaMalloc(&d, (size_t)blocks * threads * sizeof(uint32_t)));
    cudaEvent_t e0, e1;
    HRB_CUDA(cudaEventCreate(&e0));
    HRB_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        HRB_CUDA(cudaEventRecord(e0, 0));
        sadPeakKernel<<<blocks, threads>>>(d, 12345u + rep, iters);
        HRB_LAUNCH_CHECK();
        HRB_CUDA(cudaEventRecord(e1, 0));
        HRB_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        HRB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    const double sads = (double)blocks * threads * (double)iters * 64.0;  // SAD instructions (lane level)
    *gigaAbsdiffPerSec = sads * 4.0 / (best * 1e-3) / 1e9;
    return HRB_OK;
}

}  // namespace hrb
