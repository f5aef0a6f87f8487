/* hrb.h — C ABI of hopperrender_b200: HopperRender's optical-flow frame-interpolation hot path on B200.
 *
 * This is the drop-in boundary.  The reference has no FFI layer of its own: the boundary is the C++
 * class OpticalFlowCalc / OpticalFlowCalcSDR / OpticalFlowCalcHDR (HopperRender/opticalFlowCalc.h:24-138,
 * opticalFlowCalcSDR.h:13-56, opticalFlowCalcHDR.h:13-56) that CHopperRender::DeliverToRenderer drives
 * (HopperRender/HopperRender.cpp:918-924, 953-957, 1180-1186).  Each entry point below replaces one
 * member of that class; include/opticalFlowCalc*.h re-creates the class on top of this ABI so the
 * filter's host code compiles unchanged (see INTEGRATION.md).
 *
 * Conventions: plain C, opaque handle, every call returns HRB_OK (0) or an error code; the message of
 * the last error on the calling thread is available from hrb_last_error().  No exception crosses this
 * boundary.  One handle = one video stream on one GPU, used by one thread at a time; distinct handles
 * are independent (own CUDA stream unless the caller supplies one).  There is no CPU fallback: every
 * call fails with HRB_ERR_CUDA when no sm_100 device is usable.
 *
 * Strides are in ELEMENTS (pixels), as in the reference (opticalFlowCalcHDR.cpp:20): bytes = elements
 * * (is_hdr ? 2 : 1).  Frames are NV12 (8-bit) or P010 (10 significant bits in the MSBs of 16):
 * `height` luma rows of `stride` elements, then height/2 rows of interleaved U,V.
 */
#ifndef HRB_H_
#define HRB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define HRB_API __declspec(dllexport)
#else
#define HRB_API __attribute__((visibility("default")))
#endif

/* error codes */
enum {
    HRB_OK = 0,
    HRB_ERR_INVALID_ARG = 1,   /* bad pointer / geometry / mode */
    HRB_ERR_CUDA = 2,          /* a CUDA runtime call failed (replaces CHECK_ERROR, opticalFlowCalc.h:15-22) */
    HRB_ERR_BLEND_RANGE = 3,   /* blendingScalar > 1 (replaces the throw at opticalFlowCalcSDR.cpp:143-146) */
    HRB_ERR_NO_DEVICE = 4,     /* no device with enough memory (replaces detectDevices, opticalFlowCalc.cpp:97-109) */
    HRB_ERR_STATE = 5          /* call not valid in the current state (e.g. tap read without tap mode) */
};

/* frameOutputMode values (HopperRender/HopperRender.h:10-18) */
enum {
    HRB_MODE_WARPED_FRAME_12 = 0,
    HRB_MODE_WARPED_FRAME_21 = 1,
    HRB_MODE_BLENDED_FRAME = 2,
    HRB_MODE_HSV_FLOW = 3,
    HRB_MODE_GREY_FLOW = 4,
    HRB_MODE_SIDE_BY_SIDE_1 = 5,
    HRB_MODE_SIDE_BY_SIDE_2 = 6
};

typedef struct hrb_ofc hrb_ofc;

/* Constructor arguments of OpticalFlowCalcSDR/HDR (opticalFlowCalcSDR.h:15-17) + target selection. */
typedef struct hrb_ofc_desc {
    int frame_height;
    int frame_width;
    int input_stride;    /* elements; <= 0 means frame_width (opticalFlowCalcSDR.cpp:212) */
    int output_stride;   /* elements; <= 0 means frame_width (opticalFlowCalcSDR.cpp:213) */
    int delta_scalar;
    int neighbor_scalar;
    float black_level;
    float white_level;
    int max_calc_res;    /* flow height is halved until <= this (opticalFlowCalcSDR.cpp:217-222) */
    int is_hdr;          /* 0: NV12 / OpticalFlowCalcSDR, 1: P010 / OpticalFlowCalcHDR */
    int device_ordinal;  /* CUDA device; replaces detectDevices (opticalFlowCalc.cpp:45-110) */
    void* cuda_stream;   /* optional cudaStream_t to run on (NULL: the handle creates its own) */
} hrb_ofc_desc;

/* Public data members of OpticalFlowCalc (opticalFlowCalc.h:26-50). Times are in seconds. */
typedef struct hrb_ofc_state {
    int frame_width, frame_height, input_stride, output_stride;
    float output_black_level, output_white_level;
    int res_scalar;              /* m_opticalFlowResScalar */
    int flow_width, flow_height; /* m_opticalFlowFrameWidth / Height */
    int search_radius;           /* m_opticalFlowSearchRadius */
    double ofc_calc_time, ofc_avg_calc_time, ofc_peak_calc_time;
    int ofc_calc_count;
    double ofc_calc_time_sum;
    double warp_calc_time;
    int delta_scalar, neighbor_bias_scalar;
    unsigned int total_frame_delta;
    unsigned int frame_count;
} hrb_ofc_state;

/* The members the filter writes on a live object (HopperRender.cpp:1386-1389, 1448, 1457). */
typedef struct hrb_ofc_params {
    int search_radius;        /* 5..16 (config.h:8-9) */
    int delta_scalar;
    int neighbor_bias_scalar;
    float black_level;
    float white_level;
} hrb_ofc_params;

/* ---- lifecycle --------------------------------------------------------------------------------- */
/* OpticalFlowCalcSDR::OpticalFlowCalcSDR / HDR ctor (opticalFlowCalcSDR.cpp:206-325, HDR :211-332) */
HRB_API int hrb_ofc_create(hrb_ofc** out, const hrb_ofc_desc* desc);
/* ~OpticalFlowCalcSDR / HDR (opticalFlowCalcSDR.cpp:185-204) */
HRB_API void hrb_ofc_destroy(hrb_ofc* h);

/* ---- the five virtuals ------------------------------------------------------------------------- */
/* updateFrame (opticalFlowCalcSDR.cpp:19-29): upload 1.5*H*input_stride elements, rotate the three
 * input slots, ++frame_count.  The host buffer is no longer read once the call returns. */
HRB_API int hrb_ofc_update_frame(hrb_ofc* h, const uint8_t* input_planes);
/* calculateOpticalFlow (opticalFlowCalcSDR.cpp:44-139): search ladder + blur, updates total_frame_delta
 * and the calc-time statistics; blocks until the flow is complete (the reference waits too, :119-120). */
HRB_API int hrb_ofc_calculate_optical_flow(hrb_ofc* h);
/* warpFrames (opticalFlowCalcSDR.cpp:141-168): asynchronous, result in the device output frame. */
HRB_API int hrb_ofc_warp_frames(hrb_ofc* h, float blending_scalar, int frame_output_mode);
/* warpFrames for up to HRB_WARP_BATCH_MAX output frames of the SAME source pair in one pass (beyond the reference, like the
 * asynchronous calls): output frame i is what hrb_ofc_warp_frames(h, blending_scalars[i], mode) would produce, bit for bit.
 * The forward / reverse flow of a sample is fetched once for all of them and both source frames cross HBM once.  The n
 * frames go to consecutive slots of the device output ring; fetch them with n calls of hrb_ofc_download_frame(_async) (in
 * the order given), with no warp_frames / copy_frame call in between. */
#define HRB_WARP_BATCH_MAX 8
HRB_API int hrb_ofc_warp_frames_batch(hrb_ofc* h, int n, const float* blending_scalars, int frame_output_mode);
/* copyFrame (opticalFlowCalcSDR.cpp:170-183) */
HRB_API int hrb_ofc_copy_frame(hrb_ofc* h);
/* downloadFrame (opticalFlowCalcSDR.cpp:31-42): blocking read of 1.5*H*output_stride elements; sets
 * warp_calc_time. */
HRB_API int hrb_ofc_download_frame(hrb_ofc* h, uint8_t* output_planes);

/* ---- public fields ----------------------------------------------------------------------------- */
/* get_state waits for every flow calculation in flight (total_frame_delta and the calc-time statistics are those of the
 * newest one); peek_state never blocks: it reflects the calculations that have finished so far.  A caller that polls
 * fields between calculate_optical_flow_async and the warps uses peek_state so that host and GPU keep overlapping. */
HRB_API int hrb_ofc_get_state(hrb_ofc* h, hrb_ofc_state* out);
HRB_API int hrb_ofc_peek_state(hrb_ofc* h, hrb_ofc_state* out);
HRB_API int hrb_ofc_set_params(hrb_ofc* h, const hrb_ofc_params* p);
/* m_frameCount = n; the filter writes 0 on seek (HopperRender.cpp:840) */
HRB_API int hrb_ofc_set_frame_count(hrb_ofc* h, unsigned int n);
HRB_API int hrb_ofc_reset(hrb_ofc* h); /* == hrb_ofc_set_frame_count(h, 0) */

/* ---- device-resident variants (benchmark / zero-copy callers) ---------------------------------- */
/* Same as hrb_ofc_update_frame but the source is already in device memory of the handle's GPU.  It is
 * hrb_ofc_update_frame_planes with y = device_planes, uv = device_planes + H * input_stride * bpp and both pitches
 * input_stride * bpp bytes: the same checks apply and it is read on the compute stream. */
HRB_API int hrb_ofc_update_frame_device(hrb_ofc* h, const void* device_planes);
/* Device address of the output frame most recently written by warp_frames / copy_frame (for a batch: its first frame;
 * the frames of a batch sit in consecutive slots of a ring that advances with every download). */
HRB_API int hrb_ofc_output_device_ptr(hrb_ofc* h, void** out);
/* Asynchronous variants for PINNED host memory.  Transfers run on their own streams: the upload of the next source
 * frame and the downloads of the current outputs overlap the kernels (the output frame is a ring of three on the
 * device, the upload has its own input slot).
 *   update_frame_async : the buffer must stay untouched until hrb_ofc_wait_upload (or synchronize) returns.
 *   download_frame_async: hands out a ticket; the buffer is valid after hrb_ofc_wait_download(ticket) (tickets may be
 *                         waited for in any order: a wait on an old ticket waits for the newest download that reuses its slot (tickets share 16
 *                         event slots), which proves the old copy has landed — it never returns early). */
HRB_API int hrb_ofc_update_frame_async(hrb_ofc* h, const uint8_t* pinned_input_planes);
HRB_API int hrb_ofc_wait_upload(hrb_ofc* h);
HRB_API int hrb_ofc_download_frame_async(hrb_ofc* h, uint8_t* pinned_output_planes, unsigned long long* ticket);
HRB_API int hrb_ofc_wait_download(hrb_ofc* h, unsigned long long ticket);
/* calculate_optical_flow without the final host wait (statistics are resolved at the next synchronize). */
HRB_API int hrb_ofc_calculate_optical_flow_async(hrb_ofc* h);
HRB_API int hrb_ofc_synchronize(hrb_ofc* h);
/* cudaStream_t the handle launches on */
HRB_API int hrb_ofc_stream(hrb_ofc* h, void** out);
/* Pin / unpin caller-owned frame memory once (e.g. a DirectShow allocator pool) so update/download DMA directly. */
HRB_API int hrb_host_register(void* ptr, size_t bytes);
HRB_API int hrb_host_unregister(void* ptr);
HRB_API int hrb_host_alloc(void** out, size_t bytes);
HRB_API int hrb_host_free(void* ptr);

/* ---- device frame planes ------------------------------------------------------------------------------------ */
/* Source and destination frames as two planes in caller-owned memory on the handle's GPU, as hardware and CUDA decoders
 * and encoders lay them out: the chroma plane is a pointer of its own (or sits at y + pitch * aligned_height), and the
 * pitches are in BYTES.  bpp = 1 (NV12) or 2 (P010). */
typedef struct hrb_frame_planes {
    void*  y;          size_t y_pitch_bytes;   /* frame_height rows of frame_width samples */
    void*  uv;         size_t uv_pitch_bytes;  /* frame_height/2 rows of frame_width interleaved U,V samples */
} hrb_frame_planes;
/* update_frame_device with the source described by two planes: the same input-slot rotation, frame_count, flow timer
 * start and ordering behind a flow in flight.  The planes are read by one kernel on the compute stream (hrb_ofc_stream),
 * which also fills the handle's own input slot (the warps read a frame for up to three source frames): the caller may
 * overwrite or release the planes with work ordered behind that stream. */
HRB_API int hrb_ofc_update_frame_planes(hrb_ofc* h, const hrb_frame_planes* src);
/* warp_frames_batch into caller surfaces: output frame i goes to dst[i] (n in 1..HRB_WARP_BATCH_MAX) and is, bit for bit,
 * the frame warp_frames_batch puts into ring slot i, in every mode.  The output stripe (set_output_stripe) applies: only
 * its luma rows and their chroma rows are written.  No other byte of a destination is written: not the pitch padding,
 * not the rows outside the stripe, not the gap between the planes.  Every destination of one call has the same
 * (y_pitch_bytes, uv_pitch_bytes).  The warp's two-sample stores need every plane base and both pitches to be multiples of
 * 2 * bpp bytes; otherwise every item takes the general form with scalar stores (same result, slower). */
HRB_API int hrb_ofc_warp_frames_to(hrb_ofc* h, int n, const float* blending_scalars, int frame_output_mode, const hrb_frame_planes* dst);
/* copy_frame into a caller surface, with the same stripe and byte rules as warp_frames_to. */
HRB_API int hrb_ofc_copy_frame_to(hrb_ofc* h, const hrb_frame_planes* dst);
/* The _to calls do not touch the output ring, its cursor or its events: download_frame and output_device_ptr keep
 * referring to the last ring frame, and warp_calc_time stays what the ring path's downloads set.  Their results are
 * visible to work ordered behind hrb_ofc_stream.
 *
 * Every plane is checked before anything is enqueued; a failure returns HRB_ERR_INVALID_ARG with a message naming the
 * plane and the rule:
 *   - the plane is not null;
 *   - it is device or managed memory of the handle's device (cudaPointerGetAttributes): host memory, pageable or pinned,
 *     and memory of another device are refused;
 *   - its pitch is at least frame_width * bpp, and its pointer and pitch are multiples of bpp;
 *   - its extent (rows - 1) * pitch + frame_width * bpp lies inside the allocation that holds it (cuMemGetAddressRange),
 *     and below 2^31 samples;
 *   - the Y and UV planes of a frame do not overlap, and the destinations of one call are pairwise disjoint.
 * The blend scalars and the mode are checked as warp_frames_batch checks them (HRB_ERR_BLEND_RANGE for a scalar above 1,
 * HRB_ERR_INVALID_ARG for a mode outside 0..6). */

/* ---- delivery loop ------------------------------------------------------------------------------------------------ */
/* The filter's DeliverToRenderer (HopperRender.cpp:944-1211) on top of one handle: for every source frame it decides how
 * many output frames to produce, advances the blending scalar, runs the search-radius auto-tuner and applies the
 * scene-change rule that chooses warp_frames or copy_frame.  The scene-change decision is taken by a kernel on the GPU,
 * so a step never waits for a flow calculation: the warps of a step keep running beside the search of its flow.
 *
 * One step is one DeliverToRenderer call, in its order:
 *   1. the output count n (m_iNumIntFrames, :945): ceil((1 - blend) / (target / playback)) when interpolation is active,
 *      otherwise 1;
 *   2. the auto-tuner (:951, :1438-1463) when auto_adjust is on;
 *   3. calculate_optical_flow_async when active and frame_count >= 3, and the frame-delta history (:959-973);
 *   4. the warp-or-copy choice for all n output frames (:1126-1183);
 *   5. the blend-scalar advance (:1192-1197).
 * The caller does the ingest (update_frame, _async, _device or _planes) of a source frame before the step that delivers
 * it.  hrb_delivery_step writes the n frames into the output ring: fetch them with n download_frame(_async) calls, in
 * order.  hrb_delivery_step_to writes output frame i into dst[i]: the frames are ready for work ordered behind
 * hrb_ofc_stream.  Steps of more than HRB_WARP_BATCH_MAX frames run as two warp batches under the same decision.  A step
 * of more than HRB_DELIVERY_MAX_FRAMES frames (the output ring's size) cannot be delivered: create, set and new_segment
 * refuse settings whose target / playback ratio needs one, with HRB_ERR_INVALID_ARG.
 *
 * Exclusive use: while a delivery is attached to a handle, calculate_optical_flow(_async), warp_frames(_batch, _to) and
 * copy_frame(_to) on that handle return HRB_ERR_STATE (the delta history would no longer describe the flows).  Ingest,
 * downloads, get_state / peek_state and set_params stay allowed.  A handle has at most one delivery, and the delivery is
 * destroyed before its handle.  A handle in a split group or a flow batch cannot have a delivery, and a handle with a
 * delivery cannot join either (HRB_ERR_STATE).
 *
 * Outcomes: the decision of step s (warped, scene change, the rule's two deltas d1 and d2, the frame delta the step
 * appended) is copied to host memory behind the step's kernels.  hrb_delivery_outcome_of(s, wait = 0) returns
 * HRB_ERR_STATE while it is still in flight; wait = 1 blocks until it has landed.  The last HRB_DELIVERY_MAX_FRAMES steps
 * are kept (older ones: HRB_ERR_INVALID_ARG).
 *
 * Auto-tuner inputs: the newest FINISHED flow calculation's time (what peek_state reports) plus the GPU time of the
 * warps / copy of the newest step whose outputs have finished, measured by events around them.  The filter reads the
 * flow it has just computed and the time until its downloads ended; neither is available without waiting. */
#define HRB_DELIVERY_MAX_FRAMES 16
typedef struct hrb_delivery hrb_delivery;
typedef struct hrb_delivery_desc {
    long long source_frame_time;   /* 100-ns units, rtSourceFrameTime (417083 = 23.976 fps); > 0 */
    long long target_frame_time;   /* 100-ns units, rtTargetFrameTime (69444 = 144 fps); > 0 */
    int frame_output_mode;         /* 0..6 (HRB_MODE_*) */
    int scene_change_threshold;    /* m_iSceneChangeThreshold; HopperRender's default is 200 */
    int active;                    /* interpolation switched on (m_iIntActiveState != Deactivated) */
    int auto_adjust;               /* run the search-radius auto-tuner (autoAdjustSettings, HopperRender.cpp:1438-1463) */
} hrb_delivery_desc;
/* One output frame of a step: known when the step returns. */
typedef struct hrb_delivery_frame {
    unsigned int source;           /* frame_count of the source frame it belongs to */
    int index;                     /* 0 .. n-1 inside the step */
    double blend;                  /* m_dBlendingScalar the frame is warped at */
    unsigned long long step;       /* the step's number (0 for the first step of a delivery) */
} hrb_delivery_frame;
/* The decision of one step, taken on the GPU. */
typedef struct hrb_delivery_outcome {
    int warped;                    /* 1: the step's frames were warped; 0: copied (copy_frame) */
    int scene_change;              /* sceneChangeDetected of HopperRender.cpp:1126-1176 */
    long long delta1, delta2;      /* cur - average and cur - nxt of the rule (0 with fewer than 3 history entries) */
    unsigned int frame_delta;      /* total_frame_delta of the flow the step computed (0: the step computed no flow) */
} hrb_delivery_outcome;
/* The descriptor is checked before the handle: HRB_ERR_INVALID_ARG for a null out / descriptor, a mode outside 0..6, a
 * non-positive frame time, a ratio needing more than HRB_DELIVERY_MAX_FRAMES outputs per step, or a null handle. */
HRB_API int hrb_delivery_create(hrb_delivery** out, hrb_ofc* h, const hrb_delivery_desc* desc);
HRB_API void hrb_delivery_destroy(hrb_delivery* d);
/* the number of output frames the next step will produce */
HRB_API int hrb_delivery_next_count(hrb_delivery* d, int* n);
/* One step into the output ring; frames[0..n-1] describe the n frames (capacity >= n, else HRB_ERR_INVALID_ARG). */
HRB_API int hrb_delivery_step(hrb_delivery* d, hrb_delivery_frame* frames, int capacity, int* n);
/* One step into dst[0..n-1] (capacity >= n; the planes are checked as warp_frames_to checks them). */
HRB_API int hrb_delivery_step_to(hrb_delivery* d, const hrb_frame_planes* dst, int capacity, hrb_delivery_frame* frames, int* n);
HRB_API int hrb_delivery_outcome_of(hrb_delivery* d, unsigned long long step, int wait, hrb_delivery_outcome* out);
/* UpdateUserSettings (HopperRender.cpp:1355-1390): mode, threshold, activation, auto-tuner and target frame time; clears
 * the delta history.  source_frame_time must be the one the delivery was created with.  The calculator's scalars and
 * levels are set with hrb_ofc_set_params. */
HRB_API int hrb_delivery_set(hrb_delivery* d, const hrb_delivery_desc* desc);
/* NewSegment (HopperRender.cpp:834-844): playback frame time = source frame time / rate, history cleared, frame_count 0 */
HRB_API int hrb_delivery_new_segment(hrb_delivery* d, double rate);

/* ---- side data of the source frames ----------------------------------------------------------------------------- */
/* The filter reads the IMediaSideData blobs of the input sample (HDR10 / HDR10+ / Dolby Vision metadata and RPU, control
 * flags, content light level, EIA-608 captions, 3D offset: HopperRender.cpp:875-900) and sets them on EVERY output sample it
 * delivers for that source frame (:993-1022).  The library keeps them beside the frame: set_side_data attaches copies of
 * `count` blobs to the frame given to the LAST update_frame call (count 0 clears); get_side_data returns the blobs of that
 * frame for the output frames being delivered.  The pointers stay valid until the next set_side_data or destroy.  The
 * contents are opaque to the library. */
typedef struct hrb_side_data {
    uint8_t guid[16];   /* the interface id the blob was read with (IMediaSideData.h) */
    const void* data;
    size_t bytes;
} hrb_side_data;
HRB_API int hrb_ofc_set_side_data(hrb_ofc* h, const hrb_side_data* items, int count);
HRB_API int hrb_ofc_get_side_data(hrb_ofc* h, hrb_side_data* items, int capacity, int* count);

/* ---- spatial split of one stream over several GPUs ----------------------------------------------------------- */
/* Restrict warp_frames / copy_frame / download_frame to the luma rows [row_begin, row_end) (even bounds) and the
 * chroma rows that belong to them.  Every GPU of the split holds the full source frames and the full flow (the
 * search is replicated, it is not the PCIe-bound part, unless the handles form a split group, below); each produces and
 * downloads only its stripe, into the same offsets of a full-frame host buffer.  Default: the whole frame. */
HRB_API int hrb_ofc_set_output_stripe(hrb_ofc* h, int row_begin, int row_end);

/* ---- split search: one flow computed by a group of handles ----------------------------------------------------- */
/* A group of n handles ("shards", usually one per GPU; several may share a device) that together compute ONE flow.
 * Shard k owns the flow rows [b_k, b_k+1), b_k = 128 * round(k * flow_height / (n * 128)), b_0 = 0, b_n = flow_height.
 * The passes of the search ladder whose windows are at most 128 rows tall are sharded: each shard searches only the
 * windows of its stripe, and between two such iterations it copies one parent-level window row above and one below its
 * stripe from its neighbours (peer to peer between devices).  Passes with taller windows straddle stripes and run on
 * every shard over the whole frame, as on a lone handle.  After the last iteration every shard receives the other
 * shards' windows and blurs the whole field, so that afterwards EVERY handle of the group holds exactly the flow,
 * flow peak, offset array and total_frame_delta a lone calculate_optical_flow on it would have produced, bit for bit:
 * warp_frames, set_output_stripe and download_frame work on it unchanged.
 *
 * Preconditions: every handle already holds both full source frames (the caller runs update_frame /
 * update_frame_device on each of them: the search reads frame 1 at unbounded offsets); the handles agree on frame size,
 * is_hdr, res_scalar, search radius, delta / neighbour scalars and search variant (checked at create and at every
 * calculate: HRB_ERR_INVALID_ARG naming the field).  Profile and debug timeline must be off on every shard
 * (HRB_ERR_STATE otherwise).  Tap mode works: a shard records every pass; in a sharded pass only the window rows of its
 * stripe are meaningful, and the sums and layer taps are zero elsewhere.
 *
 * The group owns nothing: a handle in a group remains a normal handle (its own calculate_optical_flow still runs the
 * whole ladder), and the group must be destroyed before its handles.  Up to 64 shards. */
typedef struct hrb_split hrb_split;
/* The flow-row bounds bounds[0..n] of n shards for a flow of flow_height rows; needs no device.  HRB_ERR_INVALID_ARG for
 * n < 1, n > 64 or an n that would leave a stripe empty. */
HRB_API int hrb_split_plan(int flow_height, int n, int* bounds);
/* Shard k of the group is shards[k] (distinct handles); the handles' streams must be usable from this thread. */
HRB_API int hrb_split_create(hrb_split** out, hrb_ofc* const* shards, int n);
HRB_API void hrb_split_destroy(hrb_split* s);
/* the flow rows shard `shard` owns */
HRB_API int hrb_split_stripe(hrb_split* s, int shard, int* flow_row_begin, int* flow_row_end);
/* calculate_optical_flow on every shard at once: blocks until the flow is complete on all of them, and leaves each
 * handle in the state its own calculate_optical_flow would (flow record, statistics, buffer swap). */
HRB_API int hrb_split_calculate_optical_flow(hrb_split* s);
/* calculate_optical_flow_async on every shard at once: each shard runs its part on its flow stream (flow overlap on) or
 * its compute stream, forked and joined exactly as its own calculate_optical_flow_async would, so warp_frames issued
 * afterwards reads the previous flow.  The shards order each other with events and copy with cudaMemcpyPeerAsync
 * (cudaMemcpyAsync when two shards share a device); plain launches, no CUDA graph. */
HRB_API int hrb_split_calculate_optical_flow_async(hrb_split* s);

/* ---- flow batch: the flows of many same-size streams in one ladder --------------------------------------------- */
/* A group of n independent handles ("members", one per stream) on one device whose flows are searched together: each
 * pass of the search ladder that runs the generic kernel (every pass of a reduced-resolution flow) is ONE launch over all
 * members, and so is the blur, so n short chains of small launches become one chain of launches n times larger.  Passes
 * that run the tile or small-window kernel (full-resolution flows) run one launch per member, back to back.  Each member
 * searches its own frames into its own flow: afterwards EVERY member is in exactly the state its own
 * calculate_optical_flow(_async) would have left it in, bit for bit (offset array, both blurred flows after the swap,
 * flow peaks, raw frame delta, total_frame_delta with its own SDR / HDR divisor, flow record and calc-time statistics,
 * taps when its tap mode is on).
 *
 * The members must agree on frame width and height, res_scalar, search radius, search variant and device (checked at
 * create and at every calculate: HRB_ERR_INVALID_ARG naming the field; callers whose streams differ in radius form one
 * batch per radius).  They may differ in is_hdr, strides, delta / neighbour scalars, levels, max_calc_res (with equal
 * res_scalar) and frame history.  n must be 1..HRB_FLOW_BATCH_MAX with distinct, non-null handles
 * (HRB_ERR_INVALID_ARG).  Profile and debug timeline must be off on every member (HRB_ERR_STATE otherwise).
 *
 * The batch owns no frame or flow memory: a member remains a normal handle, and the batch must be destroyed before its
 * members.  It owns one stream (at the priority of the flow streams) on which the ladder runs; plain launches, no CUDA
 * graph. */
typedef struct hrb_flow_batch hrb_flow_batch;
#define HRB_FLOW_BATCH_MAX 64
/* members[k] is member k; the members' streams must be usable from this thread */
HRB_API int hrb_flow_batch_create(hrb_flow_batch** out, hrb_ofc* const* members, int n);
/* waits for the batch's stream, then frees it */
HRB_API void hrb_flow_batch_destroy(hrb_flow_batch* b);
/* calculate_optical_flow on every member at once: blocks until every flow is complete, and leaves each member in the
 * state its own calculate_optical_flow would (flow record, statistics, buffer swap). */
HRB_API int hrb_flow_batch_calculate_optical_flow(hrb_flow_batch* b);
/* calculate_optical_flow_async on every member at once.  The batch's stream waits for each member's compute stream (the
 * ingest of its newest frame, the last readers of the flow buffer it overwrites).  A member with flow overlap on (and
 * tap mode off) is joined the way its own asynchronous calculate joins it: warp_frames issued afterwards reads the
 * previous flow, and the next calculate, join_flow or the third update_frame is ordered behind the batch.  Every other
 * member's compute stream waits for the batch at once. */
HRB_API int hrb_flow_batch_calculate_optical_flow_async(hrb_flow_batch* b);

/* ---- test taps --------------------------------------------------------------------------------- */
/* With tap mode on, calculate_optical_flow also records, per (iteration, step) pass: the window sums,
 * the winning layer per window and the offset field after the update.  Off by default (costs memory). */
HRB_API int hrb_ofc_set_tap_mode(hrb_ofc* h, int on);
HRB_API int hrb_ofc_num_passes(hrb_ofc* h, int* out);
HRB_API int hrb_ofc_pass_info(hrb_ofc* h, int pass, int* window_size, int* iteration, int* step, int* windows_x, int* windows_y);
enum {
    HRB_TAP_WINDOW_SUMS = 0, /* uint32 [R][windows_y][windows_x] == summedUpDeltaArray at the window representatives */
    HRB_TAP_WINDOW_LAYER = 1,/* uint8  [windows_y][windows_x]    == lowestLayerArray at the window representatives */
    HRB_TAP_OFFSETS = 2      /* int16  [2][flow_h][flow_w]       == offsetArray after adjustOffsetArrayKernel */
};
HRB_API int hrb_ofc_read_pass_tap(hrb_ofc* h, int pass, int which, void* dst, size_t bytes);
enum {
    HRB_BUF_OFFSET_ARRAY = 0,     /* int16 [2][flow_h][flow_w]: m_offsetArray after the last pass */
    HRB_BUF_FLOW_FOR_WARP = 1,    /* int16 [2][flow_h][flow_w]: m_blurredOffsetArray[0] (what warpFrames reads) */
    HRB_BUF_FLOW_LATEST = 2,      /* int16 [2][flow_h][flow_w]: m_blurredOffsetArray[1] (result of the last calculate) */
    HRB_BUF_OUTPUT_FRAME = 3,     /* m_outputFrameArray */
    HRB_BUF_RAW_FRAME_DELTA = 4,  /* uint32: the raw window sum total_frame_delta is derived from */
    HRB_BUF_FLOW_PEAK = 5         /* uint32 [2]: max |value| of the flow warpFrames reads, and of the latest one (the bound the warp kernel uses to skip the mirror) */
};
HRB_API int hrb_ofc_read_buffer(hrb_ofc* h, int which, void* dst, size_t bytes);
/* overwrite a blurred flow (HRB_BUF_FLOW_FOR_WARP / HRB_BUF_FLOW_LATEST) — lets tests drive warp_frames */
HRB_API int hrb_ofc_write_flow(hrb_ofc* h, int which, const int16_t* src, size_t count);

/* ---- measurement support ----------------------------------------------------------------------- */
typedef struct hrb_ofc_profile {
    /* accumulated since the last hrb_ofc_profile_reset, GPU time from CUDA events on the handle's stream */
    double ms_ingest, ms_search, ms_blur, ms_warp, ms_copy;
    uint64_t n_ingest, n_search, n_blur, n_warp, n_copy; /* kernel launches per class */
} hrb_ofc_profile;
HRB_API int hrb_ofc_set_profile(hrb_ofc* h, int on);
HRB_API int hrb_ofc_profile_read(hrb_ofc* h, hrb_ofc_profile* out); /* synchronizes */
HRB_API int hrb_ofc_profile_reset(hrb_ofc* h);
/* Kernel selection for the search ladder: 0 = automatic (tile kernel for windows >= 16, staged small-window kernel
 * below), 1 = the generic kernel for every pass, 2 = tile kernel without TMA (cp.async staging only) and down to
 * windows of 4, 3 = like 2 with the per-pixel fallback forced for every window, 4 = like 0 but windows of 2 and 4 use the
 * lane-per-pixel-column form with a butterfly reduction instead of one lane per window.
 * Results are identical; exists for A/B measurements and parity tests. */
HRB_API int hrb_ofc_set_search_variant(hrb_ofc* h, int variant);
/* hrb_ofc_calculate_optical_flow_async runs the search on its own stream, beside the warps issued after it (they read
 * the PREVIOUS flow, opticalFlowCalcSDR.cpp:113-123,150).  on = 0 keeps everything on the compute stream.  Default 1. */
HRB_API int hrb_ofc_set_flow_overlap(hrb_ofc* h, int on);
/* Orders the compute stream (hrb_ofc_stream) behind the flow calculation still running on the flow stream, without
 * blocking the host: work a caller enqueues on the compute stream afterwards sees the finished flow. */
HRB_API int hrb_ofc_join_flow(hrb_ofc* h);
/* Debug aid: record a per-CTA timeline of every tile search kernel of the following flow calculations (16 uint64 per
 * CTA: start, boxes landed, runs done, end [globaltimer ns], SM id, block x, block y, rounds (+100 on a border tile; 5 =
 * the per-pixel remainder), warps per CTA, then 7 zero words; `words_per_pass` words for each of up to 32 passes; 0
 * switches it off).  CTA i of a pass records only if 16 * (i + 1) <= words_per_pass, so passes never overlap.  The
 * buffer is zeroed here, not per calculation.  Used by tools/cta_timeline.py. */
HRB_API int hrb_ofc_debug_timeline(hrb_ofc* h, size_t words_per_pass);
HRB_API int hrb_ofc_debug_timeline_read(hrb_ofc* h, void* dst, size_t bytes);
/* number of kernels this library has launched in this process */
HRB_API uint64_t hrb_kernel_launch_count(void);
/* packed byte-SAD instruction peak of the device (VABSDIFF4.U8.ACC issue rate), in 1e9 byte-abs-diffs/s */
HRB_API int hrb_microbench_sad_peak(int device_ordinal, double* giga_absdiff_per_s);

HRB_API const char* hrb_last_error(void);
HRB_API const char* hrb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HRB_H_ */
