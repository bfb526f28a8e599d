/*
 * vt_tracker.h — C ABI of the B200-native ViT tracker hot path (libvittrack_b200.so).
 *
 * This is the drop-in boundary for the per-frame path of frodik13/gstreamer-vit-tracker.  The
 * reference has no FFI of its own for this path: it is plain Rust calling
 *   - nv12_convert::nv12_full_to_rgb_parallel / draw_*_nv12     (src/nv12_convert.rs:46,172-343)
 *   - drawing::{draw_cursor, draw_selection, get_glyph}          (src/drawing.rs:5-100)
 *   - drawing_rgb::draw_*_rgb                                    (src/drawing_rgb.rs:30-128)
 *   - vit_tracker::VitTrack::{new, init, update}                 (call sites src/tracker_context.rs:21,88,90,120)
 *   - TrackerContext::{new, handle_command, process_frame, state_name} (src/tracker_context.rs:19-166)
 *   - TimingStats::{add_interval, add_times, fps, avg_*_ms}      (src/timing_stats.rs:17-60)
 * from the pad-probe closures (src/pipeline.rs:67-184, src/pipeline_ir.rs:100-228).  Each entry
 * point below names the reference interface it replaces; INTEGRATION.md shows the Rust
 * `extern "C"` block a maintainer would add.
 *
 * Conventions: plain pointers and sizes only; no exceptions cross the boundary; every call
 * returns vt_status (0 = ok, negative = error).  A handle is thread-compatible (calls on one
 * handle must be serialised, exactly like the reference's Arc<Mutex<TrackerContext>>,
 * src/pipeline.rs:55,111); different handles may be used concurrently from different threads.
 * Frame memory is owned by the caller and never retained after a call returns (the reference
 * borrows the mapped GstBuffer for the duration of the probe, src/pipeline.rs:96).  There is no
 * CPU fallback: without a CUDA device every device entry point fails with VT_ERR_CUDA.
 */
#ifndef VT_TRACKER_H
#define VT_TRACKER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VT_ABI_VERSION 2   /* 2: vt_config grew the SURVEY.md App. A.7 variant switches (struct_size keeps v1 callers working) */

typedef int32_t vt_status;
enum {
    VT_OK = 0,
    VT_ERR_INVALID = -1,      /* bad argument */
    VT_ERR_CUDA = -2,         /* CUDA runtime / driver failure (vt_last_error() has the text) */
    VT_ERR_WEIGHTS = -3,      /* weight file missing or malformed            ≙ VitTrack::new Err */
    VT_ERR_CROP_OUTSIDE = -4, /* crop window lies entirely outside the frame ≙ VitTrack::update Err */
    VT_ERR_NOT_INIT = -5,     /* update() before init()                       */
    VT_ERR_GLYPH = -6         /* unknown character in strict text mode        ≙ get_glyph panic, src/drawing.rs:99 */
};

/* VT_FMT_GRAY8: one byte per pixel (IR sensors; BASELINE config "IR/GRAY8 at 640x512"): the tracker sees r = g = b = gray and the
 * overlays follow the NV12 luma-plane semantics (src/nv12_convert.rs:172-343 write the Y plane only). */
/* VT_FMT_YUY2: one plane of packed 4:2:2 words Y0 U Y1 V (most UVC / V4L2 cameras; the IR camera of src/pipeline_ir.rs:27-56), rows
 * of 4 * ceil(W/2) bytes, so a packed frame is 4 * ceil(W/2) * H bytes; odd W and odd H are allowed.  The tracker sees exactly the RGB
 * of vt_convert_yuy2_rgb (BT.601 integer arithmetic of src/nv12_convert.rs:24-30,124-126 on the pixel's word); the overlays follow the
 * NV12 luma-plane semantics and write only the Y samples (byte 2x of row y), never the U / V bytes. */
/* VT_FMT_RGBA / VT_FMT_BGRA: one plane of 32-bit pixels, bytes R G B A resp. B G R A (GStreamer RGBA / RGBx resp. BGRA / BGRx;
 * DeepStream NVBUF_COLOR_FORMAT_RGBA resp. NVBUF_COLOR_FORMAT_BGRx), rows of 4W bytes, so a packed frame is 4 * W * H bytes; any W and H.
 * The tracker sees exactly the RGB24 frame made of bytes 0, 1, 2 (RGBA) resp. 2, 1, 0 (BGRA) of every pixel; the overlays follow the
 * RGB24 semantics and write each colour into its channel's byte.  Byte 3 (alpha or padding) is never read and never written.
 * vt_overlay[_current] on such a handle needs a full frame (len >= 4 * W * H).  (Values 4 and 7 are not formats.) */
/* VT_FMT_I420: planar 4:2:0, the Y plane, then the U plane, then the V plane (GStreamer I420: avdec_h264 / avdec_h265, openh264dec,
 * vp8dec / vp9dec, dav1ddec, jpegdec, videotestsrc), in GStreamer's default layout, so that a mapped buffer is handed over as it is at any
 * W and H (RU4 / RU2: rounded up to a multiple of 4 / 2):
 *   Y stride s0 = RU4(W), U / V stride s1 = RU4(ceil(W/2)),
 *   U offset = s0 * RU2(H) (odd H: the Y plane has one padding row), V offset = U offset + s1 * ceil(H/2),
 *   frame bytes = V offset + s1 * ceil(H/2)    (1920x1080: 3,110,400 = W*H*3/2; 641x481: 466,576).
 * The tracker sees pixel (x, y) as the BT.601 integer RGB of Y[y][x], U[y/2][x/2], V[y/2][x/2] (the arithmetic of NV12): for even W,
 * tracking an I420 frame equals tracking the NV12 frame of the same Y and interleaved UV.  A buffer shorter than the frame is an
 * all-black image.  The overlays follow the NV12 luma-plane semantics: they write only the Y samples of the W x H image, never U, V, the
 * Y row padding or the padding row.  I420 frames are host frames or packed device frames (vt_tracker_update_device); pitched I420
 * surfaces are refused (see vt_surface). */
typedef enum {
    VT_FMT_NV12 = 0, VT_FMT_RGB24 = 1, VT_FMT_GRAY8 = 2, VT_FMT_YUY2 = 3, VT_FMT_RGBA = 5, VT_FMT_BGRA = 6, VT_FMT_I420 = 8
} vt_format;
/* BF16X3 (default): bf16 hi + lo operands, three products per K-step, scores within ~1e-5 of the fp32 oracle.  BF16 / FP16: single-pass
 * operands, 17 % faster, score error ~1e-3 / ~3e-4 — opt-in (near-tie arg-max flips are possible at that error). */
typedef enum { VT_GEMM_FP32_SIMT = 0, VT_GEMM_TCGEN05_BF16X3 = 1, VT_GEMM_TCGEN05_BF16 = 2, VT_GEMM_TCGEN05_FP16 = 3 } vt_gemm_mode;
/* SURVEY.md App. A.7: the `vit_tracker` crate (src absent: Cargo.toml:24) wraps OpenCV's TrackerVit through opencv 0.98.1
 * (Cargo.lock:700-716) and may follow an older upstream than the 4.13 behaviour the defaults restate. */
typedef enum { VT_DECODE_CEIL4 = 0 /* cw = ceil(sqrt(w*h)*4), the crop's own c (4.13) */, VT_DECODE_4FLOOR = 1 /* cw = 4*floor(sqrt(w*h)) (older) */ } vt_decode_window;
typedef enum { VT_WINDOW_HANN = 0 /* conf * hann (4.13) */, VT_WINDOW_ONE_MINUS_HANN = 1 /* conf * (1 - hann) (older) */ } vt_window;

/* ≙ vit_tracker::BBox {x, y, width, height: i32} (uses: src/selection_state.rs:44, src/pipeline.rs:166) */
typedef struct { int32_t x, y, width, height; } vt_bbox;

/* ≙ the Ok(result) of VitTrack::update: result.success, result.score, result.bbox
 * (src/tracker_context.rs:92-94,121-123).  status != VT_OK ≙ the Err branch for that target. */
typedef struct {
    int32_t success;
    float score;
    vt_bbox bbox;
    vt_status status;
    int32_t reserved;
} vt_result;

/* Hard-coded constants of the reference become fields (SURVEY.md §5 "config / flags"). */
typedef struct {
    uint32_t struct_size;        /* sizeof(vt_config) of the caller's header: fields beyond it take their defaults (ABI evolution);
                                    0 or larger than the library's own sizeof is VT_ERR_INVALID */
    const char* weights_path;    /* ≙ MODEL_PATH, src/pipeline.rs:11 (flat "VTW1" file instead of .rknn) */
    int32_t device;              /* CUDA device ordinal */
    int32_t format;              /* vt_format of the frames handed to init/update */
    int32_t width, height;       /* ≙ the caps of src/pipeline.rs:26-36 / src/pipeline_ir.rs:27-41 */
    int32_t max_targets;         /* 1 in the reference (one VitTrack, src/tracker_context.rs:8) */
    float score_threshold;       /* TrackerVit's own threshold (0.20); <=0 selects the default */
    int32_t gemm_mode;           /* vt_gemm_mode */
    int32_t use_cuda_graph;      /* 1: replay the per-frame kernel chain from a CUDA graph */
    int32_t box_overlay;         /* 1: update() also draws rect+crosshair for gated targets (device) and
                                       copies the touched rows back into the caller's frame */
    float overlay_gate;          /* gate for box_overlay: success && score > gate (0.25, src/tracker_context.rs:93) */
    int32_t debug_capture;       /* 1: keep per-block token copies for vt_tracker_debug_tokens (disables graph replay) */
    int32_t upload_window;       /* 1: update()/submit() upload only the search windows of the active targets (2-D copies out of a
                                       pinned frame; rect_last is mirrored on the host) instead of the whole frame.  The device copy
                                       of the frame is then partial: vt_overlay_current re-uploads the whole frame when it needs it. */
    /* --- since VT_ABI_VERSION 2: variant switches of VitTrack's pre/post-processing (SURVEY.md App. A.7); all-zero = OpenCV 4.13 --- */
    int32_t pad_plus1;           /* crop padding: 0 padR = max(x2-W, 0) (4.13); 1 padR = max(x2-W+1, 0), likewise at the bottom (older) */
    int32_t decode_window;       /* vt_decode_window */
    int32_t window;              /* vt_window */
    int32_t norm_custom;         /* 0: blob = (u8/255 - mean_c)/std_c, ImageNet mean/std on the channels in memory order (App. A.4);
                                    1: blob = u8*norm_scale[c] + norm_bias[c] — any per-channel affine map: the cv2 Scalar-division quirk
                                       (SURVEY.md §8c), or scale 1 / bias 0 when the NPU model normalises internally */
    float norm_scale[3], norm_bias[3];
    int32_t reserved[4];
} vt_config;

typedef struct vt_tracker vt_tracker;

/* ------------------------------------------------------------------------------------------- */
/* library                                                                                      */
/* ------------------------------------------------------------------------------------------- */
int32_t vt_abi_version(void);
/* thread-local text of the last failure on the calling thread (never NULL) */
const char* vt_last_error(void);
void vt_config_default(vt_config* cfg);
/* pinned host memory for frames (what a GstAllocator for the upstream element would hand out) */
vt_status vt_alloc_pinned(size_t bytes, void** out);
void vt_free_pinned(void* p);
/* Validates a model file without touching the GPU — what VitTrack::new's Err branch reports up front (src/tracker_context.rs:21):
 * VT_OK and shape_out = {D, depth, heads, hidden, head_channels} when vt_tracker_create would accept the file, VT_ERR_WEIGHTS (and
 * vt_last_error()) when the file is missing, not a VTW1 file, of an unsupported shape, or its size does not match its header. */
vt_status vt_weights_probe(const char* path, int32_t shape_out[5]);

/* ------------------------------------------------------------------------------------------- */
/* VitTrack                                                                                     */
/* ------------------------------------------------------------------------------------------- */
/* ≙ VitTrack::new(model_path) (src/tracker_context.rs:21) */
vt_status vt_tracker_create(const vt_config* cfg, vt_tracker** out);
void vt_tracker_destroy(vt_tracker* t);

/* ≙ VitTrack::init(&frame, bbox) (src/tracker_context.rs:88).  `frame` is host memory in the
 * handle's format, tightly packed (NV12: w*h*3/2 bytes, src/nv12_convert.rs:48; RGB24: h*w*3,
 * src/pipeline_ir.rs:142; RGBA / BGRA: h*w*4; I420: GStreamer's layout, see vt_format).  A short NV12 buffer is treated as an all-black image
 * (src/nv12_convert.rs:48-50). */
vt_status vt_tracker_init(vt_tracker* t, int32_t target, const uint8_t* frame, size_t len, vt_bbox box);

/* ≙ VitTrack::update(&frame) (src/tracker_context.rs:90,120) for every initialised target, one
 * batched forward.  results[max_targets]; entries of targets that are not initialised get
 * status VT_ERR_NOT_INIT.  With cfg.box_overlay the rows touched by the box overlay are written
 * back into `frame` (≙ draw_rect_nv12 + draw_crosshair_nv12, src/pipeline.rs:165-168). */
vt_status vt_tracker_update(vt_tracker* t, uint8_t* frame, size_t len, vt_result* results);

/* Asynchronous pair: submit() enqueues upload + kernels on the handle's CUDA stream and returns; wait() blocks until the OLDEST
 * submitted frame's results are in host memory.  Up to two frames may be in flight per handle (rect_last lives on the device, so
 * frame t+1 can be enqueued before the result of frame t has been read): this hides the host round trip between frames.
 * `frame` must stay valid until its wait() returns.  Pageable (non-pinned) host frames cannot be pipelined (one staging buffer);
 * with cfg.upload_window a frame submitted while another is in flight gets a predicted window (the host mirror of rect_last lags by
 * one frame: its search window grown by 1/8 of its side); whatever the real window needs beyond it the crop kernel reads straight
 * from the pinned frame, so results never depend on the prediction. */
vt_status vt_tracker_submit(vt_tracker* t, uint8_t* frame, size_t len);
vt_status vt_tracker_submit_device(vt_tracker* t, uint8_t* d_frame, size_t len);  /* frame already in device memory, tracked in place */
vt_status vt_tracker_wait(vt_tracker* t, vt_result* results);

/* Stream group: the handle's n active targets are n independent video streams — ≙ n TrackerContexts (src/pipeline.rs:55: one per
 * pipeline) stepped together.  frames[i] (pinned host memory, a full frame: lens[i] >= the frame bytes of stream i's geometry) belongs
 * to the i-th active target (ascending slot order); every stream's search window is uploaded into its own device frame, all n targets
 * go through ONE batched ViT forward (from 4 streams on the GEMMs run in their many-row throughput forms), and with cfg.box_overlay
 * each stream's box is drawn into ITS frame.  results[slot] as in update().  Each target is initialised on a frame of its own stream
 * with vt_tracker_init(t, slot, frame_of_that_stream, len, box).  Results equal those of n single-target handles of the streams'
 * geometries (boxes equal, scores within the re-association noise of the kernel forms, <= 1e-5).
 * Every stream has the handle's geometry (cfg.format / width / height) unless its slot was given one of its own with
 * vt_tracker_set_stream_geometry: one group may mix cameras of different sizes and formats (e.g. a 1920x1080 NV12 visible camera and a
 * 640x512 YUY2 IR camera, src/pipeline.rs:26-36 / src/pipeline_ir.rs:27-56) in the same batched forward. */
vt_status vt_tracker_update_streams(vt_tracker* t, uint8_t* const* frames, const size_t* lens, int32_t n, vt_result* results);

/* Stream groups of mixed cameras: target slot `target` takes frames of its own format and size instead of cfg.format / width / height.
 * Once set, every call that handles that slot's frames uses it: vt_tracker_init / vt_tracker_init_surface on the slot (template crop,
 * length, pitch and template-window checks) and, for the stream of that slot, vt_tracker_update_streams, vt_tracker_update_streams_surface
 * and vt_tracker_run_streams_ring.  Everything else stays per handle (pad_plus1, decode / window switches, normalisation, box_overlay,
 * overlay_gate, upload_window).  VT_ERR_INVALID (and vt_last_error()) for: an initialised slot (vt_tracker_drop it first), frames in
 * flight, a probe (HUD) handle, an unknown format, or a width or height <= 0.  g == NULL: the slot goes back to the cfg geometry.
 * On a handle where any slot's geometry differs from cfg the single-frame entry points (update, submit, *_device, update_surface,
 * submit_surface, run_ring, vt_overlay_current) are VT_ERR_INVALID: one frame of the handle's geometry cannot serve every target. */
typedef struct { int32_t format, width, height, reserved; } vt_stream_geometry;  /* format: vt_format; reserved: 0 */
vt_status vt_tracker_set_stream_geometry(vt_tracker* t, int32_t target, const vt_stream_geometry* g);
vt_status vt_tracker_get_stream_geometry(const vt_tracker* t, int32_t target, vt_stream_geometry* out);

/* Same as update() but the frame is already in device memory (bench `value` leg, NVDEC/NVMM producers): the tracker reads the
 * caller's frame in place (no copy) and, with cfg.box_overlay, draws the box INTO it — the in-place semantics of the reference's
 * probe (src/pipeline.rs:90-100,165-168) on a device surface. */
vt_status vt_tracker_update_device(vt_tracker* t, uint8_t* d_frame, size_t len, vt_result* results);

/* A frame in device memory on the handle's GPU, in the handle's format, with any row pitch (decoder surfaces: NVDEC, NvBufSurface).
 * NV12: planes[0] = Y (H rows), planes[1] = interleaved UV ((H+1)/2 rows); RGB24 / GRAY8 / YUY2 / RGBA / BGRA: planes[0] only, planes[1]
 * ignored.  pitch[i] >= the plane's row bytes (W for Y / UV / GRAY8, 3W for RGB24, 4 * ceil(W/2) for YUY2, 4W for RGBA / BGRA: a
 * DeepStream NvBufSurface gives planes[0] = dataPtr + planeParams.offset[0], pitch[0] = planeParams.pitch[0]); planes may be separate allocations
 * and need no alignment.  A tightly packed frame d is the surface {d, d + W*H}, {W, W} (RGB24: {d, NULL}, {3W, 0}).
 * There are no I420 surfaces: a vt_surface has two planes, and hardware decoders (NVDEC, nvv4l2decoder, nvh264dec) deliver NV12, while
 * I420 comes from software decoders in host memory.  Every surface entry point (the vt_tracker_*_surface calls, vt_probe_frame_surface,
 * vt_probe_group_frame_surface) is VT_ERR_INVALID, with vt_last_error() naming I420, for an I420 handle or stream slot; a packed I420
 * device frame goes through vt_tracker_update_device / vt_tracker_submit_device.
 *
 * The surface entry points below are additive (VT_ABI_VERSION stays 2): each behaves like the entry point it names, except that the
 * frame is a surface.  The tracker reads the surface in place (nothing is copied), and with cfg.box_overlay draws the box into it: into
 * planes[0] (the Y plane for NV12 / GRAY8, the Y samples for YUY2, the image for RGB24, the colour bytes for RGBA / BGRA) with the
 * reference's clamping, so nothing is written into the pitch padding, the UV plane, the YUY2 chroma bytes or byte 3 of a 32-bit pixel.  The surface must stay valid until the call returns (submit: until the matching wait()).
 * VT_ERR_INVALID (and vt_last_error()) for a NULL surface or plane, a pitch below the plane's row bytes, a plane that is not device or
 * managed memory of cfg.device, and — synchronous calls — frames in flight.  These four vt_tracker_*_surface calls are also
 * VT_ERR_INVALID on the tracker of a probe (HUD) handle, whose surfaces go through vt_probe_frame_surface / vt_probe_group_frame_surface. */
typedef struct { uint8_t* planes[2]; size_t pitch[2]; } vt_surface;
vt_status vt_tracker_init_surface(vt_tracker* t, int32_t target, const vt_surface* s, vt_bbox box);  /* ≙ vt_tracker_init */
vt_status vt_tracker_update_surface(vt_tracker* t, const vt_surface* s, vt_result* results);         /* ≙ vt_tracker_update_device */
vt_status vt_tracker_submit_surface(vt_tracker* t, const vt_surface* s);                             /* ≙ vt_tracker_submit_device; then wait() */
/* ≙ vt_tracker_update_streams: surfaces[i] belongs to the i-th active target (n = the number of active targets, at most 16); each stream's
 * box is drawn into its own surface.  Streams may have different pitches and plane offsets, and each surface is checked against the row
 * bytes and plane count of its own stream's geometry (vt_tracker_set_stream_geometry). */
vt_status vt_tracker_update_streams_surface(vt_tracker* t, const vt_surface* surfaces, int32_t n, vt_result* results);

/* The per-buffer loop of a streaming thread, run natively (≙ the GStreamer streaming thread invoking the probe once per buffer,
 * src/pipeline.rs:65-67): n frames of a ring (`ring` frames of frame_len bytes, `stride` bytes apart, starting at index `first`,
 * wrapping) go through this handle.  `frames` is host memory for the HOST modes (pinned for pipelining) and device memory for the
 * DEVICE modes.  SYNC = vt_tracker_update[_device] per frame; PIPELINED = vt_tracker_submit[_device] / vt_tracker_wait with two frames
 * in flight.  `pristine` (nullable, host modes with cfg.box_overlay): the same ring without overlays — after a frame's wait() the
 * pixels its box overlay touched are restored from it, so a ring can be replayed on clean frames.  latency_us (nullable, n entries):
 * wall time from handing frame i in to having its result (SYNC modes).  last (nullable): results[max_targets] of the final frame.
 * Multi-stream drivers call this from one host thread per stream. */
typedef enum { VT_RUN_HOST_SYNC = 0, VT_RUN_HOST_PIPELINED = 1, VT_RUN_DEVICE_SYNC = 2, VT_RUN_DEVICE_PIPELINED = 3 } vt_run_mode;
vt_status vt_tracker_run_ring(vt_tracker* t, uint8_t* frames, size_t stride, size_t frame_len, int32_t ring, int32_t first, int32_t n,
                              int32_t mode, const uint8_t* pristine, vt_result* last, double* latency_us);
/* The same loop for a stream group (vt_tracker_update_streams per step): rings[i] = ring of stream i (pinned host memory), pristine[i]
 * (nullable array / entries) = its clean copy.  In a group of mixed geometries frame_len and stride cover the largest stream's frame;
 * each stream reads (and restores) only the bytes of its own geometry. */
vt_status vt_tracker_run_streams_ring(vt_tracker* t, uint8_t* const* rings, int32_t n_streams, size_t stride, size_t frame_len, int32_t ring,
                                      int32_t first, int32_t n, const uint8_t* const* pristine, vt_result* last, double* latency_us);

/* tracker state access (≙ rect_last inside VitTrack; used by tests for teacher forcing) */
vt_status vt_tracker_get_rect(vt_tracker* t, int32_t target, vt_bbox* out);
vt_status vt_tracker_set_rect(vt_tracker* t, int32_t target, vt_bbox box);
vt_status vt_tracker_drop(vt_tracker* t, int32_t target); /* forget a target */

/* diagnostics for parity tests: copies of device intermediates of the last update (any pointer may be NULL)
 *   search_blob  float[3*256*256]  planar CHW normalised search crop of `target`
 *   conf_win     float[256]        conf * hann
 *   size_map     float[512], off_map float[512]
 *   tokens       float[320*D]      final-LayerNorm token features */
vt_status vt_tracker_debug_read(vt_tracker* t, int32_t target, float* search_blob, float* template_blob,
                                float* conf_win, float* size_map, float* off_map, float* tokens);
int32_t vt_tracker_model_dim(const vt_tracker* t, int32_t which); /* 0 D, 1 depth, 2 heads, 3 hidden, 4 head_ch;
                                                                      5: tracker handles alive on this handle's GPU, all processes (the
                                                                         latency / throughput kernel forms switch on it) */
/* token features [320*D] after the embeddings (which = 0) or after block `which` (1..depth).  Needs
 * cfg.debug_capture = 1 at create time (captures one copy per block; disables graph replay). */
vt_status vt_tracker_debug_tokens(vt_tracker* t, int32_t target, int32_t which, float* out);
/* Device timeline of the tensor-core kernels launched since the previous call (set VT_B200_TRACE=1 in the environment before
 * vt_tracker_create; VT_ERR_INVALID otherwise): out[8 i ..] = {kernel id, t_entry, t_after_dependency_wait, t_end, 4 kernel-specific
 * marks} in ns of the GPU's global timer; *n = records written (<= max_records).  ≙ the finer per-stage timers of src/pipeline_ir.rs:126-208. */
vt_status vt_tracker_debug_trace(vt_tracker* t, unsigned long long* out, int32_t max_records, int32_t* n);
/* the handle's CUDA stream (cudaStream_t) so that callers can time on the launching stream, and a stream sync */
void* vt_tracker_stream(vt_tracker* t);
vt_status vt_tracker_sync(vt_tracker* t);

/* diagnostics: one C[M,N] = A[M,K] * W[N,K]^T (+bias, optional GELU) on host data through the tcgen05 GEMM kernel
 * (nsplit 1 = bf16, 3 = bf16x3); *err_out != 0 reports an expired pipeline wait.  N and K multiples of 64. */
vt_status vt_debug_gemm(int32_t device, int32_t M, int32_t N, int32_t K, const float* A, const float* W, const float* bias,
                        int32_t nsplit, int32_t gelu, float* C_out, int32_t* err_out);

/* ------------------------------------------------------------------------------------------- */
/* NV12 -> RGB (parity / bench entry)                                                           */
/* ------------------------------------------------------------------------------------------- */
/* ≙ nv12_full_to_rgb_parallel(nv12, width, height) -> Array3<u8>(h, w, 3) in R,G,B order
 * (src/nv12_convert.rs:46-92).  Host buffers; len < w*h*3/2 -> rgb_out is all zeros (:48-50). */
vt_status vt_convert_nv12_rgb(vt_tracker* t, const uint8_t* nv12, size_t len, uint8_t* rgb_out);
/* device-resident, batched: n_frames frames of the handle's geometry, frame i at d_nv12 + i*stride_in */
vt_status vt_convert_nv12_rgb_device(vt_tracker* t, const uint8_t* d_nv12, size_t stride_in, uint8_t* d_rgb,
                                     size_t stride_out, int32_t n_frames);

/* ------------------------------------------------------------------------------------------- */
/* format steps either side of the RGB probe (SURVEY.md §8(f) row 1)                            */
/* ------------------------------------------------------------------------------------------- */
/* ≙ the `videoconvert` YUY2 -> RGB step of src/pipeline_ir.rs:27-56 (GStreamer element; its source is not in the reference tree,
 * so this follows the reference's own BT.601 integer arithmetic, src/nv12_convert.rs:24-30,124-126, on packed 4:2:2).
 * yuy2: rows of (width*2 rounded up to 4) bytes, Y0 U Y1 V; rgb_out: h*w*3, R,G,B.  A short buffer gives a black frame. */
vt_status vt_convert_yuy2_rgb(vt_tracker* t, const uint8_t* yuy2, size_t len, int32_t width, int32_t height, uint8_t* rgb_out);
vt_status vt_convert_yuy2_rgb_device(vt_tracker* t, const uint8_t* d_yuy2, size_t stride_in, uint8_t* d_rgb, size_t stride_out, int32_t width,
                                     int32_t height, int32_t n_frames);
/* ≙ the `rgaconvert` RGB 640x512 -> 1280x1024 display upscale of src/pipeline_ir.rs:62-73 (hardware scaler element): bilinear with
 * OpenCV INTER_LINEAR fixed-point semantics, bit-exact with cv2.resize (any source / destination size). */
vt_status vt_resize_rgb(vt_tracker* t, const uint8_t* rgb, int32_t src_w, int32_t src_h, uint8_t* out, int32_t dst_w, int32_t dst_h);
vt_status vt_resize_rgb_device(vt_tracker* t, const uint8_t* d_rgb, int32_t src_w, int32_t src_h, uint8_t* d_out, int32_t dst_w, int32_t dst_h);
/* device-resident, batched: n_frames frames, frame i at d_rgb + i*stride_in -> d_out + i*stride_out (one launch) */
vt_status vt_resize_rgb_device_batch(vt_tracker* t, const uint8_t* d_rgb, size_t stride_in, int32_t src_w, int32_t src_h, uint8_t* d_out,
                                     size_t stride_out, int32_t dst_w, int32_t dst_h, int32_t n_frames);

/* ------------------------------------------------------------------------------------------- */
/* overlay                                                                                      */
/* ------------------------------------------------------------------------------------------- */
typedef enum {
    VT_OV_RECT = 0,       /* ≙ draw_rect_nv12 (src/nv12_convert.rs:172) / draw_rect_rgb (src/drawing_rgb.rs:55): x,y,w,h,a=thickness */
    VT_OV_CROSSHAIR = 1,  /* ≙ draw_crosshair_nv12 (:216) / draw_crosshair_rgb (:68): x=cx,y=cy,a=size */
    VT_OV_TEXT = 2,       /* ≙ draw_text_nv12 (:245) / draw_text_rgb (:86): x,y,a=scale,text */
    VT_OV_BACKGROUND = 3, /* ≙ draw_background_nv12 (:324; a=darkness) / draw_background_rgb (:30; fill 30) */
    VT_OV_CURSOR = 4,     /* ≙ draw_cursor (src/drawing.rs:5) / draw_cursor_rgb (src/drawing_rgb.rs:75): x,y */
    VT_OV_SELECTION = 5   /* ≙ draw_selection (src/drawing.rs:25) / draw_selection_rgb (:106): x,y=start, w,h=cursor */
} vt_overlay_kind;

typedef struct {
    int32_t kind;
    int32_t x, y, w, h;
    int32_t a;            /* thickness | size | scale | darkness */
    uint8_t r, g, b;      /* NV12: r is the luma/brightness; RGB: colour (text uses r as luma) */
    uint8_t strict_glyphs;/* text: 1 = unknown char is VT_ERR_GLYPH (RGB path panics in the reference), 0 = skip+advance (NV12 path) */
    char text[48];
} vt_overlay_cmd;

/* Applies cmds in order to a host frame (upload, draw on device, copy the touched rows back). */
vt_status vt_overlay(vt_tracker* t, uint8_t* frame, size_t len, const vt_overlay_cmd* cmds, int32_t n);
/* Same, on the device-resident copy of the frame most recently given to update()/submit(); only the
 * touched rows travel back into `frame`.  This is what the probe shim uses for pageable frames.  When the device copy is not that
 * frame (the last frame was device-resident and tracked in place, or a conversion / vt_overlay() reused the buffer) `frame` is
 * uploaded first, as vt_overlay() does. */
vt_status vt_overlay_current(vt_tracker* t, uint8_t* frame, size_t len, const vt_overlay_cmd* cmds, int32_t n);

/* ------------------------------------------------------------------------------------------- */
/* timing                                                                                       */
/* ------------------------------------------------------------------------------------------- */
/* ≙ TimingStats (src/timing_stats.rs): same 120-sample windows and accessors, plus the
 * device-timed stage breakdown (%globaltimer stamps written by the kernels) of the last frame and its rolling means. */
typedef struct {
    double fps;            /* ≙ TimingStats::fps()          1e6 / mean(interval_us) */
    double avg_conv_ms;    /* ≙ TimingStats::avg_conv_ms()  (device: preprocess stage) */
    double avg_track_ms;   /* ≙ TimingStats::avg_track_ms() (host wall time of update) */
    /* device-timed stages, last frame (ms) */
    float h2d_ms, preprocess_ms, vit_ms, decode_ms, overlay_ms, d2h_ms, total_ms;
    /* rolling means over the same 120-frame window (ms) */
    float avg_h2d_ms, avg_preprocess_ms, avg_vit_ms, avg_decode_ms, avg_overlay_ms, avg_d2h_ms, avg_total_ms;
    uint64_t frames;
    uint64_t kernel_launches;  /* kernels launched by this handle so far (graph nodes count individually) */
    uint64_t h2d_bytes, d2h_bytes; /* bytes this handle copied host->device / device->host so far */
} vt_timing;
vt_status vt_timing_get(vt_tracker* t, vt_timing* out);
/* ≙ TimingStats::add_interval / add_times for callers that keep the reference's host timers */
vt_status vt_timing_add_interval(vt_tracker* t, uint64_t us);
vt_status vt_timing_add_times(vt_tracker* t, uint64_t conv_us, uint64_t track_us);

/* ≙ TimingStats::new() as a free-standing object for callers that keep their own timers (no device needed) */
typedef struct vt_timing_stats vt_timing_stats;
vt_timing_stats* vt_timing_stats_create(void);
void vt_timing_stats_destroy(vt_timing_stats* s);
void vt_timing_stats_add_interval(vt_timing_stats* s, uint64_t us);
void vt_timing_stats_add_times(vt_timing_stats* s, uint64_t conv_us, uint64_t track_us);
double vt_timing_stats_fps(const vt_timing_stats* s);
double vt_timing_stats_avg_conv_ms(const vt_timing_stats* s);
double vt_timing_stats_avg_track_ms(const vt_timing_stats* s);

/* ------------------------------------------------------------------------------------------- */
/* host state machine (≙ TrackerContext / SelectionState / UserCommand / AppState)              */
/* ------------------------------------------------------------------------------------------- */
/* ≙ UserCommand (src/user_commands.rs:2-9); `fast` is the bool payload of the Move* variants */
typedef enum { VT_CMD_MOVE_UP = 0, VT_CMD_MOVE_DOWN, VT_CMD_MOVE_LEFT, VT_CMD_MOVE_RIGHT, VT_CMD_CONFIRM, VT_CMD_CANCEL, VT_CMD_QUIT } vt_command;
/* ≙ state_name() values (src/tracker_context.rs:157-166) */
typedef enum { VT_STATE_SELECT_START = 0, VT_STATE_SELECT_END, VT_STATE_TRACKING, VT_STATE_LOST } vt_state;
/* ≙ SelectionState (src/selection_state.rs:9-18) */
typedef struct { int32_t cursor_x, cursor_y, start_x, start_y, phase, step, fast_step; } vt_selection;

/* ≙ the keyboard reader's byte -> UserCommand map (src/raw_mode_guard.rs:65-101): returns 1 and fills cmd (vt_command) / fast
 * when `byte` maps to a command, 0 when the reference ignores it.  VT_CMD_QUIT is what clears the `running` flag there (:89-92). */
int32_t vt_command_from_key(uint8_t byte, int32_t* cmd, int32_t* fast);

typedef struct vt_context vt_context;
/* ≙ TrackerContext::new(model_path, width, height) (src/tracker_context.rs:19); creates its tracker from cfg */
vt_status vt_context_create(const vt_config* cfg, vt_context** out);
void vt_context_destroy(vt_context* c);
/* ≙ TrackerContext::handle_command (src/tracker_context.rs:36) */
vt_status vt_context_handle_command(vt_context* c, int32_t cmd, int32_t fast);
/* ≙ TrackerContext::process_frame(&frame) -> Option<BBox> (src/tracker_context.rs:64).
 * *has_bbox = 1 and *bbox filled ≙ Some(bbox). Frame in the handle's format (NV12 frames are
 * converted on the device inside the fused crop kernel; the RGB image is never materialised). */
vt_status vt_context_process_frame(vt_context* c, uint8_t* frame, size_t len, int32_t* has_bbox, vt_bbox* bbox);
/* The same state machine with the outcome of VitTrack::update supplied by the caller (err != 0 ≙ Err);
 * no device is involved.  Used to exercise the host logic without a GPU. */
vt_status vt_context_create_scripted(int32_t width, int32_t height, vt_context** out);
vt_status vt_context_process_scripted(vt_context* c, const vt_result* scripted, int32_t err, int32_t* has_bbox, vt_bbox* bbox);
int32_t vt_context_state(const vt_context* c);
const char* vt_context_state_name(const vt_context* c);            /* "SELECT START" | "SELECT END" | "TRACKING" | "LOST" */
float vt_context_current_score(const vt_context* c);                /* ≙ ctx.current_score (src/pipeline.rs:116) */
int32_t vt_context_current_bbox(const vt_context* c, vt_bbox* out); /* ≙ ctx.current_bbox (src/pipeline.rs:170); 1 = Some */
void vt_context_selection(const vt_context* c, vt_selection* out);  /* ≙ ctx.selection.clone() (src/pipeline.rs:117) */
uint64_t vt_context_lost_frames(const vt_context* c);
vt_tracker* vt_context_tracker(vt_context* c);

/* ≙ the body of the pad-probe closure, src/pipeline.rs:67-184 (NV12) / src/pipeline_ir.rs:100-228
 * (RGB24 / RGBA / BGRA, chosen by cfg.format): interval timing, process_frame, HUD + cursor/selection + box
 * overlay written in place into `frame`.  Commands are delivered beforehand with
 * vt_context_handle_command (≙ draining cmd_rx, src/pipeline.rs:84-88).  hud_override (may be
 * NULL) replaces the timing-dependent HUD strings so that pixel parity is testable:
 * {fps_line, timing_line}. */
vt_status vt_probe_frame(vt_context* c, uint8_t* frame, size_t len, const char* const* hud_override);
/* ≙ vt_probe_frame on a pitched device surface of the context's geometry (vt_surface rules above): the probe's HUD, cursor / selection
 * and box are drawn in place into the surface's plane 0 (Y / RGB / the Y samples of YUY2 / the colour bytes of RGBA / BGRA), never into
 * pitch padding, the UV plane, YUY2 chroma bytes or byte 3 of a 32-bit pixel; nothing is copied between host and device but the result block.  A confirm frame initialises the tracker on this
 * surface.  VT_ERR_INVALID (and vt_last_error()) for a NULL surface, a surface that fails the vt_surface checks, or a probe-group member.
 * A context may take host frames on one call and surfaces on the next. */
vt_status vt_probe_frame_surface(vt_context* c, const vt_surface* s, const char* const* hud_override);

/* The same loop over vt_probe_frame (the drop-in call): n frames of a host ring through the context, HUD drawn into every frame.
 * `pristine` (nullable): after each probe the HUD region and the box of that frame are restored from it. */
vt_status vt_context_run_ring(vt_context* c, uint8_t* frames, size_t stride, size_t frame_len, int32_t ring, int32_t first, int32_t n,
                              const char* const* hud_override, const uint8_t* pristine, double* latency_us);

/* ---- probe groups: the drop-in probe for up to 16 cameras in one batched forward (additive; VT_ABI_VERSION stays 2) ----------------
 * ≙ n TrackerContext::new (one per pipeline, src/pipeline.rs:55) sharing ONE tracker handle with max_targets = n_streams (1..16): stream i
 * is member context i and target slot i.  Each stream behaves exactly like a single vt_context probing the same frames with the same
 * commands, but one group step runs ONE batched forward over the streams whose state machine calls VitTrack on that frame (TRACKING:
 * update; SELECT END with a pending confirm: init on that stream's frame, then update) and draws every stream's HUD, cursor / selection and
 * box in place — each with the HUD style of its format (luma: NV12 / GRAY8 / YUY2; RGB: RGB24 / RGBA / BGRA) — with ONE synchronisation for the whole step.
 * A stream that leaves TRACKING, or whose confirm fails the gate, gives up its slot (tracking resumes only through a fresh init).
 * Timing: the group keeps one TimingStats (on its tracker) and every stream is probed once per step, so every stream's FPS / conv / trk
 * HUD line shows the group's step figures. */
typedef struct vt_probe_group vt_probe_group;
/* geoms: NULL = every stream has cfg's format / width / height; else n_streams entries (validated as vt_tracker_set_stream_geometry). */
vt_status vt_probe_group_create(const vt_config* cfg, int32_t n_streams, const vt_stream_geometry* geoms, vt_probe_group** out);
void vt_probe_group_destroy(vt_probe_group* g);
int32_t vt_probe_group_size(const vt_probe_group* g);  /* VT_ERR_INVALID for NULL */
/* The borrowed member context of stream i (NULL when out of range): vt_context_handle_command and every read accessor (state, state_name,
 * current_score, current_bbox, selection, lost_frames, vt_context_tracker) work on it; the frame entry points (vt_probe_frame,
 * vt_context_process_frame, vt_context_run_ring) are VT_ERR_INVALID on a member; vt_context_destroy on a member does nothing.
 * The shared tracker (vt_context_tracker of any member) refuses every frame entry point (init / update / submit / stream-group / ring
 * calls); vt_tracker_get_rect / set_rect (stream i = target i), vt_tracker_debug_read, vt_timing_get and vt_tracker_stream stay usable. */
vt_context* vt_probe_group_context(vt_probe_group* g, int32_t stream);
/* ≙ the n pad-probe closures each invoked once for one buffer of its camera.  frames[i]: pinned host frame of stream i (vt_alloc_pinned),
 * full length for its geometry (lens[i] >= its frame bytes); a pageable, short or NULL frame is VT_ERR_INVALID with a message.
 * hud_override as in vt_probe_frame, for every stream. */
vt_status vt_probe_group_frame(vt_probe_group* g, uint8_t* const* frames, const size_t* lens, const char* const* hud_override);
/* ≙ vt_probe_group_frame with surfaces[i] the current surface of stream i (n = vt_probe_group_size(g)); each checked against stream i's
 * geometry; one batched forward, one synchronisation, every stream's HUD drawn into its own surface.  VT_ERR_INVALID (and
 * vt_last_error()) for a NULL group or array, n != the group's size, or a surface that fails the vt_surface checks for its stream. */
vt_status vt_probe_group_frame_surface(vt_probe_group* g, const vt_surface* surfaces, int32_t n, const char* const* hud_override);
/* ≙ vt_context_run_ring for a group: n steps, stream i's frames from rings[i] (pinned host memory; `ring` frames, `stride` apart, frame_len
 * bytes each), pristine[i] (nullable; pristine itself nullable) restores what each step drew, latency_us[step] (nullable). */
vt_status vt_probe_group_run_ring(vt_probe_group* g, uint8_t* const* rings, size_t stride, size_t frame_len, int32_t ring, int32_t first,
                                  int32_t n, const char* const* hud_override, const uint8_t* const* pristine, double* latency_us);

#ifdef __cplusplus
}
#endif
#endif /* VT_TRACKER_H */
