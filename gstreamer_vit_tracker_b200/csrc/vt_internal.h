// vt_internal.h — shared declarations of libvittrack_b200 (not installed; the public ABI is include/vt_tracker.h)
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "vt_tracker.h"

namespace vt {

constexpr int kNTz = 64;        // template tokens (128/16)^2
constexpr int kNTx = 256;       // search tokens (256/16)^2
constexpr int kNTok = 320;      // joint sequence
constexpr int kPatchK = 768;    // 3*16*16
constexpr int kSearch = 256;
constexpr int kTemplate = 128;
constexpr int kMap = 16;        // score map side
constexpr int kWindow = 120;    // TimingStats window (src/timing_stats.rs:19)
constexpr int kMaxCmds = 32;

void set_error(const char* fmt, ...);
// caller's vt_config (any struct_size the ABI ever had) -> the library's full struct with defaults for what the caller's header lacks
vt_status resolve_config(const vt_config* in, vt_config* out);

// GRAY8 frames are a bare luma plane, YUY2 frames carry one Y sample per pixel and I420 frames lead with a Y plane: all are drawn on
// with the NV12 (Y plane) overlay semantics
__host__ __device__ inline bool format_is_luma(int fmt) {
    return fmt == VT_FMT_NV12 || fmt == VT_FMT_GRAY8 || fmt == VT_FMT_YUY2 || fmt == VT_FMT_I420;
}
__host__ __device__ inline int overlay_format(int fmt) { return format_is_luma(fmt) ? VT_FMT_NV12 : fmt; }
// RGBA / BGRA: 32-bit pixels whose byte 3 (alpha or padding) is never read or written; tracked and drawn on as the RGB24 frame of their
// colour bytes
__host__ __device__ inline bool format_is_rgb32(int fmt) { return fmt == VT_FMT_RGBA || fmt == VT_FMT_BGRA; }
// byte offsets of R, G and B within a pixel of an RGB format (RGB24 / RGBA: 0 1 2; BGRA: 2 1 0): every reader and writer of colour bytes
// takes the channel order from here
struct RgbOffsets {
    int r, g, b;
};
__host__ __device__ inline RgbOffsets fmt_rgb_offsets(int fmt) { return fmt == VT_FMT_BGRA ? RgbOffsets{2, 1, 0} : RgbOffsets{0, 1, 2}; }

// ---- plane geometry of a format: every site that addresses plane 0 (Y / RGB / gray / packed YUY2 / RGBA / BGRA) goes through these
// bytes between horizontally adjacent pixels of plane 0: the RGB triple, the 32-bit RGBA / BGRA pixel, the Y sample (YUY2: Y0 U Y1 V,
// every second byte)
__host__ __device__ inline int fmt_px_step(int fmt) {
    return fmt == VT_FMT_RGB24 ? 3 : format_is_rgb32(fmt) ? 4 : fmt == VT_FMT_YUY2 ? 2 : 1;
}
// bytes of one packed row of plane 0 (YUY2: whole pixel-pair words, 4 * ceil(W / 2): odd widths pad the last word; I420: the Y stride,
// RU4(W), as GStreamer lays it out)
__host__ __device__ inline size_t fmt_row_bytes(int fmt, int W) {
    return fmt == VT_FMT_YUY2 ? (size_t)4 * (size_t)((W + 1) / 2)
         : fmt == VT_FMT_I420 ? (size_t)((W + 3) & ~3)
                              : (size_t)W * (size_t)fmt_px_step(fmt);
}
// I420 in GStreamer's default layout (include/vt_tracker.h): the Y plane of RU2(H) rows (odd H: one padding row), then the U plane,
// then the V plane, each ceil(H / 2) rows of i420_chroma_pitch(W) = RU4(ceil(W / 2)) bytes.  These two and fmt_row_bytes are the one
// place that knows that layout.
__host__ __device__ inline size_t i420_chroma_pitch(int W) { return (size_t)(((W + 1) / 2 + 3) & ~3); }
// the U plane's offset in the frame; the V plane starts i420_chroma_pitch(W) * ceil(H / 2) bytes after it
__host__ __device__ inline size_t i420_u_offset(int W, int H) { return fmt_row_bytes(VT_FMT_I420, W) * (size_t)((H + 1) & ~1); }
// bytes of a packed frame, every plane
__host__ __device__ inline size_t fmt_frame_bytes(int fmt, int W, int H) {
    if (fmt == VT_FMT_I420) return i420_u_offset(W, H) + 2 * i420_chroma_pitch(W) * (size_t)((H + 1) / 2);
    return fmt == VT_FMT_NV12 ? (size_t)W * H + (size_t)((H + 1) / 2) * W + (W & 1) : fmt_row_bytes(fmt, W) * (size_t)H;
}
// the shortest buffer that is a frame; anything shorter is an all-black image (NV12: src/nv12_convert.rs:48-50)
__host__ __device__ inline size_t fmt_valid_bytes(int fmt, int W, int H) {
    return fmt == VT_FMT_NV12 ? (size_t)W * H * 3 / 2 : fmt_frame_bytes(fmt, W, H);
}
// Geometry of the frames of one stream: the handle's (cfg.format / width / height), or a target slot's own in a stream group of mixed
// cameras (vt_tracker_set_stream_geometry)
struct StreamGeom {
    int32_t fmt, W, H;
    size_t bytes() const { return fmt_frame_bytes(fmt, W, H); }
    bool operator==(const StreamGeom& o) const { return fmt == o.fmt && W == o.W && H == o.H; }
};
// the formats and sizes a handle's frames may have (vt_tracker_create's cfg, vt_tracker_set_stream_geometry)
inline bool geometry_ok(int fmt, int W, int H) {
    return W > 0 && H > 0 && (format_is_luma(fmt) || fmt == VT_FMT_RGB24 || format_is_rgb32(fmt));
}
// the bytes [*o0, *o1) of a plane-0 row that hold the pixels x0 .. x1 - 1 (YUY2: the whole words of those pixels)
__host__ __device__ inline void fmt_col_span(int fmt, long long x0, long long x1, size_t* o0, size_t* o1) {
    if (fmt == VT_FMT_YUY2) *o0 = (size_t)(2 * (x0 & ~1LL)), *o1 = (size_t)(4 * ((x1 + 1) / 2));
    else *o0 = (size_t)(x0 * fmt_px_step(fmt)), *o1 = (size_t)(x1 * fmt_px_step(fmt));
}

#define VT_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ::vt::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return VT_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

// Launch with optional programmatic dependent launch (the kernel calls griddepcontrol.wait before touching anything the
// preceding kernel of the stream wrote) and an optional thread-block cluster along x.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, int cluster_x, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = s;
    cudaLaunchAttribute attr[2];
    unsigned n = 0;
    if (pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster_x > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = (unsigned)cluster_x, attr[n].val.clusterDim.y = 1, attr[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = attr, cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- TimingStats, src/timing_stats.rs:3-60 (same window, same arithmetic) -------------------------
template <typename T>
struct Ring {
    T v[kWindow];
    int head = 0, len = 0;
    void push(T x) {
        if (len >= kWindow) head = (head + 1) % kWindow, --len;
        v[(head + len) % kWindow] = x;
        ++len;
    }
    double mean() const {
        if (!len) return 0.0;
        double s = 0;
        for (int i = 0; i < len; ++i) s += (double)v[(head + i) % kWindow];
        return s / len;
    }
};
struct TimingStats {
    Ring<uint64_t> intervals, conv, track;
    void add_interval(uint64_t us) { intervals.push(us); }
    void add_times(uint64_t c, uint64_t t) { conv.push(c), track.push(t); }
    double fps() const {
        if (!intervals.len) return 0.0;
        const double avg = intervals.mean();
        return avg > 0.0 ? 1000000.0 / avg : 0.0;
    }
    double avg_conv_ms() const { return conv.len ? conv.mean() / 1000.0 : 0.0; }
    double avg_track_ms() const { return track.len ? track.mean() / 1000.0 : 0.0; }
};

// ---- per-target device state -----------------------------------------------------------------
struct TargetState {       // lives in device memory, one per target slot
    int32_t rect[4];       // rect_last x, y, w, h  (≙ TrackerVit::rect_last)
    int32_t active;        // 1 after init
    int32_t crop_err;      // set by the crop kernel when the window is entirely outside the frame
    int32_t pad[2];
};

struct DeviceResult {      // written by the decode kernel, copied to pinned host memory
    int32_t success;
    float score;
    int32_t bbox[4];
    int32_t status;
    int32_t best;          // argmax index (diagnostic)
};

// Device-side stage stamps (%globaltimer, ns), copied to the host together with the results: they replace cudaEvent records
// inside the per-frame graph (an event node between two kernels breaks the programmatic-dependent-launch edge) and the seven
// cudaEventElapsedTime queries per frame (~20 us of host time).
enum { ST_SUBMIT = 0, ST_PRE, ST_VIT, ST_DEC, ST_DEC_END, ST_OVL_END, ST_COUNT = 8 };
__device__ __forceinline__ unsigned long long device_time_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
    return t;
}
// One frame as the kernels read and draw it, built on the host by packed_ref / surface_ref (tracker_frame.cu): always complete, the
// kernels apply no defaults.  A host frame only ever goes with a PACKED device frame of the same layout (the handle's or a stream's own
// buffer, into which windows of the host frame are uploaded), so the crop kernel's fall-back and the overlay mirror address the host
// frame with the device frame's pitches and chroma offset; a surface or a device frame tracked in place has none.
struct FrameRef {
    const uint8_t* plane[2];      // plane 0 (Y / RGB / gray / YUY2 / RGBA / BGRA); NV12 chroma plane, I420 U plane (always packed: the V
                                  // plane follows it at pitch[1] * ceil(H / 2)), else null
    size_t pitch[2];              // their row pitches in bytes (packed frames: fmt_row_bytes, W; I420: i420_chroma_pitch)
    uint8_t* host;                // the caller's PINNED host frame (device-mapped under UVA) or null: zero-copy target of the overlay mirror
                                  // and the crop kernel's fall-back source for pixels outside the uploaded windows
    alignas(16) int32_t geom[4];  // {format, width, height, valid}; valid 0: the buffer was short -> black image (src/nv12_convert.rs:48-50)
};
// A frame's (or a probe-group stream's) HUD: the overlay command list of the probe and the background-dim handshake
struct OverlayCmdDev;
struct HudCtl {
    const OverlayCmdDev* list;  // in pinned host memory (or the device copy the stamp kernel wrote), n entries
    int32_t n;
    int32_t bg_on_device;       // the region a leading HUD background dim reads was uploaded with the windows: read it from the device frame
    int32_t bg_ready;           // set by the host-pass CTA of the overlay kernel once its copy of that region is in registers (reset per frame)
};
// Per-frame control block in device memory: the addresses and parameters that change from frame to frame reach the kernels of the
// (captured once, replayed) per-frame graph through it.  Written by stamp_kernel at the start of every frame, outside the graph.
constexpr int kMaxWin = 16;
struct FrameCtl {
    // the frames this step reads and draws into: frames[0] for every target of a single-frame handle (n_frames = 1); active target i's
    // OWN frame frames[i] in a stream group or the forward of a probe group (n_frames = n: a group may mix cameras, and the captured graph
    // does not change with the mix).  target_frame() is the one reader of this rule.  (The scalars first: a kernel's first load of the
    // block brings frames[0] into the same cache line.)
    int32_t n_frames;
    int32_t n_win;             // -1: the whole device frame holds this frame; else win[i] = the region that does, for active target i
    uint32_t* hblk;            // pinned host result block of the frame's queue slot
    HudCtl hud;                // this frame's HUD (probe)
    FrameRef frames[kMaxWin];
    int32_t win[kMaxWin][4];   // x0, y0, x1, y1 (exclusive), even-aligned
};
__host__ __device__ inline const FrameRef& target_frame(const FrameCtl& c, int i) { return c.frames[i < c.n_frames ? i : 0]; }
// Probe groups (vt_probe_group_frame): the control block of a group's handle.  Its FrameCtl part addresses the streams that take part in
// the step's forward by active-target index, as for a stream group (the crop reads it); the per-stream table addresses EVERY stream of the
// group by its index, which is also its target slot: CTA pair x of the step's last kernel (probe_group_overlay_kernel) draws stream x.
struct ProbeStreamCtl {
    FrameRef frame;  // the stream's device frame (its search window, if it takes part, and its HUD region uploaded this step) beside its
                     // pinned host frame, or its surface (vt_probe_group_frame_surface: drawn in place)
    HudCtl hud;      // its HUD list in the pinned block of the step's queue slot; the handshake of its pair of CTAs
    int32_t slot;    // its target slot when it takes part in this step's forward, else -1 (the HUD of a stream without result)
};
struct ProbeGroupCtl {
    FrameCtl f;                  // first: every kernel of the forward reads it through the same pointer
    ProbeStreamCtl s[kMaxWin];
};
// h_list / n / d_list (optional): the frame's HUD list travels in the kernel's parameter block and is written to d_list, so the overlay
// kernel reads it from device memory (from the pinned block it was a PCIe round trip at the head of the frame's last kernel)
constexpr int kHudInline = 12;
cudaError_t launch_stamp(unsigned long long* stamp, FrameCtl* d_ctl, const FrameCtl& ctl, cudaStream_t s, const OverlayCmdDev* h_list = nullptr,
                         int n = 0, OverlayCmdDev* d_list = nullptr);
// the same for a probe group's control block (its HUD lists stay in the pinned block: each CTA pair reads its stream's list there)
cudaError_t launch_stamp_group(unsigned long long* stamp, ProbeGroupCtl* d_ctl, const ProbeGroupCtl& ctl, cudaStream_t s);
// last kernel of a frame: result block -> the pinned host block ctl->hblk (zero-copy stores)
cudaError_t launch_publish(const void* d_blk, const FrameCtl* d_ctl, size_t bytes, cudaStream_t s, bool pdl);

// ---- pixel kernels (pixel.cu) ------------------------------------------------------------------
struct FrameDesc {
    FrameRef frame;        // read only when ctl is null (the template pass of vt_tracker_init)
    // When non-null the frames (and the valid windows / host fall-back) are read from this per-frame control block: the per-frame graph
    // is captured once, while vt_tracker_update_device tracks straight out of the caller's device frame (no device->device copy) and
    // window uploads change from frame to frame.
    const FrameCtl* ctl;
    int32_t pad_plus1;     // App. A.7: 1 = the crop treats the last column / row of the frame as padding (older OpenCV: padR = x2-W+1)
};

cudaError_t launch_nv12_to_rgb(const uint8_t* d_nv12, size_t stride_in, uint8_t* d_rgb, size_t stride_out, int width, int height,
                               int n_frames, cudaStream_t s);

cudaError_t launch_yuy2_to_rgb(const uint8_t* d_yuy2, size_t stride_in, uint8_t* d_rgb, size_t stride_out, int width, int height,
                               int n_frames, cudaStream_t s);
cudaError_t launch_resize_rgb_linear(const uint8_t* d_src, int sw, int sh, uint8_t* d_dst, int dw, int dh, cudaStream_t s);
// batched form: taps per destination column / row precomputed (xt[dw] = {x0, x1, a0, a1}, yt[dh] = {y0, y1, b0, b1}); needs
// (dw * 3) % 16 == 0, 16-byte aligned destination and strides
// max_src_rows: the largest number of source rows any tile of 16 destination rows needs (0 = unknown): up to 12 the tiled separable kernel runs
cudaError_t launch_resize_rgb_tab(const uint8_t* d_src, size_t stride_in, int sw, int sh, uint8_t* d_dst, size_t stride_out, int dw, int dh,
                                  int n_frames, const int4* d_xt, const int4* d_yt, cudaStream_t s, int max_src_rows = 0);

// fused crop + (NV12->RGB) + bilinear resize + normalise -> patch-major tokens A[target][n_tok][768]
// slots: list of target slot indices processed (device array), n = count. factor 2 -> 128 template, 4 -> 256 search
// p_hi / p_lo (nullable): the same values as a bf16 (hi, lo) split, the A operand of the tensor-core patch-embed GEMM
cudaError_t launch_crop_resize_norm(FrameDesc f, TargetState* d_state, const int32_t* d_slots, int n, int factor, int out_size,
                                    const float* d_norm_lut, float* d_patches, size_t patches_stride, __nv_bfloat16* p_hi,
                                    __nv_bfloat16* p_lo, cudaStream_t s, unsigned long long* stamp = nullptr);

struct OverlayCmdDev {     // device-side copy of vt_overlay_cmd with resolved glyph rows
    int32_t kind, x, y, w, h, a;
    uint8_t r, g, b, nchar;
    uint8_t glyph[48][7];  // rows per character; 0xFF in row 0 marks "unknown: skip"
    uint8_t known[48];
    // per-frame HUD lists (probe): the frame's outcome is only known on the device when the overlay kernel runs, so the host queues the
    // commands of both outcomes and the kernel picks:
    uint8_t cond;          // 0 always; 1 only when the gate passed (status ok && success && score > gate); 2 only when it did not
    uint8_t from_result;   // 0 as given; 1 RECT = the result's bbox; 2 CROSSHAIR at the bbox centre; 3 TEXT + "<round(score*100)>%"
                           //   (digit glyphs '0'..'9' in glyph[37..46], '%' in glyph[47])
    uint8_t pad_[2];
};
enum { VT_HUD_ALWAYS = 0, VT_HUD_IF_PASS = 1, VT_HUD_IF_FAIL = 2 };
enum { VT_HUD_GIVEN = 0, VT_HUD_RESULT_RECT = 1, VT_HUD_RESULT_CROSS = 2, VT_HUD_SCORE_TEXT = 3 };
constexpr int kHudDigitSlot = 37, kHudPercentSlot = 47;
// (overlay kernels: `format` is the frame's vt_format; they draw with the semantics of overlay_format(format))
cudaError_t launch_overlay(uint8_t* d_frame, size_t len, int width, int height, int format, const OverlayCmdDev* d_cmds, int n,
                           cudaStream_t s);
// device-side box overlay straight from the decode result (rect thickness 3 + crosshair 15, src/pipeline.rs:165-168) into each target's
// frame of the control block; also the frame's last kernel: runs the per-frame HUD list of the control block (if any), mirrors the
// touched pixels into the pinned host frame and publishes the result block.  draw_box = 0: HUD list only (probe: the box is part of the
// list).  n = 0 is legal with a HUD list (frames on which no tracker ran).
cudaError_t launch_box_overlay(const DeviceResult* d_res, const int32_t* d_slots, int n, float gate, const FrameCtl* d_ctl,
                               unsigned long long* stamp_end, cudaStream_t s, bool pdl, const void* d_blk, size_t blk_bytes, int draw_box);
// the last kernel of a probe group's step: the same drawing as launch_box_overlay in HUD mode, one CTA pair per stream of the group
// (n_streams, whether or not the stream took part in the forward), each with its stream's frames, geometry, slot and HUD list from d_ctl
cudaError_t launch_group_overlay(int n_streams, const DeviceResult* d_res, float gate, const ProbeGroupCtl* d_ctl, unsigned long long* stamp_end,
                                 cudaStream_t s, bool pdl, const void* d_blk, size_t blk_bytes);

// ---- live handles per GPU across processes (handle_registry.cpp) ----------------------------------------------------------------
void registry_add(int device, int delta);
int registry_total(int device);
void registry_sweep(int device);

// ---- probe support (tracker_frame.cu; used by host_state.cpp) -----------------------------------------------------------------
// One synchronisation per probed frame: the HUD of src/pipeline.rs:125-174 is queued BEFORE the frame's result exists, as the
// commands of both outcomes; the frame's last kernel picks by the gate and takes box / score digits from the decode result.
struct HudCmd {
    vt_overlay_cmd cmd;
    uint8_t cond;         // VT_HUD_ALWAYS / VT_HUD_IF_PASS / VT_HUD_IF_FAIL
    uint8_t from_result;  // VT_HUD_GIVEN / VT_HUD_RESULT_RECT / VT_HUD_RESULT_CROSS / VT_HUD_SCORE_TEXT
};
void tracker_enable_hud(vt_tracker* t);                                   // before the handle's first frame
// the list of the NEXT submit on this handle (probe groups: of stream `stream` in the next group step)
vt_status tracker_set_hud(vt_tracker* t, const HudCmd* cmds, int n, int stream = 0);
// a frame on which no tracker runs (SELECT / LOST states): upload what the list reads, draw, mirror, publish — then vt_tracker_wait
vt_status tracker_submit_hud_only(vt_tracker* t, uint8_t* frame, size_t len);
// Probe groups (host_state.cpp: vt_probe_group).  tracker_make_group turns a fresh handle (max_targets = n, slot geometries set) into the
// tracker of a group of n streams: HUD mode, a ProbeGroupCtl, and every public frame entry point refused.  Stream i is target slot i.
vt_status tracker_make_group(vt_tracker* t, int n);
// VitTrack::init of stream i's target on its full pinned frame (no public-entry-point check); the slot joins the next step's forward
vt_status tracker_group_init(vt_tracker* t, int stream, const uint8_t* frame, size_t len, vt_bbox box);
// takes the stream's target out of the forward (device state cleared; the slot list reaches the device with the next step)
vt_status tracker_group_drop(vt_tracker* t, int stream);
bool tracker_group_active(const vt_tracker* t, int stream);
// one group step: frames[i] (pinned, full length: checked by the caller) of every stream, the HUD lists staged with tracker_set_hud; the
// streams whose slot is active run one batched forward, and the step's last kernel draws every stream's HUD — then vt_tracker_wait.
// surfs (else null): surfs[i] is stream i's device surface (checked by the caller), tracked and drawn into in place
vt_status tracker_submit_group(vt_tracker* t, uint8_t* const* frames, const size_t* lens, const vt_surface* surfs = nullptr);
// Probe (HUD) handles on the caller's device surfaces (vt_probe_frame_surface, vt_probe_group_frame_surface); the public surface calls
// refuse those handles.  tracker_check_surface: the vt_surface rules for a frame of slot `stream`'s geometry (a single probe: 0).
vt_status tracker_check_surface(const vt_tracker* t, int stream, const vt_surface* s, const char* where);
// VitTrack::init of `target` on the surface (no public-entry-point checks; a probe group's stream i is target i)
vt_status tracker_init_surface(vt_tracker* t, int32_t target, const vt_surface* s, vt_bbox box, const char* where);
// a single probe's frame on the surface with the staged HUD list: forward = false for a frame on which no tracker runs — then vt_tracker_wait
vt_status tracker_submit_surface(vt_tracker* t, const vt_surface* s, bool forward, const char* where);
bool frame_is_pinned(const void* p);
// copies the region of a frame that a box overlay (rect thickness 3 + crosshair 15) / the probe HUD touched back from a clean copy
void restore_box_region(uint8_t* frame, const uint8_t* clean, int fmt, int W, int H, const vt_bbox& b);
void restore_rect_region(uint8_t* frame, const uint8_t* clean, int fmt, int W, int H, long long x0, long long y0, long long x1, long long y1);

// ---- ViT kernels (vit.cu) ----------------------------------------------------------------------
struct GemmArgs {
    const float* A;        // activations, row-major
    int64_t lda;
    const float* W;        // [N, K] row-major (torch Linear layout)
    const float* bias;     // [N] or null
    float* C;
    int64_t ldc;
    int M, N, K;
    // optional LayerNorm over the K axis of A (K == feature dim)
    const float* ln_g;
    const float* ln_b;
    // epilogue
    int gelu;              // exact erf GELU
    int relu;
    int residual;          // C = C + result
    const float* pos;      // [a_rows_in, N] added per row (pos-embed), or null
    // row maps: logical row m -> physical row (m / rows_in) * rows_stride + row_off + (m % rows_in)
    int a_rows_in, a_rows_stride, a_row_off;
    int c_rows_in, c_rows_stride, c_row_off;
    // im2col mode for the 3x3 head conv: K = 9*feat, tap-major; A rows are 16x16 grid tokens
    int im2col_feat;       // 0 = off, else feature dim D
};
cudaError_t launch_gemm_simt(const GemmArgs& g, cudaStream_t s);
cudaError_t launch_layernorm(const float* x, int64_t ldx, const float* g, const float* b, float* y, int64_t ldy, int M, int D,
                             int rows_in, int rows_stride, int row_off, cudaStream_t s);
// LayerNorm whose output is written as a bf16 (hi, lo) split [M, D] (dense rows) for the tensor-core GEMMs
cudaError_t launch_layernorm_split(const float* x, int64_t ldx, const float* g, const float* b, __nv_bfloat16* hi, __nv_bfloat16* lo, int M,
                                   int D, int rows_in, int rows_stride, int row_off, cudaStream_t s, bool pdl = false);
// Sum of np partial GEMM results (fixed order) + bias + an fp32 addend row, fused with the following LayerNorm; one warp per row m:
//   v = add[(add_period ? m % add_period : xrow) * D ..] + bias + sum_j P[j][m, :]
//   X[xrow, :] = v                      xrow = (m / period) * x_rows + m % period + x_row_off
//   ln_hi/lo[lrow, :] = split(LN(v))    lrow = (m / period) * ln_rows + m % period + ln_row_off   (skipped when m % period + ln_row_off < 0)
// MLP: add = X (residual), add_period = 0.  Patch embed: add = pos_x, add_period = 256, rows land at 64.. of every target.
#ifdef __CUDACC__
// Single-pass fp16 operands (VT_GEMM_TCGEN05_FP16): the small kernels that write a GEMM operand take a null `lo` pointer as "hi only,
// fp16 values" — the 16 bits of the fp16 value go where the bf16 hi part would.
__device__ __forceinline__ unsigned short operand_bits(float v, bool f16) {
    return f16 ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
#endif
struct ReduceLnArgs {
    const float* P;
    int np;
    int64_t p_stride;         // elements between partials
    const float *bias, *add;
    int add_period;
    float* X;
    int M, D, period, x_rows, x_row_off;
    const float *ln_g, *ln_b;
    __nv_bfloat16 *ln_hi, *ln_lo;
    int ln_rows, ln_row_off;
};
// front: latency mode (reduce_ln_kernel FRONT)
cudaError_t launch_reduce_ln(const ReduceLnArgs& a, cudaStream_t s, bool pdl, bool front = false);
// 3x3 head conv partials (one per tap) -> + bias, ReLU -> 1x1 conv -> sigmoid / hann / arg-max / bbox decode (App. A.5-A.6).
// 16 CTAs per target (one map row each); the last one to finish merges the 16 row candidates and updates rect_last.
cudaError_t launch_head_decode(const float* P, int np, int64_t p_stride, int head_ch, const float* b1, const float* w2, const float* b2,
                               const float* hann, TargetState* d_state, const int32_t* d_slots, int n, float threshold, DeviceResult* d_res,
                               float* d_maps, float* d_cand, unsigned* d_counters, unsigned long long* stamps, cudaStream_t s, bool pdl,
                               int decode_window = 0, const int* tc_err = nullptr, bool front = false);
// qkv: [B*320, 3D]; out: [B*320, D] fp32 (nullable) and/or bf16 split (nullable)
cudaError_t launch_attention(const float* qkv, float* out, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, int B, int D, int heads,
                             cudaStream_t s);
// head 1x1 conv + sigmoid + hann + argmax + bbox decode, one CTA per target
cudaError_t launch_decode(const float* h1, int head_ch, const float* w2, const float* b2, const float* hann, TargetState* d_state,
                          const int32_t* d_slots, int n, float threshold, DeviceResult* d_res, float* d_maps, unsigned long long* stamps,
                          cudaStream_t s, int decode_window = 0);

// ---- tensor-core GEMM (gemm_tc.cu) ------------------------------------------------------------------
struct TcOut {                // dense output [planes][batch][heads][rows][cols] the epilogue copies staged tiles into
    uint8_t* base;
    int64_t row_bytes, plane_bytes;
    int rows, heads, batch;
};
struct TcGemmArgs {
    int M, N, K;
    int conv_feat;            // 0, or the feature dim D of the 3x3 head conv (A gathered from the [B,16,16,D] grid by TMA)
    const float* bias;        // [N] or null
    const float* pos;         // [pos_rows, N] added to row (m % pos_rows), or null
    int pos_rows;
    int gelu, relu;
    int residual;             // add the fp32 tile read through maps.R (flat [rows][N], same rows as the tile) before storing
    // Output addressing: row m of the GEMM is (target m / period + batch_off, row-in-target m % period + <x>_row_off) of the
    // dense [targets][heads][rows][cols] outputs (TcOut); rows outside a target's range are skipped.
    int period, batch_off;
    int c_on, c_row_off;      // fp32 tile -> c
    TcOut c, o[6], ln_out[2], p;
    int o_mode;               // 0 off; 1 bf16 split tile -> o[0] (hi), o[1] (lo); 2 QKV scatter -> o[0..5] = Q, K, V^T (hi, lo);
                              // 3 staged in shared memory only (A operand of the chained GEMM)
    int dup_ln;               // set at launch ("spread" form): replica 0 stores the fp32 tile, 1 the LayerNorm hi tile, 2 the lo tile
    int dup_hl;               // set at launch ("spread" form): replica z = 0 stores the bf16 hi tiles, z = 1 the lo tiles
    int chain_slices;         // set at launch ("spread" form): the chained product is computed in 3 column slices by 3 replicas of the tile
    int kb_per_split;         // split-K: 64-wide k-blocks per blockIdx.z slice (0 = no split); the fp32 partial tile of slice z goes to
                              // plane z of c and bias / activations / residual must be off
    int chain_n;              // N2 of a chained second GEMM (0 = off): P[blockIdx.x] = tile x W2[:, n0..n0+64)^T -> p (plane blockIdx.x)
    int o_row_off;
    // LayerNorm of the full output row fused into the epilogue (cluster of N / 64 CTAs): y = LN(row) * g + b -> ln_out[0] (hi), ln_out[1] (lo)
    const float *ln_g, *ln_b; // null = off
    int ln_row_off;
    int* err;                 // set to 1 if a bounded mbarrier wait expired
    unsigned long long* trace; // device timeline buffer (diagnostics) or null
    int trace_id;
};
struct TcMaps {               // kernel parameter block (__grid_constant__): the TMA load descriptors
    CUtensorMap Ahi, Alo, Bhi, Blo, R, B2hi, B2lo;
    CUtensorMap Ahi64, Alo64, B2hiHalf, B2loHalf;  // 64-row tiles (q64): A in boxes of 64 rows, W2 in boxes of N2 / 2 rows (one slice)
};
struct TcGemmPlan {           // one GEMM on 128 x 64 (or 64 x 64: q64) output tiles
    TcMaps maps;
    TcGemmArgs args;
};
bool tc_plan_init(TcGemmPlan* p, const __nv_bfloat16* Ahi, const __nv_bfloat16* Alo, uint64_t a_rows, const __nv_bfloat16* Whi,
                  const __nv_bfloat16* Wlo, int N, int K, int conv_feat, int conv_batch);
bool tc_plan_chain(TcGemmPlan* p, const __nv_bfloat16* W2hi, const __nv_bfloat16* W2lo, int N2, float* P, uint64_t rows, uint64_t batch);
// dense outputs [planes][batch][heads][rows][cols] (elem_bytes 2 = bf16, 4 = fp32), V^T [batch][heads][64][tokens], and the flat fp32
// residual source (TMA load)
TcOut tc_out(void* base, int elem_bytes, int64_t cols, int rows, int heads, int batch, int planes);
TcOut tc_out_vt(void* base, int tokens, int heads, int batch);
bool tc_resid_map(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols);
cudaError_t tc_gemm_setup();
// spread: latency mode — tiles are replicated over idle SMs so that each replica stores a share of the epilogue output (only when the
// whole grid still fits in one wave of kSpreadCtas CTAs)
constexpr int kSpreadCtas = 132;
// q64 (latency mode, bf16x3, plans that tc_gemm_q64_supported accepts): 64-row tiles with M = 64 UMMAs — the QKV scatter as hi / lo
// replicas (2 CTAs per tile), the chained FC1 as two replicas of N2 / 2 chained columns each; any other plan is rejected
cudaError_t tc_gemm_launch(const TcGemmPlan& p, int M, int nsplit, cudaStream_t s, bool pdl, bool spread = false, bool q64 = false);
bool tc_gemm_q64_supported(const TcGemmPlan& p, int nsplit);
// A-stationary throughput form (gemm_as.cu) of a plain 64-column-tile plan with K <= 192 whose epilogue is a bf16 (hi, lo) tile store or
// the QKV scatter: one CTA per (128-row tile, range of 64-column chunks), the activation tile resident in shared memory, two TMEM
// accumulators (main loop of chunk i + 1 under the epilogue of chunk i).  Bit-identical to tc_gemm_launch on the same plan.
cudaError_t tc_gemm_as_setup();
bool tc_gemm_as_supported(const TcGemmPlan& p);
// forced_split > 0: that many CTAs per row tile instead of as many as fit one wave (VT_B200_AS_SPLIT)
cudaError_t tc_gemm_as_launch(const TcGemmPlan& p, int M, int nsplit, cudaStream_t s, bool pdl, int sm_count, int forced_split);
// chained MLP in the A-stationary form (bf16x3): plan = an FC1 plan with tc_plan_chain applied; the GELU'd hidden tile goes back into
// tensor memory as the A operand of the chained product, which accumulates over all hidden chunks of the CTA; *planes partial planes
// (CTAs per row tile) are written to the chain output for reduce_ln_kernel
bool tc_gemm_as_mlp_supported(const TcGemmPlan& p, int nsplit);
cudaError_t tc_gemm_as_mlp_launch(const TcGemmPlan& p, int M, cudaStream_t s, bool pdl, int sm_count, int forced_split, int* planes);
struct TcAttentionPlan {      // kernel parameter block (__grid_constant__)
    CUtensorMap mQhi, mQlo, mKhi, mKlo, mVhi, mVlo;
    CUtensorMap mQ64hi, mQ64lo;      // Q in boxes of 64 rows (VT_ATT_CHAIN_Q64)
    CUtensorMap mW2hi, mW2lo;        // chained form: W_proj [D][D], boxes of 64 x 64
    __nv_bfloat16 *out_hi, *out_lo;  // [B][320][D]: the proj GEMM's A operand
    float* p2;                       // chained form: fp32 partial proj products, plane h = head h: [heads][batch][320][D]
    int64_t p2_plane;                // elements per plane
    int D, chain;                    // chain: set at launch
};
bool tc_attention_plan_init(TcAttentionPlan* p, const __nv_bfloat16* Qhi, const __nv_bfloat16* Qlo, const __nv_bfloat16* Khi, const __nv_bfloat16* Klo,
                            const __nv_bfloat16* Vthi, const __nv_bfloat16* Vtlo, int batch_heads, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, int D,
                            int batch);
bool tc_attention_plan_chain(TcAttentionPlan* p, const __nv_bfloat16* Whi, const __nv_bfloat16* Wlo, float* P2, int64_t plane_elems);
cudaError_t tc_attention_setup();
// form: plain; DUP = two replicas per tile storing the hi / lo output tiles; CHAIN = proj folded in (D / 64 replicas per tile, each
// stores one kAttChainW-column slice of the head's partial proj product; needs tc_attention_plan_chain); CHAIN_Q64 = CHAIN on 64-row query
// tiles (M = 64 UMMAs: five tiles instead of 128 + 128 + 64, half the exponentials per CTA) — the latter three are "spread" forms
enum { VT_ATT_PLAIN = 0, VT_ATT_DUP = 1, VT_ATT_CHAIN = 2, VT_ATT_CHAIN_Q64 = 3 };
constexpr int kAttChainW = 32;  // columns of the partial proj product per replica CTA of the chained form (32 or 64)
cudaError_t tc_attention_launch(const TcAttentionPlan& p, int B, int heads, int nsplit, int* err, cudaStream_t s, bool pdl,
                                unsigned long long* trace = nullptr, int form = VT_ATT_PLAIN);
cudaError_t launch_split_bf16(const float* x, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t n, cudaStream_t s);

}  // namespace vt
