// tracker_state.h — the vt_tracker handle and the internals shared by the tracker translation units:
//   tracker_create.cu  weight files, device buffers, GEMM / attention plan wiring, vt_tracker_create / destroy
//   tracker_frame.cu   the per-frame path: upload, kernel chain (CUDA graph), submit / wait, init / update entry points
//   tracker_abi.cu     convert / format / overlay / timing / diagnostics entry points of include/vt_tracker.h
#pragma once

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "tc_common.cuh"
#include "vt_internal.h"

namespace vt {

struct BlockW {
    const float *ln1_g, *ln1_b, *qkv_w, *qkv_b, *proj_w, *proj_b, *ln2_g, *ln2_b, *fc1_w, *fc1_b, *fc2_w, *fc2_b;
};

// One device copy of a weight file (fp32 master + bf16 hi / lo split) shared by every handle of that device: with many streams per GPU
// the 45 MB stay L2 resident once instead of once per stream.  Keyed by device, path, size and mtime; freed with the last handle.
struct WeightSet {
    int device = 0;
    float* d_weights = nullptr;
    __nv_bfloat16 *w_hi = nullptr, *w_lo = nullptr;
    __nv_bfloat16* w_f16 = nullptr;  // fp16 copy for handles in VT_GEMM_TCGEN05_FP16 mode (made on first use)
    size_t n = 0;
    int32_t hdr[7] = {0, 0, 0, 0, 0, 0, 0};
    std::mutex split_mutex;
    ~WeightSet() {
        cudaSetDevice(device);
        if (d_weights) cudaFree(d_weights);
        if (w_hi) cudaFree(w_hi);
        if (w_lo) cudaFree(w_lo);
        if (w_f16) cudaFree(w_f16);
    }
};
// Live tracker handles per device, counted across processes (handle_registry.cpp).  With one or two streams on a GPU most SMs idle
// during a frame, and the "spread" GEMM forms trade them for latency (tiles replicated so that each replica stores a share of the
// epilogue output); with more streams SM time is the budget and the plain forms are used.  Read at every frame: the graph variant
// follows the handle count.
constexpr int kMaxDevices = 64, kSpreadMaxHandles = 2, kUnchainTargets = 8;

// Environment switches of a handle, read by read_switches at create (meaning and defaults: DESIGN.md §9).
struct Switches {
    bool spread = true, att_chain = true, att_q64 = true, gemm_q64 = true, as_mlp = true, trace = false, hostprof = false;
    int unchain_n = kUnchainTargets, as_rows = 1024, as_split = 0, win_shrink = 0;
};

// The kernel forms the model shape allows on the tensor-core path (shape_forms): vt_tracker_create sizes the buffers and wires the
// plans from them, forward_forms picks the forms of every forward among them.
struct ShapeForms {
    bool fuse_ln = false;       // LayerNorm fused into the producing GEMM's epilogue (else layernorm_split kernels)
    bool chain_mlp = false;     // FC2 partial products inside the FC1 kernel + reduce_ln
    bool tc_attention = false;  // tensor-core attention (else the SIMT attention kernel)
    bool att_chain = false;     // proj folded into the attention kernel (per-head partials in Pbuf + reduce_ln)
    bool split_k = false;       // patch embed and 3x3 head conv as split-K partials + reduce_ln / head_decode
};

}  // namespace vt

using namespace vt;  // internal header of the tracker translation units only: the handle below names vt:: types throughout

struct vt_tracker {
    vt_config cfg;
    int D = 0, depth = 0, heads = 0, hidden = 0, head_ch = 0;
    int W = 0, H = 0, fmt = 0, maxT = 1;
    size_t frame_bytes = 0;
    float threshold = 0.2f;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_ovl[2] = {};  // around vt_overlay's kernel (overlay_ms)
    Switches sw;

    // weights (one device allocation, shared between the handles of a device: WeightSet)
    std::shared_ptr<WeightSet> wset;
    float* d_weights = nullptr;
    size_t n_weights = 0;
    const float *patch_w, *patch_b, *pos_z, *pos_x, *lnf_g, *lnf_b, *h1_w, *h1_b, *h2_w, *h2_b;
    std::vector<BlockW> blk;
    float *d_lut = nullptr, *d_hann = nullptr;

    // frame + state
    uint8_t* d_frame = nullptr;
    uint8_t* d_sframes[kMaxWin] = {};  // stream groups: one device frame per stream (allocated on first use, grown with its geometry)
    size_t d_sframe_bytes[kMaxWin] = {};
    uint8_t* d_frames[2] = {nullptr, nullptr};  // double buffer: d_frame points at the one most recently filled (queue slot s uses [s])
    cudaStream_t copy_stream = nullptr;          // uploads of pipelined host frames overlap the in-flight frame's kernels
    cudaEvent_t ev_up[2] = {nullptr, nullptr};
    uint8_t* d_rgb = nullptr;  // lazily allocated, vt_convert_nv12_rgb
    uint8_t *d_fmt_in = nullptr, *d_fmt_out = nullptr;  // lazily grown scratch of the format entry points (YUY2, resize)
    size_t fmt_in_cap = 0, fmt_out_cap = 0;
    int rsz_max_src_rows = 0;            // source rows needed by the neediest 16-row destination tile of that geometry
    int4* d_rsz_taps = nullptr;          // resize taps of the last geometry: [dw] column taps then [dh] row taps
    int rsz_geom[4] = {0, 0, 0, 0};      // sw, sh, dw, dh they were built for
    uint8_t* h_stage = nullptr;  // pinned staging for non-pinned callers
    size_t h_stage_bytes = 0;    // bytes of h_stage and of each d_frames[i]: the largest frame of the cfg and the slot geometries, + 256
    // what the device frame buffer t->d_frame holds: the whole host frame most recently given to update()/submit()/init() (what
    // vt_overlay_current draws on), or something else (search windows only, a convert / overlay scratch upload, nothing: the last frame
    // was tracked in place in the caller's device memory)
    bool d_frame_is_last_host_frame = false;
    TargetState* d_state = nullptr;
    int32_t* d_slots = nullptr;
    // one device block [DeviceResult x maxT][u64 stamps x ST_COUNT][int tc_err, pad] written into the pinned host block of the frame's queue slot by the frame's last kernel
    DeviceResult *d_res = nullptr, *h_res = nullptr;
    size_t res_block_bytes = 0;
    unsigned long long *d_stamps = nullptr, *h_stamps = nullptr;
    int* h_tc_err = nullptr;
    FrameCtl* d_ctl = nullptr;         // per-frame control block (frames, result block address, valid windows, HUD list)
    // probe HUD (host_state.cpp): the frame's last kernel runs a per-frame command list; the list of the NEXT submit is staged in the
    // pinned block of that submit's queue slot by tracker_set_hud()
    bool hud_mode = false;
    OverlayCmdDev* h_hud[2] = {nullptr, nullptr};
    OverlayCmdDev* d_hud[2] = {nullptr, nullptr};  // device copies of the lists (written by the stamp kernel from its parameter block)
    // (per stream of a probe group; [0] on every other handle)
    int hud_next_n[kMaxWin] = {};
    int hud_next_rmw[kMaxWin][4] = {};  // region the list reads before it writes (NV12 background dim): x0, y0, x1, y1; empty = none
    size_t hud_next_bytes[kMaxWin] = {};  // pixels the list touches (device -> host accounting)
    // probe group of group_n streams (vt_probe_group, tracker_make_group): stream i = target slot i; d_ctl is a ProbeGroupCtl; the public
    // frame entry points are refused
    int group_n = 0;
    int32_t* h_slots = nullptr;  // pinned: the active slot list of the next group step (uploaded ahead of the step's kernels)
    bool inflight_mirrored = false;
    float* d_maps = nullptr;
    OverlayCmdDev *d_cmds = nullptr, *h_cmds = nullptr;
    std::vector<int> active;          // slot indices, ascending
    std::vector<vt_bbox> rect_mirror; // host mirror of rect_last (valid after wait)
    std::vector<int> inited;
    std::vector<StreamGeom> geom;     // per slot: the geometry of its stream's frames (the cfg one unless vt_tracker_set_stream_geometry)

    // activations
    float *patches_x = nullptr, *patches_z = nullptr, *Zemb = nullptr, *X = nullptr, *QKV = nullptr, *ATT = nullptr, *HID = nullptr,
          *Yf = nullptr, *H1 = nullptr, *d_dbg = nullptr;
    int debug_capture = 0;

    // tensor-core mode (gemm_mode != VT_GEMM_FP32_SIMT): bf16 (hi, lo) copies of the weights and of every GEMM A operand
    int nsplit = 0;  // 0 = fp32 SIMT, 1 = bf16, 2 = fp16 (single pass), 3 = bf16x3
    bool f16 = false;  // nsplit == 2: the operand "hi" buffers hold fp16 values, the "lo" buffers are unused (kernels get null)
    __nv_bfloat16 *w_hi = nullptr, *w_lo = nullptr;
    __nv_bfloat16 *px_hi = nullptr, *px_lo = nullptr, *pz_hi = nullptr, *pz_lo = nullptr, *ln_hi = nullptr, *ln_lo = nullptr, *att_hi = nullptr,
                  *att_lo = nullptr, *hid_hi = nullptr, *hid_lo = nullptr, *yf_hi = nullptr, *yf_lo = nullptr;
    __nv_bfloat16 *q_hi = nullptr, *q_lo = nullptr, *k_hi = nullptr, *k_lo = nullptr, *vt_hi = nullptr, *vt_lo = nullptr;
    __nv_bfloat16 *zln_hi = nullptr, *zln_lo = nullptr;  // LN1 (block 0) of the template tokens, [B][64][D], computed at init
    float* Pbuf = nullptr;      // [planes][B][320][D] fp32 partials: chained MLP (hidden / 64), chained attention (heads), patch-embed K-slices (4)
    float *Phead = nullptr, *d_cand = nullptr;  // [9 taps][B][256][head_ch] conv partials; [B][16][8] row candidates of the decode
    unsigned* d_counters = nullptr;
    int sm_count = 148;         // SMs of the device (grid sizing of the throughput forms)
    bool counted = false;       // this handle is included in g_live_handles
    TcAttentionPlan plan_att;
    int* d_tc_err = nullptr;
    unsigned long long* d_trace = nullptr;  // VT_B200_TRACE=1: device timeline of the chain (vt_tracker_debug_trace)
    TcGemmPlan plan_patch_x, plan_patch_z, plan_head;
    struct BlockPlans {
        TcGemmPlan qkv, proj, fc1, fc2;
        TcAttentionPlan att;  // plan_att + this block's W_proj maps (chained form)
    };
    std::vector<BlockPlans> plans;

    std::map<int, cudaGraphExec_t> graphs;
    int kernels_per_frame = 0;
    uint64_t kernel_launches = 0, frames = 0, h2d_bytes = 0, d2h_bytes = 0;

    // in-flight frames: a queue of depth kQueue.  rect_last lives on the device, so frame t+1 can be enqueued before the results of
    // frame t have been read back; every slot has its own pinned result block and completion event.
    static constexpr int kQueue = 2;
    struct Slot {
        uint8_t* frame = nullptr;  // caller's host frame (null for device-resident frames)
        size_t len = 0;
        bool mirrored = false, pageable = false;
        size_t hud_bytes = 0;      // pixels this frame's HUD list touches
        std::chrono::steady_clock::time_point t_submit;
    } q[kQueue];
    int q_head = 0, q_count = 0;
    DeviceResult* h_blk[kQueue] = {nullptr, nullptr};
    cudaEvent_t q_done[kQueue] = {nullptr, nullptr};
    bool in_flight = false;          // q_count > 0
    uint8_t* inflight_frame = nullptr;
    std::chrono::steady_clock::time_point t_submit;

    // VT_B200_HOSTPROF=1: host-side wall time of the submit / wait phases, printed at destroy (diagnostics)
    double hp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t hp_n = 0;

    TimingStats stats;
    Ring<float> r_h2d, r_pre, r_vit, r_dec, r_ovl, r_d2h, r_tot;
    float last[7] = {0, 0, 0, 0, 0, 0, 0};
};

namespace vt {

bool is_pinned(const void* p);
// The one home of the geometry decision: the handle's own (cfg) geometry, and the geometry of target slot `slot`'s frames, which every
// site that reads, uploads, checks or draws into a slot's frames goes through.  A uniform handle is one whose slots all hold the cfg one.
inline StreamGeom cfg_geom(const vt_tracker* t) { return StreamGeom{t->fmt, t->W, t->H}; }
inline const StreamGeom& slot_geom(const vt_tracker* t, int slot) { return t->geom[slot]; }
// A packed frame of geometry g at `base` as the kernels read it, beside the caller's pinned host frame `host` (or null); valid = false:
// the buffer was short (tracker_frame.cu, with surface_ref the only constructors of a FrameRef)
FrameRef packed_ref(const StreamGeom& g, const uint8_t* base, uint8_t* host, bool valid);
// VT_ERR_INVALID (with a message naming `where`) on a handle where a slot's geometry differs from cfg: single-frame entry points
vt_status check_uniform_geometry(const vt_tracker* t, const char* where);
// vt_overlay_cmd -> device form (glyph rows resolved); VT_ERR_GLYPH for an unknown character in strict mode
vt_status fill_cmd_dev(const vt_overlay_cmd& c, OverlayCmdDev& d);
void bind_slot(vt_tracker* t, int slot);
ShapeForms shape_forms(const vt_tracker* t);
// rows of the frame touched by a rect / crosshair (reference clamping), span bookkeeping and the device -> host row copies
bool rect_rows(int fmt, long long H, int y, int h, int th, long long& r0, long long& r1);
bool cross_rows(long long H, int cy, int size, long long& r0, long long& r1);
void merge_spans(std::vector<std::pair<int, int>>& spans);
vt_status download_rows(vt_tracker* t, uint8_t* frame, size_t len, const std::vector<std::pair<int, int>>& spans, bool* staged);
void unstage_rows(vt_tracker* t, uint8_t* frame, size_t len, const std::vector<std::pair<int, int>>& spans);

#define VT_LAUNCH(call)                                                                   \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            ::vt::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return VT_ERR_CUDA;                                                           \
        }                                                                                 \
        ++launches;                                                                       \
    } while (0)

}  // namespace vt
