// tracker_frame.cu — the per-frame path of vt_tracker: per-handle CUDA stream, CUDA-graph replay of the per-frame
// kernel chain, and the VitTrack::init / ::update entry points of include/vt_tracker.h.
//
// Per frame (update/submit):   H2D frame (pinned, cudaMemcpyAsync on the handle's stream)
//   -> K2 crop+convert+resize+normalise (search window of every active target, rect_last read on device)
//   -> template-token gather -> patch-embed GEMM -> depth x [LN+QKV, attention, proj+res, LN+FC1+GELU, FC2+res]
//   -> final LN -> 3x3 head conv (im2col GEMM) -> K8 decode (updates rect_last on device)
//   -> optional K9 box overlay -> results published into the pinned host block by the last kernel (+ touched rows for pageable frames).
// rect_last never leaves the device between frames, so consecutive frames can be enqueued without a
// host round trip.
#include "tracker_state.h"

extern "C" int vt_glyph_rows(int ch, uint8_t rows[7]);  // host_state.cpp

namespace vt {

// template tokens (fixed since init) -> rows 0..63 of every target's sequence: residual stream X and, on the fused-LN
// tensor-core path, their block-0 LN1 as the bf16 split A operand of the first QKV GEMM.
// Independent of the crop kernel ahead of it: launched as its programmatic dependent, it does its copies WHILE the crop runs and only
// then waits for it, so that the patch GEMM behind (whose dependency wait covers this kernel only) still starts after the crop.
__global__ void gather_template_kernel(float* __restrict__ X, const float* __restrict__ Zemb, const int32_t* __restrict__ slots, int D,
                                       uint32_t* __restrict__ ln_hi, uint32_t* __restrict__ ln_lo, const uint32_t* __restrict__ zln_hi,
                                       const uint32_t* __restrict__ zln_lo, unsigned long long* stamp) {
    tc::pdl_launch_dependents();
    const int bi = blockIdx.y;
    const int n = kNTz * D;
    const size_t so = (size_t)slots[bi] * n, xo = (size_t)bi * kNTok * D;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        X[xo + i] = Zemb[so + i];
        if (ln_hi && i < n / 2) {
            ln_hi[xo / 2 + i] = zln_hi[so / 2 + i];
            if (ln_lo) ln_lo[xo / 2 + i] = zln_lo[so / 2 + i];
        }
    }
    tc::pdl_wait();  // the crop kernel has completed: end of the preprocess stage
    if (stamp && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) *stamp = device_time_ns();
}

static GemmArgs gemm_args(const float* A, int64_t lda, const float* W, const float* bias, float* C, int64_t ldc, int M, int N, int K) {
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.A = A, g.lda = lda, g.W = W, g.bias = bias, g.C = C, g.ldc = ldc, g.M = M, g.N = N, g.K = K;
    g.a_rows_in = g.c_rows_in = 1 << 30;
    return g;
}

// The kernel forms of one forward, a function of the handle, n and spread (latency mode: few live handles on the GPU, run_forward):
// the graph key (n, spread) determines them.
constexpr int kAttSimt = -1;  // ForwardForms::att: launch_attention (else a VT_ATT_* form of tc_attention_launch)
struct ForwardForms {
    int patch_slices = 0;      // patch-embed K-slices summed by reduce_ln: 0 (unsplit), 4, or 2 (merged, from kUnchainTargets targets)
    int head_planes = 0;       // head-conv partial planes summed by head_decode: 9, 3 (merged), or 0 (unsplit: H1 + decode_kernel)
    bool ln_split = false;     // LayerNorm as separate layernorm_split kernels
    bool qkv_as = false;       // QKV in the A-stationary form
    int att = kAttSimt;
    bool proj_in_att = false;  // proj folded into the attention kernel + reduce_ln, instead of the proj GEMM
    bool mlp_chain = false;    // FC2 partial products inside the FC1 kernel + reduce_ln (else FC1 stores the hidden tile, FC2 GEMM)
    bool mlp_as = false;       // FC1 (with the chained product: gemm_as_mlp_kernel) in the A-stationary form
    bool gemm_q64 = false;     // QKV and the chained FC1 on 64-row tiles (tc_gemm_launch q64)
    bool spread = false;       // latency-mode replicas of the one-tile GEMMs (tc_gemm_launch picks them from the plan)
    bool pdl = true;           // programmatic dependent launch along the chain (off under debug_capture)
};

// FC1 without the chained product: it stores the hidden tile for the FC2 GEMM
static TcGemmPlan unchained_fc1(TcGemmPlan p) {
    p.args.chain_n = 0, p.args.o_mode = 1;
    return p;
}

static ForwardForms forward_forms(const vt_tracker* t, int n, bool spread) {
    ForwardForms f;
    f.pdl = !t->debug_capture;
    if (!t->nsplit) return f;
    const ShapeForms sf = shape_forms(t);
    const vt_tracker::BlockPlans& p = t->plans[0];  // every block's plans have the same shape
    const int M = n * kNTok, att_w = t->heads * (t->D / kAttChainW);
    f.spread = spread;
    // Many targets: the split-K forms of patch embed (4 K-slices) and head conv (one 3x3 tap per slice) are shaped for one target's
    // three row tiles; from 8 targets on they are 384 / 576 short CTAs (2.6 / 3.9 waves), so the slices are merged — 2 K-slices, 3 taps
    // per slice: a third of the partial planes, CTAs that run three times as many MMAs per prologue.
    f.patch_slices = sf.split_k ? (n >= kUnchainTargets ? 2 : 4) : 0;
    f.head_planes = sf.split_k ? (n >= kUnchainTargets ? 3 : 9) : 0;
    f.ln_split = !sf.fuse_ln;
    // many rows (cfg4, stream groups): the A-stationary form — activation tile resident, epilogue of chunk i under the main loop of i + 1
    const bool as_form = t->sw.as_rows > 0 && M >= t->sw.as_rows;
    f.qkv_as = as_form && tc_gemm_as_supported(p.qkv);
    // Latency mode: the proj GEMM is folded into the attention kernel (per-head partial products, D / kAttChainW replicas per tile) and
    // reduce_ln adds the heads + bias + residual and applies LN2 — one kernel and one dependency edge less per block.  64-row query
    // tiles (5 per sequence) when that grid still fits one wave: each CTA computes half the exponentials.
    if (sf.tc_attention) {
        const bool chain = spread && sf.att_chain && t->sw.att_chain;
        f.att = chain && t->sw.att_q64 && n * 5 * att_w <= kSpreadCtas ? VT_ATT_CHAIN_Q64
                : chain && n * 3 * att_w <= kSpreadCtas            ? VT_ATT_CHAIN
                : spread                                            ? VT_ATT_DUP
                                                                    : VT_ATT_PLAIN;
    }
    f.proj_in_att = f.att == VT_ATT_CHAIN || f.att == VT_ATT_CHAIN_Q64;
    // Chained form (FC2 partial products inside the FC1 kernel, summed by reduce_ln): shortest critical path for a few targets.
    // From kUnchainTargets targets on the 12 fp32 partial planes per row tile cost more than the hidden round trip
    // (cfg4, 16 targets: ViT stage 905 -> 819 us unchained), so FC1 writes the hidden tile and FC2 runs as its own GEMM.
    // ... except in the A-stationary form, where a CTA accumulates the chained product over all of its hidden chunks (3 planes
    // per row tile at 5120 rows, and no hidden round trip at all)
    const bool as_mlp = as_form && sf.chain_mlp && t->sw.as_mlp && tc_gemm_as_mlp_supported(p.fc1, t->nsplit);
    f.mlp_chain = as_mlp || (sf.chain_mlp && n < t->sw.unchain_n);
    f.mlp_as = f.mlp_chain ? as_mlp : as_form && tc_gemm_as_supported(unchained_fc1(p.fc1));
    // Latency mode: QKV and the chained FC1 on 64-row tiles (M = 64 UMMAs: five tiles instead of 128 + 128 + 64, half the epilogue per
    // CTA) when both grids of two replicas per tile still fit one wave — one target
    const int tiles64 = (M + 63) / 64;
    f.gemm_q64 = spread && t->sw.gemm_q64 && !f.qkv_as && f.mlp_chain && !f.mlp_as && tc_gemm_q64_supported(p.qkv, t->nsplit) &&
                 tc_gemm_q64_supported(p.fc1, t->nsplit) && (p.qkv.args.N / 64) * tiles64 * 2 <= kSpreadCtas &&
                 (p.fc1.args.N / 64) * tiles64 * 2 <= kSpreadCtas;
    return f;
}

// Enqueues crop -> ViT -> decode (-> box overlay) for the n active targets on t->stream.
static vt_status enqueue_forward(vt_tracker* t, int n, int& launches, const ForwardForms& f) {
    const int D = t->D, Hd = t->hidden, C = t->head_ch;
    cudaStream_t s = t->stream;
    const FrameDesc fd{FrameRef{}, t->d_ctl, t->cfg.pad_plus1};  // the frames from d_ctl
    auto LO = [&](__nv_bfloat16* p) { return t->f16 ? nullptr : p; };  // fp16 mode: "hi only" (see vt_internal.h: operand_bits)
    VT_LAUNCH(launch_crop_resize_norm(fd, t->d_state, t->d_slots, n, 4, kSearch, t->d_lut, t->patches_x, (size_t)kNTx * kPatchK, t->px_hi,
                                      LO(t->px_lo), s, t->d_stamps + ST_PRE));
    {
        dim3 grid((kNTz * D + 255) / 256, n);
        const bool ln = t->nsplit && !f.ln_split;  // LN1 of block 0 for the template rows (the search rows get it after the patch embed)
        VT_LAUNCH(launch_ex(gather_template_kernel, grid, dim3(256), 0, s, f.pdl, 1, t->X, (const float*)t->Zemb, (const int32_t*)t->d_slots, D,
                            ln ? (uint32_t*)t->ln_hi : nullptr, (uint32_t*)LO(t->ln_lo), (const uint32_t*)t->zln_hi, (const uint32_t*)t->zln_lo,
                            t->d_stamps + ST_VIT));
    }
    const int M = n * kNTok;
    if (t->nsplit == 0) {
        // ---------------- fp32 CUDA-core path ----------------
        {
            GemmArgs g = gemm_args(t->patches_x, kPatchK, t->patch_w, t->patch_b, t->X, D, n * kNTx, D, kPatchK);
            g.pos = t->pos_x;
            g.c_rows_in = kNTx, g.c_rows_stride = kNTok, g.c_row_off = kNTz;
            VT_LAUNCH(launch_gemm_simt(g, s));
        }
        if (t->debug_capture) VT_CUDA(cudaMemcpyAsync(t->d_dbg, t->X, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, s));
        for (int l = 0; l < t->depth; ++l) {
            const BlockW& b = t->blk[l];
            {
                GemmArgs g = gemm_args(t->X, D, b.qkv_w, b.qkv_b, t->QKV, 3 * D, M, 3 * D, D);
                g.ln_g = b.ln1_g, g.ln_b = b.ln1_b;
                VT_LAUNCH(launch_gemm_simt(g, s));
            }
            VT_LAUNCH(launch_attention(t->QKV, t->ATT, nullptr, nullptr, n, D, t->heads, s));
            {
                GemmArgs g = gemm_args(t->ATT, D, b.proj_w, b.proj_b, t->X, D, M, D, D);
                g.residual = 1;
                VT_LAUNCH(launch_gemm_simt(g, s));
            }
            {
                GemmArgs g = gemm_args(t->X, D, b.fc1_w, b.fc1_b, t->HID, Hd, M, Hd, D);
                g.ln_g = b.ln2_g, g.ln_b = b.ln2_b, g.gelu = 1;
                VT_LAUNCH(launch_gemm_simt(g, s));
            }
            {
                GemmArgs g = gemm_args(t->HID, Hd, b.fc2_w, b.fc2_b, t->X, D, M, D, Hd);
                g.residual = 1;
                VT_LAUNCH(launch_gemm_simt(g, s));
            }
            if (t->debug_capture)
                VT_CUDA(cudaMemcpyAsync(t->d_dbg + (size_t)(l + 1) * t->maxT * kNTok * D, t->X, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, s));
        }
        VT_LAUNCH(launch_layernorm(t->X, D, t->lnf_g, t->lnf_b, t->Yf, D, n * kNTx, D, kNTx, kNTok, kNTz, s));
        {
            GemmArgs g = gemm_args(t->Yf, D, t->h1_w, t->h1_b, t->H1, C, n * kNTx, C, 9 * D);
            g.relu = 1, g.im2col_feat = D;
            g.a_rows_in = kNTx, g.a_rows_stride = kNTx, g.a_row_off = 0;
            VT_LAUNCH(launch_gemm_simt(g, s));
        }
    } else {
        // ---------------- tensor-core path: tcgen05 GEMMs fed by TMA, bf16 (x3 split) operands, fp32 TMEM accumulators ----------------
        const int ns = t->nsplit;
        TcGemmPlan pp = t->plan_patch_x;
        if (f.patch_slices) pp.args.kb_per_split = kPatchK / 64 / f.patch_slices;
        VT_LAUNCH(tc_gemm_launch(pp, n * kNTx, ns, s, f.pdl));  // unsplit: + LN1 of block 0 for the search rows (fused)
        if (f.patch_slices) {  // X[64.., :] = pos_x + patch_b + sum of the K-slices; LN1 of block 0
            ReduceLnArgs r{};
            r.P = t->Pbuf, r.np = f.patch_slices, r.p_stride = (int64_t)t->maxT * kNTx * D, r.bias = t->patch_b, r.add = t->pos_x, r.add_period = kNTx;
            r.X = t->X, r.M = n * kNTx, r.D = D, r.period = kNTx, r.x_rows = kNTok, r.x_row_off = kNTz;
            r.ln_g = t->blk[0].ln1_g, r.ln_b = t->blk[0].ln1_b, r.ln_hi = t->ln_hi, r.ln_lo = LO(t->ln_lo), r.ln_rows = kNTok, r.ln_row_off = kNTz;
            VT_LAUNCH(launch_reduce_ln(r, s, f.pdl, f.spread));
        }
        if (t->debug_capture) VT_CUDA(cudaMemcpyAsync(t->d_dbg, t->X, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, s));
        for (int l = 0; l < t->depth; ++l) {
            const BlockW& b = t->blk[l];
            const vt_tracker::BlockPlans& p = t->plans[l];
            if (f.ln_split) VT_LAUNCH(launch_layernorm_split(t->X, D, b.ln1_g, b.ln1_b, t->ln_hi, LO(t->ln_lo), M, D, 1 << 30, 0, 0, s, f.pdl));
            if (f.qkv_as)
                VT_LAUNCH(tc_gemm_as_launch(p.qkv, M, ns, s, f.pdl, t->sm_count, t->sw.as_split));
            else
                VT_LAUNCH(tc_gemm_launch(p.qkv, M, ns, s, f.pdl, f.spread, f.gemm_q64));
            if (f.att == kAttSimt)
                VT_LAUNCH(launch_attention(t->QKV, nullptr, t->att_hi, LO(t->att_lo), n, D, t->heads, s));
            else
                VT_LAUNCH(tc_attention_launch(f.proj_in_att ? p.att : t->plan_att, n, t->heads, ns, t->d_tc_err, s, f.pdl, t->d_trace, f.att));
            if (f.proj_in_att) {
                ReduceLnArgs r{};
                r.P = t->Pbuf, r.np = t->heads, r.p_stride = (int64_t)t->maxT * kNTok * D, r.bias = b.proj_b, r.add = t->X, r.add_period = 0;
                r.X = t->X, r.M = M, r.D = D, r.period = kNTok, r.x_rows = kNTok, r.x_row_off = 0;
                r.ln_g = b.ln2_g, r.ln_b = b.ln2_b, r.ln_hi = t->ln_hi, r.ln_lo = LO(t->ln_lo), r.ln_rows = kNTok, r.ln_row_off = 0;
                VT_LAUNCH(launch_reduce_ln(r, s, f.pdl, f.spread));
            } else {  // fused: + LN2
                VT_LAUNCH(tc_gemm_launch(p.proj, M, ns, s, f.pdl && f.att != kAttSimt, f.spread));
            }
            if (f.ln_split) VT_LAUNCH(launch_layernorm_split(t->X, D, b.ln2_g, b.ln2_b, t->ln_hi, LO(t->ln_lo), M, D, 1 << 30, 0, 0, s, f.pdl));
            int planes = Hd / 64;
            const TcGemmPlan fc1 = f.mlp_chain ? p.fc1 : unchained_fc1(p.fc1);
            if (f.mlp_as && f.mlp_chain)
                VT_LAUNCH(tc_gemm_as_mlp_launch(fc1, M, s, f.pdl, t->sm_count, t->sw.as_split, &planes));
            else if (f.mlp_as)
                VT_LAUNCH(tc_gemm_as_launch(fc1, M, ns, s, f.pdl, t->sm_count, t->sw.as_split));
            else
                VT_LAUNCH(tc_gemm_launch(fc1, M, ns, s, f.pdl, f.spread && f.mlp_chain, f.gemm_q64));
            if (f.mlp_chain) {  // X += fc2_b + sum of the partials; LN1 of the next block / the final LN of the search rows
                const bool last = l + 1 == t->depth;
                ReduceLnArgs r{};
                r.P = t->Pbuf, r.np = planes, r.p_stride = (int64_t)t->maxT * kNTok * D, r.bias = b.fc2_b, r.add = t->X, r.add_period = 0;
                r.X = t->X, r.M = M, r.D = D, r.period = kNTok, r.x_rows = kNTok, r.x_row_off = 0;
                r.ln_g = last ? t->lnf_g : t->blk[l + 1].ln1_g, r.ln_b = last ? t->lnf_b : t->blk[l + 1].ln1_b;
                r.ln_hi = last ? t->yf_hi : t->ln_hi, r.ln_lo = LO(last ? t->yf_lo : t->ln_lo);
                r.ln_rows = last ? kNTx : kNTok, r.ln_row_off = last ? -kNTz : 0;
                VT_LAUNCH(launch_reduce_ln(r, s, f.pdl, f.spread));
            } else {
                VT_LAUNCH(tc_gemm_launch(p.fc2, M, ns, s, f.pdl));  // fused: + LN1 of the next block / the final LN of the search rows
            }
            if (t->debug_capture)
                VT_CUDA(cudaMemcpyAsync(t->d_dbg + (size_t)(l + 1) * t->maxT * kNTok * D, t->X, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, s));
        }
        if (f.ln_split) VT_LAUNCH(launch_layernorm_split(t->X, D, t->lnf_g, t->lnf_b, t->yf_hi, LO(t->yf_lo), n * kNTx, D, kNTx, kNTok, kNTz, s, f.pdl));
        TcGemmPlan ph = t->plan_head;
        if (f.head_planes) ph.args.kb_per_split = 9 * (D / 64) / f.head_planes;  // 3x3 taps per slice
        VT_LAUNCH(tc_gemm_launch(ph, n * kNTx, ns, s, f.pdl));
    }
    if (f.head_planes)
        VT_LAUNCH(launch_head_decode(t->Phead, f.head_planes, (int64_t)t->maxT * kNTx * C, C, t->h1_b, t->h2_w, t->h2_b, t->d_hann, t->d_state, t->d_slots,
                                     n, t->threshold, t->d_res, t->d_maps, t->d_cand, t->d_counters, t->d_stamps, s, f.pdl, t->cfg.decode_window,
                                     t->d_tc_err, f.spread));
    else
        VT_LAUNCH(launch_decode(t->H1, C, t->h2_w, t->h2_b, t->d_hann, t->d_state, t->d_slots, n, t->threshold, t->d_res, t->d_maps, t->d_stamps, s,
                                t->cfg.decode_window));
    if (t->group_n)  // probe group: every stream's HUD (one CTA pair per stream of the group, not per target of the forward), mirror, publish
        VT_LAUNCH(launch_group_overlay(t->group_n, t->d_res, t->cfg.overlay_gate, reinterpret_cast<const ProbeGroupCtl*>(t->d_ctl),
                                       t->d_stamps + ST_OVL_END, s, f.pdl, t->d_res, t->res_block_bytes));
    else if (t->cfg.box_overlay || t->hud_mode)  // box overlay and / or the frame's HUD list, pinned-frame mirror, ... and publishes the result block
        VT_LAUNCH(launch_box_overlay(t->d_res, t->d_slots, n, t->cfg.overlay_gate, t->d_ctl, t->d_stamps + ST_OVL_END, s, f.pdl, t->d_res,
                                     t->res_block_bytes, t->cfg.box_overlay | (t->hud_mode ? 1 << 16 : 0)));
    else  // results, stage stamps and the error flag -> the pinned host block of this frame's queue slot
        VT_LAUNCH(launch_publish(t->d_res, t->d_ctl, t->res_block_bytes, s, f.pdl));
    return VT_OK;
}

static vt_status run_forward(vt_tracker* t) {
    const int n = (int)t->active.size();
    if (n == 0) return VT_OK;
    int launches = 0;
    const int dev = t->cfg.device;
    const bool spread = t->sw.spread && dev >= 0 && dev < kMaxDevices && registry_total(dev) <= kSpreadMaxHandles;
    const ForwardForms f = forward_forms(t, n, spread);
    if (!t->cfg.use_cuda_graph || t->debug_capture) {
        vt_status st = enqueue_forward(t, n, launches, f);
        t->kernel_launches += launches;
        t->kernels_per_frame = launches;
        return st;
    }
    const int key = n * 2 + (spread ? 1 : 0);
    auto it = t->graphs.find(key);
    if (it == t->graphs.end()) {
        cudaGraph_t graph = nullptr;
        VT_CUDA(cudaStreamBeginCapture(t->stream, cudaStreamCaptureModeThreadLocal));
        vt_status st = enqueue_forward(t, n, launches, f);
        cudaError_t e = cudaStreamEndCapture(t->stream, &graph);
        if (st != VT_OK) {
            if (graph) cudaGraphDestroy(graph);
            return st;
        }
        if (e != cudaSuccess) {
            set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
            return VT_ERR_CUDA;
        }
        cudaGraphExec_t exec = nullptr;
        VT_CUDA(cudaGraphInstantiate(&exec, graph, 0));
        cudaGraphDestroy(graph);
        it = t->graphs.emplace(key, exec).first;
        t->kernels_per_frame = launches;
    }
    VT_CUDA(cudaGraphLaunch(it->second, t->stream));
    t->kernel_launches += t->kernels_per_frame;
    return VT_OK;
}

static vt_status sync_slots(vt_tracker* t) {
    if (!t->active.empty())
        VT_CUDA(cudaMemcpyAsync(t->d_slots, t->active.data(), sizeof(int32_t) * t->active.size(), cudaMemcpyHostToDevice, t->stream));
    VT_CUDA(cudaStreamSynchronize(t->stream));  // t->active is pageable: make the copy complete before it can change
    return VT_OK;
}

// Search window of a target in frame coordinates (App. A.1 with factor 4), grown by `margin_div` (0 = exact; d: by c / d on every side,
// at least 16 px — used when the host's copy of rect_last lags by one frame), clipped to the frame and grown to even coordinates
// (NV12 chroma pairs).  Returns false when the window misses the frame.
static bool search_window(const StreamGeom& g, const vt_bbox& r, int margin_div, int& x0, int& y0, int& x1, int& y1) {
    if (r.width <= 0 || r.height <= 0) return false;
    const int c = (int)ceil(sqrt((double)(int)((long long)r.width * r.height)) * 4.0);
    const int m = margin_div > 0 ? std::max(16, c / margin_div) : 0;
    const long long wx = (long long)r.x + (r.width - c) / 2 - m, wy = (long long)r.y + (r.height - c) / 2 - m, e = (long long)c + 2 * m;
    x0 = (int)std::max(wx, 0LL) & ~1, y0 = (int)std::max(wy, 0LL) & ~1;
    x1 = (int)std::min((std::min(wx + e, (long long)g.W) + 1) & ~1LL, (long long)g.W);
    y1 = (int)std::min((std::min(wy + e, (long long)g.H) + 1) & ~1LL, (long long)g.H);
    return x1 > x0 && y1 > y0;
}

// What travels host -> device for one frame (PCIe is the end-to-end roofline, SURVEY.md §8(d)): the whole frame, or — cfg.upload_window,
// pinned frame — only the search window of every active target (+ the region a HUD list reads before writing).  The fused crop kernel
// reads nothing else; should the real window leave the uploaded one (pipelined frames: rect_mirror lags by one frame and the window
// is a prediction), the crop kernel fetches the missing pixels straight from the pinned host frame, so the result never depends on
// the prediction.
struct UploadPlan {
    bool whole = true;
    int n_win = 0;
    int win[kMaxWin][4];
    bool has_rmw = false;
    int rmw[4] = {0, 0, 0, 0};
    size_t bytes = 0;
};
// Window uploads need windows whose pixels carry their own chroma: even x0 (NV12 chroma pairs, YUY2 words) and, for NV12, even y0.
// YUY2 takes any W and H: a window that ends on an odd last column copies that column's whole word, and chroma is per row.  RGBA / BGRA
// take any W and H: a window is whole 4-byte pixels, each with its own colour.  I420 takes any W and H: the chroma planes are copied
// over the blocks [x0 / 2, ceil(x1 / 2)) x [y0 / 2, ceil(y1 / 2)), which hold the chroma of every pixel of the window.
static bool windows_allowed(const StreamGeom& g) {
    return g.fmt == VT_FMT_YUY2 || format_is_rgb32(g.fmt) || g.fmt == VT_FMT_I420 || (!(g.W % 2) && !((g.H % 2) && g.fmt == VT_FMT_NV12));
}
// I420: the chroma blocks under the window w, [cx, cx + cw) x [cy, cy + ch), in each of the U and V planes
static void i420_chroma_window(const int* w, size_t& cx, size_t& cy, size_t& cw, size_t& ch) {
    cx = (size_t)(w[0] / 2), cy = (size_t)(w[1] / 2), cw = (size_t)((w[2] + 1) / 2) - cx, ch = (size_t)((w[3] + 1) / 2) - cy;
}
// bytes of plane 0 that hold the pixels [x0, x1) x [y0, y1) of a packed frame (YUY2: whole words)
static size_t plane0_bytes(const StreamGeom& g, int x0, int y0, int x1, int y1) {
    size_t o0, o1;
    fmt_col_span(g.fmt, x0, x1, &o0, &o1);
    return (o1 - o0) * (size_t)(y1 - y0);
}
// bytes of the window w = (x0, y0, x1, y1): plane 0 and, for NV12, the chroma rows under it (I420: the chroma blocks, in U and in V)
static size_t window_bytes(const StreamGeom& g, const int* w) {
    if (g.fmt == VT_FMT_I420) {
        size_t cx, cy, cw, ch;
        i420_chroma_window(w, cx, cy, cw, ch);
        return plane0_bytes(g, w[0], w[1], w[2], w[3]) + 2 * cw * ch;
    }
    return plane0_bytes(g, w[0], w[1], w[2], w[3]) + (g.fmt == VT_FMT_NV12 ? (size_t)(w[2] - w[0]) * ((w[3] - w[1]) / 2) : 0);
}
// one 2D copy of the window w of a packed frame out of plane 0 (+ one of the NV12 chroma rows under it when `chroma`; I420: one 3D copy
// of depth 2, its slices the U and the V plane, so that a window costs two copy calls as for NV12)
static vt_status copy_window(const StreamGeom& g, uint8_t* dst, const uint8_t* src, const int* w, bool chroma, cudaMemcpyKind kind,
                             cudaStream_t stream) {
    const size_t row = fmt_row_bytes(g.fmt, g.W), rows = (size_t)(w[3] - w[1]);
    size_t o0, o1;
    fmt_col_span(g.fmt, w[0], w[2], &o0, &o1);
    const size_t o = (size_t)w[1] * row + o0;
    VT_CUDA(cudaMemcpy2DAsync(dst + o, row, src + o, row, o1 - o0, rows, kind, stream));
    if (chroma && g.fmt == VT_FMT_NV12) {
        const size_t W = (size_t)g.W, uvo = W * g.H + (size_t)(w[1] / 2) * W + w[0];
        VT_CUDA(cudaMemcpy2DAsync(dst + uvo, W, src + uvo, W, (size_t)(w[2] - w[0]), rows / 2, kind, stream));
    } else if (chroma && g.fmt == VT_FMT_I420) {
        size_t cx, cy, cw, ch;
        i420_chroma_window(w, cx, cy, cw, ch);
        const size_t cp = i420_chroma_pitch(g.W), crows = (size_t)((g.H + 1) / 2), uo = i420_u_offset(g.W, g.H);
        cudaMemcpy3DParms p = {};
        p.srcPtr = make_cudaPitchedPtr(const_cast<uint8_t*>(src + uo), cp, cp, crows);
        p.dstPtr = make_cudaPitchedPtr(dst + uo, cp, cp, crows);
        p.srcPos = p.dstPos = make_cudaPos(cx, cy, 0);
        p.extent = make_cudaExtent(cw, ch, 2);
        p.kind = kind;
        VT_CUDA(cudaMemcpy3DAsync(&p, stream));
    }
    return VT_OK;
}

static void plan_upload(vt_tracker* t, size_t len, bool pinned_host, bool lagging, const int* rmw, UploadPlan& p) {
    p = UploadPlan();
    const StreamGeom g = cfg_geom(t);  // (single-frame calls: a handle of uniform geometry)
    const bool valid = len >= fmt_valid_bytes(g.fmt, g.W, g.H);
    if (!t->cfg.upload_window || !pinned_host || !valid || len < t->frame_bytes || (int)t->active.size() > kMaxWin || !windows_allowed(g) ||
        (t->active.empty() && !t->hud_mode))
        return;
    size_t bytes = 0;
    int k = 0;
    for (int s : t->active) {
        int* w = p.win[k++];
        if (!search_window(g, t->rect_mirror[s], lagging ? 8 : 0, w[0], w[1], w[2], w[3])) {
            w[0] = w[1] = w[2] = w[3] = 0;  // the window misses the frame: the crop kernel flags it; nothing to read
            continue;
        }
        const int sh = t->sw.win_shrink;  // diagnostics: windows too small on purpose exercise the crop kernel's pinned-frame fall-back
        if (sh > 0 && w[2] - w[0] > 4 * sh && w[3] - w[1] > 4 * sh) w[0] += sh, w[1] += sh, w[2] -= sh, w[3] -= sh;
        bytes += window_bytes(g, w);
    }
    if (rmw && rmw[2] > rmw[0] && rmw[3] > rmw[1] && format_is_luma(t->fmt)) {
        p.has_rmw = true;
        p.rmw[0] = std::max(rmw[0], 0), p.rmw[1] = std::max(rmw[1], 0), p.rmw[2] = std::min(rmw[2], t->W), p.rmw[3] = std::min(rmw[3], t->H);
        if (p.rmw[2] > p.rmw[0] && p.rmw[3] > p.rmw[1]) bytes += plane0_bytes(g, p.rmw[0], p.rmw[1], p.rmw[2], p.rmw[3]);
        else p.has_rmw = false;
    }
    if (bytes * 2 > t->frame_bytes) return;  // not worth the extra copies
    p.whole = false, p.n_win = k, p.bytes = bytes;
}

// g: the geometry of the frame (the cfg one; vt_tracker_init: the slot's)
static vt_status do_upload(vt_tracker* t, const StreamGeom& g, const uint8_t* frame, size_t len, const UploadPlan& p, bool device_src,
                           cudaStream_t stream) {
    if (!stream) stream = t->stream;
    const size_t frame_bytes = g.bytes();
    size_t n = std::min(len, frame_bytes);
    if (len < fmt_valid_bytes(g.fmt, g.W, g.H) && g.fmt == VT_FMT_NV12) n = 0;  // src/nv12_convert.rs:48-50 -> black image
    if (n == 0) return VT_OK;
    const cudaMemcpyKind kind = device_src ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (!p.whole) {
        for (int i = 0; i < p.n_win; ++i) {
            const int* w = p.win[i];
            if (w[2] == w[0] || w[3] == w[1]) continue;
            vt_status st = copy_window(g, t->d_frame, frame, w, true, kind, stream);
            if (st != VT_OK) return st;
        }
        if (p.has_rmw) {  // plane 0 only (the luma background dim reads and writes Y)
            vt_status st = copy_window(g, t->d_frame, frame, p.rmw, false, kind, stream);
            if (st != VT_OK) return st;
        }
        if (!device_src) t->h2d_bytes += p.bytes;
        t->d_frame_is_last_host_frame = false;  // only windows of the frame are on the device
        return VT_OK;
    }
    const bool pinned = device_src || is_pinned(frame);
    t->d_frame_is_last_host_frame = !device_src && n >= frame_bytes;
    if (!device_src) t->h2d_bytes += n;
    if (pinned) {
        VT_CUDA(cudaMemcpyAsync(t->d_frame, frame, n, kind, stream));
    } else {
        memcpy(t->h_stage, frame, n);
        VT_CUDA(cudaMemcpyAsync(t->d_frame, t->h_stage, n, cudaMemcpyHostToDevice, stream));
    }
    return VT_OK;
}

static void fill_results(vt_tracker* t, vt_result* results) {
    for (int s = 0; s < t->maxT; ++s) {
        vt_result r;
        memset(&r, 0, sizeof(r));
        if (!t->inited[s]) {
            r.status = VT_ERR_NOT_INIT;
        } else {
            const DeviceResult& d = t->h_res[s];
            r.success = d.success, r.score = d.score, r.status = d.status;
            r.bbox = vt_bbox{d.bbox[0], d.bbox[1], d.bbox[2], d.bbox[3]};
            if (d.status == VT_OK && d.success) t->rect_mirror[s] = r.bbox;
        }
        if (results) results[s] = r;
    }
}

// Rows touched by a rect / crosshair, following the reference's clamping exactly
// (src/nv12_convert.rs:181-212,224-241; src/drawing_rgb.rs:55-73).  Returns false if nothing is drawn.
bool rect_rows(int fmt, long long H, int y, int h, int th, long long& r0, long long& r1) {
    if (H <= 0) return false;
    if (format_is_luma(fmt)) {
        const long long y1 = std::max(y, 0);
        const long long sum = (long long)(int32_t)((uint32_t)y + (uint32_t)h);
        const long long y2 = sum < 0 ? H - 1 : std::min(sum, H - 1);  // negative i32 -> huge usize -> clamped
        const long long t = std::max(th, 1);
        r0 = std::min(y1, std::max(0LL, y2 - t + 1));
        r1 = std::max(y2, std::min(y1 + t - 1, H - 1));
    } else {  // rows y+t, y+rh-1-t (t < thickness) and y..y+rh-1, each bounds-checked per pixel
        const long long t = std::max(th, 1);
        r0 = std::min<long long>(y, (long long)y + h - t), r1 = std::max<long long>((long long)y + h - 1, (long long)y + t - 1);
        if (r1 < 0 || r0 > H - 1) return false;
    }
    r0 = std::max(0LL, std::min(r0, H - 1)), r1 = std::max(0LL, std::min(r1, H - 1));
    return r1 >= r0;
}
bool cross_rows(long long H, int cy, int size, long long& r0, long long& r1) {
    const long long c = std::max(cy, 0), s = std::max(size, 0);
    r0 = std::max(0LL, std::min(c - s, H - 1)), r1 = std::max(0LL, std::min(c + s, H - 1));
    return r1 >= r0;
}

// rows of the frame touched by the box overlay of the current results, merged
static void box_rows(const vt_tracker* t, std::vector<std::pair<int, int>>& spans) {
    for (int s : t->active) {
        const DeviceResult& d = t->h_res[s];
        if (d.status != VT_OK || !d.success || !(d.score > t->cfg.overlay_gate)) continue;
        long long r0, r1;
        if (rect_rows(t->fmt, t->H, d.bbox[1], d.bbox[3], 3, r0, r1)) spans.emplace_back((int)r0, (int)r1);
        if (cross_rows(t->H, d.bbox[1] + d.bbox[3] / 2, 15, r0, r1)) spans.emplace_back((int)r0, (int)r1);
    }
}

void merge_spans(std::vector<std::pair<int, int>>& spans) {
    std::sort(spans.begin(), spans.end());
    std::vector<std::pair<int, int>> out;
    for (auto& sp : spans) {
        if (!out.empty() && sp.first <= out.back().second + 8) out.back().second = std::max(out.back().second, sp.second);
        else out.push_back(sp);
    }
    spans.swap(out);
}

// device -> host copy of whole rows [r0, r1] of the drawable plane (Y plane for NV12, the image for RGB24 / RGBA / BGRA)
vt_status download_rows(vt_tracker* t, uint8_t* frame, size_t len, const std::vector<std::pair<int, int>>& spans, bool* staged) {
    const size_t pitch = fmt_row_bytes(t->fmt, t->W);
    const bool pinned = is_pinned(frame);
    *staged = !pinned;
    for (auto& sp : spans) {
        const size_t off = (size_t)sp.first * pitch;
        size_t n = (size_t)(sp.second - sp.first + 1) * pitch;
        if (off >= len) continue;
        n = std::min(n, len - off);
        t->d2h_bytes += n;
        VT_CUDA(cudaMemcpyAsync((pinned ? frame : t->h_stage) + off, t->d_frame + off, n, cudaMemcpyDeviceToHost, t->stream));
    }
    return VT_OK;
}
void unstage_rows(vt_tracker* t, uint8_t* frame, size_t len, const std::vector<std::pair<int, int>>& spans) {
    const size_t pitch = fmt_row_bytes(t->fmt, t->W);
    for (auto& sp : spans) {
        const size_t off = (size_t)sp.first * pitch;
        size_t n = (size_t)(sp.second - sp.first + 1) * pitch;
        if (off >= len) continue;
        memcpy(frame + off, t->h_stage + off, std::min(n, len - off));
    }
}

static void collect_timing(vt_tracker* t) {
    // stage boundaries stamped on the device (ns): submit, crop start, ViT start, decode start, decode end, overlay end
    const unsigned long long* st = t->h_stamps;
    auto span = [&](int a, int b) { return st[b] > st[a] && st[a] ? (float)((double)(st[b] - st[a]) * 1e-6) : 0.f; };
    const bool ovl = t->cfg.box_overlay || t->hud_mode;
    const int last_dev = ovl ? ST_OVL_END : ST_DEC_END;
    const float wall = (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t->t_submit).count();
    float ms[7];
    ms[0] = span(ST_SUBMIT, ST_PRE), ms[1] = span(ST_PRE, ST_VIT), ms[2] = span(ST_VIT, ST_DEC), ms[3] = span(ST_DEC, ST_DEC_END);
    ms[4] = ovl ? span(ST_DEC_END, ST_OVL_END) : 0.f;
    const float dev = span(ST_SUBMIT, last_dev);
    ms[5] = wall > dev ? wall - dev : 0.f;  // results (and overlay rows) back in host memory + completion latency, host clock
    ms[6] = wall;
    if (t->active.empty()) ms[1] = ms[2] = ms[3] = ms[4] = 0.f;
    memcpy(t->last, ms, sizeof(ms));
    t->r_h2d.push(ms[0]), t->r_pre.push(ms[1]), t->r_vit.push(ms[2]), t->r_dec.push(ms[3]), t->r_ovl.push(ms[4]), t->r_d2h.push(ms[5]),
        t->r_tot.push(ms[6]);
}

static inline double now_us() {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// The two constructors of a FrameRef.  A packed frame of geometry g at `base` (NV12: the chroma plane right behind the Y plane; I420:
// plane 1 is the U plane, the V plane follows it), beside the caller's pinned host frame `host` (or null); valid = false: the buffer was
// short, the crop reads a black image.
FrameRef packed_ref(const StreamGeom& g, const uint8_t* base, uint8_t* host, bool valid) {
    const bool nv12 = g.fmt == VT_FMT_NV12, i420 = g.fmt == VT_FMT_I420;
    const uint8_t* p1 = nv12 ? base + (size_t)g.W * g.H : i420 ? base + i420_u_offset(g.W, g.H) : nullptr;
    const size_t pitch1 = nv12 ? (size_t)g.W : i420 ? i420_chroma_pitch(g.W) : 0;
    return FrameRef{{base, p1}, {fmt_row_bytes(g.fmt, g.W), pitch1}, host, {g.fmt, g.W, g.H, valid ? 1 : 0}};
}
// the caller's surface s (checked by check_surface), read and drawn into in place
static FrameRef surface_ref(const StreamGeom& g, const vt_surface& s) {
    const bool nv12 = g.fmt == VT_FMT_NV12;
    return FrameRef{{s.planes[0], nv12 ? s.planes[1] : nullptr}, {s.pitch[0], nv12 ? s.pitch[1] : 0}, nullptr, {g.fmt, g.W, g.H, 1}};
}

// The caller's surface (include/vt_tracker.h: vt_surface): every plane of the format present, a pitch that holds a row, and device (or
// managed) memory of the handle's GPU, for a frame of geometry g.  `i` >= 0 names the surface of a stream group in the message.
static vt_status check_surface(const vt_tracker* t, const StreamGeom& g, const vt_surface* s, const char* where, int i) {
    if (g.fmt == VT_FMT_I420) {  // (three planes: a vt_surface has two, and the crop kernel addresses V by the packed layout)
        set_error("%s: surface %d: I420 frames are not taken as surfaces (host frames or packed device frames only: "
                  "vt_tracker_update_device / vt_tracker_submit_device)", where, i);
        return VT_ERR_INVALID;
    }
    if (!s) {
        set_error("%s: surface %d is null", where, i);
        return VT_ERR_INVALID;
    }
    const int np = g.fmt == VT_FMT_NV12 ? 2 : 1;
    for (int p = 0; p < np; ++p) {
        const size_t row = fmt_row_bytes(g.fmt, g.W);  // (NV12: the chroma rows are W bytes as well)
        if (!s->planes[p]) {
            set_error("%s: surface %d: plane %d is null", where, i, p);
            return VT_ERR_INVALID;
        }
        if (s->pitch[p] < row) {
            set_error("%s: surface %d: pitch[%d] = %zu is smaller than the plane's row (%zu bytes)", where, i, p, s->pitch[p], row);
            return VT_ERR_INVALID;
        }
        cudaPointerAttributes a;
        const cudaError_t e = cudaPointerGetAttributes(&a, s->planes[p]);
        if (e != cudaSuccess) cudaGetLastError();  // (not a sticky error: clear it)
        if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != t->cfg.device) {
            set_error("%s: surface %d: plane %d is not device memory of GPU %d", where, i, p, t->cfg.device);
            return VT_ERR_INVALID;
        }
    }
    return VT_OK;
}

// Checks shared by the surface entry points: a synchronous call finds no frame in flight.
static vt_status surface_call(vt_tracker* t, const char* where, bool sync) {
    if (sync && t->q_count) {
        set_error("%s: frames are in flight (submit/wait); drain them first", where);
        return VT_ERR_INVALID;
    }
    VT_CUDA(cudaSetDevice(t->cfg.device));
    return VT_OK;
}

// The end of every submit: the queue slot's completion event, the result block's device -> host bytes, one more frame in flight
static vt_status finish_submit(vt_tracker* t, int slot) {
    VT_CUDA(cudaEventRecord(t->q_done[slot], t->stream));
    t->d2h_bytes += t->res_block_bytes;
    ++t->q_count;
    t->in_flight = true;
    return VT_OK;
}

// surf: a pitched device surface tracked in place (frame / d_src unused)
static vt_status submit_common(vt_tracker* t, uint8_t* frame, const uint8_t* d_src, size_t len, bool forward = true, const vt_surface* surf = nullptr) {
    if (t->q_count >= vt_tracker::kQueue) {
        set_error("%d frames are already in flight on this handle", t->q_count);
        return VT_ERR_INVALID;
    }
    const bool pinned = d_src || surf || is_pinned(frame);
    if (t->q_count > 0 && (!pinned || t->q[t->q_head].pageable)) {
        set_error("pageable host frames are staged through one buffer and cannot be pipelined: wait() first or use pinned frames");
        return VT_ERR_INVALID;
    }
    const double hp0 = t->sw.hostprof ? now_us() : 0;
    const int slot = (t->q_head + t->q_count) % vt_tracker::kQueue;
    vt_tracker::Slot& q = t->q[slot];
    q.t_submit = std::chrono::steady_clock::now();
    q.frame = d_src || surf ? nullptr : frame, q.len = len, q.pageable = !pinned;
    // the caller's pinned frame is device-mapped under UVA: zero-copy target of the overlay mirror, fall-back source of the crop kernel
    uint8_t* const host_frame = (frame && !d_src && !surf && pinned && len >= t->frame_bytes) ? frame : nullptr;
    // this frame's HUD list (staged by tracker_set_hud in this slot's pinned block)
    const int n_hud = t->hud_mode ? t->hud_next_n[0] : 0;
    q.hud_bytes = n_hud ? t->hud_next_bytes[0] : 0;
    q.mirrored = host_frame && (t->cfg.box_overlay || n_hud > 0);
    // device-resident frame: track (and draw the box) straight in the caller's device memory — no device->device copy.  A full-length
    // packed device frame is tracked in place like a surface.
    const StreamGeom g = cfg_geom(t);
    const bool in_place = surf || (d_src && len >= t->frame_bytes);
    if (!in_place) t->d_frame = t->d_frames[slot];  // the slot's own frame buffer: the other one may still be read by the frame in flight
    const bool lagging = t->q_count > 0;  // a frame is in flight: rect_mirror is one frame old, the windows are predictions
    UploadPlan plan;
    if (!in_place && !d_src) plan_upload(t, len, host_frame != nullptr, lagging, n_hud ? t->hud_next_rmw[0] : nullptr, plan);
    if (!in_place && !d_src && lagging) {
        // pipelined host frame: upload on the copy stream while the frame in flight computes; the main stream picks it up through an event
        vt_status st = do_upload(t, g, frame, len, plan, false, t->copy_stream);
        if (st != VT_OK) return st;
        VT_CUDA(cudaEventRecord(t->ev_up[slot], t->copy_stream));
        VT_CUDA(cudaStreamWaitEvent(t->stream, t->ev_up[slot], 0));
    }
    FrameCtl ctl;
    memset(&ctl, 0, sizeof(ctl));
    ctl.frames[0] = surf ? surface_ref(g, *surf) : packed_ref(g, in_place ? d_src : t->d_frame, host_frame, len >= fmt_valid_bytes(g.fmt, g.W, g.H));
    ctl.n_frames = 1, ctl.hblk = reinterpret_cast<uint32_t*>(t->h_blk[slot]);
    ctl.hud.list = n_hud ? t->h_hud[slot] : nullptr, ctl.hud.n = n_hud;
    const bool hud_inline = n_hud > 0 && n_hud <= kHudInline && t->d_hud[slot] != nullptr;
    if (hud_inline) ctl.hud.list = t->d_hud[slot];
    ctl.n_win = plan.whole ? -1 : plan.n_win;
    if (!plan.whole) memcpy(ctl.win, plan.win, sizeof(ctl.win));
    ctl.hud.bg_on_device = (n_hud && (in_place || d_src || plan.whole || plan.has_rmw)) ? 1 : 0;  // the dimmed region is in the device frame
    t->hud_next_n[0] = 0;
    VT_CUDA(launch_stamp(t->d_stamps + ST_SUBMIT, t->d_ctl, ctl, t->stream, hud_inline ? t->h_hud[slot] : nullptr, n_hud, t->d_hud[slot]));
    ++t->kernel_launches;
    if (in_place) {
        t->d_frame_is_last_host_frame = false;  // tracked in the caller's device memory: the internal buffer holds an older frame
    } else if (d_src) {  // short device frame: device->device copy of what there is (NV12: black frame, src/nv12_convert.rs:48-50)
        vt_status st = do_upload(t, g, d_src, len, plan, true, nullptr);
        if (st != VT_OK) return st;
    } else if (!lagging) {
        vt_status st = do_upload(t, g, frame, len, plan, false, nullptr);  // the host mirror of rect_last is exact: the search windows suffice
        if (st != VT_OK) return st;
    }
    const double hp1 = t->sw.hostprof ? now_us() : 0;
    const bool ran = forward && !t->active.empty();
    if (ran) {
        vt_status st = run_forward(t);
        if (st != VT_OK) return st;
    } else if (n_hud > 0) {  // no tracker runs on this frame (SELECT / LOST states of the probe): HUD list + publish only
        cudaError_t e = launch_box_overlay(t->d_res, t->d_slots, 0, t->cfg.overlay_gate, t->d_ctl, t->d_stamps + ST_OVL_END, t->stream, false,
                                           t->d_res, t->res_block_bytes, 0);
        if (e != cudaSuccess) {
            set_error("overlay launch failed: %s", cudaGetErrorString(e));
            return VT_ERR_CUDA;
        }
        ++t->kernel_launches;
    }
    const double hp2 = t->sw.hostprof ? now_us() : 0;
    // the result block reaches t->h_blk[slot] through the last kernel of the frame; nothing ran: copy it
    if (!ran && n_hud == 0) VT_CUDA(cudaMemcpyAsync(t->h_blk[slot], t->d_res, t->res_block_bytes, cudaMemcpyDeviceToHost, t->stream));
    const vt_status st = finish_submit(t, slot);
    if (st == VT_OK && t->sw.hostprof) t->hp[0] += hp1 - hp0, t->hp[1] += hp2 - hp1, t->hp[2] += now_us() - hp2;
    return st;
}

// Stream i's device frame d_sframes[i] holds a frame of `bytes` (+ 256), grown only between synchronous group steps: nothing in flight
// reads the old buffer
static vt_status ensure_stream_frame(vt_tracker* t, int i, size_t bytes) {
    if (t->d_sframe_bytes[i] >= bytes + 256) return VT_OK;
    if (t->d_sframes[i]) VT_CUDA(cudaFree(t->d_sframes[i]));
    t->d_sframes[i] = nullptr, t->d_sframe_bytes[i] = 0;
    VT_CUDA(cudaMalloc(&t->d_sframes[i], bytes + 256));
    VT_CUDA(cudaMemsetAsync(t->d_sframes[i], 0, bytes + 256, t->stream));
    t->d_sframe_bytes[i] = bytes + 256;
    return VT_OK;
}

// One stream of a group step that takes part in the forward: its full pinned host frame `frame`, of target slot `slot`'s geometry, goes
// into the device frame d_sframes[buf] — whole (and *whole = true), or with cfg.upload_window only the search window around the slot's
// rect_last.  win: the uploaded window (empty: the window misses the frame, the crop kernel flags it); *ref: the stream's frame.
static vt_status stage_stream(vt_tracker* t, int buf, int slot, uint8_t* frame, int* win, FrameRef* ref, bool* whole) {
    const StreamGeom& g = slot_geom(t, slot);
    vt_status st = ensure_stream_frame(t, buf, g.bytes());
    if (st != VT_OK) return st;
    uint8_t* dst = t->d_sframes[buf];
    const bool all = !t->cfg.upload_window || !windows_allowed(g);
    if (all) {
        VT_CUDA(cudaMemcpyAsync(dst, frame, g.bytes(), cudaMemcpyHostToDevice, t->stream));
        t->h2d_bytes += g.bytes();
        win[0] = win[1] = 0, win[2] = g.W, win[3] = g.H;
    } else if (search_window(g, t->rect_mirror[slot], 0, win[0], win[1], win[2], win[3])) {
        st = copy_window(g, dst, frame, win, true, cudaMemcpyHostToDevice, t->stream);
        if (st != VT_OK) return st;
        t->h2d_bytes += window_bytes(g, win);
    } else {
        win[0] = win[1] = win[2] = win[3] = 0;
    }
    *ref = packed_ref(g, dst, frame, true);
    if (whole) *whole = all;
    return VT_OK;
}

// Stream group: the n active targets of the handle are n independent video streams (one target each, each of its slot's geometry),
// stepped together through ONE batched forward (M = 320 n rows: from 1024 rows on the GEMMs run in their throughput forms).  frames[i] is
// the pinned host frame of the i-th active target; each target's search window is uploaded into that target's own device frame and the
// box overlay is mirrored into that target's host frame.  Or surfs[i] (frames / lens unused) is the i-th target's device surface, read
// and drawn into in place.  Stream i's geometry travels in the control block (ctl.frames[i]), so one captured graph per stream count
// serves any mix of sizes and formats.  Synchronous (rect_mirror is exact: the windows are the real search windows).
static vt_status submit_streams(vt_tracker* t, uint8_t* const* frames, const size_t* lens, const vt_surface* surfs, int n) {
    const char* where = surfs ? "vt_tracker_update_streams_surface" : "vt_tracker_update_streams";
    if (t->q_count > 0 || t->hud_mode) {
        set_error("%s: frames are in flight on this handle, or it is a probe (HUD) handle", where);
        return VT_ERR_INVALID;
    }
    if (n != (int)t->active.size() || n <= 0 || n > kMaxWin) {
        set_error("%s: %d frames for %d active targets (one frame per active target, at most %d)", where, n, (int)t->active.size(), kMaxWin);
        return VT_ERR_INVALID;
    }
    for (int i = 0; i < n; ++i) {
        const StreamGeom& g = slot_geom(t, t->active[i]);
        if (surfs) {
            const vt_status st = check_surface(t, g, &surfs[i], where, i);
            if (st != VT_OK) return st;
        } else if (!frames[i] || lens[i] < g.bytes() || !is_pinned(frames[i])) {
            set_error("%s: frame %d must be a full frame (%zu bytes for its %dx%d format %d, got %zu) in pinned host memory (vt_alloc_pinned)",
                      where, i, g.bytes(), g.W, g.H, g.fmt, frames[i] ? lens[i] : (size_t)0);
            return VT_ERR_INVALID;
        }
    }
    const int slot = t->q_head;
    vt_tracker::Slot& q = t->q[slot];
    q.t_submit = std::chrono::steady_clock::now();
    q.frame = surfs ? nullptr : frames[0], q.len = surfs ? 0 : lens[0], q.pageable = false, q.hud_bytes = 0, q.mirrored = !surfs;
    FrameCtl ctl;
    memset(&ctl, 0, sizeof(ctl));
    for (int i = 0; i < n; ++i) {
        if (surfs) {  // in place: nothing to upload, the whole surface holds the frame
            ctl.frames[i] = surface_ref(slot_geom(t, t->active[i]), surfs[i]);
            continue;
        }
        vt_status st = stage_stream(t, i, t->active[i], frames[i], ctl.win[i], &ctl.frames[i], nullptr);
        if (st != VT_OK) return st;
    }
    ctl.n_frames = n, ctl.hblk = reinterpret_cast<uint32_t*>(t->h_blk[slot]);
    ctl.n_win = surfs ? -1 : n;
    t->d_frame_is_last_host_frame = false;
    VT_CUDA(launch_stamp(t->d_stamps + ST_SUBMIT, t->d_ctl, ctl, t->stream));
    ++t->kernel_launches;
    vt_status st = run_forward(t);
    if (st != VT_OK) return st;
    return finish_submit(t, slot);
}

static vt_status wait_common(vt_tracker* t, vt_result* results) {
    if (t->q_count == 0) {
        set_error("no frame in flight");
        return VT_ERR_INVALID;
    }
    const int slot = t->q_head;
    const vt_tracker::Slot q = t->q[slot];
    t->q_head = (t->q_head + 1) % vt_tracker::kQueue;
    --t->q_count;
    t->in_flight = t->q_count > 0;
    t->t_submit = q.t_submit, t->inflight_frame = q.frame, t->inflight_mirrored = q.mirrored;
    const size_t len = q.len;
    const double hp0 = t->sw.hostprof ? now_us() : 0;
    VT_CUDA(cudaEventSynchronize(t->q_done[slot]));
    bind_slot(t, slot);
    const double hp1 = t->sw.hostprof ? now_us() : 0;
    if (*t->h_tc_err) {  // travels with the results; reset on the device for the next frame
        cudaMemsetAsync(t->d_tc_err, 0, sizeof(int), t->stream);
        *t->h_tc_err = 0;
        set_error("tcgen05 path: a bounded mbarrier wait expired (pipeline protocol error)");
        return VT_ERR_CUDA;
    }
    fill_results(t, results);
    const double hp2 = t->sw.hostprof ? now_us() : 0;
    if (q.hud_bytes && t->inflight_mirrored) t->d2h_bytes += q.hud_bytes;  // HUD pixels mirrored into the pinned frame
    if (t->cfg.box_overlay && t->inflight_frame && t->inflight_mirrored) {
        // the overlay kernel wrote the box pixels straight into the caller's pinned frame: count them as device->host traffic
        for (int sl : t->active) {
            const DeviceResult& d = t->h_res[sl];
            if (d.status == VT_OK && d.success && d.score > t->cfg.overlay_gate) t->d2h_bytes += 6ull * (size_t)(std::max(d.bbox[2], 0) + std::max(d.bbox[3], 0)) + 62;
        }
    } else if (t->cfg.box_overlay && t->inflight_frame) {  // pageable frame (never pipelined): copy the touched rows back
        std::vector<std::pair<int, int>> spans;
        box_rows(t, spans);
        merge_spans(spans);
        if (!spans.empty()) {
            bool staged = false;
            vt_status st = download_rows(t, t->inflight_frame, len, spans, &staged);
            if (st != VT_OK) return st;
            VT_CUDA(cudaStreamSynchronize(t->stream));
            if (staged) unstage_rows(t, t->inflight_frame, len, spans);
        }
    }
    const double hp3 = t->sw.hostprof ? now_us() : 0;
    collect_timing(t);
    ++t->frames;
    if (t->sw.hostprof) t->hp[3] += hp1 - hp0, t->hp[4] += hp2 - hp1, t->hp[5] += hp3 - hp2, t->hp[6] += now_us() - hp3, ++t->hp_n;
    return VT_OK;
}

// ---- ring replay support ----------------------------------------------------------------------------------------------------------
// [x0, x1) x [y0, y1) of the drawable plane (Y plane / luma for NV12, I420 and GRAY8, the RGB image for RGB24, the whole pixel-pair
// words for YUY2, the whole 4-byte pixels for RGBA / BGRA), clipped to the frame
void restore_rect_region(uint8_t* frame, const uint8_t* clean, int fmt, int W, int H, long long x0, long long y0, long long x1, long long y1) {
    x0 = std::max(x0, 0LL), y0 = std::max(y0, 0LL), x1 = std::min<long long>(x1, W), y1 = std::min<long long>(y1, H);
    if (x1 <= x0 || y1 <= y0) return;
    const size_t pitch = fmt_row_bytes(fmt, W);
    size_t o0, o1;
    fmt_col_span(fmt, x0, x1, &o0, &o1);
    for (long long y = y0; y < y1; ++y) {
        const size_t o = (size_t)y * pitch + o0;
        memcpy(frame + o, clean + o, o1 - o0);
    }
}
// a box overlay touches the box outline (inclusive x..x+w, y..y+h in the luma formats) and a +-15 px crosshair at its centre
void restore_box_region(uint8_t* frame, const uint8_t* clean, int fmt, int W, int H, const vt_bbox& b) {
    if (b.width < 0 || b.height < 0 || b.width > 4 * W || b.height > 4 * H) {  // wrapped / absurd geometry: restore everything
        restore_rect_region(frame, clean, fmt, W, H, 0, 0, W, H);
        return;
    }
    restore_rect_region(frame, clean, fmt, W, H, (long long)b.x - 16, (long long)b.y - 16, (long long)b.x + b.width + 17, (long long)b.y + b.height + 17);
}

// ---- probe support --------------------------------------------------------------------------------------------------------------
void tracker_enable_hud(vt_tracker* t) {
    if (t && t->graphs.empty()) t->hud_mode = true;  // (the frame's last kernel is part of the captured graph)
}

// Stages the HUD list of the NEXT submit in the pinned block of the queue slot that submit will use.  A probe group's block holds one
// list of up to kMaxCmds commands per stream: stream i's at [i * kMaxCmds], drawn on stream i's frame (its geometry).
vt_status tracker_set_hud(vt_tracker* t, const HudCmd* cmds, int n, int stream) {
    if (!t || !t->hud_mode || n < 0 || n > kMaxCmds || (n > 0 && !cmds) || stream < 0 || stream >= std::max(t->group_n, 1)) {
        set_error("tracker_set_hud: invalid argument (HUD mode %d, %d commands, stream %d)", t ? (int)t->hud_mode : -1, n, stream);
        return VT_ERR_INVALID;
    }
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const int slot = (t->q_head + t->q_count) % vt_tracker::kQueue;
    if (!t->h_hud[slot])
        VT_CUDA(cudaHostAlloc(&t->h_hud[slot], sizeof(OverlayCmdDev) * kMaxCmds * std::max(t->group_n, 1), cudaHostAllocDefault));
    if (!t->d_hud[slot] && !t->group_n) VT_CUDA(cudaMalloc(&t->d_hud[slot], sizeof(OverlayCmdDev) * kHudInline));
    const StreamGeom& g = slot_geom(t, stream);  // (a single probe: the cfg geometry)
    int rmw[4] = {0, 0, 0, 0};
    size_t bytes = 0;
    for (int i = 0; i < n; ++i) {
        OverlayCmdDev& d = t->h_hud[slot][stream * kMaxCmds + i];
        const vt_overlay_cmd& c = cmds[i].cmd;
        vt_status st = fill_cmd_dev(c, d);
        if (st != VT_OK) return st;
        d.cond = cmds[i].cond, d.from_result = cmds[i].from_result;
        if (d.from_result == VT_HUD_SCORE_TEXT) {  // digit and '%' glyphs for the device-side "{:.0}%" of the score
            if (d.nchar > 32) {
                set_error("tracker_set_hud: score text prefix too long");
                return VT_ERR_INVALID;
            }
            for (int k = 0; k <= 10; ++k) {
                uint8_t rows[7];
                const int ch = k < 10 ? '0' + k : '%';
                if (vt_glyph_rows(ch, rows) == 0) d.known[kHudDigitSlot + k] = 1, memcpy(d.glyph[kHudDigitSlot + k], rows, 7);
            }
        }
        if (c.kind == VT_OV_BACKGROUND && format_is_luma(g.fmt) && c.x >= 0 && c.y >= 0 && c.w > 0 && c.h > 0) {
            // the luma background dim reads before it writes (src/nv12_convert.rs:324-343): that region must be on the device
            const int x1 = (int)std::min<long long>((long long)c.x + c.w, g.W), y1 = (int)std::min<long long>((long long)c.y + c.h, g.H);
            if (rmw[2] <= rmw[0]) rmw[0] = c.x, rmw[1] = c.y, rmw[2] = x1, rmw[3] = y1;
            else rmw[0] = std::min(rmw[0], c.x), rmw[1] = std::min(rmw[1], c.y), rmw[2] = std::max(rmw[2], x1), rmw[3] = std::max(rmw[3], y1);
            bytes += (size_t)std::max(0, x1 - c.x) * std::max(0, y1 - c.y);
        } else if (c.kind == VT_OV_TEXT) {
            bytes += (size_t)35 * std::max(c.a, 0) * std::max(c.a, 0) * d.nchar;
        } else {
            bytes += 1024;  // rect / crosshair / cursor / selection outlines
        }
    }
    t->hud_next_n[stream] = n, t->hud_next_bytes[stream] = bytes;
    memcpy(t->hud_next_rmw[stream], rmw, sizeof(rmw));
    return VT_OK;
}

// The template window must intersect the frame (cv2 raises an ROI assertion otherwise, App. A.1)
static vt_status check_template_window(const vt_tracker* t, const StreamGeom& g, vt_bbox box, const char* where) {
    if (box.width <= 0 || box.height <= 0) {
        set_error("%s: empty box", where);
        return VT_ERR_CROP_OUTSIDE;
    }
    const int c = (int)ceil(sqrt((double)((long long)box.width * box.height)) * 2.0);
    const int x1 = box.x + (box.width - c) / 2, y1 = box.y + (box.height - c) / 2;
    const int pp = t->cfg.pad_plus1;
    const int pl = std::max(0, -x1), pt = std::max(0, -y1), pr = std::max(x1 + c - g.W + pp, 0), pb = std::max(y1 + c - g.H + pp, 0);
    if (c - pl - pr <= 0 || c - pt - pb <= 0) {
        set_error("%s: template window lies outside the frame", where);
        return VT_ERR_CROP_OUTSIDE;
    }
    return VT_OK;
}

// The template pass of vt_tracker_init[_surface] on the device frame fd: template crop -> patch embed (+ LN1 of block 0) of `target`,
// which then joins the active targets with rect_last = box.
static vt_status init_template(vt_tracker* t, int32_t target, vt_bbox box, const FrameDesc& fd) {
    TargetState hs;
    memset(&hs, 0, sizeof(hs));
    hs.rect[0] = box.x, hs.rect[1] = box.y, hs.rect[2] = box.width, hs.rect[3] = box.height, hs.active = 1;
    int32_t slot = target;
    VT_CUDA(cudaMemcpyAsync(t->d_state + target, &hs, sizeof(hs), cudaMemcpyHostToDevice, t->stream));
    // d_slots is reused as a one-element list for the template pass, then restored
    VT_CUDA(cudaMemcpyAsync(t->d_slots, &slot, sizeof(slot), cudaMemcpyHostToDevice, t->stream));
    int launches = 0;
    VT_LAUNCH(launch_crop_resize_norm(fd, t->d_state, t->d_slots, 1, 2, kTemplate, t->d_lut, t->patches_z, (size_t)kNTz * kPatchK, t->pz_hi,
                                      t->f16 ? nullptr : t->pz_lo, t->stream));
    if (t->nsplit == 0) {
        GemmArgs g = gemm_args(t->patches_z, kPatchK, t->patch_w, t->patch_b, t->Zemb + (size_t)target * kNTz * t->D, t->D, kNTz, t->D, kPatchK);
        g.pos = t->pos_z;
        g.c_rows_in = kNTz, g.c_rows_stride = kNTz, g.c_row_off = 0;
        VT_LAUNCH(launch_gemm_simt(g, t->stream));
    } else {
        TcGemmPlan p = t->plan_patch_z;
        p.args.batch_off = target;
        VT_LAUNCH(tc_gemm_launch(p, kNTz, t->nsplit, t->stream, false));
        VT_LAUNCH(launch_layernorm_split(t->Zemb + (size_t)target * kNTz * t->D, t->D, t->blk[0].ln1_g, t->blk[0].ln1_b, t->zln_hi + (size_t)target * kNTz * t->D,
                                         t->f16 ? nullptr : t->zln_lo + (size_t)target * kNTz * t->D, kNTz, t->D, 1 << 30, 0, 0, t->stream, false));
    }
    t->kernel_launches += launches;
    VT_CUDA(cudaStreamSynchronize(t->stream));
    if (!t->inited[target]) {
        t->inited[target] = 1;
        t->active.push_back(target);
        std::sort(t->active.begin(), t->active.end());
    }
    t->rect_mirror[target] = box;
    return sync_slots(t);
}

vt_status check_uniform_geometry(const vt_tracker* t, const char* where) {
    for (int s = 0; s < t->maxT; ++s)
        if (!(slot_geom(t, s) == cfg_geom(t))) {
            set_error("%s: slot %d has a stream geometry of its own (vt_tracker_set_stream_geometry): this handle takes frames through the "
                      "stream-group calls only", where, s);
            return VT_ERR_INVALID;
        }
    return VT_OK;
}

// d_frames[0..1] and h_stage hold any frame vt_tracker_init is given: the largest of the cfg and the slot geometries
static vt_status grow_frame_buffers(vt_tracker* t, size_t bytes) {
    if (bytes <= t->h_stage_bytes) return VT_OK;
    VT_CUDA(cudaStreamSynchronize(t->stream));
    for (uint8_t*& f : t->d_frames) {
        VT_CUDA(cudaFree(f));
        f = nullptr;
    }
    VT_CUDA(cudaFreeHost(t->h_stage));
    t->h_stage = nullptr, t->h_stage_bytes = 0, t->d_frame = nullptr, t->d_frame_is_last_host_frame = false;
    for (uint8_t*& f : t->d_frames) {
        VT_CUDA(cudaMalloc(&f, bytes));
        VT_CUDA(cudaMemset(f, 0, bytes));
    }
    VT_CUDA(cudaHostAlloc(&t->h_stage, bytes, cudaHostAllocDefault));
    t->h_stage_bytes = bytes, t->d_frame = t->d_frames[0];
    return VT_OK;
}

// VitTrack::init of `target` on a host frame of the slot's geometry (the whole frame is uploaded)
static vt_status init_from_host(vt_tracker* t, int32_t target, const uint8_t* frame, size_t len, vt_bbox box) {
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const StreamGeom& g = slot_geom(t, target);
    vt_status st = check_template_window(t, g, box, "vt_tracker_init");
    if (st != VT_OK) return st;
    st = do_upload(t, g, frame, len, UploadPlan(), false, nullptr);  // the whole frame
    if (st != VT_OK) return st;
    const bool valid = len >= fmt_valid_bytes(g.fmt, g.W, g.H);
    return init_template(t, target, box, FrameDesc{packed_ref(g, t->d_frame, nullptr, valid), nullptr, t->cfg.pad_plus1});
}

// The tracker of a probe group steps its streams through vt_probe_group_frame only: every public frame entry point refuses it.
static bool group_refused(const vt_tracker* t, const char* where) {
    if (!t->group_n) return false;
    set_error("%s: this handle is the tracker of a probe group; its frames go through vt_probe_group_frame / vt_probe_group_run_ring", where);
    return true;
}

// The public surface calls refuse a probe (HUD) handle: the probe's state machine stages a HUD list for every frame of that handle, so
// its surfaces go through vt_probe_frame_surface / vt_probe_group_frame_surface (tracker_init_surface / tracker_submit_surface below).
static bool hud_refused(const vt_tracker* t, const char* where) {
    if (!t->hud_mode) return false;
    set_error("%s: a probe (HUD) handle takes surfaces through vt_probe_frame_surface / vt_probe_group_frame_surface only", where);
    return true;
}

vt_status tracker_check_surface(const vt_tracker* t, int stream, const vt_surface* s, const char* where) {
    return check_surface(t, slot_geom(t, stream), s, where, stream);
}

// VitTrack::init of `target` on a surface of the slot's geometry, read in place
vt_status tracker_init_surface(vt_tracker* t, int32_t target, const vt_surface* s, vt_bbox box, const char* where) {
    if (t->in_flight) {
        set_error("%s: a frame is in flight", where);
        return VT_ERR_INVALID;
    }
    vt_status st = surface_call(t, where, true);
    if (st == VT_OK) st = check_surface(t, slot_geom(t, target), s, where, 0);
    const StreamGeom& g = slot_geom(t, target);
    if (st == VT_OK) st = check_template_window(t, g, box, where);
    if (st != VT_OK) return st;
    return init_template(t, target, box, FrameDesc{surface_ref(g, *s), nullptr, t->cfg.pad_plus1});
}

vt_status tracker_submit_surface(vt_tracker* t, const vt_surface* s, bool forward, const char* where) {
    vt_status st = surface_call(t, where, false);
    if (st == VT_OK) st = check_surface(t, cfg_geom(t), s, where, 0);
    if (st != VT_OK) return st;
    return submit_common(t, nullptr, nullptr, 0, forward, s);
}

}  // namespace vt

using namespace vt;

extern "C" {

vt_status vt_tracker_init(vt_tracker* t, int32_t target, const uint8_t* frame, size_t len, vt_bbox box) {
    if (!t || !frame || target < 0 || target >= t->maxT) {
        set_error("vt_tracker_init: invalid argument");
        return VT_ERR_INVALID;
    }
    if (t->in_flight) {
        set_error("vt_tracker_init: a frame is in flight");
        return VT_ERR_INVALID;
    }
    if (group_refused(t, "vt_tracker_init")) return VT_ERR_INVALID;
    return init_from_host(t, target, frame, len, box);
}

vt_status vt_tracker_init_surface(vt_tracker* t, int32_t target, const vt_surface* s, vt_bbox box) {
    if (!t || !s || target < 0 || target >= t->maxT) {
        set_error("vt_tracker_init_surface: invalid argument");
        return VT_ERR_INVALID;
    }
    if (group_refused(t, "vt_tracker_init_surface") || hud_refused(t, "vt_tracker_init_surface")) return VT_ERR_INVALID;
    return tracker_init_surface(t, target, s, box, "vt_tracker_init_surface");
}

vt_status vt_tracker_set_stream_geometry(vt_tracker* t, int32_t target, const vt_stream_geometry* g) {
    if (!t || target < 0 || target >= t->maxT) {
        set_error("vt_tracker_set_stream_geometry: invalid handle or target slot");
        return VT_ERR_INVALID;
    }
    if (t->hud_mode) {
        set_error("vt_tracker_set_stream_geometry: a probe (HUD) handle tracks one stream of the handle's geometry");
        return VT_ERR_INVALID;
    }
    if (t->in_flight) {
        set_error("vt_tracker_set_stream_geometry: frames are in flight (submit/wait); drain them first");
        return VT_ERR_INVALID;
    }
    if (t->inited[target]) {
        set_error("vt_tracker_set_stream_geometry: slot %d is initialised; vt_tracker_drop it first", target);
        return VT_ERR_INVALID;
    }
    const StreamGeom ng = g ? StreamGeom{g->format, g->width, g->height} : cfg_geom(t);
    if (g && (!geometry_ok(ng.fmt, ng.W, ng.H) || g->reserved != 0)) {
        set_error("vt_tracker_set_stream_geometry: format %d, %d x %d (reserved %d) is not a frame geometry (a vt_format, width and height > 0, "
                  "reserved 0)", g->format, g->width, g->height, g->reserved);
        return VT_ERR_INVALID;
    }
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const vt_status st = grow_frame_buffers(t, ng.bytes() + 256);
    if (st != VT_OK) return st;
    t->geom[target] = ng;
    return VT_OK;
}

vt_status vt_tracker_get_stream_geometry(const vt_tracker* t, int32_t target, vt_stream_geometry* out) {
    if (!t || !out || target < 0 || target >= t->maxT) {
        set_error("vt_tracker_get_stream_geometry: invalid argument");
        return VT_ERR_INVALID;
    }
    const StreamGeom& g = slot_geom(t, target);
    out->format = g.fmt, out->width = g.W, out->height = g.H, out->reserved = 0;
    return VT_OK;
}

vt_status vt_tracker_drop(vt_tracker* t, int32_t target) {
    if (!t || target < 0 || target >= t->maxT || t->in_flight) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    if (t->inited[target]) {
        t->inited[target] = 0;
        t->active.erase(std::remove(t->active.begin(), t->active.end(), target), t->active.end());
        VT_CUDA(cudaMemsetAsync(t->d_state + target, 0, sizeof(TargetState), t->stream));
    }
    return sync_slots(t);
}

vt_status vt_tracker_submit(vt_tracker* t, uint8_t* frame, size_t len) {
    if (!t || !frame) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_submit")) return VT_ERR_INVALID;
    vt_status st = check_uniform_geometry(t, "vt_tracker_submit");
    if (st != VT_OK) return st;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    return submit_common(t, frame, nullptr, len);
}

}  // extern "C"
namespace vt {
vt_status tracker_submit_hud_only(vt_tracker* t, uint8_t* frame, size_t len) {
    if (!t || !frame) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    return submit_common(t, frame, nullptr, len, false);
}

vt_status tracker_make_group(vt_tracker* t, int n) {
    if (!t || n < 1 || n > kMaxWin || n != t->maxT || !t->graphs.empty() || t->q_count || t->group_n) {
        set_error("tracker_make_group: needs a fresh handle with max_targets = %d (1..%d)", n, kMaxWin);
        return VT_ERR_INVALID;
    }
    VT_CUDA(cudaSetDevice(t->cfg.device));
    VT_CUDA(cudaFree(t->d_ctl));
    t->d_ctl = nullptr;
    VT_CUDA(cudaMalloc(&t->d_ctl, sizeof(ProbeGroupCtl)));
    VT_CUDA(cudaMemset(t->d_ctl, 0, sizeof(ProbeGroupCtl)));
    VT_CUDA(cudaHostAlloc(&t->h_slots, sizeof(int32_t) * kMaxWin, cudaHostAllocDefault));
    for (int i = 0; i < n; ++i) {  // one device frame per stream, of its geometry: every stream's HUD is drawn into it at every step
        const vt_status st = ensure_stream_frame(t, i, slot_geom(t, i).bytes());
        if (st != VT_OK) return st;
    }
    tracker_enable_hud(t);
    t->group_n = n;
    return VT_OK;
}

vt_status tracker_group_init(vt_tracker* t, int stream, const uint8_t* frame, size_t len, vt_bbox box) {
    if (!t || !t->group_n || stream < 0 || stream >= t->group_n || !frame || t->in_flight) {
        set_error("tracker_group_init: invalid argument");
        return VT_ERR_INVALID;
    }
    return init_from_host(t, stream, frame, len, box);
}

vt_status tracker_group_drop(vt_tracker* t, int stream) {
    if (!t || !t->group_n || stream < 0 || stream >= t->group_n || t->in_flight) {
        set_error("tracker_group_drop: invalid argument");
        return VT_ERR_INVALID;
    }
    if (t->inited[stream]) {
        t->inited[stream] = 0;
        t->active.erase(std::remove(t->active.begin(), t->active.end(), stream), t->active.end());
        VT_CUDA(cudaSetDevice(t->cfg.device));
        VT_CUDA(cudaMemsetAsync(t->d_state + stream, 0, sizeof(TargetState), t->stream));
    }
    return VT_OK;
}

bool tracker_group_active(const vt_tracker* t, int stream) { return t && stream >= 0 && stream < t->group_n && t->inited[stream]; }

// One probe-group step.  The streams whose slot is active (stream i = slot i, ascending) run ONE batched forward: each one's search window
// is uploaded into its own device frame and the crop addresses them by active-target index, as in a stream group.  The step's last kernel
// runs one CTA pair per stream of the group: the stream's HUD list (both outcomes for a stream in the forward, picked by its own result),
// drawn on its device frame and mirrored into its pinned host frame.  With no stream in the forward that kernel is the whole step.
// Every luma stream's HUD region is uploaded with the windows, so that — as in the single probe — the device pass dims its own copy of the
// region while the host pass reads the pinned frame.  Or surfs[i] (frames / lens unused; checked by the caller) is stream i's device
// surface: read and drawn into in place, nothing uploaded and nothing mirrored.  Synchronous (rect_mirror is exact: the windows are the
// real search windows).
vt_status tracker_submit_group(vt_tracker* t, uint8_t* const* frames, const size_t* lens, const vt_surface* surfs) {
    const int n = t ? t->group_n : 0;
    if (!n || t->q_count) {
        set_error("tracker_submit_group: not the tracker of a probe group, or a step is in flight");
        return VT_ERR_INVALID;
    }
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const int slot = t->q_head;
    vt_tracker::Slot& q = t->q[slot];
    q.t_submit = std::chrono::steady_clock::now();
    q.frame = surfs ? nullptr : frames[0], q.len = surfs ? 0 : lens[0], q.pageable = false, q.mirrored = !surfs, q.hud_bytes = 0;
    ProbeGroupCtl ctl;
    memset(&ctl, 0, sizeof(ctl));
    const int k_act = (int)t->active.size();
    for (int i = 0, k = 0; i < n; ++i) {  // every stream of the group, by stream index; the forward's targets by active-target index k
        const StreamGeom& g = slot_geom(t, i);
        ProbeStreamCtl& e = ctl.s[i];
        const bool fwd = k < k_act && t->active[k] == i;  // (active is ascending)
        bool whole = surfs != nullptr;  // in place: the whole surface holds the frame
        if (surfs) {
            e.frame = surface_ref(g, surfs[i]);
        } else if (fwd) {
            vt_status st = stage_stream(t, i, i, frames[i], ctl.f.win[k], &e.frame, &whole);
            if (st != VT_OK) return st;
        } else {
            e.frame = packed_ref(g, t->d_sframes[i], frames[i], true);
        }
        if (fwd) ctl.f.frames[k++] = e.frame;
        e.hud.n = t->hud_next_n[i];
        e.hud.list = e.hud.n ? t->h_hud[slot] + (size_t)i * kMaxCmds : nullptr;
        e.slot = t->inited[i] ? i : -1;
        const int* r = t->hud_next_rmw[i];
        int w[4] = {std::max(r[0], 0), std::max(r[1], 0), std::min(r[2], g.W), std::min(r[3], g.H)};
        if (e.hud.n && whole) {
            e.hud.bg_on_device = 1;
        } else if (e.hud.n && w[2] > w[0] && w[3] > w[1]) {  // plane 0 only (the luma background dim reads and writes Y)
            vt_status st = copy_window(g, t->d_sframes[i], frames[i], w, false, cudaMemcpyHostToDevice, t->stream);
            if (st != VT_OK) return st;
            t->h2d_bytes += plane0_bytes(g, w[0], w[1], w[2], w[3]);
            e.hud.bg_on_device = 1;
        }
        if (e.hud.n) q.hud_bytes += t->hud_next_bytes[i];
        t->hud_next_n[i] = 0;
    }
    ctl.f.n_frames = k_act, ctl.f.hblk = reinterpret_cast<uint32_t*>(t->h_blk[slot]);
    ctl.f.n_win = surfs ? -1 : k_act;
    if (k_act) {  // (drops since the last step changed the list: it reaches the device ahead of the step's kernels)
        memcpy(t->h_slots, t->active.data(), sizeof(int32_t) * (size_t)k_act);
        VT_CUDA(cudaMemcpyAsync(t->d_slots, t->h_slots, sizeof(int32_t) * (size_t)k_act, cudaMemcpyHostToDevice, t->stream));
    }
    t->d_frame_is_last_host_frame = false;
    VT_CUDA(launch_stamp_group(t->d_stamps + ST_SUBMIT, reinterpret_cast<ProbeGroupCtl*>(t->d_ctl), ctl, t->stream));
    ++t->kernel_launches;
    if (k_act) {
        vt_status st = run_forward(t);
        if (st != VT_OK) return st;
    } else {  // no stream in the forward: every stream's HUD in one launch
        cudaError_t e = launch_group_overlay(n, t->d_res, t->cfg.overlay_gate, reinterpret_cast<const ProbeGroupCtl*>(t->d_ctl),
                                             t->d_stamps + ST_OVL_END, t->stream, false, t->d_res, t->res_block_bytes);
        if (e != cudaSuccess) {
            set_error("probe group overlay launch failed: %s", cudaGetErrorString(e));
            return VT_ERR_CUDA;
        }
        ++t->kernel_launches;
    }
    return finish_submit(t, slot);
}
}  // namespace vt
extern "C" {

vt_status vt_tracker_submit_device(vt_tracker* t, uint8_t* d_frame, size_t len) {
    if (!t || !d_frame) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_submit_device")) return VT_ERR_INVALID;
    vt_status st = check_uniform_geometry(t, "vt_tracker_submit_device");
    if (st != VT_OK) return st;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    return submit_common(t, nullptr, d_frame, len);
}

vt_status vt_tracker_wait(vt_tracker* t, vt_result* results) {
    if (!t) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    return wait_common(t, results);
}

vt_status vt_tracker_update(vt_tracker* t, uint8_t* frame, size_t len, vt_result* results) {
    if (!t || !frame) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_update")) return VT_ERR_INVALID;
    vt_status st = check_uniform_geometry(t, "vt_tracker_update");
    if (st != VT_OK) return st;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    if (t->q_count) {
        set_error("vt_tracker_update: frames are in flight (submit/wait); drain them first");
        return VT_ERR_INVALID;
    }
    st = submit_common(t, frame, nullptr, len);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

vt_status vt_tracker_update_streams(vt_tracker* t, uint8_t* const* frames, const size_t* lens, int32_t n, vt_result* results) {
    if (!t || !frames || !lens) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_update_streams")) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    vt_status st = submit_streams(t, frames, lens, nullptr, n);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

vt_status vt_tracker_update_device(vt_tracker* t, uint8_t* d_frame, size_t len, vt_result* results) {
    if (!t || !d_frame) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_update_device")) return VT_ERR_INVALID;
    vt_status st = check_uniform_geometry(t, "vt_tracker_update_device");
    if (st != VT_OK) return st;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    if (t->q_count) {
        set_error("vt_tracker_update_device: frames are in flight (submit/wait); drain them first");
        return VT_ERR_INVALID;
    }
    st = submit_common(t, nullptr, d_frame, len);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

vt_status vt_tracker_update_surface(vt_tracker* t, const vt_surface* s, vt_result* results) {
    if (!t || !s) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_update_surface")) return VT_ERR_INVALID;
    if (hud_refused(t, "vt_tracker_update_surface")) return VT_ERR_INVALID;
    vt_status st = check_uniform_geometry(t, "vt_tracker_update_surface");
    if (st == VT_OK) st = surface_call(t, "vt_tracker_update_surface", true);
    if (st == VT_OK) st = check_surface(t, cfg_geom(t), s, "vt_tracker_update_surface", 0);
    if (st == VT_OK) st = submit_common(t, nullptr, nullptr, 0, true, s);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

vt_status vt_tracker_submit_surface(vt_tracker* t, const vt_surface* s) {
    if (!t || !s) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_submit_surface")) return VT_ERR_INVALID;
    if (hud_refused(t, "vt_tracker_submit_surface")) return VT_ERR_INVALID;
    vt_status st = check_uniform_geometry(t, "vt_tracker_submit_surface");
    if (st != VT_OK) return st;
    return tracker_submit_surface(t, s, true, "vt_tracker_submit_surface");
}

vt_status vt_tracker_update_streams_surface(vt_tracker* t, const vt_surface* surfaces, int32_t n, vt_result* results) {
    if (!t || !surfaces) return VT_ERR_INVALID;
    if (group_refused(t, "vt_tracker_update_streams_surface")) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    vt_status st = submit_streams(t, nullptr, nullptr, surfaces, n);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

// ≙ the streaming thread's per-buffer loop (src/pipeline.rs:65-67), natively: see include/vt_tracker.h
vt_status vt_tracker_run_ring(vt_tracker* t, uint8_t* frames, size_t stride, size_t frame_len, int32_t ring, int32_t first, int32_t n, int32_t mode,
                              const uint8_t* pristine, vt_result* last, double* latency_us) {
    if (!t || !frames || ring <= 0 || first < 0 || n < 0 || mode < VT_RUN_HOST_SYNC || mode > VT_RUN_DEVICE_PIPELINED || frame_len > stride) {
        set_error("vt_tracker_run_ring: invalid argument");
        return VT_ERR_INVALID;
    }
    if (t->q_count) {
        set_error("vt_tracker_run_ring: frames are in flight; drain them first");
        return VT_ERR_INVALID;
    }
    if (group_refused(t, "vt_tracker_run_ring")) return VT_ERR_INVALID;
    if (check_uniform_geometry(t, "vt_tracker_run_ring") != VT_OK) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const bool device = mode >= VT_RUN_DEVICE_SYNC, pipelined = mode == VT_RUN_HOST_PIPELINED || mode == VT_RUN_DEVICE_PIPELINED;
    std::vector<vt_result> res((size_t)t->maxT);
    auto fr = [&](int i) { return frames + (size_t)((first + i) % ring) * stride; };
    auto restore = [&](int i) {  // undo what the box overlay of frame i drew (host rings only)
        if (!pristine || device || !t->cfg.box_overlay) return;
        const uint8_t* clean = pristine + (size_t)((first + i) % ring) * stride;
        for (int s : t->active) {
            const vt_result& r = res[s];
            if (r.status == VT_OK && r.success && r.score > t->cfg.overlay_gate) restore_box_region(fr(i), clean, t->fmt, t->W, t->H, r.bbox);
        }
    };
    vt_status st = VT_OK;
    if (!pipelined) {
        for (int i = 0; i < n && st == VT_OK; ++i) {
            const auto t0 = std::chrono::steady_clock::now();
            st = submit_common(t, device ? nullptr : fr(i), device ? fr(i) : nullptr, frame_len);
            if (st == VT_OK) st = wait_common(t, res.data());
            if (latency_us) latency_us[i] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
            restore(i);
        }
    } else {
        for (int i = 0; i < n && st == VT_OK; ++i) {
            st = submit_common(t, device ? nullptr : fr(i), device ? fr(i) : nullptr, frame_len);
            if (st == VT_OK && i > 0) {
                st = wait_common(t, res.data());
                restore(i - 1);
            }
        }
        while (t->q_count && st == VT_OK) {
            st = wait_common(t, res.data());
            restore(n - 1);
        }
        if (st != VT_OK)  // leave no frame in flight behind an error
            while (t->q_count) wait_common(t, nullptr);
    }
    if (last && st == VT_OK && n > 0) memcpy(last, res.data(), sizeof(vt_result) * (size_t)t->maxT);
    return st;
}

// vt_tracker_run_ring for a stream group: stream i's ring starts at rings[i] (pinned host memory; `ring` frames, `stride` apart)
vt_status vt_tracker_run_streams_ring(vt_tracker* t, uint8_t* const* rings, int32_t n_streams, size_t stride, size_t frame_len, int32_t ring,
                                      int32_t first, int32_t n, const uint8_t* const* pristine, vt_result* last, double* latency_us) {
    if (!t || !rings || n_streams <= 0 || n_streams > kMaxWin || ring <= 0 || first < 0 || n < 0 || frame_len > stride) {
        set_error("vt_tracker_run_streams_ring: invalid argument");
        return VT_ERR_INVALID;
    }
    if (group_refused(t, "vt_tracker_run_streams_ring")) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    std::vector<vt_result> res((size_t)t->maxT);
    uint8_t* fr[kMaxWin];
    size_t lens[kMaxWin];
    vt_status st = VT_OK;
    for (int i = 0; i < n && st == VT_OK; ++i) {
        const size_t off = (size_t)((first + i) % ring) * stride;
        for (int k = 0; k < n_streams; ++k) fr[k] = rings[k] + off, lens[k] = frame_len;
        const auto t0 = std::chrono::steady_clock::now();
        st = submit_streams(t, fr, lens, nullptr, n_streams);
        if (st == VT_OK) st = wait_common(t, res.data());
        if (latency_us) latency_us[i] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
        if (st == VT_OK && pristine && t->cfg.box_overlay)  // undo what the box overlays drew: the rings are replayed on clean frames
            for (int k = 0; k < n_streams && k < (int)t->active.size(); ++k) {
                const vt_result& r = res[t->active[k]];
                const StreamGeom& g = slot_geom(t, t->active[k]);
                if (pristine[k] && r.status == VT_OK && r.success && r.score > t->cfg.overlay_gate)
                    restore_box_region(fr[k], pristine[k] + off, g.fmt, g.W, g.H, r.bbox);
            }
    }
    if (last && st == VT_OK && n > 0) memcpy(last, res.data(), sizeof(vt_result) * (size_t)t->maxT);
    return st;
}

vt_status vt_tracker_get_rect(vt_tracker* t, int32_t target, vt_bbox* out) {
    if (!t || !out || target < 0 || target >= t->maxT) return VT_ERR_INVALID;
    if (!t->inited[target]) return VT_ERR_NOT_INIT;
    *out = t->rect_mirror[target];
    return VT_OK;
}

vt_status vt_tracker_set_rect(vt_tracker* t, int32_t target, vt_bbox box) {
    if (!t || target < 0 || target >= t->maxT || t->in_flight) return VT_ERR_INVALID;
    if (!t->inited[target]) return VT_ERR_NOT_INIT;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    int32_t r[4] = {box.x, box.y, box.width, box.height};
    VT_CUDA(cudaMemcpyAsync(&t->d_state[target].rect[0], r, sizeof(r), cudaMemcpyHostToDevice, t->stream));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    t->rect_mirror[target] = box;
    return VT_OK;
}

}  // extern "C"
