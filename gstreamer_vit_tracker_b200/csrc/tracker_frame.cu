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

// Enqueues crop -> ViT -> decode (-> box overlay) for the n active targets on t->stream.
static vt_status enqueue_forward(vt_tracker* t, int n, int& launches, bool record_events, bool capturing, bool spread) {
    const int D = t->D, Hd = t->hidden, C = t->head_ch;
    (void)record_events, (void)capturing;  // stage times come from device stamps (ST_*), not from event nodes
    cudaStream_t s = t->stream;
    FrameDesc fd{t->d_frame, t->W, t->H, t->fmt, t->frame_valid, t->d_ctl, t->cfg.pad_plus1};
    auto LO = [&](__nv_bfloat16* p) { return t->f16 ? nullptr : p; };  // fp16 mode: "hi only" (see vt_internal.h: operand_bits)
    VT_LAUNCH(launch_crop_resize_norm(fd, t->d_state, t->d_slots, n, 4, kSearch, t->d_lut, t->patches_x, (size_t)kNTx * kPatchK, t->px_hi,
                                      LO(t->px_lo), s, t->d_stamps + ST_PRE));
    {
        dim3 grid((kNTz * D + 255) / 256, n);
        const bool f = t->fuse_ln;
        VT_LAUNCH(launch_ex(gather_template_kernel, grid, dim3(256), 0, s, t->pdl && !t->debug_capture, 1, t->X, (const float*)t->Zemb,
                            (const int32_t*)t->d_slots, D, f ? (uint32_t*)t->ln_hi : nullptr, (uint32_t*)LO(t->ln_lo), (const uint32_t*)t->zln_hi,
                            (const uint32_t*)t->zln_lo, t->d_stamps + ST_VIT));
    }
    const int M = n * kNTok;
    int head_np = 9;
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
        const bool pdl = t->pdl && !t->debug_capture, fuse = t->fuse_ln;
        // Many targets: the split-K forms of patch embed (4 K-slices) and head conv (one 3x3 tap per slice) are shaped for one target's
        // three row tiles; from 8 targets on they are 384 / 576 short CTAs (2.6 / 3.9 waves), so the slices are merged — 2 K-slices, 3 taps
        // per slice: a third of the partial planes, CTAs that run three times as many MMAs per prologue.
        const bool merge_slices = t->split_k && n >= kUnchainTargets && !getenv("VT_B200_NO_MERGE_SLICES");
        int patch_np = 4;
        if (merge_slices) {
            TcGemmPlan pp = t->plan_patch_x;
            pp.args.kb_per_split = kPatchK / 64 / 2, patch_np = 2;
            VT_LAUNCH(tc_gemm_launch(pp, n * kNTx, ns, s, pdl));
        } else {
            VT_LAUNCH(tc_gemm_launch(t->plan_patch_x, n * kNTx, ns, s, pdl));  // fused: + LN1 of block 0 for the search rows
        }
        if (t->split_k) {  // X[64.., :] = pos_x + patch_b + sum of the K-slices; LN1 of block 0
            ReduceLnArgs r{};
            r.P = t->Pbuf, r.np = patch_np, r.p_stride = (int64_t)t->maxT * kNTx * D, r.bias = t->patch_b, r.add = t->pos_x, r.add_period = kNTx;
            r.X = t->X, r.M = n * kNTx, r.D = D, r.period = kNTx, r.x_rows = kNTok, r.x_row_off = kNTz;
            r.ln_g = t->blk[0].ln1_g, r.ln_b = t->blk[0].ln1_b, r.ln_hi = t->ln_hi, r.ln_lo = LO(t->ln_lo), r.ln_rows = kNTok, r.ln_row_off = kNTz;
            VT_LAUNCH(launch_reduce_ln(r, s, pdl));
        }
        if (t->debug_capture) VT_CUDA(cudaMemcpyAsync(t->d_dbg, t->X, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, s));
        for (int l = 0; l < t->depth; ++l) {
            const BlockW& b = t->blk[l];
            const vt_tracker::BlockPlans& p = t->plans[l];
            if (!fuse) VT_LAUNCH(launch_layernorm_split(t->X, D, b.ln1_g, b.ln1_b, t->ln_hi, LO(t->ln_lo), M, D, 1 << 30, 0, 0, s, pdl));
            // many rows (cfg4, stream groups): the A-stationary form — activation tile resident, epilogue of chunk i under the main loop of i + 1
            const bool as_form = t->as_rows > 0 && M >= t->as_rows;
            const bool tp_mcast = t->tp_rows > 0 && M >= t->tp_rows;
            if (as_form && tc_gemm_as_supported(p.qkv))
                VT_LAUNCH(tc_gemm_as_launch(p.qkv, M, ns, s, pdl, t->sm_count));
            else
                VT_LAUNCH(tc_gemm_launch(p.qkv, M, ns, s, pdl, spread));
            // Latency mode: the proj GEMM is folded into the attention kernel (per-head partial products, D / kAttChainW replicas per
            // tile) and reduce_ln adds the heads + bias + residual and applies LN2 — one kernel and one dependency edge less per block.
            // 64-row query tiles (5 per sequence) when that grid still fits one wave: each CTA computes half the exponentials.
            const bool att_q64 = spread && t->att_chain_ok && t->att_q64 && n * t->heads * 5 * (D / kAttChainW) <= kSpreadCtas;
            const bool att_chain = att_q64 || (spread && t->att_chain_ok && n * t->heads * 3 * (D / kAttChainW) <= kSpreadCtas);
            if (t->tc_attention)
                VT_LAUNCH(tc_attention_launch(att_chain ? p.att : t->plan_att, n, t->heads, ns, t->d_tc_err, s, pdl, t->d_trace,
                                              att_q64 ? VT_ATT_CHAIN_Q64 : att_chain ? VT_ATT_CHAIN : (spread ? VT_ATT_DUP : VT_ATT_PLAIN)));
            else
                VT_LAUNCH(launch_attention(t->QKV, nullptr, t->att_hi, LO(t->att_lo), n, D, t->heads, s));
            if (att_chain) {
                ReduceLnArgs r{};
                r.P = t->Pbuf, r.np = t->heads, r.p_stride = (int64_t)t->maxT * kNTok * D, r.bias = b.proj_b, r.add = t->X, r.add_period = 0;
                r.X = t->X, r.M = M, r.D = D, r.period = kNTok, r.x_rows = kNTok, r.x_row_off = 0;
                r.ln_g = b.ln2_g, r.ln_b = b.ln2_b, r.ln_hi = t->ln_hi, r.ln_lo = LO(t->ln_lo), r.ln_rows = kNTok, r.ln_row_off = 0;
                VT_LAUNCH(launch_reduce_ln(r, s, pdl));
            } else {
                VT_LAUNCH(tc_gemm_launch(p.proj, M, ns, s, pdl && t->tc_attention, spread && !tp_mcast, tp_mcast));  // fused: + LN2
            }
            if (!fuse) VT_LAUNCH(launch_layernorm_split(t->X, D, b.ln2_g, b.ln2_b, t->ln_hi, LO(t->ln_lo), M, D, 1 << 30, 0, 0, s, pdl));
            // Chained form (FC2 partial products inside the FC1 kernel, summed by reduce_ln): shortest critical path for a few targets.
            // From kUnchainTargets targets on the 12 fp32 partial planes per row tile cost more than the hidden round trip
            // (cfg4, 16 targets: ViT stage 905 -> 819 us unchained), so FC1 writes the hidden tile and FC2 runs as its own GEMM.
            // ... except in the A-stationary form, where a CTA accumulates the chained product over all of its hidden chunks (3 planes
            // per row tile at 5120 rows, and no hidden round trip at all)
            const bool as_mlp = as_form && t->chain_mlp && t->as_mlp && tc_gemm_as_mlp_supported(p.fc1, ns);
            const bool chain = as_mlp || (t->chain_mlp && n < t->unchain_n);
            int planes = (int)(Hd / 64);
            if (as_mlp) {
                VT_LAUNCH(tc_gemm_as_mlp_launch(p.fc1, M, s, pdl, t->sm_count, &planes, t->fuse_ln ? &p.fc2 : nullptr));
            } else if (chain) {
                VT_LAUNCH(tc_gemm_launch(p.fc1, M, ns, s, pdl, spread));
            } else {
                TcGemmPlan fc1 = p.fc1;
                fc1.args.chain_n = 0, fc1.args.o_mode = 1;
                if (as_form && tc_gemm_as_supported(fc1))
                    VT_LAUNCH(tc_gemm_as_launch(fc1, M, ns, s, pdl, t->sm_count));
                else
                    VT_LAUNCH(tc_gemm_launch(fc1, M, ns, s, pdl));
            }
            if (chain && planes == 0) {
                // (reduced inside the MLP kernel's clusters)
            } else if (chain) {  // X += fc2_b + sum of the partials; LN1 of the next block / the final LN of the search rows
                const bool last = l + 1 == t->depth;
                ReduceLnArgs r{};
                r.P = t->Pbuf, r.np = planes, r.p_stride = (int64_t)t->maxT * kNTok * D, r.bias = b.fc2_b, r.add = t->X, r.add_period = 0;
                r.X = t->X, r.M = M, r.D = D, r.period = kNTok, r.x_rows = kNTok, r.x_row_off = 0;
                r.ln_g = last ? t->lnf_g : t->blk[l + 1].ln1_g, r.ln_b = last ? t->lnf_b : t->blk[l + 1].ln1_b;
                r.ln_hi = last ? t->yf_hi : t->ln_hi, r.ln_lo = LO(last ? t->yf_lo : t->ln_lo);
                r.ln_rows = last ? kNTx : kNTok, r.ln_row_off = last ? -kNTz : 0;
                VT_LAUNCH(launch_reduce_ln(r, s, pdl));
            } else {
                VT_LAUNCH(tc_gemm_launch(p.fc2, M, ns, s, pdl, false, tp_mcast));  // fused: + LN1 of the next block / the final LN of the search rows
            }
            if (t->debug_capture)
                VT_CUDA(cudaMemcpyAsync(t->d_dbg + (size_t)(l + 1) * t->maxT * kNTok * D, t->X, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, s));
        }
        if (!fuse) VT_LAUNCH(launch_layernorm_split(t->X, D, t->lnf_g, t->lnf_b, t->yf_hi, LO(t->yf_lo), n * kNTx, D, kNTx, kNTok, kNTz, s, pdl));
        if (merge_slices) {
            TcGemmPlan ph = t->plan_head;
            ph.args.kb_per_split = 3 * (D / 64), head_np = 3;
            VT_LAUNCH(tc_gemm_launch(ph, n * kNTx, ns, s, pdl));
        } else {
            VT_LAUNCH(tc_gemm_launch(t->plan_head, n * kNTx, ns, s, pdl));
        }
    }
    if (t->nsplit && t->split_k)
        VT_LAUNCH(launch_head_decode(t->Phead, head_np, (int64_t)t->maxT * kNTx * C, C, t->h1_b, t->h2_w, t->h2_b, t->d_hann, t->d_state, t->d_slots, n,
                                     t->threshold, t->d_res, t->d_maps, t->d_cand, t->d_counters, t->d_stamps, s, t->pdl && !t->debug_capture,
                                     t->cfg.decode_window, t->d_tc_err));
    else
        VT_LAUNCH(launch_decode(t->H1, C, t->h2_w, t->h2_b, t->d_hann, t->d_state, t->d_slots, n, t->threshold, t->d_res, t->d_maps, t->d_stamps, s,
                                t->cfg.decode_window));
    if (t->cfg.box_overlay || t->hud_mode)  // box overlay and / or the frame's HUD list, pinned-frame mirror, ... and publishes the result block
        VT_LAUNCH(launch_box_overlay(t->frame_bytes, t->W, t->H, overlay_format(t->fmt), t->d_res, t->d_slots, n, t->cfg.overlay_gate, t->d_ctl,
                                     t->d_stamps + ST_OVL_END, s, t->pdl && !t->debug_capture, t->d_res, t->res_block_bytes,
                                     t->cfg.box_overlay | (getenv("VT_B200_HUD_SKIP") ? atoi(getenv("VT_B200_HUD_SKIP")) << 8 : 0) |
                                         ((t->hud_mode && !getenv("VT_B200_HUD_ONE_CTA")) ? 1 << 16 : 0)));
    else  // results, stage stamps and the error flag -> the pinned host block of this frame's queue slot
        VT_LAUNCH(launch_publish(t->d_res, t->d_ctl, t->res_block_bytes, s, t->pdl && !t->debug_capture));
    return VT_OK;
}

static vt_status run_forward(vt_tracker* t) {
    const int n = (int)t->active.size();
    if (n == 0) return VT_OK;
    int launches = 0;
    const int dev = t->cfg.device;
    const bool spread = t->spread_ok && dev >= 0 && dev < kMaxDevices && registry_total(dev) <= kSpreadMaxHandles;
    if (!t->cfg.use_cuda_graph || t->debug_capture) {
        vt_status st = enqueue_forward(t, n, launches, true, false, spread);
        t->kernel_launches += launches;
        t->kernels_per_frame = launches;
        return st;
    }
    const int key = (n * 2 + (t->frame_valid ? 1 : 0)) * 2 + (spread ? 1 : 0);  // frame_valid is a kernel parameter baked into the graph
    auto it = t->graphs.find(key);
    if (it == t->graphs.end()) {
        cudaGraph_t graph = nullptr;
        VT_CUDA(cudaStreamBeginCapture(t->stream, cudaStreamCaptureModeThreadLocal));
        vt_status st = enqueue_forward(t, n, launches, true, true, spread);
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
static bool search_window(const vt_tracker* t, const vt_bbox& r, int margin_div, int& x0, int& y0, int& x1, int& y1) {
    if (r.width <= 0 || r.height <= 0) return false;
    const int c = (int)ceil(sqrt((double)(int)((long long)r.width * r.height)) * 4.0);
    const int m = margin_div > 0 ? std::max(16, c / margin_div) : 0;
    const long long wx = (long long)r.x + (r.width - c) / 2 - m, wy = (long long)r.y + (r.height - c) / 2 - m, e = (long long)c + 2 * m;
    x0 = (int)std::max(wx, 0LL) & ~1, y0 = (int)std::max(wy, 0LL) & ~1;
    x1 = (int)std::min((std::min(wx + e, (long long)t->W) + 1) & ~1LL, (long long)t->W);
    y1 = (int)std::min((std::min(wy + e, (long long)t->H) + 1) & ~1LL, (long long)t->H);
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
static void plan_upload(vt_tracker* t, size_t len, bool pinned_host, bool lagging, const int* rmw, UploadPlan& p) {
    p = UploadPlan();
    const bool valid = (t->fmt == VT_FMT_NV12) ? (len >= (size_t)t->W * t->H * 3 / 2) : (len >= t->frame_bytes);
    if (!t->cfg.upload_window || !pinned_host || !valid || len < t->frame_bytes || (int)t->active.size() > kMaxWin || (t->W % 2) ||
        ((t->H % 2) && t->fmt == VT_FMT_NV12) || (t->active.empty() && !t->hud_mode))
        return;
    const size_t bpp2 = t->fmt == VT_FMT_NV12 ? 3 : (t->fmt == VT_FMT_GRAY8 ? 2 : 6);  // bytes per pixel x 2
    size_t bytes = 0;
    int k = 0;
    for (int s : t->active) {
        int* w = p.win[k++];
        if (!search_window(t, t->rect_mirror[s], lagging ? 8 : 0, w[0], w[1], w[2], w[3])) {
            w[0] = w[1] = w[2] = w[3] = 0;  // the window misses the frame: the crop kernel flags it; nothing to read
            continue;
        }
        if (t->win_shrink > 0 && w[2] - w[0] > 4 * t->win_shrink && w[3] - w[1] > 4 * t->win_shrink)
            w[0] += t->win_shrink, w[1] += t->win_shrink, w[2] -= t->win_shrink, w[3] -= t->win_shrink;
        bytes += (size_t)(w[2] - w[0]) * (w[3] - w[1]) * bpp2 / 2;
    }
    if (rmw && rmw[2] > rmw[0] && rmw[3] > rmw[1] && format_is_luma(t->fmt)) {
        p.has_rmw = true;
        p.rmw[0] = std::max(rmw[0], 0), p.rmw[1] = std::max(rmw[1], 0), p.rmw[2] = std::min(rmw[2], t->W), p.rmw[3] = std::min(rmw[3], t->H);
        if (p.rmw[2] > p.rmw[0] && p.rmw[3] > p.rmw[1]) bytes += (size_t)(p.rmw[2] - p.rmw[0]) * (p.rmw[3] - p.rmw[1]);
        else p.has_rmw = false;
    }
    if (bytes * 2 > t->frame_bytes) return;  // not worth the extra copies
    p.whole = false, p.n_win = k, p.bytes = bytes;
}

static vt_status do_upload(vt_tracker* t, const uint8_t* frame, size_t len, const UploadPlan& p, bool device_src, cudaStream_t stream) {
    if (!stream) stream = t->stream;
    size_t n = std::min(len, t->frame_bytes);
    t->frame_valid = (t->fmt == VT_FMT_NV12) ? (len >= (size_t)t->W * t->H * 3 / 2) : (len >= t->frame_bytes);
    if (!t->frame_valid && t->fmt == VT_FMT_NV12) n = 0;  // src/nv12_convert.rs:48-50 -> black image
    if (n == 0) return VT_OK;
    const cudaMemcpyKind kind = device_src ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (!p.whole) {
        const size_t W = (size_t)t->W;
        for (int i = 0; i < p.n_win; ++i) {
            const int* w = p.win[i];
            const size_t cols = (size_t)(w[2] - w[0]), rows = (size_t)(w[3] - w[1]);
            if (!cols || !rows) continue;
            if (t->fmt == VT_FMT_GRAY8) {
                const size_t o = (size_t)w[1] * W + w[0];
                VT_CUDA(cudaMemcpy2DAsync(t->d_frame + o, W, frame + o, W, cols, rows, kind, stream));
            } else if (t->fmt == VT_FMT_NV12) {
                const size_t yo = (size_t)w[1] * W + w[0], uvo = W * t->H + (size_t)(w[1] / 2) * W + w[0];
                VT_CUDA(cudaMemcpy2DAsync(t->d_frame + yo, W, frame + yo, W, cols, rows, kind, stream));
                VT_CUDA(cudaMemcpy2DAsync(t->d_frame + uvo, W, frame + uvo, W, cols, rows / 2, kind, stream));
            } else {
                const size_t pitch = W * 3, o = (size_t)w[1] * pitch + (size_t)w[0] * 3;
                VT_CUDA(cudaMemcpy2DAsync(t->d_frame + o, pitch, frame + o, pitch, cols * 3, rows, kind, stream));
            }
        }
        if (p.has_rmw) {  // luma plane only (the NV12 / GRAY8 background dim reads and writes Y)
            const size_t o = (size_t)p.rmw[1] * W + p.rmw[0];
            VT_CUDA(cudaMemcpy2DAsync(t->d_frame + o, W, frame + o, W, (size_t)(p.rmw[2] - p.rmw[0]), (size_t)(p.rmw[3] - p.rmw[1]), kind, stream));
        }
        if (!device_src) t->h2d_bytes += p.bytes;
        t->d_frame_is_last_host_frame = false;  // only windows of the frame are on the device
        return VT_OK;
    }
    const bool pinned = device_src || is_pinned(frame);
    t->d_frame_is_last_host_frame = !device_src && n >= t->frame_bytes;
    if (!device_src) t->h2d_bytes += n;
    if (pinned) {
        VT_CUDA(cudaMemcpyAsync(t->d_frame, frame, n, kind, stream));
    } else {
        memcpy(t->h_stage, frame, n);
        VT_CUDA(cudaMemcpyAsync(t->d_frame, t->h_stage, n, cudaMemcpyHostToDevice, stream));
    }
    return VT_OK;
}

// whole-frame upload (init, and the callers outside the per-frame path)
vt_status upload_frame(vt_tracker* t, const uint8_t* frame, size_t len, bool allow_window, bool device_src, cudaStream_t stream) {
    (void)allow_window;
    return do_upload(t, frame, len, UploadPlan(), device_src, stream);
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

// device -> host copy of whole rows [r0, r1] of the drawable plane (Y plane for NV12, the image for RGB24)
vt_status download_rows(vt_tracker* t, uint8_t* frame, size_t len, const std::vector<std::pair<int, int>>& spans, bool* staged) {
    const size_t pitch = (size_t)t->W * (format_is_luma(t->fmt) ? 1 : 3);
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
    const size_t pitch = (size_t)t->W * (format_is_luma(t->fmt) ? 1 : 3);
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
    if (getenv("VT_B200_STAMPDBG") && ovl) {  // diagnostics: overlay kernel prologue end / dependency satisfied / end, relative to the decode end
        static double acc[3] = {0, 0, 0};
        static int cnt = 0;
        acc[0] += (double)((long long)st[6] - (long long)st[ST_DEC_END]), acc[1] += (double)((long long)st[7] - (long long)st[ST_DEC_END]);
        acc[2] += (double)((long long)st[ST_OVL_END] - (long long)st[ST_DEC_END]);
        if (++cnt % 50 == 0) fprintf(stderr, "[vt stampdbg] overlay vs decode end: prologue done %+.2f us, dependency satisfied %+.2f us, end %+.2f us\n",
                                     acc[0] / cnt * 1e-3, acc[1] / cnt * 1e-3, acc[2] / cnt * 1e-3);
    }
    memcpy(t->last, ms, sizeof(ms));
    t->r_h2d.push(ms[0]), t->r_pre.push(ms[1]), t->r_vit.push(ms[2]), t->r_dec.push(ms[3]), t->r_ovl.push(ms[4]), t->r_d2h.push(ms[5]),
        t->r_tot.push(ms[6]);
}

static inline double now_us() {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static vt_status submit_common(vt_tracker* t, uint8_t* frame, const uint8_t* d_src, size_t len, bool forward = true) {
    if (t->q_count >= vt_tracker::kQueue) {
        set_error("%d frames are already in flight on this handle", t->q_count);
        return VT_ERR_INVALID;
    }
    const bool pinned = d_src || is_pinned(frame);
    if (t->q_count > 0 && (!pinned || t->q[t->q_head].pageable)) {
        set_error("pageable host frames are staged through one buffer and cannot be pipelined: wait() first or use pinned frames");
        return VT_ERR_INVALID;
    }
    const double hp0 = t->hostprof ? now_us() : 0;
    const int slot = (t->q_head + t->q_count) % vt_tracker::kQueue;
    vt_tracker::Slot& q = t->q[slot];
    q.t_submit = std::chrono::steady_clock::now();
    q.frame = d_src ? nullptr : frame, q.len = len, q.pageable = !pinned;
    // the caller's pinned frame is device-mapped under UVA: zero-copy target of the overlay mirror, fall-back source of the crop kernel
    uint8_t* const host_frame = (frame && !d_src && pinned && len >= t->frame_bytes) ? frame : nullptr;
    // this frame's HUD list (staged by tracker_set_hud in this slot's pinned block)
    const int n_hud = t->hud_mode ? t->hud_next_n : 0;
    q.hud_bytes = n_hud ? t->hud_next_bytes : 0;
    q.mirrored = host_frame && (t->cfg.box_overlay || n_hud > 0);
    // device-resident frame: track (and draw the box) straight in the caller's device memory — no device->device copy
    const bool in_place = d_src && len >= t->frame_bytes;
    if (!in_place) t->d_frame = t->d_frames[slot];  // the slot's own frame buffer: the other one may still be read by the frame in flight
    const bool lagging = t->q_count > 0;  // a frame is in flight: rect_mirror is one frame old, the windows are predictions
    UploadPlan plan;
    // (the region a HUD list dims is read by the overlay kernel straight from the pinned host frame: it needs no upload of its own)
    static const bool bg_from_host = getenv("VT_B200_HUD_BG_FROM_HOST") != nullptr;  // (measured slower: profiles/r2_final.md)
    if (!in_place && !d_src)
        plan_upload(t, len, host_frame != nullptr, lagging, (n_hud && !(bg_from_host && host_frame && t->hud_next_bg_leads)) ? t->hud_next_rmw : nullptr, plan);
    if (!in_place && !d_src && lagging) {
        // pipelined host frame: upload on the copy stream while the frame in flight computes; the main stream picks it up through an event
        vt_status st = do_upload(t, frame, len, plan, false, t->copy_stream);
        if (st != VT_OK) return st;
        VT_CUDA(cudaEventRecord(t->ev_up[slot], t->copy_stream));
        VT_CUDA(cudaStreamWaitEvent(t->stream, t->ev_up[slot], 0));
    }
    FrameCtl ctl;
    memset(&ctl, 0, sizeof(ctl));
    ctl.frame = in_place ? d_src : t->d_frame, ctl.host_frame = host_frame, ctl.hblk = reinterpret_cast<uint32_t*>(t->h_blk[slot]);
    ctl.hud = n_hud ? t->h_hud[slot] : nullptr, ctl.n_hud = n_hud;
    const bool hud_inline = n_hud > 0 && n_hud <= kHudInline && t->d_hud[slot] != nullptr;
    if (hud_inline) ctl.hud = t->d_hud[slot];
    ctl.n_win = plan.whole ? -1 : plan.n_win;
    if (!plan.whole) memcpy(ctl.win, plan.win, sizeof(ctl.win));
    ctl.bg_on_device = (n_hud && (in_place || d_src || plan.whole || plan.has_rmw)) ? 1 : 0;  // the dimmed region is in the device frame
    t->hud_next_n = 0;
    VT_CUDA(launch_stamp(t->d_stamps + ST_SUBMIT, t->d_ctl, ctl, t->stream, hud_inline ? t->h_hud[slot] : nullptr, n_hud, t->d_hud[slot]));
    ++t->kernel_launches;
    if (in_place) {
        t->frame_valid = 1;
        t->d_frame_is_last_host_frame = false;  // tracked in the caller's device memory: the internal buffer holds an older frame
    } else if (d_src) {  // short device frame: device->device copy of what there is (NV12: black frame, src/nv12_convert.rs:48-50)
        vt_status st = do_upload(t, d_src, len, plan, true, nullptr);
        if (st != VT_OK) return st;
    } else if (!lagging) {
        vt_status st = do_upload(t, frame, len, plan, false, nullptr);  // the host mirror of rect_last is exact: the search windows suffice
        if (st != VT_OK) return st;
    }
    const double hp1 = t->hostprof ? now_us() : 0;
    const bool ran = forward && !t->active.empty();
    if (ran) {
        vt_status st = run_forward(t);
        if (st != VT_OK) return st;
    } else if (n_hud > 0) {  // no tracker runs on this frame (SELECT / LOST states of the probe): HUD list + publish only
        cudaError_t e = launch_box_overlay(t->frame_bytes, t->W, t->H, overlay_format(t->fmt), t->d_res, t->d_slots, 0, t->cfg.overlay_gate, t->d_ctl,
                                           t->d_stamps + ST_OVL_END, t->stream, false, t->d_res, t->res_block_bytes, 0);
        if (e != cudaSuccess) {
            set_error("overlay launch failed: %s", cudaGetErrorString(e));
            return VT_ERR_CUDA;
        }
        ++t->kernel_launches;
    }
    const double hp2 = t->hostprof ? now_us() : 0;
    // the result block reaches t->h_blk[slot] through the last kernel of the frame; nothing ran: copy it
    if (!ran && n_hud == 0) VT_CUDA(cudaMemcpyAsync(t->h_blk[slot], t->d_res, t->res_block_bytes, cudaMemcpyDeviceToHost, t->stream));
    VT_CUDA(cudaEventRecord(t->q_done[slot], t->stream));
    t->d2h_bytes += t->res_block_bytes;
    if (t->hostprof) t->hp[0] += hp1 - hp0, t->hp[1] += hp2 - hp1, t->hp[2] += now_us() - hp2;
    ++t->q_count;
    t->in_flight = true;
    return VT_OK;
}

// Stream group: the n active targets of the handle are n independent video streams (one target each, same geometry), stepped together
// through ONE batched forward (M = 320 n rows: from 1024 rows on the GEMMs run in their throughput forms).  frames[i] is the pinned
// host frame of the i-th active target; each target's search window is uploaded into that target's own device frame and the box overlay
// is mirrored into that target's host frame.  Synchronous (rect_mirror is exact: the windows are the real search windows).
static vt_status submit_streams(vt_tracker* t, uint8_t* const* frames, const size_t* lens, int n) {
    if (t->q_count > 0 || t->hud_mode) {
        set_error("vt_tracker_update_streams: frames are in flight on this handle, or it is a probe (HUD) handle");
        return VT_ERR_INVALID;
    }
    if (n != (int)t->active.size() || n <= 0 || n > kMaxWin) {
        set_error("vt_tracker_update_streams: %d frames for %d active targets (one frame per active target, at most %d)", n, (int)t->active.size(), kMaxWin);
        return VT_ERR_INVALID;
    }
    for (int i = 0; i < n; ++i)
        if (!frames[i] || lens[i] < t->frame_bytes || !is_pinned(frames[i])) {
            set_error("vt_tracker_update_streams: frame %d must be a full frame in pinned host memory (vt_alloc_pinned)", i);
            return VT_ERR_INVALID;
        }
    const int slot = t->q_head;
    vt_tracker::Slot& q = t->q[slot];
    q.t_submit = std::chrono::steady_clock::now();
    q.frame = frames[0], q.len = lens[0], q.pageable = false, q.hud_bytes = 0, q.mirrored = true;
    FrameCtl ctl;
    memset(&ctl, 0, sizeof(ctl));
    const bool windows = t->cfg.upload_window && !(t->W % 2) && !((t->H % 2) && t->fmt == VT_FMT_NV12);
    const size_t W = (size_t)t->W;
    for (int i = 0; i < n; ++i) {
        if (!t->d_sframes[i]) {
            VT_CUDA(cudaMalloc(&t->d_sframes[i], t->frame_bytes + 256));
            VT_CUDA(cudaMemsetAsync(t->d_sframes[i], 0, t->frame_bytes + 256, t->stream));
        }
        uint8_t* dst = t->d_sframes[i];
        const uint8_t* src = frames[i];
        int* w = ctl.win[i];
        if (!windows) {
            VT_CUDA(cudaMemcpyAsync(dst, src, t->frame_bytes, cudaMemcpyHostToDevice, t->stream));
            t->h2d_bytes += t->frame_bytes;
            w[0] = w[1] = 0, w[2] = t->W, w[3] = t->H;
        } else if (search_window(t, t->rect_mirror[t->active[i]], 0, w[0], w[1], w[2], w[3])) {
            const size_t cols = (size_t)(w[2] - w[0]), rows = (size_t)(w[3] - w[1]);
            if (t->fmt == VT_FMT_GRAY8) {
                const size_t o = (size_t)w[1] * W + w[0];
                VT_CUDA(cudaMemcpy2DAsync(dst + o, W, src + o, W, cols, rows, cudaMemcpyHostToDevice, t->stream));
                t->h2d_bytes += cols * rows;
            } else if (t->fmt == VT_FMT_NV12) {
                const size_t yo = (size_t)w[1] * W + w[0], uvo = W * t->H + (size_t)(w[1] / 2) * W + w[0];
                VT_CUDA(cudaMemcpy2DAsync(dst + yo, W, src + yo, W, cols, rows, cudaMemcpyHostToDevice, t->stream));
                VT_CUDA(cudaMemcpy2DAsync(dst + uvo, W, src + uvo, W, cols, rows / 2, cudaMemcpyHostToDevice, t->stream));
                t->h2d_bytes += cols * rows * 3 / 2;
            } else {
                const size_t pitch = W * 3, o = (size_t)w[1] * pitch + (size_t)w[0] * 3;
                VT_CUDA(cudaMemcpy2DAsync(dst + o, pitch, src + o, pitch, cols * 3, rows, cudaMemcpyHostToDevice, t->stream));
                t->h2d_bytes += cols * rows * 3;
            }
        } else {
            w[0] = w[1] = w[2] = w[3] = 0;  // the window misses the frame: the crop kernel flags it
        }
        ctl.frames[i] = dst, ctl.host_frames[i] = frames[i];
    }
    ctl.frame = t->d_sframes[0], ctl.host_frame = frames[0], ctl.hblk = reinterpret_cast<uint32_t*>(t->h_blk[slot]);
    ctl.n_win = n;
    t->frame_valid = 1, t->d_frame_is_last_host_frame = false;
    VT_CUDA(launch_stamp(t->d_stamps + ST_SUBMIT, t->d_ctl, ctl, t->stream));
    ++t->kernel_launches;
    vt_status st = run_forward(t);
    if (st != VT_OK) return st;
    VT_CUDA(cudaEventRecord(t->q_done[slot], t->stream));
    t->d2h_bytes += t->res_block_bytes;
    ++t->q_count;
    t->in_flight = true;
    return VT_OK;
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
    const double hp0 = t->hostprof ? now_us() : 0;
    VT_CUDA(cudaEventSynchronize(t->q_done[slot]));
    bind_slot(t, slot);
    const double hp1 = t->hostprof ? now_us() : 0;
    if (*t->h_tc_err) {  // travels with the results; reset on the device for the next frame
        cudaMemsetAsync(t->d_tc_err, 0, sizeof(int), t->stream);
        *t->h_tc_err = 0;
        set_error("tcgen05 path: a bounded mbarrier wait expired (pipeline protocol error)");
        return VT_ERR_CUDA;
    }
    fill_results(t, results);
    const double hp2 = t->hostprof ? now_us() : 0;
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
    const double hp3 = t->hostprof ? now_us() : 0;
    collect_timing(t);
    ++t->frames;
    if (t->hostprof) t->hp[3] += hp1 - hp0, t->hp[4] += hp2 - hp1, t->hp[5] += hp3 - hp2, t->hp[6] += now_us() - hp3, ++t->hp_n;
    return VT_OK;
}

// ---- ring replay support ----------------------------------------------------------------------------------------------------------
// [x0, x1) x [y0, y1) of the drawable plane (Y plane / luma for NV12 and GRAY8, the RGB image otherwise), clipped to the frame
void restore_rect_region(uint8_t* frame, const uint8_t* clean, int fmt, int W, int H, long long x0, long long y0, long long x1, long long y1) {
    x0 = std::max(x0, 0LL), y0 = std::max(y0, 0LL), x1 = std::min<long long>(x1, W), y1 = std::min<long long>(y1, H);
    if (x1 <= x0 || y1 <= y0) return;
    const size_t bpp = format_is_luma(fmt) ? 1 : 3, pitch = (size_t)W * bpp;
    for (long long y = y0; y < y1; ++y) {
        const size_t o = (size_t)y * pitch + (size_t)x0 * bpp;
        memcpy(frame + o, clean + o, (size_t)(x1 - x0) * bpp);
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

// Stages the HUD list of the NEXT submit in the pinned block of the queue slot that submit will use.
vt_status tracker_set_hud(vt_tracker* t, const HudCmd* cmds, int n) {
    if (!t || !t->hud_mode || n < 0 || n > kMaxCmds || (n > 0 && !cmds)) {
        set_error("tracker_set_hud: invalid argument (HUD mode %d, %d commands)", t ? (int)t->hud_mode : -1, n);
        return VT_ERR_INVALID;
    }
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const int slot = (t->q_head + t->q_count) % vt_tracker::kQueue;
    if (!t->h_hud[slot]) VT_CUDA(cudaHostAlloc(&t->h_hud[slot], sizeof(OverlayCmdDev) * kMaxCmds, cudaHostAllocDefault));
    if (!t->d_hud[slot]) VT_CUDA(cudaMalloc(&t->d_hud[slot], sizeof(OverlayCmdDev) * kHudInline));
    int rmw[4] = {0, 0, 0, 0};
    size_t bytes = 0;
    for (int i = 0; i < n; ++i) {
        OverlayCmdDev& d = t->h_hud[slot][i];
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
        if (c.kind == VT_OV_BACKGROUND && format_is_luma(t->fmt) && c.x >= 0 && c.y >= 0 && c.w > 0 && c.h > 0) {
            // the luma background dim reads before it writes (src/nv12_convert.rs:324-343): that region must be on the device
            const int x1 = (int)std::min<long long>((long long)c.x + c.w, t->W), y1 = (int)std::min<long long>((long long)c.y + c.h, t->H);
            if (rmw[2] <= rmw[0]) rmw[0] = c.x, rmw[1] = c.y, rmw[2] = x1, rmw[3] = y1;
            else rmw[0] = std::min(rmw[0], c.x), rmw[1] = std::min(rmw[1], c.y), rmw[2] = std::max(rmw[2], x1), rmw[3] = std::max(rmw[3], y1);
            bytes += (size_t)std::max(0, x1 - c.x) * std::max(0, y1 - c.y);
        } else if (c.kind == VT_OV_TEXT) {
            bytes += (size_t)35 * std::max(c.a, 0) * std::max(c.a, 0) * d.nchar;
        } else {
            bytes += 1024;  // rect / crosshair / cursor / selection outlines
        }
    }
    int n_bg = 0;
    for (int i = 0; i < n; ++i) n_bg += cmds[i].cmd.kind == VT_OV_BACKGROUND;
    t->hud_next_bg_leads = n_bg == 1 && cmds[0].cmd.kind == VT_OV_BACKGROUND && cmds[0].cond == VT_HUD_ALWAYS;
    t->hud_next_n = n, t->hud_next_bytes = bytes;
    memcpy(t->hud_next_rmw, rmw, sizeof(rmw));
    return VT_OK;
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
    VT_CUDA(cudaSetDevice(t->cfg.device));
    // the template window must intersect the frame (cv2 raises an ROI assertion otherwise, App. A.1)
    {
        if (box.width <= 0 || box.height <= 0) {
            set_error("vt_tracker_init: empty box");
            return VT_ERR_CROP_OUTSIDE;
        }
        const int c = (int)ceil(sqrt((double)((long long)box.width * box.height)) * 2.0);
        const int x1 = box.x + (box.width - c) / 2, y1 = box.y + (box.height - c) / 2;
        const int pp = t->cfg.pad_plus1;
        const int pl = std::max(0, -x1), pt = std::max(0, -y1), pr = std::max(x1 + c - t->W + pp, 0), pb = std::max(y1 + c - t->H + pp, 0);
        if (c - pl - pr <= 0 || c - pt - pb <= 0) {
            set_error("vt_tracker_init: template window lies outside the frame");
            return VT_ERR_CROP_OUTSIDE;
        }
    }
    vt_status st = upload_frame(t, frame, len);
    if (st != VT_OK) return st;
    TargetState hs;
    memset(&hs, 0, sizeof(hs));
    hs.rect[0] = box.x, hs.rect[1] = box.y, hs.rect[2] = box.width, hs.rect[3] = box.height, hs.active = 1;
    int32_t slot = target;
    VT_CUDA(cudaMemcpyAsync(t->d_state + target, &hs, sizeof(hs), cudaMemcpyHostToDevice, t->stream));
    // d_slots is reused as a one-element list for the template pass, then restored
    VT_CUDA(cudaMemcpyAsync(t->d_slots, &slot, sizeof(slot), cudaMemcpyHostToDevice, t->stream));
    FrameDesc fd{t->d_frame, t->W, t->H, t->fmt, t->frame_valid, nullptr, t->cfg.pad_plus1};
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
}  // namespace vt
extern "C" {

vt_status vt_tracker_submit_device(vt_tracker* t, uint8_t* d_frame, size_t len) {
    if (!t || !d_frame) return VT_ERR_INVALID;
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
    VT_CUDA(cudaSetDevice(t->cfg.device));
    if (t->q_count) {
        set_error("vt_tracker_update: frames are in flight (submit/wait); drain them first");
        return VT_ERR_INVALID;
    }
    vt_status st = submit_common(t, frame, nullptr, len);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

vt_status vt_tracker_update_streams(vt_tracker* t, uint8_t* const* frames, const size_t* lens, int32_t n, vt_result* results) {
    if (!t || !frames || !lens) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    vt_status st = submit_streams(t, frames, lens, n);
    if (st != VT_OK) return st;
    return wait_common(t, results);
}

vt_status vt_tracker_update_device(vt_tracker* t, uint8_t* d_frame, size_t len, vt_result* results) {
    if (!t || !d_frame) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    if (t->q_count) {
        set_error("vt_tracker_update_device: frames are in flight (submit/wait); drain them first");
        return VT_ERR_INVALID;
    }
    vt_status st = submit_common(t, nullptr, d_frame, len);
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
    VT_CUDA(cudaSetDevice(t->cfg.device));
    std::vector<vt_result> res((size_t)t->maxT);
    uint8_t* fr[kMaxWin];
    size_t lens[kMaxWin];
    vt_status st = VT_OK;
    for (int i = 0; i < n && st == VT_OK; ++i) {
        const size_t off = (size_t)((first + i) % ring) * stride;
        for (int k = 0; k < n_streams; ++k) fr[k] = rings[k] + off, lens[k] = frame_len;
        const auto t0 = std::chrono::steady_clock::now();
        st = submit_streams(t, fr, lens, n_streams);
        if (st == VT_OK) st = wait_common(t, res.data());
        if (latency_us) latency_us[i] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
        if (st == VT_OK && pristine && t->cfg.box_overlay)  // undo what the box overlays drew: the rings are replayed on clean frames
            for (int k = 0; k < n_streams && k < (int)t->active.size(); ++k) {
                const vt_result& r = res[t->active[k]];
                if (pristine[k] && r.status == VT_OK && r.success && r.score > t->cfg.overlay_gate)
                    restore_box_region(fr[k], pristine[k] + off, t->fmt, t->W, t->H, r.bbox);
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
