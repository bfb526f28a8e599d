// tracker_abi.cu — the entry points of include/vt_tracker.h around the per-frame path: diagnostics read-backs, the NV12 -> RGB
// parity / bench entry, the format steps either side of the RGB probe, explicit overlay commands and TimingStats.
#include "tracker_state.h"

using namespace vt;

extern "C" {

// patch-major [tokens][768] -> planar CHW blob
static void patches_to_chw(const std::vector<float>& p, int size, float* chw) {
    const int nt = size / 16;
    for (int tok = 0; tok < nt * nt; ++tok)
        for (int c = 0; c < 3; ++c)
            for (int py = 0; py < 16; ++py)
                for (int px = 0; px < 16; ++px)
                    chw[(size_t)c * size * size + (size_t)((tok / nt) * 16 + py) * size + (tok % nt) * 16 + px] =
                        p[(size_t)tok * kPatchK + c * 256 + py * 16 + px];
}

vt_status vt_tracker_debug_read(vt_tracker* t, int32_t target, float* search_blob, float* template_blob, float* conf_win, float* size_map,
                                float* off_map, float* tokens) {
    if (!t || target < 0 || target >= t->maxT || t->in_flight) return VT_ERR_INVALID;
    if (!t->inited[target]) return VT_ERR_NOT_INIT;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    const int bi = (int)(std::find(t->active.begin(), t->active.end(), target) - t->active.begin());
    if (search_blob) {
        std::vector<float> p((size_t)kNTx * kPatchK);
        VT_CUDA(cudaMemcpy(p.data(), t->patches_x + (size_t)bi * kNTx * kPatchK, p.size() * sizeof(float), cudaMemcpyDeviceToHost));
        patches_to_chw(p, kSearch, search_blob);
    }
    if (template_blob) {  // patches_z holds the most recently initialised template
        std::vector<float> p((size_t)kNTz * kPatchK);
        VT_CUDA(cudaMemcpy(p.data(), t->patches_z, p.size() * sizeof(float), cudaMemcpyDeviceToHost));
        patches_to_chw(p, kTemplate, template_blob);
    }
    if (conf_win || size_map || off_map) {
        float m[1280];
        VT_CUDA(cudaMemcpy(m, t->d_maps + (size_t)target * 1280, sizeof(m), cudaMemcpyDeviceToHost));
        if (conf_win) memcpy(conf_win, m, 256 * sizeof(float));
        if (size_map) memcpy(size_map, m + 256, 512 * sizeof(float));
        if (off_map) memcpy(off_map, m + 768, 512 * sizeof(float));
    }
    if (tokens) {  // final-LN search-token features [256, D] placed at rows 64..319; template rows zero
        memset(tokens, 0, sizeof(float) * kNTok * t->D);
        if (t->nsplit) {  // the tensor-core path keeps only the bf16 split of the final LN: recompute the fp32 copy from X
            VT_CUDA(launch_layernorm(t->X, t->D, t->lnf_g, t->lnf_b, t->Yf, t->D, (int)t->active.size() * kNTx, t->D, kNTx, kNTok, kNTz, t->stream));
            VT_CUDA(cudaStreamSynchronize(t->stream));
        }
        VT_CUDA(cudaMemcpy(tokens + (size_t)kNTz * t->D, t->Yf + (size_t)bi * kNTx * t->D, sizeof(float) * kNTx * t->D, cudaMemcpyDeviceToHost));
    }
    return VT_OK;
}

// Device timeline of the kernels launched since the last call (VT_B200_TRACE=1 at create): out[8 i ..] = {kernel id, t_entry,
// t_after_pdl_wait, t_end, 4 kernel-specific marks} in ns; returns the number of records (<= max_records) through *n and resets the counter.
vt_status vt_tracker_debug_trace(vt_tracker* t, unsigned long long* out, int32_t max_records, int32_t* n) {
    if (!t || !out || !n || !t->d_trace) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    unsigned long long cnt = 0;
    VT_CUDA(cudaMemcpy(&cnt, t->d_trace, 8, cudaMemcpyDeviceToHost));
    const int32_t k = (int32_t)std::min<unsigned long long>(std::min<unsigned long long>(cnt, 2048), (unsigned long long)std::max(max_records, 0));
    if (k > 0) VT_CUDA(cudaMemcpy(out, t->d_trace + 1, (size_t)k * 64, cudaMemcpyDeviceToHost));
    VT_CUDA(cudaMemset(t->d_trace, 0, 8));
    *n = k;
    return VT_OK;
}

// which: 0 embeddings, 1..depth block outputs (needs cfg.debug_capture = 1)
vt_status vt_tracker_debug_tokens(vt_tracker* t, int32_t target, int32_t which, float* out) {
    if (!t || !out || target < 0 || target >= t->maxT || !t->debug_capture || which < 0 || which > t->depth) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    const int bi = (int)(std::find(t->active.begin(), t->active.end(), target) - t->active.begin());
    VT_CUDA(cudaMemcpy(out, t->d_dbg + ((size_t)which * t->maxT + bi) * kNTok * t->D, sizeof(float) * kNTok * t->D, cudaMemcpyDeviceToHost));
    return VT_OK;
}

// ---- NV12 -> RGB -------------------------------------------------------------------------------
vt_status vt_convert_nv12_rgb(vt_tracker* t, const uint8_t* nv12, size_t len, uint8_t* rgb_out) {
    if (!t || !nv12 || !rgb_out || t->in_flight) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const size_t W = t->W, H = t->H, out_bytes = W * H * 3;
    if (t->fmt != VT_FMT_NV12) {
        set_error("vt_convert_nv12_rgb: the handle was not created for NV12 frames");
        return VT_ERR_INVALID;
    }
    if (len < W * H * 3 / 2) {  // src/nv12_convert.rs:48-50
        memset(rgb_out, 0, out_bytes);
        return VT_OK;
    }
    t->d_frame_is_last_host_frame = false;  // the frame buffer is reused as the conversion's input
    if (!t->d_rgb) VT_CUDA(cudaMalloc(&t->d_rgb, out_bytes + 256));
    const size_t n = std::min(len, t->frame_bytes);
    const bool pin_in = is_pinned(nv12), pin_out = is_pinned(rgb_out);
    if (!pin_in) memcpy(t->h_stage, nv12, n);
    VT_CUDA(cudaMemcpyAsync(t->d_frame, pin_in ? nv12 : t->h_stage, n, cudaMemcpyHostToDevice, t->stream));
    cudaError_t e = launch_nv12_to_rgb(t->d_frame, t->frame_bytes, t->d_rgb, out_bytes, t->W, t->H, 1, t->stream);
    if (e != cudaSuccess) {
        set_error("nv12_to_rgb launch failed: %s", cudaGetErrorString(e));
        return VT_ERR_CUDA;
    }
    ++t->kernel_launches;
    if (pin_out) {
        VT_CUDA(cudaMemcpyAsync(rgb_out, t->d_rgb, out_bytes, cudaMemcpyDeviceToHost, t->stream));
        VT_CUDA(cudaStreamSynchronize(t->stream));
    } else {
        VT_CUDA(cudaStreamSynchronize(t->stream));
        VT_CUDA(cudaMemcpy(rgb_out, t->d_rgb, out_bytes, cudaMemcpyDeviceToHost));
    }
    return VT_OK;
}

vt_status vt_convert_nv12_rgb_device(vt_tracker* t, const uint8_t* d_nv12, size_t stride_in, uint8_t* d_rgb, size_t stride_out,
                                     int32_t n_frames) {
    if (!t || !d_nv12 || !d_rgb || n_frames <= 0) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    cudaError_t e = launch_nv12_to_rgb(d_nv12, stride_in, d_rgb, stride_out, t->W, t->H, n_frames, t->stream);
    if (e != cudaSuccess) {
        set_error("nv12_to_rgb launch failed: %s", cudaGetErrorString(e));
        return VT_ERR_CUDA;
    }
    ++t->kernel_launches;
    return VT_OK;
}

// ---- format steps either side of the RGB probe (SURVEY.md §8(f) row 1) ---------------------------------------------------------------
static vt_status fmt_scratch(vt_tracker* t, size_t in_bytes, size_t out_bytes) {
    if (in_bytes > t->fmt_in_cap) {
        if (t->d_fmt_in) cudaFree(t->d_fmt_in);
        t->d_fmt_in = nullptr, t->fmt_in_cap = 0;
        VT_CUDA(cudaMalloc(&t->d_fmt_in, in_bytes + 256));
        t->fmt_in_cap = in_bytes;
    }
    if (out_bytes > t->fmt_out_cap) {
        if (t->d_fmt_out) cudaFree(t->d_fmt_out);
        t->d_fmt_out = nullptr, t->fmt_out_cap = 0;
        VT_CUDA(cudaMalloc(&t->d_fmt_out, out_bytes + 256));
        t->fmt_out_cap = out_bytes;
    }
    return VT_OK;
}

vt_status vt_convert_yuy2_rgb_device(vt_tracker* t, const uint8_t* d_yuy2, size_t stride_in, uint8_t* d_rgb, size_t stride_out, int32_t width,
                                     int32_t height, int32_t n_frames) {
    if (!t || !d_yuy2 || !d_rgb || width <= 0 || height <= 0 || n_frames <= 0) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    VT_CUDA(launch_yuy2_to_rgb(d_yuy2, stride_in, d_rgb, stride_out, width, height, n_frames, t->stream));
    ++t->kernel_launches;
    return VT_OK;
}

vt_status vt_convert_yuy2_rgb(vt_tracker* t, const uint8_t* yuy2, size_t len, int32_t width, int32_t height, uint8_t* rgb_out) {
    if (!t || !yuy2 || !rgb_out || width <= 0 || height <= 0 || t->in_flight) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const size_t in_bytes = (((size_t)width * 2 + 3) & ~(size_t)3) * height, out_bytes = (size_t)width * height * 3;
    if (len < in_bytes) {  // short buffer -> black frame, as the NV12 path (src/nv12_convert.rs:48-50)
        memset(rgb_out, 0, out_bytes);
        return VT_OK;
    }
    vt_status st = fmt_scratch(t, in_bytes, out_bytes);
    if (st != VT_OK) return st;
    VT_CUDA(cudaMemcpyAsync(t->d_fmt_in, yuy2, in_bytes, cudaMemcpyHostToDevice, t->stream));
    VT_CUDA(launch_yuy2_to_rgb(t->d_fmt_in, in_bytes, t->d_fmt_out, out_bytes, width, height, 1, t->stream));
    ++t->kernel_launches;
    VT_CUDA(cudaMemcpyAsync(rgb_out, t->d_fmt_out, out_bytes, cudaMemcpyDeviceToHost, t->stream));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    t->h2d_bytes += in_bytes, t->d2h_bytes += out_bytes;
    return VT_OK;
}

// OpenCV INTER_LINEAR taps (SURVEY.md App. A.3) of every destination index, host side: the arithmetic of lin_tap() in pixel.cu
static void resize_taps(int s, int d, bool clamp_frac, std::vector<int32_t>& out /* 4 per index: i0, i1, a0, a1 */) {
    const double scale = 1.0 / ((double)d / (double)s);
    out.resize((size_t)d * 4);
    for (int i = 0; i < d; ++i) {
        float f = (float)(((double)i + 0.5) * scale - 0.5);
        int ix = (int)floorf(f);
        f -= (float)ix;
        if (clamp_frac) {  // horizontal taps clamp the fraction at the borders ...
            if (ix < 0) ix = 0, f = 0.f;
            if (ix >= s - 1) ix = s - 1, f = 0.f;
        }
        const int a0 = (int)lrintf((1.f - f) * 2048.f), a1 = (int)lrintf(f * 2048.f);
        int i0 = ix, i1 = ix + 1;
        if (clamp_frac) i1 = std::min(i1, s - 1);
        else i0 = std::min(std::max(i0, 0), s - 1), i1 = std::min(std::max(i1, 0), s - 1);  // ... vertical taps clamp the row index
        out[4 * i] = i0, out[4 * i + 1] = i1, out[4 * i + 2] = a0, out[4 * i + 3] = a1;
    }
}

vt_status vt_resize_rgb_device_batch(vt_tracker* t, const uint8_t* d_rgb, size_t stride_in, int32_t sw, int32_t sh, uint8_t* d_out, size_t stride_out,
                                     int32_t dw, int32_t dh, int32_t n_frames) {
    if (!t || !d_rgb || !d_out || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || n_frames <= 0) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const bool fast = ((size_t)dw * 3) % 16 == 0 && stride_out % 16 == 0 && reinterpret_cast<uintptr_t>(d_out) % 16 == 0 && dh <= 65535 && n_frames <= 65535;
    if (!fast) {  // odd geometry: the per-pixel kernel, frame by frame
        for (int i = 0; i < n_frames; ++i) {
            VT_CUDA(launch_resize_rgb_linear(d_rgb + (size_t)i * stride_in, sw, sh, d_out + (size_t)i * stride_out, dw, dh, t->stream));
            ++t->kernel_launches;
        }
        return VT_OK;
    }
    if (t->rsz_geom[0] != sw || t->rsz_geom[1] != sh || t->rsz_geom[2] != dw || t->rsz_geom[3] != dh || !t->d_rsz_taps) {
        std::vector<int32_t> xt, yt;
        resize_taps(sw, dw, true, xt);
        resize_taps(sh, dh, false, yt);
        VT_CUDA(cudaStreamSynchronize(t->stream));  // an earlier launch may still read the old tables
        if (t->d_rsz_taps) cudaFree(t->d_rsz_taps);
        t->d_rsz_taps = nullptr;
        VT_CUDA(cudaMalloc(&t->d_rsz_taps, sizeof(int4) * ((size_t)dw + dh)));
        VT_CUDA(cudaMemcpy(t->d_rsz_taps, xt.data(), sizeof(int4) * dw, cudaMemcpyHostToDevice));
        VT_CUDA(cudaMemcpy(t->d_rsz_taps + dw, yt.data(), sizeof(int4) * dh, cudaMemcpyHostToDevice));
        t->rsz_geom[0] = sw, t->rsz_geom[1] = sh, t->rsz_geom[2] = dw, t->rsz_geom[3] = dh;
        t->rsz_max_src_rows = 0;
        for (int d0 = 0; d0 < dh; d0 += 16) {  // tiles of 16 destination rows (kRszTileRows)
            const int d1 = std::min(d0 + 16, (int)dh) - 1;
            t->rsz_max_src_rows = std::max(t->rsz_max_src_rows, yt[4 * d1 + 1] - yt[4 * d0] + 1);
        }
    }
    VT_CUDA(launch_resize_rgb_tab(d_rgb, stride_in, sw, sh, d_out, stride_out, dw, dh, n_frames, t->d_rsz_taps, t->d_rsz_taps + dw, t->stream,
                                  t->rsz_max_src_rows));
    ++t->kernel_launches;
    return VT_OK;
}

vt_status vt_resize_rgb_device(vt_tracker* t, const uint8_t* d_rgb, int32_t sw, int32_t sh, uint8_t* d_out, int32_t dw, int32_t dh) {
    return vt_resize_rgb_device_batch(t, d_rgb, (size_t)sw * sh * 3, sw, sh, d_out, (size_t)dw * dh * 3, dw, dh, 1);
}

vt_status vt_resize_rgb(vt_tracker* t, const uint8_t* rgb, int32_t sw, int32_t sh, uint8_t* out, int32_t dw, int32_t dh) {
    if (!t || !rgb || !out || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || t->in_flight) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    const size_t in_bytes = (size_t)sw * sh * 3, out_bytes = (size_t)dw * dh * 3;
    vt_status st = fmt_scratch(t, in_bytes, out_bytes);
    if (st != VT_OK) return st;
    VT_CUDA(cudaMemcpyAsync(t->d_fmt_in, rgb, in_bytes, cudaMemcpyHostToDevice, t->stream));
    st = vt_resize_rgb_device_batch(t, t->d_fmt_in, in_bytes, sw, sh, t->d_fmt_out, out_bytes, dw, dh, 1);
    if (st != VT_OK) return st;
    VT_CUDA(cudaMemcpyAsync(out, t->d_fmt_out, out_bytes, cudaMemcpyDeviceToHost, t->stream));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    t->h2d_bytes += in_bytes, t->d2h_bytes += out_bytes;
    return VT_OK;
}

// exposed for bench.py: stream handle so that device-side timing happens on the launching stream
void* vt_tracker_stream(vt_tracker* t) { return t ? (void*)t->stream : nullptr; }
vt_status vt_tracker_sync(vt_tracker* t) {
    if (!t) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    VT_CUDA(cudaStreamSynchronize(t->stream));
    return VT_OK;
}

// ---- overlay -------------------------------------------------------------------------------------
int vt_glyph_rows(int ch, uint8_t rows[7]);  // host_state.cpp

}  // extern "C"
namespace vt {
vt_status fill_cmd_dev(const vt_overlay_cmd& c, OverlayCmdDev& d) {
    memset(&d, 0, sizeof(d));
    d.kind = c.kind, d.x = c.x, d.y = c.y, d.w = c.w, d.h = c.h, d.a = c.a, d.r = c.r, d.g = c.g, d.b = c.b;
    if (c.kind < VT_OV_RECT || c.kind > VT_OV_SELECTION) {
        set_error("vt_overlay: unknown command kind %d", c.kind);
        return VT_ERR_INVALID;
    }
    if (c.kind == VT_OV_TEXT) {
        const size_t len = strnlen(c.text, sizeof(c.text));
        d.nchar = (uint8_t)len;
        for (size_t k = 0; k < len; ++k) {
            uint8_t rows[7];
            if (vt_glyph_rows((unsigned char)c.text[k], rows) == 0) {
                d.known[k] = 1;
                memcpy(d.glyph[k], rows, 7);
            } else if (c.strict_glyphs) {
                set_error("vt_overlay: no glyph for character 0x%02x", (unsigned char)c.text[k]);
                return VT_ERR_GLYPH;
            }
        }
    }
    return VT_OK;
}
}  // namespace vt
extern "C" {

static vt_status build_cmds(vt_tracker* t, const vt_overlay_cmd* cmds, int n, std::vector<std::pair<int, int>>& spans) {
    if (n < 0 || n > kMaxCmds) {
        set_error("vt_overlay: at most %d commands", kMaxCmds);
        return VT_ERR_INVALID;
    }
    const long long H = t->H;
    for (int i = 0; i < n; ++i) {
        const vt_overlay_cmd& c = cmds[i];
        OverlayCmdDev& d = t->h_cmds[i];
        const vt_status fs = fill_cmd_dev(c, d);
        if (fs != VT_OK) return fs;
        long long r0 = 0, r1 = -1;
        switch (c.kind) {
            case VT_OV_RECT:
                if (!rect_rows(t->fmt, H, c.y, c.h, c.a, r0, r1)) r0 = 0, r1 = -1;
                break;
            case VT_OV_CROSSHAIR:
                if (!cross_rows(H, c.y, c.a, r0, r1)) r0 = 0, r1 = -1;
                break;
            case VT_OV_TEXT: r0 = c.y, r1 = (long long)c.y + 7LL * std::max(c.a, 0); break;
            case VT_OV_BACKGROUND:
                r0 = c.y, r1 = (long long)c.y + c.h;
                if (!format_is_luma(t->fmt) && (long long)c.y + c.h < 0) r0 = 0, r1 = H - 1;  // (y+bh) as usize wraps, src/drawing_rgb.rs:45
                break;
            case VT_OV_CURSOR: {
                const long long yc = std::max(0LL, std::min<long long>(c.y, H - 1));  // src/drawing.rs:7 clamps, the RGB path does not
                r0 = std::min<long long>(c.y, yc) - 26, r1 = std::max<long long>(c.y, yc) + 26;
                break;
            }
            case VT_OV_SELECTION: r0 = std::min(c.y, c.h), r1 = std::max(c.y, c.h); break;
            default: set_error("vt_overlay: unknown command kind %d", c.kind); return VT_ERR_INVALID;
        }
        if (r1 >= r0 && r1 >= 0 && r0 <= H - 1) spans.emplace_back((int)std::max(0LL, r0), (int)std::min(r1, H - 1));
    }
    return VT_OK;
}

static vt_status overlay_impl(vt_tracker* t, uint8_t* frame, size_t len, const vt_overlay_cmd* cmds, int32_t n, bool upload) {
    if (!t || !frame || (n > 0 && !cmds) || t->in_flight) return VT_ERR_INVALID;
    VT_CUDA(cudaSetDevice(t->cfg.device));
    // RGBA / BGRA: a full frame, so that every drawn pixel is whole (RGB24 writes are bounds-checked per pixel against len instead)
    const size_t need = format_is_luma(t->fmt) || format_is_rgb32(t->fmt) ? fmt_row_bytes(t->fmt, t->W) * t->H : 0;
    if (len < need) {
        set_error("vt_overlay: frame shorter than its Y plane (YUY2 / RGBA / BGRA: than the packed frame)");
        return VT_ERR_INVALID;
    }
    std::vector<std::pair<int, int>> spans;
    vt_status st = build_cmds(t, cmds, n, spans);
    if (st != VT_OK) return st;
    if (n == 0) return VT_OK;
    VT_CUDA(cudaEventRecord(t->ev_ovl[0], t->stream));
    if (upload) {
        const size_t nb = std::min(len, t->frame_bytes);
        t->d_frame_is_last_host_frame = false;
        if (is_pinned(frame)) {
            VT_CUDA(cudaMemcpyAsync(t->d_frame, frame, nb, cudaMemcpyHostToDevice, t->stream));
        } else {
            memcpy(t->h_stage, frame, nb);
            VT_CUDA(cudaMemcpyAsync(t->d_frame, t->h_stage, nb, cudaMemcpyHostToDevice, t->stream));
        }
    }
    VT_CUDA(cudaMemcpyAsync(t->d_cmds, t->h_cmds, sizeof(OverlayCmdDev) * n, cudaMemcpyHostToDevice, t->stream));
    cudaError_t e = launch_overlay(t->d_frame, std::min(len, t->frame_bytes), t->W, t->H, t->fmt, t->d_cmds, n, t->stream);
    if (e != cudaSuccess) {
        set_error("overlay launch failed: %s", cudaGetErrorString(e));
        return VT_ERR_CUDA;
    }
    ++t->kernel_launches;
    VT_CUDA(cudaEventRecord(t->ev_ovl[1], t->stream));
    merge_spans(spans);
    bool staged = false;
    st = download_rows(t, frame, len, spans, &staged);
    if (st != VT_OK) return st;
    VT_CUDA(cudaStreamSynchronize(t->stream));
    if (staged) unstage_rows(t, frame, len, spans);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, t->ev_ovl[0], t->ev_ovl[1]) == cudaSuccess) t->last[4] = ms;
    else cudaGetLastError();
    return VT_OK;
}

vt_status vt_overlay(vt_tracker* t, uint8_t* frame, size_t len, const vt_overlay_cmd* cmds, int32_t n) {
    return overlay_impl(t, frame, len, cmds, n, true);
}
vt_status vt_overlay_current(vt_tracker* t, uint8_t* frame, size_t len, const vt_overlay_cmd* cmds, int32_t n) {
    if (t && check_uniform_geometry(t, "vt_overlay_current") != VT_OK) return VT_ERR_INVALID;
    if (t && t->cfg.upload_window) {
        set_error("vt_overlay_current needs the whole frame on the device: create the handle with upload_window = 0");
        return VT_ERR_INVALID;
    }
    // The device copy must BE the frame most recently given to update()/submit(): after a device-resident frame (tracked in place in
    // the caller's memory), a conversion or an explicit vt_overlay() it is something else — upload `frame` instead of drawing on a
    // stale image (the caller's frame is the same picture by contract).
    return overlay_impl(t, frame, len, cmds, n, t ? !t->d_frame_is_last_host_frame : false);
}

// ---- timing --------------------------------------------------------------------------------------
vt_status vt_timing_get(vt_tracker* t, vt_timing* o) {
    if (!t || !o) return VT_ERR_INVALID;
    memset(o, 0, sizeof(*o));
    o->fps = t->stats.fps(), o->avg_conv_ms = t->stats.avg_conv_ms(), o->avg_track_ms = t->stats.avg_track_ms();
    o->h2d_ms = t->last[0], o->preprocess_ms = t->last[1], o->vit_ms = t->last[2], o->decode_ms = t->last[3], o->overlay_ms = t->last[4];
    o->d2h_ms = t->last[5], o->total_ms = t->last[6];
    o->avg_h2d_ms = (float)t->r_h2d.mean(), o->avg_preprocess_ms = (float)t->r_pre.mean(), o->avg_vit_ms = (float)t->r_vit.mean();
    o->avg_decode_ms = (float)t->r_dec.mean(), o->avg_overlay_ms = (float)t->r_ovl.mean(), o->avg_d2h_ms = (float)t->r_d2h.mean();
    o->avg_total_ms = (float)t->r_tot.mean();
    o->frames = t->frames, o->kernel_launches = t->kernel_launches;
    o->h2d_bytes = t->h2d_bytes, o->d2h_bytes = t->d2h_bytes;
    return VT_OK;
}
vt_status vt_timing_add_interval(vt_tracker* t, uint64_t us) {
    if (!t) return VT_ERR_INVALID;
    t->stats.add_interval(us);
    return VT_OK;
}
vt_status vt_timing_add_times(vt_tracker* t, uint64_t conv_us, uint64_t track_us) {
    if (!t) return VT_ERR_INVALID;
    t->stats.add_times(conv_us, track_us);
    return VT_OK;
}

}  // extern "C"
