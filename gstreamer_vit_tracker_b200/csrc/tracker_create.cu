// tracker_create.cu — vt_tracker construction: VTW1 weight files (one device copy per file and device, shared between handles),
// device buffers, and the wiring of the tensor-core GEMM / attention plans of every block (≙ VitTrack::new,
// /root/reference/src/tracker_context.rs:21).
#include "tracker_state.h"

namespace vt {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::mutex g_weight_mutex;
static std::map<std::string, std::weak_ptr<WeightSet>> g_weight_cache;

bool frame_is_pinned(const void* p) { return is_pinned(p); }
bool is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// Header of a VTW1 file: magic, shape, and the float count the shape implies — checked against the file size BEFORE anything is
// allocated (the file comes from outside: negative or absurd header fields must not turn into a huge allocation or an overflow).
static vt_status read_weight_header(const char* path, FILE** f_out, int32_t hdr[7], size_t* n_out, struct stat* sb_out) {
    struct stat sb;
    if (!path || stat(path, &sb) != 0 || !S_ISREG(sb.st_mode)) {
        set_error("cannot open weight file %s", path ? path : "(null)");
        return VT_ERR_WEIGHTS;
    }
    FILE* f = fopen(path, "rb");
    if (!f) {
        set_error("cannot open weight file %s", path);
        return VT_ERR_WEIGHTS;
    }
    char magic[4];
    if (fread(magic, 1, 4, f) != 4 || memcmp(magic, "VTW1", 4) != 0 || fread(hdr, 4, 7, f) != 7) {
        fclose(f);
        set_error("%s is not a VTW1 weight file", path);
        return VT_ERR_WEIGHTS;
    }
    const long long Dl = hdr[0], L = hdr[1], heads = hdr[2], Hl = hdr[3], Cl = hdr[4];
    if (Dl <= 0 || Dl > 1024 || Dl % 32 || L <= 0 || L > 64 || Hl <= 0 || Hl > 8192 || Hl % 32 || Cl <= 0 || Cl > 1024 || Cl % 32 || heads <= 0 ||
        Dl % heads || (Dl / heads != 16 && Dl / heads != 32 && Dl / heads != 64)) {
        fclose(f);
        set_error("unsupported model shape D=%d depth=%d heads=%d hidden=%d head_ch=%d", hdr[0], hdr[1], hdr[2], hdr[3], hdr[4]);
        return VT_ERR_WEIGHTS;
    }
    const size_t D = (size_t)Dl, H = (size_t)Hl, C = (size_t)Cl;
    const size_t n = D * kPatchK + D + kNTz * D + kNTx * D + (size_t)L * (4 * D + 3 * D * D + 3 * D + D * D + D + H * D + H + D * H + D) + 2 * D +
                     C * D * 9 + C + 5 * C + 5;
    if ((unsigned long long)sb.st_size != 32ull + 4ull * n) {
        fclose(f);
        set_error("weight file %s: %lld bytes, the header implies %llu", path, (long long)sb.st_size, 32ull + 4ull * n);
        return VT_ERR_WEIGHTS;
    }
    *n_out = n;
    if (sb_out) *sb_out = sb;
    if (f_out) *f_out = f;
    else fclose(f);
    return VT_OK;
}

static vt_status load_weights(vt_tracker* t, const char* path) {
    struct stat sb;
    if (!path || stat(path, &sb) != 0) {
        set_error("cannot open weight file %s", path ? path : "(null)");
        return VT_ERR_WEIGHTS;
    }
    char key[1200];
    snprintf(key, sizeof(key), "%d|%s|%lld|%lld", t->cfg.device, path, (long long)sb.st_size, (long long)sb.st_mtime);
    std::lock_guard<std::mutex> lock(g_weight_mutex);
    std::shared_ptr<WeightSet> ws = g_weight_cache[key].lock();
    if (!ws) {
        FILE* f = nullptr;
        int32_t hdr[7];
        size_t n = 0;
        vt_status hs = read_weight_header(path, &f, hdr, &n, nullptr);
        if (hs != VT_OK) return hs;
        const size_t D = hdr[0], C = hdr[4];
        std::vector<float> host(n);
        const size_t got = fread(host.data(), sizeof(float), n, f);
        fclose(f);
        if (got != n) {
            set_error("weight file %s is truncated (%zu of %zu floats)", path, got, n);
            return VT_ERR_WEIGHTS;
        }
        // head conv weight [C, D, 3, 3] -> [C, tap, D] so that the im2col K axis is tap-major
        const size_t h1_off = n - (5 + 5 * C + C + C * D * 9);
        {
            std::vector<float> re(C * D * 9);
            for (size_t c = 0; c < C; ++c)
                for (size_t d = 0; d < D; ++d)
                    for (size_t tap = 0; tap < 9; ++tap) re[(c * 9 + tap) * D + d] = host[h1_off + (c * D + d) * 9 + tap];
            std::copy(re.begin(), re.end(), host.begin() + h1_off);
        }
        ws = std::make_shared<WeightSet>();
        ws->device = t->cfg.device, ws->n = n;
        memcpy(ws->hdr, hdr, sizeof(hdr));
        VT_CUDA(cudaMalloc(&ws->d_weights, n * sizeof(float)));
        VT_CUDA(cudaMemcpy(ws->d_weights, host.data(), n * sizeof(float), cudaMemcpyHostToDevice));
        g_weight_cache[key] = ws;
    }
    t->wset = ws;
    t->D = ws->hdr[0], t->depth = ws->hdr[1], t->heads = ws->hdr[2], t->hidden = ws->hdr[3], t->head_ch = ws->hdr[4];
    const size_t D = t->D, H = t->hidden, C = t->head_ch;
    t->n_weights = ws->n;
    t->d_weights = ws->d_weights;
    const float* p = t->d_weights;
    auto take = [&](size_t cnt) {
        const float* r = p;
        p += cnt;
        return r;
    };
    t->patch_w = take(D * kPatchK), t->patch_b = take(D), t->pos_z = take(kNTz * D), t->pos_x = take(kNTx * D);
    t->blk.resize(t->depth);
    for (auto& b : t->blk) {
        b.ln1_g = take(D), b.ln1_b = take(D), b.qkv_w = take(3 * D * D), b.qkv_b = take(3 * D);
        b.proj_w = take(D * D), b.proj_b = take(D), b.ln2_g = take(D), b.ln2_b = take(D);
        b.fc1_w = take(H * D), b.fc1_b = take(H), b.fc2_w = take(D * H), b.fc2_b = take(D);
    }
    t->lnf_g = take(D), t->lnf_b = take(D), t->h1_w = take(C * D * 9), t->h1_b = take(C), t->h2_w = take(5 * C), t->h2_b = take(5);
    return VT_OK;
}

void bind_slot(vt_tracker* t, int slot) {
    t->h_res = t->h_blk[slot];
    t->h_stamps = reinterpret_cast<unsigned long long*>(t->h_res + t->maxT);
    t->h_tc_err = reinterpret_cast<int*>(t->h_stamps + ST_COUNT);
}

static void read_switches(vt_tracker* t) {
    Switches& s = t->sw;
    s.spread = !getenv("VT_B200_NO_SPREAD");
    s.att_chain = !getenv("VT_B200_NO_ATT_CHAIN");
    s.att_q64 = !getenv("VT_B200_ATT_Q128");
    s.gemm_q64 = !getenv("VT_B200_GEMM_Q128");
    if (const char* e = getenv("VT_B200_UNCHAIN_N")) s.unchain_n = atoi(e);
    if (const char* e = getenv("VT_B200_AS_ROWS")) s.as_rows = atoi(e);
    s.as_mlp = !getenv("VT_B200_NO_AS_MLP");
    if (const char* e = getenv("VT_B200_AS_SPLIT")) s.as_split = atoi(e);
    s.trace = getenv("VT_B200_TRACE") != nullptr;
    s.hostprof = getenv("VT_B200_HOSTPROF") != nullptr;
    if (const char* e = getenv("VT_B200_WINDOW_SHRINK")) s.win_shrink = atoi(e) & ~1;
}

ShapeForms shape_forms(const vt_tracker* t) {
    ShapeForms f;
    const int D = t->D, Hd = t->hidden, C = t->head_ch;
    f.fuse_ln = D / 64 <= 8;  // a LayerNorm cluster holds at most 8 column tiles
    f.chain_mlp = f.fuse_ln && D <= 192;
    f.tc_attention = D / t->heads == 64;
    f.att_chain = f.chain_mlp && f.tc_attention && Hd / 64 >= t->heads;
    f.split_k = f.chain_mlp && Hd / 64 >= 4 && (C == 64 || C == 128);
    return f;
}

}  // namespace vt

using namespace vt;

extern "C" {

int32_t vt_abi_version(void) { return VT_ABI_VERSION; }
const char* vt_last_error(void) { return vt::g_err; }

void vt_config_default(vt_config* c) {
    if (!c) return;
    memset(c, 0, sizeof(*c));
    c->struct_size = sizeof(vt_config);
    c->format = VT_FMT_NV12;
    c->width = 1920, c->height = 1080;  // src/pipeline.rs:26-27
    c->max_targets = 1;
    c->score_threshold = 0.20f;
    c->gemm_mode = VT_GEMM_TCGEN05_BF16X3;  // the parity-safe tensor-core path; VT_GEMM_FP32_SIMT is the numerically anchoring fallback
    c->use_cuda_graph = 1;
    c->box_overlay = 0;
    c->overlay_gate = 0.25f;  // src/tracker_context.rs:93,122
    // App. A.7 switches: all zero = the OpenCV 4.13 behaviour with the intended normalisation
    for (int k = 0; k < 3; ++k) c->norm_scale[k] = 1.f, c->norm_bias[k] = 0.f;  // (only read with norm_custom = 1)
}

vt_status vt_weights_probe(const char* path, int32_t shape_out[5]) {
    int32_t hdr[7];
    size_t n = 0;
    vt_status st = read_weight_header(path, nullptr, hdr, &n, nullptr);
    if (st == VT_OK && shape_out) memcpy(shape_out, hdr, 5 * sizeof(int32_t));
    return st;
}

vt_status vt_alloc_pinned(size_t bytes, void** out) {
    if (!out) return VT_ERR_INVALID;
    VT_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
    return VT_OK;
}
void vt_free_pinned(void* p) {
    if (p) cudaFreeHost(p);
}

void vt_tracker_destroy(vt_tracker* t) {
    if (!t) return;
    if (t->sw.hostprof && t->hp_n) {
        const double n = (double)t->hp_n;
        fprintf(stderr, "[vt hostprof] frames %llu  submit: upload %.1f  graph launch %.1f  result copy+event %.1f | wait: stream sync %.1f  "
                        "err check+results %.1f  overlay rows %.1f  timing %.1f (us / frame)\n",
                (unsigned long long)t->hp_n, t->hp[0] / n, t->hp[1] / n, t->hp[2] / n, t->hp[3] / n, t->hp[4] / n, t->hp[5] / n, t->hp[6] / n);
    }
    cudaSetDevice(t->cfg.device);
    if (t->counted) registry_add(t->cfg.device, -1);
    if (t->stream) cudaStreamSynchronize(t->stream);
    for (auto& kv : t->graphs) cudaGraphExecDestroy(kv.second);
    for (auto& e : t->ev_ovl)
        if (e) cudaEventDestroy(e);
    if (t->d_rsz_taps) cudaFree(t->d_rsz_taps);
    if (t->d_fmt_in) cudaFree(t->d_fmt_in);
    if (t->d_fmt_out) cudaFree(t->d_fmt_out);
    if (t->copy_stream) cudaStreamSynchronize(t->copy_stream), cudaStreamDestroy(t->copy_stream);
    for (auto& e : t->ev_up)
        if (e) cudaEventDestroy(e);
    for (uint8_t* f : t->d_sframes) cudaFree(f);
    void* dev[] = {t->d_lut, t->d_hann, t->d_frames[0], t->d_frames[1], t->d_rgb, t->d_state, t->d_slots, t->d_res, t->d_maps, t->d_cmds,
                   t->patches_x, t->patches_z, t->Zemb, t->X, t->QKV, t->ATT, t->HID, t->Yf, t->H1, t->d_dbg,
                   t->px_hi, t->px_lo, t->pz_hi, t->pz_lo, t->ln_hi, t->ln_lo, t->att_hi, t->att_lo,
                   t->hid_hi, t->hid_lo, t->yf_hi, t->yf_lo, t->q_hi, t->q_lo, t->k_hi, t->k_lo, t->vt_hi, t->vt_lo, t->zln_hi, t->zln_lo, t->d_trace, t->Pbuf, t->Phead, t->d_cand, t->d_counters};
    for (void* p : dev)
        if (p) cudaFree(p);
    if (t->h_stage) cudaFreeHost(t->h_stage);
    for (int i = 0; i < vt_tracker::kQueue; ++i) {
        if (t->h_blk[i]) cudaFreeHost(t->h_blk[i]);
        if (t->q_done[i]) cudaEventDestroy(t->q_done[i]);
    }
    if (t->d_ctl) cudaFree(t->d_ctl);
    for (auto& h : t->d_hud)
        if (h) cudaFree(h);
    for (auto& h : t->h_hud)
        if (h) cudaFreeHost(h);
    if (t->h_cmds) cudaFreeHost(t->h_cmds);
    if (t->h_slots) cudaFreeHost(t->h_slots);
    if (t->stream) cudaStreamDestroy(t->stream);
    delete t;
}

}  // extern "C"

namespace vt {
// The caller's struct may be older (smaller) than the library's: copy what it has over the defaults.
vt_status resolve_config(const vt_config* in, vt_config* out) {
    constexpr size_t kMin = offsetof(vt_config, max_targets) + sizeof(int32_t);
    if (!in || !out || in->struct_size < kMin || in->struct_size > sizeof(vt_config)) {
        set_error("vt_config: struct_size %u is not a size this library knows (%zu..%zu): call vt_config_default() first", in ? in->struct_size : 0u,
                  kMin, sizeof(vt_config));
        return VT_ERR_INVALID;
    }
    vt_config_default(out);
    memcpy(out, in, in->struct_size);
    out->struct_size = (uint32_t)sizeof(vt_config);
    return VT_OK;
}
}  // namespace vt

extern "C" {

vt_status vt_tracker_create(const vt_config* cfg_in, vt_tracker** out) {
    vt_config cfg_full;
    if (!out) return VT_ERR_INVALID;
    {
        const vt_status rs = resolve_config(cfg_in, &cfg_full);
        if (rs != VT_OK) return rs;
    }
    const vt_config* cfg = &cfg_full;
    if (!cfg->weights_path || cfg->max_targets <= 0 || cfg->max_targets > 64 || !geometry_ok(cfg->format, cfg->width, cfg->height)) {
        set_error("vt_tracker_create: invalid configuration");
        return VT_ERR_INVALID;
    }
    if (cfg->gemm_mode < VT_GEMM_FP32_SIMT || cfg->gemm_mode > VT_GEMM_TCGEN05_FP16) {
        set_error("vt_tracker_create: unknown gemm_mode %d", cfg->gemm_mode);
        return VT_ERR_INVALID;
    }
    if ((cfg->pad_plus1 | cfg->decode_window | cfg->window | cfg->norm_custom) & ~1) {
        set_error("vt_tracker_create: pad_plus1 / decode_window / window / norm_custom are 0 or 1 (SURVEY.md App. A.7)");
        return VT_ERR_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        set_error("no CUDA device: libvittrack_b200 has no CPU fallback");
        return VT_ERR_CUDA;
    }
    VT_CUDA(cudaSetDevice(cfg->device));
    vt_tracker* t = new vt_tracker();
    t->cfg = *cfg;
    t->cfg.weights_path = nullptr;
    t->W = cfg->width, t->H = cfg->height, t->fmt = cfg->format, t->maxT = cfg->max_targets;
    t->frame_bytes = fmt_frame_bytes(t->fmt, t->W, t->H);
    t->threshold = cfg->score_threshold > 0.f ? cfg->score_threshold : 0.20f;
    t->debug_capture = cfg->debug_capture;
    read_switches(t);
    auto fail = [&](vt_status st) {
        vt_tracker_destroy(t);
        return st;
    };
    vt_status st = load_weights(t, cfg->weights_path);
    if (st != VT_OK) return fail(st);
#define VT_TRY(call)                                                                                             \
    do {                                                                                                         \
        cudaError_t e_ = (call);                                                                                 \
        if (e_ != cudaSuccess) {                                                                                 \
            set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);             \
            return fail(VT_ERR_CUDA);                                                                            \
        }                                                                                                        \
    } while (0)
    VT_TRY(cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking));
    for (auto& e : t->ev_ovl) VT_TRY(cudaEventCreate(&e));
    const size_t D = t->D, Hd = t->hidden, C = t->head_ch, B = t->maxT;
    // A.4 normalisation LUT: (v/255 - mean_c)/std_c in double, rounded once to fp32 (channels in memory order)
    {
        const double mean[3] = {0.485, 0.456, 0.406}, stdv[3] = {0.229, 0.224, 0.225};
        float lut[768];
        for (int c = 0; c < 3; ++c)
            for (int v = 0; v < 256; ++v)
                lut[c * 256 + v] = cfg->norm_custom ? (float)((double)v * (double)cfg->norm_scale[c] + (double)cfg->norm_bias[c])  // App. A.7
                                                    : (float)(((double)v / 255.0 - mean[c]) / stdv[c]);
        VT_TRY(cudaMalloc(&t->d_lut, sizeof(lut)));
        VT_TRY(cudaMemcpy(t->d_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
        // A.5 hann window, fp32 exactly as OpenCV builds it
        float h1[16], hann[256];
        for (int i = 0; i < 16; ++i) h1[i] = 0.5f * (1.f - cosf((float)(2 * M_PI / 17) * (float)(i + 1)));
        for (int y = 0; y < 16; ++y)
            for (int x = 0; x < 16; ++x) hann[y * 16 + x] = cfg->window == VT_WINDOW_ONE_MINUS_HANN ? 1.f - h1[y] * h1[x] : h1[y] * h1[x];
        VT_TRY(cudaMalloc(&t->d_hann, sizeof(hann)));
        VT_TRY(cudaMemcpy(t->d_hann, hann, sizeof(hann), cudaMemcpyHostToDevice));
    }
    for (int i = 0; i < 2; ++i) {
        VT_TRY(cudaMalloc(&t->d_frames[i], t->frame_bytes + 256));
        VT_TRY(cudaMemset(t->d_frames[i], 0, t->frame_bytes + 256));
        VT_TRY(cudaEventCreateWithFlags(&t->ev_up[i], cudaEventDisableTiming));
    }
    t->d_frame = t->d_frames[0];
    VT_TRY(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
    t->h_stage_bytes = t->frame_bytes + 256;
    VT_TRY(cudaHostAlloc(&t->h_stage, t->h_stage_bytes, cudaHostAllocDefault));
    VT_TRY(cudaMalloc(&t->d_state, sizeof(TargetState) * B));
    VT_TRY(cudaMemset(t->d_state, 0, sizeof(TargetState) * B));
    VT_TRY(cudaMalloc(&t->d_slots, sizeof(int32_t) * B));
    t->res_block_bytes = sizeof(DeviceResult) * B + sizeof(unsigned long long) * ST_COUNT + 2 * sizeof(int);
    VT_TRY(cudaMalloc(&t->d_res, t->res_block_bytes));
    VT_TRY(cudaMemset(t->d_res, 0, t->res_block_bytes));
    for (int i = 0; i < vt_tracker::kQueue; ++i) {
        VT_TRY(cudaHostAlloc(&t->h_blk[i], t->res_block_bytes, cudaHostAllocDefault));
        memset(t->h_blk[i], 0, t->res_block_bytes);
        VT_TRY(cudaEventCreateWithFlags(&t->q_done[i], cudaEventDisableTiming));
    }
    t->d_stamps = reinterpret_cast<unsigned long long*>(t->d_res + B);
    t->d_tc_err = reinterpret_cast<int*>(t->d_stamps + ST_COUNT);
    bind_slot(t, 0);
    {
        FrameCtl ctl;
        memset(&ctl, 0, sizeof(ctl));
        ctl.frames[0] = packed_ref(cfg_geom(t), t->d_frame, nullptr, true);
        ctl.n_frames = 1, ctl.n_win = -1;
        VT_TRY(cudaMalloc(&t->d_ctl, sizeof(FrameCtl)));
        VT_TRY(cudaMemcpy(t->d_ctl, &ctl, sizeof(ctl), cudaMemcpyHostToDevice));
    }
    VT_TRY(cudaMalloc(&t->d_maps, sizeof(float) * 1280 * B));
    VT_TRY(cudaMemset(t->d_maps, 0, sizeof(float) * 1280 * B));
    VT_TRY(cudaMalloc(&t->d_cmds, sizeof(OverlayCmdDev) * kMaxCmds));
    VT_TRY(cudaHostAlloc(&t->h_cmds, sizeof(OverlayCmdDev) * kMaxCmds, cudaHostAllocDefault));
    VT_TRY(cudaMalloc(&t->patches_x, sizeof(float) * B * kNTx * kPatchK));
    VT_TRY(cudaMalloc(&t->patches_z, sizeof(float) * kNTz * kPatchK));
    VT_TRY(cudaMalloc(&t->Zemb, sizeof(float) * B * kNTz * D));
    VT_TRY(cudaMalloc(&t->X, sizeof(float) * B * kNTok * D));
    VT_TRY(cudaMalloc(&t->QKV, sizeof(float) * B * kNTok * 3 * D));
    VT_TRY(cudaMalloc(&t->ATT, sizeof(float) * B * kNTok * D));
    VT_TRY(cudaMalloc(&t->HID, sizeof(float) * B * kNTok * Hd));
    VT_TRY(cudaMalloc(&t->Yf, sizeof(float) * B * kNTx * D));
    VT_TRY(cudaMalloc(&t->H1, sizeof(float) * B * kNTx * C));
    VT_TRY(cudaMemset(t->patches_x, 0, sizeof(float) * B * kNTx * kPatchK));
    VT_TRY(cudaMemset(t->patches_z, 0, sizeof(float) * kNTz * kPatchK));
    if (t->debug_capture) VT_TRY(cudaMalloc(&t->d_dbg, sizeof(float) * (size_t)(t->depth + 1) * B * kNTok * D));
    t->nsplit = cfg->gemm_mode == VT_GEMM_TCGEN05_BF16X3 ? 3 : (cfg->gemm_mode == VT_GEMM_TCGEN05_BF16 ? 1 : (cfg->gemm_mode == VT_GEMM_TCGEN05_FP16 ? 2 : 0));
    t->f16 = t->nsplit == 2;
    if (t->nsplit) {
        if (D % 64 || Hd % 64 || C % 64) {
            set_error("the tcgen05 path needs D, hidden and head_ch to be multiples of 64 (D=%zu hidden=%zu head_ch=%zu)", D, Hd, C);
            return fail(VT_ERR_WEIGHTS);
        }
        VT_TRY(tc_gemm_setup());
        VT_TRY(tc_gemm_as_setup());
        VT_TRY(cudaDeviceGetAttribute(&t->sm_count, cudaDevAttrMultiProcessorCount, cfg->device));
        const ShapeForms sf = shape_forms(t);
        const size_t p_planes = std::max({sf.chain_mlp ? Hd / 64 : 0, sf.att_chain ? (size_t)t->heads : 0, sf.split_k ? (size_t)4 : 0});
        if (p_planes) VT_TRY(cudaMalloc(&t->Pbuf, sizeof(float) * p_planes * B * kNTok * D));
        if (sf.split_k) {
            VT_TRY(cudaMalloc(&t->Phead, sizeof(float) * 9 * B * kNTx * C));
            VT_TRY(cudaMalloc(&t->d_cand, sizeof(float) * B * 16 * 8));
            VT_TRY(cudaMalloc(&t->d_counters, sizeof(unsigned) * B));
            VT_TRY(cudaMemset(t->d_counters, 0, sizeof(unsigned) * B));
        }
        {   // bf16 (hi, lo) split of the shared weights: done once per WeightSet
            std::lock_guard<std::mutex> lock(t->wset->split_mutex);
            if (!t->wset->w_hi) {
                const size_t nw = t->n_weights;
                VT_TRY(cudaMalloc(&t->wset->w_hi, nw * 2));
                VT_TRY(cudaMalloc(&t->wset->w_lo, nw * 2));
                VT_TRY(launch_split_bf16(t->d_weights, t->wset->w_hi, t->wset->w_lo, nw, t->stream));
                VT_TRY(cudaStreamSynchronize(t->stream));
            }
            t->w_hi = t->wset->w_hi, t->w_lo = t->wset->w_lo;
            if (t->f16) {  // single-pass fp16 operands: an fp16 copy of the weights stands in for the hi part
                if (!t->wset->w_f16) {
                    VT_TRY(cudaMalloc(&t->wset->w_f16, t->n_weights * 2));
                    VT_TRY(launch_split_bf16(t->d_weights, t->wset->w_f16, nullptr, t->n_weights, t->stream));
                    VT_TRY(cudaStreamSynchronize(t->stream));
                }
                t->w_hi = t->wset->w_f16;
            }
        }
        auto balloc = [&](__nv_bfloat16** hi, __nv_bfloat16** lo, size_t n) -> cudaError_t {
            cudaError_t e = cudaMalloc(hi, n * 2);
            if (e == cudaSuccess) e = cudaMalloc(lo, n * 2);
            if (e == cudaSuccess) e = cudaMemset(*hi, 0, n * 2);
            if (e == cudaSuccess) e = cudaMemset(*lo, 0, n * 2);
            return e;
        };
        VT_TRY(balloc(&t->px_hi, &t->px_lo, B * kNTx * kPatchK));
        VT_TRY(balloc(&t->pz_hi, &t->pz_lo, (size_t)128 * kPatchK));  // one 128-row tile; rows 64..127 stay zero
        VT_TRY(balloc(&t->ln_hi, &t->ln_lo, B * kNTok * D));
        VT_TRY(balloc(&t->zln_hi, &t->zln_lo, B * kNTz * D));
        VT_TRY(balloc(&t->att_hi, &t->att_lo, B * kNTok * D));
        VT_TRY(balloc(&t->hid_hi, &t->hid_lo, B * kNTok * Hd));
        VT_TRY(balloc(&t->yf_hi, &t->yf_lo, B * kNTx * D));
        if (sf.tc_attention) {
            const size_t nq = B * t->heads * kNTok * 64;
            VT_TRY(balloc(&t->q_hi, &t->q_lo, nq));
            VT_TRY(balloc(&t->k_hi, &t->k_lo, nq));
            VT_TRY(balloc(&t->vt_hi, &t->vt_lo, nq));
            VT_TRY(tc_attention_setup());
            if (!tc_attention_plan_init(&t->plan_att, t->q_hi, t->q_lo, t->k_hi, t->k_lo, t->vt_hi, t->vt_lo, (int)(B * t->heads), t->att_hi, t->att_lo, (int)D, (int)B))
                return fail(VT_ERR_CUDA);
        }
        auto whi = [&](const float* w) { return t->w_hi + (w - t->d_weights); };
        auto wlo = [&](const float* w) { return t->w_lo + (w - t->d_weights); };
        bool ok = true;
        const uint64_t rows = B * kNTok;
        // outputs of the GEMM epilogues (TcOut: dense [planes][targets][heads][rows][cols]) and the flat residual TMA source
        CUtensorMap mXres;
        ok &= tc_resid_map(&mXres, t->X, B * kNTok, D);
        const int Bi = (int)B, Di = (int)D;
        const TcOut oX = tc_out(t->X, 4, Di, kNTok, 1, Bi, 1);
        const TcOut oLn[2] = {tc_out(t->ln_hi, 2, Di, kNTok, 1, Bi, 1), tc_out(t->ln_lo, 2, Di, kNTok, 1, Bi, 1)};
        const TcOut oYf[2] = {tc_out(t->yf_hi, 2, Di, kNTx, 1, Bi, 1), tc_out(t->yf_lo, 2, Di, kNTx, 1, Bi, 1)};
        const TcOut oHid[2] = {tc_out(t->hid_hi, 2, (int)Hd, kNTok, 1, Bi, 1), tc_out(t->hid_lo, 2, (int)Hd, kNTok, 1, Bi, 1)};
        const TcOut oH1 = tc_out(t->H1, 4, (int)C, kNTx, 1, Bi, 1), oZ = tc_out(t->Zemb, 4, Di, kNTz, 1, Bi, 1);
        const TcOut oQKV = tc_out(t->QKV, 4, 3 * Di, kNTok, 1, Bi, 1);
        TcOut oQ[6] = {};
        if (sf.tc_attention) {
            oQ[0] = tc_out(t->q_hi, 2, 64, kNTok, t->heads, Bi, 1), oQ[1] = tc_out(t->q_lo, 2, 64, kNTok, t->heads, Bi, 1);
            oQ[2] = tc_out(t->k_hi, 2, 64, kNTok, t->heads, Bi, 1), oQ[3] = tc_out(t->k_lo, 2, 64, kNTok, t->heads, Bi, 1);
            oQ[4] = tc_out_vt(t->vt_hi, kNTok, t->heads, Bi), oQ[5] = tc_out_vt(t->vt_lo, kNTok, t->heads, Bi);
        }
        // patch embed (search): A = patches [B*256, 768] -> X rows 64.. of every target, + pos_x
        ok &= tc_plan_init(&t->plan_patch_x, t->px_hi, t->px_lo, B * kNTx, whi(t->patch_w), wlo(t->patch_w), (int)D, kPatchK, 0, 0);
        {
            TcGemmArgs& a = t->plan_patch_x.args;
            a.bias = t->patch_b, a.pos = t->pos_x, a.pos_rows = kNTx;
            a.period = kNTx, a.c_on = 1, a.c_row_off = kNTz, a.c = oX;
            if (sf.split_k) {  // 4 x K = 192 slices -> fp32 partials [4][B][256][D]; bias, pos, LN1 happen in reduce_ln_kernel
                a.bias = nullptr, a.pos = nullptr, a.c_row_off = 0, a.kb_per_split = kPatchK / 64 / 4;
                a.c = tc_out(t->Pbuf, 4, Di, kNTx, 1, Bi, 4);
            } else if (sf.fuse_ln) {  // LN1 of block 0 for the search rows, straight into the first QKV GEMM's A operand
                a.ln_g = t->blk[0].ln1_g, a.ln_b = t->blk[0].ln1_b, a.ln_row_off = kNTz;
                a.ln_out[0] = oLn[0], a.ln_out[1] = oLn[1];
            }
        }
        // patch embed (template, at init): one 128-row tile whose rows 64.. are clipped; batch_off = the target slot, set per call
        ok &= tc_plan_init(&t->plan_patch_z, t->pz_hi, t->pz_lo, 128, whi(t->patch_w), wlo(t->patch_w), (int)D, kPatchK, 0, 0);
        {
            TcGemmArgs& a = t->plan_patch_z.args;
            a.bias = t->patch_b, a.pos = t->pos_z, a.pos_rows = kNTz;
            a.period = 128, a.c_on = 1, a.c = oZ;
        }
        t->plans.resize(t->depth);
        for (int l = 0; l < t->depth && ok; ++l) {
            const BlockW& b = t->blk[l];
            vt_tracker::BlockPlans& p = t->plans[l];
            ok &= tc_plan_init(&p.qkv, t->ln_hi, t->ln_lo, rows, whi(b.qkv_w), wlo(b.qkv_w), (int)(3 * D), (int)D, 0, 0);
            p.qkv.args.bias = b.qkv_b, p.qkv.args.period = kNTok;
            if (sf.tc_attention) {
                p.qkv.args.o_mode = 2;
                for (int i = 0; i < 6; ++i) p.qkv.args.o[i] = oQ[i];
            } else {
                p.qkv.args.c_on = 1, p.qkv.args.c = oQKV;
            }
            ok &= tc_plan_init(&p.proj, t->att_hi, t->att_lo, rows, whi(b.proj_w), wlo(b.proj_w), (int)D, (int)D, 0, 0);
            p.proj.args.bias = b.proj_b, p.proj.args.period = kNTok, p.proj.args.residual = 1, p.proj.args.c_on = 1;
            p.proj.maps.R = mXres, p.proj.args.c = oX;
            if (sf.fuse_ln) p.proj.args.ln_g = b.ln2_g, p.proj.args.ln_b = b.ln2_b, p.proj.args.ln_out[0] = oLn[0], p.proj.args.ln_out[1] = oLn[1];
            ok &= tc_plan_init(&p.fc1, t->ln_hi, t->ln_lo, rows, whi(b.fc1_w), wlo(b.fc1_w), (int)Hd, (int)D, 0, 0);
            p.fc1.args.bias = b.fc1_b, p.fc1.args.gelu = 1, p.fc1.args.period = kNTok, p.fc1.args.o_mode = 1;
            p.fc1.args.o[0] = oHid[0], p.fc1.args.o[1] = oHid[1];
            if (sf.chain_mlp) ok &= tc_plan_chain(&p.fc1, whi(b.fc2_w), wlo(b.fc2_w), (int)D, t->Pbuf, kNTok, B);
            if (sf.att_chain) {
                p.att = t->plan_att;
                ok &= tc_attention_plan_chain(&p.att, whi(b.proj_w), wlo(b.proj_w), t->Pbuf, (int64_t)B * kNTok * D);
            }
            ok &= tc_plan_init(&p.fc2, t->hid_hi, t->hid_lo, rows, whi(b.fc2_w), wlo(b.fc2_w), (int)D, (int)Hd, 0, 0);
            p.fc2.args.bias = b.fc2_b, p.fc2.args.period = kNTok, p.fc2.args.residual = 1, p.fc2.args.c_on = 1;
            p.fc2.maps.R = mXres, p.fc2.args.c = oX;
            if (sf.fuse_ln) {
                TcGemmArgs& a = p.fc2.args;
                if (l + 1 < t->depth) {
                    a.ln_g = t->blk[l + 1].ln1_g, a.ln_b = t->blk[l + 1].ln1_b, a.ln_out[0] = oLn[0], a.ln_out[1] = oLn[1];
                } else {  // final LN, search rows only -> the head conv's [B,16,16,D] grid (the template rows fall outside and are clipped)
                    a.ln_g = t->lnf_g, a.ln_b = t->lnf_b, a.ln_row_off = -kNTz, a.ln_out[0] = oYf[0], a.ln_out[1] = oYf[1];
                }
            }
        }
        // 3x3 head conv: A gathered by TMA from the [B,16,16,D] final-LN grid (zero fill = zero padding), weights [C][tap][D]
        ok &= tc_plan_init(&t->plan_head, t->yf_hi, t->yf_lo, 0, whi(t->h1_w), wlo(t->h1_w), (int)C, (int)(9 * D), (int)D, (int)B);
        t->plan_head.args.bias = t->h1_b, t->plan_head.args.relu = 1, t->plan_head.args.period = kNTx, t->plan_head.args.c_on = 1;
        t->plan_head.args.c = oH1;
        if (sf.split_k) {  // one tap per slice -> fp32 partials [9][B][256][C]; bias, ReLU, 1x1 conv and decode in head_decode_kernel
            t->plan_head.args.bias = nullptr, t->plan_head.args.relu = 0, t->plan_head.args.kb_per_split = (int)(D / 64);
            t->plan_head.args.c = tc_out(t->Phead, 4, (int)C, kNTx, 1, Bi, 9);
        }
        if (!ok) return fail(VT_ERR_CUDA);
        for (TcGemmPlan* p : {&t->plan_patch_x, &t->plan_patch_z, &t->plan_head}) p->args.err = t->d_tc_err;
        for (auto& p : t->plans) p.qkv.args.err = p.proj.args.err = p.fc1.args.err = p.fc2.args.err = t->d_tc_err;
        if (t->sw.trace) {
            VT_TRY(cudaMalloc(&t->d_trace, tc::kTraceWords * 8));
            VT_TRY(cudaMemset(t->d_trace, 0, tc::kTraceWords * 8));
            t->plan_patch_x.args.trace = t->plan_head.args.trace = t->d_trace;
            t->plan_patch_x.args.trace_id = 1, t->plan_head.args.trace_id = 6;
            for (auto& p : t->plans) {
                p.qkv.args.trace = p.proj.args.trace = p.fc1.args.trace = p.fc2.args.trace = t->d_trace;
                p.qkv.args.trace_id = 2, p.proj.args.trace_id = 3, p.fc1.args.trace_id = 4, p.fc2.args.trace_id = 5;
            }
        }
    }
    t->rect_mirror.assign(B, vt_bbox{0, 0, 0, 0});
    t->inited.assign(B, 0);
    t->geom.assign(B, cfg_geom(t));
    VT_TRY(cudaStreamSynchronize(t->stream));
#undef VT_TRY
    if (t->cfg.device >= 0 && t->cfg.device < kMaxDevices) {
        registry_add(t->cfg.device, +1), t->counted = true;
        registry_sweep(t->cfg.device);
    }
    *out = t;
    return VT_OK;
}

int32_t vt_tracker_model_dim(const vt_tracker* t, int32_t which) {
    if (!t) return 0;
    switch (which) {
        case 0: return t->D;
        case 1: return t->depth;
        case 2: return t->heads;
        case 3: return t->hidden;
        case 5: return registry_total(t->cfg.device);
        default: return t->head_ch;
    }
}

}  // extern "C"
