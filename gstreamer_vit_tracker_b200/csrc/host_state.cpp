// host_state.cpp — host-side mirror of the reference's control logic around the device path:
//   SelectionState   ≙ /root/reference/src/selection_state.rs:1-45
//   TrackerContext   ≙ /root/reference/src/tracker_context.rs:7-167 (+ AppState, src/app_state.rs)
//   probe body       ≙ src/pipeline.rs:67-184 (NV12) and src/pipeline_ir.rs:100-228 (RGB24)
//   glyph lookup     ≙ src/drawing.rs:52-100
// The reference is Rust; no Rust toolchain exists in the build image, so the host side is C++ with
// the same names, argument meaning and error behaviour behind the C ABI of include/vt_tracker.h.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <string>
#include <vector>

#include "vt_internal.h"

namespace {

// 5x7 font, MSB-left 5-bit rows; same 40 characters as the reference table.
struct Glyph {
    char ch;
    uint8_t rows[7];
};
const Glyph kFont[] = {
    {'0', {14, 17, 19, 21, 25, 17, 14}}, {'1', {4, 12, 4, 4, 4, 4, 14}},      {'2', {14, 17, 1, 6, 8, 16, 31}},
    {'3', {14, 17, 1, 6, 1, 17, 14}},    {'4', {2, 6, 10, 18, 31, 2, 2}},     {'5', {31, 16, 30, 1, 1, 17, 14}},
    {'6', {6, 8, 16, 30, 17, 17, 14}},   {'7', {31, 1, 2, 4, 8, 8, 8}},       {'8', {14, 17, 17, 14, 17, 17, 14}},
    {'9', {14, 17, 17, 15, 1, 2, 12}},   {'.', {0, 0, 0, 0, 0, 12, 12}},      {':', {0, 12, 12, 0, 12, 12, 0}},
    {'-', {0, 0, 0, 31, 0, 0, 0}},       {' ', {0, 0, 0, 0, 0, 0, 0}},        {'F', {31, 16, 30, 16, 16, 16, 16}},
    {'P', {30, 17, 30, 16, 16, 16, 16}}, {'S', {14, 17, 16, 14, 1, 17, 14}},  {'T', {31, 4, 4, 4, 4, 4, 4}},
    {'R', {30, 17, 30, 20, 18, 17, 17}}, {'A', {14, 17, 31, 17, 17, 17, 17}}, {'C', {14, 17, 16, 16, 16, 17, 14}},
    {'K', {17, 18, 20, 24, 20, 18, 17}}, {'I', {14, 4, 4, 4, 4, 4, 14}},      {'N', {17, 25, 21, 19, 17, 17, 17}},
    {'G', {14, 17, 16, 23, 17, 17, 14}}, {'E', {31, 16, 30, 16, 16, 16, 31}}, {'L', {16, 16, 16, 16, 16, 16, 31}},
    {'O', {14, 17, 17, 17, 17, 17, 14}}, {'D', {28, 18, 17, 17, 17, 18, 28}}, {'%', {25, 26, 4, 4, 8, 11, 19}},
    {'s', {0, 0, 14, 16, 14, 1, 30}},    {'c', {0, 0, 14, 16, 16, 17, 14}},   {'o', {0, 0, 14, 17, 17, 17, 14}},
    {'r', {0, 0, 22, 25, 16, 16, 16}},   {'e', {0, 0, 14, 17, 31, 16, 14}},   {'m', {0, 0, 26, 21, 21, 17, 17}},
    {'t', {8, 8, 28, 8, 8, 9, 6}},       {'k', {16, 16, 18, 20, 24, 20, 18}}, {'n', {0, 0, 22, 25, 17, 17, 17}},
    {'v', {0, 0, 17, 17, 17, 10, 4}},
};

// ≙ SelectionState (src/selection_state.rs)
struct SelectionState {
    int32_t cursor_x, cursor_y, start_x, start_y;
    int32_t phase;  // 0 MovingToStart, 1 SelectingArea
    int32_t step, fast_step;
    SelectionState(int w, int h) : cursor_x(w / 2), cursor_y(h / 2), start_x(w / 2), start_y(h / 2), phase(0), step(10), fast_step(50) {}
    static int clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
    void move_cursor(int dx, int dy, bool fast, int w, int h) {
        const int s = fast ? fast_step : step;
        cursor_x = clamp(cursor_x + dx * s, 0, w - 1);
        cursor_y = clamp(cursor_y + dy * s, 0, h - 1);
    }
    vt_bbox get_bbox() const {
        const int w = start_x > cursor_x ? start_x - cursor_x : cursor_x - start_x;
        const int h = start_y > cursor_y ? start_y - cursor_y : cursor_y - start_y;
        return vt_bbox{start_x < cursor_x ? start_x : cursor_x, start_y < cursor_y ? start_y : cursor_y, w > 20 ? w : 20, h > 20 ? h : 20};
    }
};

enum class AppState { Selecting, Tracking, Lost };

}  // namespace

struct vt_context {
    vt_tracker* tracker = nullptr;
    vt_config cfg;
    AppState state = AppState::Selecting;
    uint64_t lost_frames = 0;
    SelectionState selection;
    bool has_bbox = false;
    vt_bbox current_bbox{0, 0, 0, 0};
    float current_score = 0.f;
    int32_t frame_width, frame_height;
    bool pending_confirm = false;
    bool frame_on_device = false;  // the tracker saw (uploaded) the frame during this process_frame call
    // probe state (≙ the Arc<...> captured by the closure, src/pipeline.rs:55-63)
    uint64_t frame_num = 0;
    bool have_last = false;
    std::chrono::steady_clock::time_point last_time;
    vt_probe_group* group = nullptr;  // member of a probe group: borrowed (the group owns it and the tracker), frames go through the group
    vt_context(int w, int h) : selection(w, h), frame_width(w), frame_height(h) {}
};

// ≙ n TrackerContexts (one per pipeline, src/pipeline.rs:55) sharing one tracker handle: stream i = member i = target slot i
struct vt_probe_group {
    vt_tracker* tracker = nullptr;
    std::vector<vt_context*> members;
    // probe state of the group step (one interval per step: every stream is probed once per step)
    uint64_t frame_num = 0;
    bool have_last = false;
    std::chrono::steady_clock::time_point last_time;
};

namespace {
// the single-context frame entry points refuse a group member
bool member_refused(const vt_context* c, const char* where) {
    if (!c || !c->group) return false;
    vt::set_error("%s: this context is a member of a probe group; its frames go through vt_probe_group_frame / vt_probe_group_run_ring", where);
    return true;
}
}  // namespace

extern "C" {

int vt_glyph_rows(int ch, uint8_t rows[7]) {
    for (const Glyph& g : kFont)
        if (g.ch == (char)ch) {
            memcpy(rows, g.rows, 7);
            return 0;
        }
    return -1;
}

vt_status vt_context_create(const vt_config* cfg, vt_context** out) {
    if (!cfg || !out) return VT_ERR_INVALID;
    *out = nullptr;
    vt_config c;
    const vt_status rs = vt::resolve_config(cfg, &c);
    if (rs != VT_OK) return rs;
    c.max_targets = 1;   // one VitTrack per TrackerContext (src/tracker_context.rs:8)
    c.box_overlay = 0;   // the probe queues explicit overlay commands (the box is one of them)
    vt_tracker* t = nullptr;
    vt_status st = vt_tracker_create(&c, &t);  // ≙ VitTrack::new(model_path)?, src/tracker_context.rs:21
    if (st != VT_OK) return st;
    vt::tracker_enable_hud(t);  // the frame's last kernel runs the probe's HUD list (one synchronisation per probed frame)
    vt_context* ctx = new vt_context(c.width, c.height);
    ctx->tracker = t;
    ctx->cfg = c;
    ctx->cfg.weights_path = nullptr;
    *out = ctx;
    return VT_OK;
}

void vt_context_destroy(vt_context* c) {
    if (!c || c->group) return;  // (a group member is destroyed with its group)
    if (c->tracker) vt_tracker_destroy(c->tracker);
    delete c;
}

// ≙ the byte -> UserCommand match of the keyboard reader, src/raw_mode_guard.rs:65-101.  Returns 1 and fills cmd / fast when the
// byte maps to a command, 0 when it is ignored (the '[' of escape sequences and everything else).
int32_t vt_command_from_key(uint8_t byte, int32_t* cmd, int32_t* fast) {
    int c = -1, f = 0;
    switch (byte) {
        case 10: case 13: case 32: c = VT_CMD_CONFIRM; break;                       // Enter, Space
        case 87: case 119: case 73: case 105: c = VT_CMD_MOVE_UP; break;            // W w I i
        case 83: case 115: case 75: case 107: c = VT_CMD_MOVE_DOWN; break;          // S s K k
        case 65: case 97: case 74: case 106: c = VT_CMD_MOVE_LEFT; break;           // A a J j
        case 68: case 100: case 76: case 108: c = VT_CMD_MOVE_RIGHT; break;         // D d L l
        case 84: case 116: c = VT_CMD_MOVE_UP, f = 1; break;                        // T t   fast
        case 71: case 103: c = VT_CMD_MOVE_DOWN, f = 1; break;                      // G g
        case 70: case 102: c = VT_CMD_MOVE_LEFT, f = 1; break;                      // F f
        case 72: case 104: c = VT_CMD_MOVE_RIGHT, f = 1; break;                     // H h
        case 82: case 114: case 27: c = VT_CMD_CANCEL; break;                       // R r Escape
        case 81: case 113: c = VT_CMD_QUIT; break;                                  // Q q
        default: break;                                                             // 91 '[' and the rest: ignored
    }
    if (c < 0) return 0;
    if (cmd) *cmd = c;
    if (fast) *fast = f;
    return 1;
}

vt_status vt_context_handle_command(vt_context* c, int32_t cmd, int32_t fast) {  // src/tracker_context.rs:36-61
    if (!c) return VT_ERR_INVALID;
    const int w = c->frame_width, h = c->frame_height;
    switch (cmd) {
        case VT_CMD_MOVE_UP: c->selection.move_cursor(0, -1, fast != 0, w, h); break;
        case VT_CMD_MOVE_DOWN: c->selection.move_cursor(0, 1, fast != 0, w, h); break;
        case VT_CMD_MOVE_LEFT: c->selection.move_cursor(-1, 0, fast != 0, w, h); break;
        case VT_CMD_MOVE_RIGHT: c->selection.move_cursor(1, 0, fast != 0, w, h); break;
        case VT_CMD_CONFIRM: c->pending_confirm = true; break;
        case VT_CMD_CANCEL:
            c->state = AppState::Selecting;
            c->selection = SelectionState(w, h);
            c->has_bbox = false;
            break;
        case VT_CMD_QUIT: break;
        default: return VT_ERR_INVALID;
    }
    return VT_OK;
}

}  // extern "C"

namespace {
// outcome of VitTrack::init + update as the state machine sees it: ok=false ≙ Err(e)
struct UpdateOutcome {
    bool ok;
    vt_result r;
};

// ≙ TrackerContext::process_frame, src/tracker_context.rs:64-155.  `init_and_update(bb)` runs
// tracker.init(frame, bb) followed by tracker.update(frame) (:88-90); `update()` runs tracker.update(frame) (:120).
// A device/tracker error maps to the reference's Err branches (selection reset / Lost) and never propagates.
template <typename InitUpdate, typename Update>
void process_frame_core(vt_context* c, InitUpdate init_and_update, Update update, int32_t* has_bbox, vt_bbox* bbox) {
    *has_bbox = 0;
    switch (c->state) {
        case AppState::Selecting:
            if (c->pending_confirm) {
                c->pending_confirm = false;
                if (c->selection.phase == 0) {  // :71-80
                    c->selection.start_x = c->selection.cursor_x;
                    c->selection.start_y = c->selection.cursor_y;
                    c->selection.phase = 1;
                } else {  // :81-112
                    const UpdateOutcome o = init_and_update(c->selection.get_bbox());
                    if (o.ok && o.r.success && o.r.score > 0.25f) {
                        c->current_bbox = o.r.bbox, c->has_bbox = true;
                        c->current_score = o.r.score;
                        c->state = AppState::Tracking;
                        *has_bbox = 1, *bbox = o.r.bbox;
                        return;
                    }
                    c->selection = SelectionState(c->frame_width, c->frame_height);  // low score (:100-103) or Err (:105-109)
                }
            }
            return;
        case AppState::Tracking: {  // :117-140
            c->pending_confirm = false;
            const UpdateOutcome o = update();
            if (o.ok) {
                if (o.r.success && o.r.score > 0.25f) {
                    c->current_bbox = o.r.bbox, c->has_bbox = true;
                    c->current_score = o.r.score;
                    *has_bbox = 1, *bbox = o.r.bbox;
                } else {
                    c->state = AppState::Lost, c->lost_frames = 0;
                    c->current_score = 0.f;
                }
            } else {
                c->state = AppState::Lost, c->lost_frames = 0;
            }
            return;
        }
        case AppState::Lost:  // :142-153
            c->pending_confirm = false;
            if (c->lost_frames > 60) {
                c->state = AppState::Selecting;
                c->selection = SelectionState(c->frame_width, c->frame_height);
                c->has_bbox = false;
            } else {
                c->lost_frames += 1;
            }
            return;
    }
}
}  // namespace

extern "C" {

vt_status vt_context_process_frame(vt_context* c, uint8_t* frame, size_t len, int32_t* has_bbox, vt_bbox* bbox) {
    if (!c || !c->tracker || !frame || !has_bbox || !bbox || member_refused(c, "vt_context_process_frame")) return VT_ERR_INVALID;
    c->frame_on_device = false;
    auto upd = [&]() {
        UpdateOutcome o;
        const vt_status st = vt_tracker_update(c->tracker, frame, len, &o.r);
        if (st == VT_OK) c->frame_on_device = true;
        o.ok = st == VT_OK && o.r.status == VT_OK;
        return o;
    };
    auto init_upd = [&](vt_bbox bb) {
        vt_tracker_init(c->tracker, 0, frame, len, bb);  // return value ignored, like the reference (:88)
        return upd();
    };
    process_frame_core(c, init_upd, upd, has_bbox, bbox);
    return VT_OK;
}

// State machine without a device: the outcome of update() is scripted by the caller (err != 0 ≙ Err).
vt_status vt_context_create_scripted(int32_t width, int32_t height, vt_context** out) {
    if (!out || width <= 0 || height <= 0) return VT_ERR_INVALID;
    vt_context* ctx = new vt_context(width, height);
    memset(&ctx->cfg, 0, sizeof(ctx->cfg));
    ctx->cfg.width = width, ctx->cfg.height = height;
    *out = ctx;
    return VT_OK;
}
vt_status vt_context_process_scripted(vt_context* c, const vt_result* scripted, int32_t err, int32_t* has_bbox, vt_bbox* bbox) {
    if (!c || !has_bbox || !bbox || (!err && !scripted)) return VT_ERR_INVALID;
    auto upd = [&]() {
        UpdateOutcome o;
        o.ok = !err;
        if (scripted) o.r = *scripted;
        return o;
    };
    process_frame_core(c, [&](vt_bbox) { return upd(); }, upd, has_bbox, bbox);
    return VT_OK;
}

int32_t vt_context_state(const vt_context* c) {  // src/tracker_context.rs:157-166
    if (!c) return -1;
    if (c->state == AppState::Selecting) return c->selection.phase == 0 ? VT_STATE_SELECT_START : VT_STATE_SELECT_END;
    return c->state == AppState::Tracking ? VT_STATE_TRACKING : VT_STATE_LOST;
}
const char* vt_context_state_name(const vt_context* c) {
    static const char* const names[4] = {"SELECT START", "SELECT END", "TRACKING", "LOST"};
    const int s = vt_context_state(c);
    return s < 0 ? "" : names[s];
}
float vt_context_current_score(const vt_context* c) { return c ? c->current_score : 0.f; }
int32_t vt_context_current_bbox(const vt_context* c, vt_bbox* out) {
    if (!c || !c->has_bbox) return 0;
    if (out) *out = c->current_bbox;
    return 1;
}
void vt_context_selection(const vt_context* c, vt_selection* o) {
    if (!c || !o) return;
    const SelectionState& s = c->selection;
    *o = vt_selection{s.cursor_x, s.cursor_y, s.start_x, s.start_y, s.phase, s.step, s.fast_step};
}
uint64_t vt_context_lost_frames(const vt_context* c) { return c ? c->lost_frames : 0; }
vt_tracker* vt_context_tracker(vt_context* c) { return c ? c->tracker : nullptr; }

// ≙ TimingStats as a free-standing object (src/timing_stats.rs:3-60)
struct vt_timing_stats {
    vt::TimingStats s;
};
vt_timing_stats* vt_timing_stats_create(void) { return new vt_timing_stats(); }
void vt_timing_stats_destroy(vt_timing_stats* s) { delete s; }
// (a null object reads as the empty TimingStats: every accessor of src/timing_stats.rs:36-60 returns 0.0 then)
void vt_timing_stats_add_interval(vt_timing_stats* s, uint64_t us) {
    if (s) s->s.add_interval(us);
}
void vt_timing_stats_add_times(vt_timing_stats* s, uint64_t conv_us, uint64_t track_us) {
    if (s) s->s.add_times(conv_us, track_us);
}
double vt_timing_stats_fps(const vt_timing_stats* s) { return s ? s->s.fps() : 0.0; }
double vt_timing_stats_avg_conv_ms(const vt_timing_stats* s) { return s ? s->s.avg_conv_ms() : 0.0; }
double vt_timing_stats_avg_track_ms(const vt_timing_stats* s) { return s ? s->s.avg_track_ms() : 0.0; }

static vt_overlay_cmd make_cmd(int kind, int x, int y, int w, int h, int a, uint8_t r, uint8_t g, uint8_t b, const char* text = nullptr,
                               int strict = 0) {
    vt_overlay_cmd c;
    memset(&c, 0, sizeof(c));
    c.kind = kind, c.x = x, c.y = y, c.w = w, c.h = h, c.a = a, c.r = r, c.g = g, c.b = b, c.strict_glyphs = (uint8_t)strict;
    if (text) snprintf(c.text, sizeof(c.text), "%s", text);
    return c;
}

// HUD strings of one probe invocation (src/pipeline.rs:126-156 / src/pipeline_ir.rs:168-190)
struct HudText {
    char fps[48], timing[48];
};
static void hud_text(vt_context* c, bool nv12, const char* const* hud_override, HudText& h) {
    vt_timing tm;
    vt_timing_get(c->tracker, &tm);
    snprintf(h.fps, sizeof(h.fps), "FPS: %.0f", tm.fps);
    if (nv12) snprintf(h.timing, sizeof(h.timing), "conv:%.1fms trk:%.1fms", tm.avg_conv_ms, tm.avg_track_ms);
    else snprintf(h.timing, sizeof(h.timing), "trk:%.1fms", tm.avg_track_ms);
    if (hud_override && hud_override[0]) snprintf(h.fps, sizeof(h.fps), "%s", hud_override[0]);
    if (hud_override && hud_override[1]) snprintf(h.timing, sizeof(h.timing), "%s", hud_override[1]);
}

// The overlay of one probe invocation as a command list, draw order of the reference (src/pipeline.rs:125-174 /
// src/pipeline_ir.rs:165-202: background, state, FPS, timing, score, cursor / selection, box + crosshair).
// `state` = state_name() after process_frame; score / box as ctx.current_score / the box the reference would draw.
// cond / from_result != 0 are used by the one-synchronisation path, where score and box come from the device-side result.
static void hud_commands(const vt_context* c, bool nv12, int state, const HudText& h, bool draw_box, const vt_bbox& b, float score, uint8_t cond,
                         bool from_result, std::vector<vt::HudCmd>& out) {
    static const char* const names[4] = {"SELECT START", "SELECT END", "TRACKING", "LOST"};
    const bool tracking = state == VT_STATE_TRACKING, selecting = state == VT_STATE_SELECT_START || state == VT_STATE_SELECT_END;
    const int strict = nv12 ? 0 : 1;  // the RGB path looks glyphs up with get_glyph, which panics (src/drawing.rs:99)
    auto push = [&](const vt_overlay_cmd& cmd, uint8_t cnd, uint8_t fr = vt::VT_HUD_GIVEN) { out.push_back(vt::HudCmd{cmd, cnd, fr}); };
    char score_line[48];
    snprintf(score_line, sizeof(score_line), "score: %.0f%%", score * 100.0f);
    push(make_cmd(VT_OV_TEXT, 15, 15, 0, 0, 2, 255, 0, 0, names[state], strict), cond);
    if (cond != vt::VT_HUD_IF_FAIL) {  // (the lines common to both outcomes are queued once, with the first variant)
        push(make_cmd(VT_OV_TEXT, 15, 40, 0, 0, 2, 255, 0, 0, h.fps, strict), vt::VT_HUD_ALWAYS);
        push(make_cmd(VT_OV_TEXT, 15, 65, 0, 0, 1, 200, 0, 0, h.timing, strict), vt::VT_HUD_ALWAYS);
    }
    if (tracking) {
        if (from_result) push(make_cmd(VT_OV_TEXT, nv12 ? 250 : 200, 15, 0, 0, 2, 255, 0, 0, "score: ", strict), cond, vt::VT_HUD_SCORE_TEXT);
        else push(make_cmd(VT_OV_TEXT, nv12 ? 250 : 200, 15, 0, 0, 2, 255, 0, 0, score_line, strict), cond);
    }
    const vt_selection sel{c->selection.cursor_x, c->selection.cursor_y, c->selection.start_x, c->selection.start_y, c->selection.phase, 0, 0};
    if (selecting) {
        // (the fail variant of a confirm frame shows the reset selection: cursor back in the centre, src/tracker_context.rs:100-109)
        const bool reset = cond == vt::VT_HUD_IF_FAIL;
        const int cx = reset ? c->frame_width / 2 : sel.cursor_x, cy = reset ? c->frame_height / 2 : sel.cursor_y;
        if (nv12) push(make_cmd(VT_OV_CURSOR, cx, cy, 0, 0, 0, 255, 0, 0), cond);
        else push(make_cmd(VT_OV_CURSOR, cx, cy, 0, 0, 0, 0, 255, 0), cond);
        if (!reset && state == VT_STATE_SELECT_END) {
            if (nv12) push(make_cmd(VT_OV_SELECTION, sel.start_x, sel.start_y, sel.cursor_x, sel.cursor_y, 0, 255, 0, 0), cond);
            else push(make_cmd(VT_OV_SELECTION, sel.start_x, sel.start_y, sel.cursor_x, sel.cursor_y, 0, 255, 255, 0), cond);
        }
    }
    if (draw_box) {
        const uint8_t r = nv12 ? 255 : 0, g = nv12 ? 0 : 255;
        push(make_cmd(VT_OV_RECT, b.x, b.y, b.width, b.height, 3, r, g, 0), cond, from_result ? vt::VT_HUD_RESULT_RECT : vt::VT_HUD_GIVEN);
        push(make_cmd(VT_OV_CROSSHAIR, b.x + b.width / 2, b.y + b.height / 2, 0, 0, 15, r, g, 0), cond,
             from_result ? vt::VT_HUD_RESULT_CROSS : vt::VT_HUD_GIVEN);
    }
}

static void probe_log(vt_context* c, bool nv12, uint64_t num) {
    const uint64_t every = nv12 ? 120 : 60;  // src/pipeline.rs:176 / src/pipeline_ir.rs:210
    static const bool log_enabled = getenv("VT_PROBE_LOG") != nullptr;  // the reference prints unconditionally
    if (log_enabled && num % every == 0 && num > 0) {
        vt_timing tm;
        vt_timing_get(c->tracker, &tm);
        printf("\r[%s] FPS: %.0f | conv: %.1fms | track: %.1fms\r\n", vt_context_state_name(c), tm.fps, tm.avg_conv_ms, tm.avg_track_ms);
    }
}

// Pageable frames: process_frame (one synchronisation), then the overlay as explicit commands on the device copy of the frame and a
// copy of the touched rows back (a second synchronisation).
static vt_status probe_two_step(vt_context* c, uint8_t* frame, size_t len, const char* const* hud_override, bool nv12) {
    vt_tracker* t = c->tracker;
    // conversion + tracking, src/pipeline.rs:104-120.  The conversion is fused into the crop kernel, so
    // `conv` is the device-timed preprocess stage of this frame and `track` the wall time of process_frame.
    const auto t1 = std::chrono::steady_clock::now();
    int32_t has = 0;
    vt_bbox bb{0, 0, 0, 0};
    vt_status st = vt_context_process_frame(c, frame, len, &has, &bb);
    if (st != VT_OK) return st;
    const uint64_t track_us = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t1).count();
    vt_timing tm;
    vt_timing_get(t, &tm);
    vt_timing_add_times(t, c->frame_on_device ? (uint64_t)(tm.preprocess_ms * 1000.f) : 0, track_us);
    HudText h;
    hud_text(c, nv12, hud_override, h);
    const int state = vt_context_state(c);
    std::vector<vt::HudCmd> hud;
    if (nv12) hud.push_back(vt::HudCmd{make_cmd(VT_OV_BACKGROUND, 10, 10, 400, 80, 150, 0, 0, 0), vt::VT_HUD_ALWAYS, vt::VT_HUD_GIVEN});
    const bool draw_box = has || (state == VT_STATE_TRACKING && c->has_bbox);
    hud_commands(c, nv12, state, h, draw_box, has ? bb : c->current_bbox, c->current_score, vt::VT_HUD_ALWAYS, false, hud);
    std::vector<vt_overlay_cmd> cmds;
    for (const vt::HudCmd& hc : hud) cmds.push_back(hc.cmd);
    return c->frame_on_device ? vt_overlay_current(t, frame, len, cmds.data(), (int32_t)cmds.size())
                              : vt_overlay(t, frame, len, cmds.data(), (int32_t)cmds.size());
}

// Pinned frames and device surfaces: ONE synchronisation per probed frame.  Everything in the HUD except score / box / the state after
// the gate is known before the frame runs; the list carries the commands of both outcomes and the frame's last kernel picks by the gate,
// renders the score digits and the box from the device-side result and mirrors the touched pixels into the pinned frame (a surface,
// surf != null, is drawn in place: frame / len unused).  The timing line shows the rolling means up to the PREVIOUS frame (this frame's
// own conv / track times exist only once it has completed; the text is timing dependent and not part of pixel parity, SURVEY.md §8 a16).
static vt_status probe_one_sync(vt_context* c, uint8_t* frame, size_t len, const vt_surface* surf, const char* const* hud_override, bool nv12) {
    vt_tracker* t = c->tracker;
    static const char* const where = "vt_probe_frame_surface";
    const auto t1 = std::chrono::steady_clock::now();
    HudText h;
    hud_text(c, nv12, hud_override, h);
    // what process_frame will do with this frame (src/tracker_context.rs:64-155)
    const bool init_update = c->state == AppState::Selecting && c->pending_confirm && c->selection.phase == 1;
    const bool update = c->state == AppState::Tracking;
    std::vector<vt::HudCmd> hud;
    if (nv12) hud.push_back(vt::HudCmd{make_cmd(VT_OV_BACKGROUND, 10, 10, 400, 80, 150, 0, 0, 0), vt::VT_HUD_ALWAYS, vt::VT_HUD_GIVEN});
    int32_t has = 0;
    vt_bbox bb{0, 0, 0, 0};
    vt_status st;
    if (!init_update && !update) {
        // no tracker call on this frame: the state machine steps on the host first, the HUD shows the new state
        process_frame_core(c, [&](vt_bbox) { return UpdateOutcome{false, vt_result{}}; }, [&]() { return UpdateOutcome{false, vt_result{}}; }, &has, &bb);
        hud_commands(c, nv12, vt_context_state(c), h, false, bb, c->current_score, vt::VT_HUD_ALWAYS, false, hud);
        if ((st = vt::tracker_set_hud(t, hud.data(), (int)hud.size())) != VT_OK) return st;
        if ((st = surf ? vt::tracker_submit_surface(t, surf, false, where) : vt::tracker_submit_hud_only(t, frame, len)) != VT_OK) return st;
        vt_result r;
        st = vt_tracker_wait(t, &r);
        if (st != VT_OK) return st;
        vt_timing_add_times(t, 0, (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t1).count());
        return VT_OK;
    }
    if (init_update) {  // return value ignored, like the reference (:88)
        if (surf) vt::tracker_init_surface(t, 0, surf, c->selection.get_bbox(), where);
        else vt_tracker_init(t, 0, frame, len, c->selection.get_bbox());
    }
    // both outcomes: gate passed -> TRACKING + score + box; failed -> LOST (tracking frame) / SELECT START with the selection reset (confirm frame)
    hud_commands(c, nv12, VT_STATE_TRACKING, h, true, bb, 0.f, vt::VT_HUD_IF_PASS, true, hud);
    hud_commands(c, nv12, update ? VT_STATE_LOST : VT_STATE_SELECT_START, h, false, bb, 0.f, vt::VT_HUD_IF_FAIL, false, hud);
    if ((st = vt::tracker_set_hud(t, hud.data(), (int)hud.size())) != VT_OK) return st;
    UpdateOutcome o;
    memset(&o.r, 0, sizeof(o.r));
    st = surf ? vt::tracker_submit_surface(t, surf, true, where) : vt_tracker_submit(t, frame, len);
    if (st == VT_OK) st = vt_tracker_wait(t, &o.r);
    o.ok = st == VT_OK && o.r.status == VT_OK;
    c->frame_on_device = st == VT_OK;
    // the state machine consumes the outcome exactly as in process_frame (the device applied the same gate to the same fp32 score)
    process_frame_core(c, [&](vt_bbox) { return o; }, [&]() { return o; }, &has, &bb);
    const uint64_t track_us = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t1).count();
    vt_timing tm;
    vt_timing_get(t, &tm);
    vt_timing_add_times(t, c->frame_on_device ? (uint64_t)(tm.preprocess_ms * 1000.f) : 0, track_us);
    return VT_OK;
}

// ≙ the streaming thread invoking the probe once per buffer (src/pipeline.rs:65-67): n frames of a host ring through vt_probe_frame
vt_status vt_context_run_ring(vt_context* c, uint8_t* frames, size_t stride, size_t frame_len, int32_t ring, int32_t first, int32_t n,
                              const char* const* hud_override, const uint8_t* pristine, double* latency_us) {
    if (!c || !c->tracker || !frames || ring <= 0 || first < 0 || n < 0 || frame_len > stride || member_refused(c, "vt_context_run_ring"))
        return VT_ERR_INVALID;
    const int fmt = c->cfg.format, W = c->frame_width, H = c->frame_height;
    for (int i = 0; i < n; ++i) {
        uint8_t* fr = frames + (size_t)((first + i) % ring) * stride;
        const auto t0 = std::chrono::steady_clock::now();
        const vt_status st = vt_probe_frame(c, fr, frame_len, hud_override);
        if (latency_us) latency_us[i] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
        if (st != VT_OK) return st;
        if (pristine) {  // HUD block (background 10,10 400x80 resp. the text lines up to x = 410) and the box drawn this frame
            const uint8_t* clean = pristine + (size_t)((first + i) % ring) * stride;
            vt::restore_rect_region(fr, clean, fmt, W, H, 10, 10, 412, 92);
            if (c->state == AppState::Tracking && c->has_bbox) vt::restore_box_region(fr, clean, fmt, W, H, c->current_bbox);
            else if (c->state == AppState::Selecting) vt::restore_rect_region(fr, clean, fmt, W, H, 0, 0, W, H);  // cursor / selection: rare, whole frame
        }
    }
    return VT_OK;
}

}  // extern "C"

// ≙ the pad-probe closure body: src/pipeline.rs:67-184 (NV12) / src/pipeline_ir.rs:100-228 (RGB24), on a host frame or a checked surface
static vt_status probe_frame(vt_context* c, uint8_t* frame, size_t len, const vt_surface* surf, const char* const* hud_override) {
    vt_tracker* t = c->tracker;
    const bool nv12 = vt::format_is_luma(c->cfg.format);  // GRAY8 / YUY2 frames take the luma-plane HUD of src/pipeline.rs:125-174
    // interval timing, src/pipeline.rs:69-79
    const auto now = std::chrono::steady_clock::now();
    if (c->have_last) vt_timing_add_interval(t, (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(now - c->last_time).count());
    c->last_time = now, c->have_last = true;
    const uint64_t num = c->frame_num++;
    const size_t need = vt::fmt_valid_bytes(c->cfg.format, c->frame_width, c->frame_height);
    const vt_status st = (surf || (len >= need && vt::frame_is_pinned(frame))) ? probe_one_sync(c, frame, len, surf, hud_override, nv12)
                                                                                         : probe_two_step(c, frame, len, hud_override, nv12);
    if (st != VT_OK) return st;
    probe_log(c, nv12, num);
    return VT_OK;
}

extern "C" {

vt_status vt_probe_frame(vt_context* c, uint8_t* frame, size_t len, const char* const* hud_override) {
    if (!c || !c->tracker || !frame || member_refused(c, "vt_probe_frame")) return VT_ERR_INVALID;
    return probe_frame(c, frame, len, nullptr, hud_override);
}

vt_status vt_probe_frame_surface(vt_context* c, const vt_surface* s, const char* const* hud_override) {
    if (!c || !c->tracker || !s) {
        vt::set_error("vt_probe_frame_surface: null context (or a context without a tracker) or surface");
        return VT_ERR_INVALID;
    }
    if (member_refused(c, "vt_probe_frame_surface")) return VT_ERR_INVALID;
    const vt_status st = vt::tracker_check_surface(c->tracker, 0, s, "vt_probe_frame_surface");  // before the state machine steps
    if (st != VT_OK) return st;
    return probe_frame(c, nullptr, 0, s, hud_override);
}

// ---- probe groups: n cameras, one batched forward and one synchronisation per step (include/vt_tracker.h) ----------------------
vt_status vt_probe_group_create(const vt_config* cfg, int32_t n_streams, const vt_stream_geometry* geoms, vt_probe_group** out) {
    if (out) *out = nullptr;
    if (!cfg || !out) {
        vt::set_error("vt_probe_group_create: null config or output");
        return VT_ERR_INVALID;
    }
    if (n_streams < 1 || n_streams > vt::kMaxWin) {
        vt::set_error("vt_probe_group_create: %d streams (a group has 1..%d)", n_streams, vt::kMaxWin);
        return VT_ERR_INVALID;
    }
    vt_config c;
    vt_status st = vt::resolve_config(cfg, &c);
    if (st != VT_OK) return st;
    for (int i = 0; geoms && i < n_streams; ++i)  // (the rule of vt_tracker_set_stream_geometry, checked before anything is allocated)
        if (!vt::geometry_ok(geoms[i].format, geoms[i].width, geoms[i].height) || geoms[i].reserved != 0) {
            vt::set_error("vt_probe_group_create: stream %d: format %d, %d x %d (reserved %d) is not a frame geometry", i, geoms[i].format,
                          geoms[i].width, geoms[i].height, geoms[i].reserved);
            return VT_ERR_INVALID;
        }
    c.max_targets = n_streams;  // one VitTrack per TrackerContext: one target slot per stream
    c.box_overlay = 0;          // the probe queues explicit overlay commands (the box is one of them)
    vt_tracker* t = nullptr;
    if ((st = vt_tracker_create(&c, &t)) != VT_OK) return st;
    for (int i = 0; geoms && i < n_streams && st == VT_OK; ++i) st = vt_tracker_set_stream_geometry(t, i, &geoms[i]);  // before HUD mode
    if (st == VT_OK) st = vt::tracker_make_group(t, n_streams);
    if (st != VT_OK) {
        vt_tracker_destroy(t);
        return st;
    }
    vt_probe_group* g = new vt_probe_group();
    g->tracker = t;
    for (int i = 0; i < n_streams; ++i) {
        vt_stream_geometry sg;
        vt_tracker_get_stream_geometry(t, i, &sg);
        vt_context* ctx = new vt_context(sg.width, sg.height);
        ctx->tracker = t, ctx->group = g;
        ctx->cfg = c;
        ctx->cfg.weights_path = nullptr, ctx->cfg.format = sg.format, ctx->cfg.width = sg.width, ctx->cfg.height = sg.height, ctx->cfg.max_targets = 1;
        g->members.push_back(ctx);
    }
    *out = g;
    return VT_OK;
}

void vt_probe_group_destroy(vt_probe_group* g) {
    if (!g) return;
    if (g->tracker) vt_tracker_destroy(g->tracker);
    for (vt_context* c : g->members) delete c;
    delete g;
}

int32_t vt_probe_group_size(const vt_probe_group* g) { return g ? (int32_t)g->members.size() : VT_ERR_INVALID; }

vt_context* vt_probe_group_context(vt_probe_group* g, int32_t stream) {
    return g && stream >= 0 && stream < (int32_t)g->members.size() ? g->members[(size_t)stream] : nullptr;
}

// ≙ probe_one_sync for every stream of the group at once: each stream predicts whether its state machine calls VitTrack on this frame
// (TRACKING: update; SELECT END with a pending confirm: init on this stream's frame into its slot, then update).  The others step their
// state machines on the host first and queue their final HUD; those that take part queue the HUD of both outcomes, and the step's last
// kernel picks per stream by that stream's own result.  A stream that leaves TRACKING, or whose confirm fails the gate, gives up its slot:
// LOST and SELECT never call update, and tracking resumes only through a fresh init.
// frames / lens: every stream's pinned frame, or surfs: every stream's device surface (checked by the caller)
static vt_status probe_group_step(vt_probe_group* g, uint8_t* const* frames, const size_t* lens, const vt_surface* surfs,
                                  const char* const* hud_override) {
    vt_tracker* t = g->tracker;
    const int n = (int)g->members.size();
    const auto now = std::chrono::steady_clock::now();  // interval timing, src/pipeline.rs:69-79 (one probe per stream and step)
    if (g->have_last) vt_timing_add_interval(t, (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(now - g->last_time).count());
    g->last_time = now, g->have_last = true;
    const uint64_t num = g->frame_num++;
    const auto t1 = std::chrono::steady_clock::now();
    std::vector<bool> part((size_t)n, false);
    std::vector<vt::HudCmd> hud;
    vt_status st;
    bool any = false;
    for (int i = 0; i < n; ++i) {
        vt_context* c = g->members[(size_t)i];
        const bool nv12 = vt::format_is_luma(c->cfg.format);
        HudText h;
        hud_text(c, nv12, hud_override, h);
        // what process_frame will do with this frame (src/tracker_context.rs:64-155)
        const bool init_update = c->state == AppState::Selecting && c->pending_confirm && c->selection.phase == 1;
        const bool update = c->state == AppState::Tracking;
        part[(size_t)i] = init_update || update;
        any = any || part[(size_t)i];
        hud.clear();
        if (nv12) hud.push_back(vt::HudCmd{make_cmd(VT_OV_BACKGROUND, 10, 10, 400, 80, 150, 0, 0, 0), vt::VT_HUD_ALWAYS, vt::VT_HUD_GIVEN});
        int32_t has = 0;
        vt_bbox bb{0, 0, 0, 0};
        if (!part[(size_t)i]) {
            // no tracker call on this frame: the state machine steps on the host first, the HUD shows the new state; a slot still held
            // (Cancel while tracking) leaves the forward
            if (vt::tracker_group_active(t, i) && (st = vt::tracker_group_drop(t, i)) != VT_OK) return st;
            process_frame_core(c, [&](vt_bbox) { return UpdateOutcome{false, vt_result{}}; }, [&]() { return UpdateOutcome{false, vt_result{}}; }, &has, &bb);
            hud_commands(c, nv12, vt_context_state(c), h, false, bb, c->current_score, vt::VT_HUD_ALWAYS, false, hud);
        } else {
            if (init_update && surfs)  // return value ignored (:88)
                vt::tracker_init_surface(t, i, &surfs[i], c->selection.get_bbox(), "vt_probe_group_frame_surface");
            else if (init_update)
                vt::tracker_group_init(t, i, frames[i], lens[i], c->selection.get_bbox());
            // both outcomes: gate passed -> TRACKING + score + box; failed -> LOST (tracking frame) / SELECT START, selection reset (confirm)
            hud_commands(c, nv12, VT_STATE_TRACKING, h, true, bb, 0.f, vt::VT_HUD_IF_PASS, true, hud);
            hud_commands(c, nv12, update ? VT_STATE_LOST : VT_STATE_SELECT_START, h, false, bb, 0.f, vt::VT_HUD_IF_FAIL, false, hud);
        }
        if ((st = vt::tracker_set_hud(t, hud.data(), (int)hud.size(), i)) != VT_OK) return st;
    }
    std::vector<vt_result> res((size_t)n);
    memset(res.data(), 0, sizeof(vt_result) * res.size());
    st = vt::tracker_submit_group(t, frames, lens, surfs);
    if (st == VT_OK) st = vt_tracker_wait(t, res.data());
    if (st != VT_OK && !any) return st;  // (nothing was drawn; with streams in the forward a failed step is their Err, as in probe_one_sync)
    for (int i = 0; i < n; ++i) {
        if (!part[(size_t)i]) continue;
        vt_context* c = g->members[(size_t)i];
        UpdateOutcome o;
        o.r = res[(size_t)i];
        o.ok = st == VT_OK && o.r.status == VT_OK;
        c->frame_on_device = st == VT_OK;
        int32_t has = 0;
        vt_bbox bb{0, 0, 0, 0};
        // the state machine consumes the outcome exactly as in process_frame (the device applied the same gate to the same fp32 score)
        process_frame_core(c, [&](vt_bbox) { return o; }, [&]() { return o; }, &has, &bb);
        if (c->state != AppState::Tracking && vt::tracker_group_active(t, i)) vt::tracker_group_drop(t, i);
    }
    const uint64_t track_us = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t1).count();
    vt_timing tm;
    vt_timing_get(t, &tm);
    vt_timing_add_times(t, any && st == VT_OK ? (uint64_t)(tm.preprocess_ms * 1000.f) : 0, track_us);
    for (vt_context* c : g->members) probe_log(c, vt::format_is_luma(c->cfg.format), num);  // one line per stream, with its state
    return VT_OK;
}

vt_status vt_probe_group_frame(vt_probe_group* g, uint8_t* const* frames, const size_t* lens, const char* const* hud_override) {
    if (!g || !g->tracker || !frames || !lens) {
        vt::set_error("vt_probe_group_frame: null group, frames or lengths");
        return VT_ERR_INVALID;
    }
    const int n = (int)g->members.size();
    for (int i = 0; i < n; ++i) {
        const vt_context* c = g->members[(size_t)i];
        const size_t need = vt::fmt_frame_bytes(c->cfg.format, c->frame_width, c->frame_height);
        if (!frames[i] || lens[i] < need || !vt::frame_is_pinned(frames[i])) {
            vt::set_error("vt_probe_group_frame: frame %d must be a full frame (%zu bytes for its %dx%d format %d, got %zu) in pinned host memory "
                          "(vt_alloc_pinned)", i, need, c->frame_width, c->frame_height, c->cfg.format, frames[i] ? lens[i] : (size_t)0);
            return VT_ERR_INVALID;
        }
    }
    return probe_group_step(g, frames, lens, nullptr, hud_override);
}

vt_status vt_probe_group_frame_surface(vt_probe_group* g, const vt_surface* surfaces, int32_t n, const char* const* hud_override) {
    if (!g || !g->tracker || !surfaces) {
        vt::set_error("vt_probe_group_frame_surface: null group or surfaces");
        return VT_ERR_INVALID;
    }
    if (n != (int32_t)g->members.size()) {
        vt::set_error("vt_probe_group_frame_surface: %d surfaces for a group of %d streams (one per stream)", n, (int)g->members.size());
        return VT_ERR_INVALID;
    }
    for (int i = 0; i < n; ++i) {  // each against its stream's geometry, before any state machine steps
        const vt_status st = vt::tracker_check_surface(g->tracker, i, &surfaces[i], "vt_probe_group_frame_surface");
        if (st != VT_OK) return st;
    }
    return probe_group_step(g, nullptr, nullptr, surfaces, hud_override);
}

// ≙ vt_context_run_ring for a group: n steps, stream i's frames from its own ring
vt_status vt_probe_group_run_ring(vt_probe_group* g, uint8_t* const* rings, size_t stride, size_t frame_len, int32_t ring, int32_t first,
                                  int32_t n, const char* const* hud_override, const uint8_t* const* pristine, double* latency_us) {
    if (!g || !g->tracker || !rings || ring <= 0 || first < 0 || n < 0 || frame_len > stride) {
        vt::set_error("vt_probe_group_run_ring: invalid argument");
        return VT_ERR_INVALID;
    }
    const int ns = (int)g->members.size();
    std::vector<uint8_t*> fr((size_t)ns);
    std::vector<size_t> lens((size_t)ns, frame_len);
    for (int i = 0; i < n; ++i) {
        const size_t off = (size_t)((first + i) % ring) * stride;
        for (int k = 0; k < ns; ++k) fr[(size_t)k] = rings[k] + off;
        const auto t0 = std::chrono::steady_clock::now();
        const vt_status st = vt_probe_group_frame(g, fr.data(), lens.data(), hud_override);
        if (latency_us) latency_us[i] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
        if (st != VT_OK) return st;
        for (int k = 0; pristine && k < ns; ++k) {  // what vt_context_run_ring restores, per stream
            const vt_context* c = g->members[(size_t)k];
            if (!pristine[k]) continue;
            const uint8_t* clean = pristine[k] + off;
            const int fmt = c->cfg.format, W = c->frame_width, H = c->frame_height;
            vt::restore_rect_region(fr[(size_t)k], clean, fmt, W, H, 10, 10, 412, 92);
            if (c->state == AppState::Tracking && c->has_bbox) vt::restore_box_region(fr[(size_t)k], clean, fmt, W, H, c->current_bbox);
            else if (c->state == AppState::Selecting) vt::restore_rect_region(fr[(size_t)k], clean, fmt, W, H, 0, 0, W, H);
        }
    }
    return VT_OK;
}

}  // extern "C"
