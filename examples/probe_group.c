/* probe_group.c — the reference's two-camera deployment (the visible pipeline of src/pipeline.rs, 1920x1080 NV12, and the IR pipeline of
 * src/pipeline_ir.rs, 640x512 YUY2, each with its own TrackerContext, state machine and HUD) as ONE probe group: every step probes one
 * buffer of each camera with vt_probe_group_frame — one batched forward over the cameras that are tracking, both HUDs drawn in place, one
 * synchronisation.  The keyboard of each pipeline is scripted: a key string per camera, one key byte per step fed through
 * vt_command_from_key ('.' = no key), so the selection, confirm, tracking and cancel flow of the reference runs unattended.
 *
 *   gcc -std=c99 -Iinclude examples/probe_group.c -Lgstreamer_vit_tracker_b200 -lvittrack_b200 -o probe_group
 *   ./probe_group model.vtw visible.nv12 ir.yuy2 [visible-keys [ir-keys]]
 *
 * visible.nv12: tightly packed 1920x1080 NV12 frames; ir.yuy2: packed 640x512 YUY2 frames.  The default scripts move each cursor, set
 * the start point, drag a selection and confirm it.  Prints every camera's state once per 30 steps.  Needs a B200: there is no CPU
 * fallback. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "vt_tracker.h"

static int fail(const char* what) {
    fprintf(stderr, "%s: %s\n", what, vt_last_error());
    return 1;
}

int main(int argc, char** argv) {
    if (argc < 4 || argc > 6) {
        fprintf(stderr, "usage: %s model.vtw visible.nv12 ir.yuy2 [visible-keys [ir-keys]]\n", argv[0]);
        return 2;
    }
    /* stream 0: the visible camera; stream 1: the IR camera */
    vt_stream_geometry cams[2];
    cams[0].format = VT_FMT_NV12, cams[0].width = 1920, cams[0].height = 1080, cams[0].reserved = 0;
    cams[1].format = VT_FMT_YUY2, cams[1].width = 640, cams[1].height = 512, cams[1].reserved = 0;
    const char* keys[2] = {argc > 4 ? argv[4] : "ffw ddddss .", argc > 5 ? argv[5] : "aw dddss ."};
    vt_config cfg;
    vt_config_default(&cfg);
    cfg.weights_path = argv[1];
    cfg.format = cams[0].format, cfg.width = cams[0].width, cfg.height = cams[0].height;
    cfg.upload_window = 1; /* only the search windows and the HUD regions travel over PCIe */

    vt_probe_group* grp = NULL;
    if (vt_probe_group_create(&cfg, 2, cams, &grp) != VT_OK) return fail("vt_probe_group_create");

    const char* path[2] = {argv[2], argv[3]};
    size_t bytes[2];
    bytes[0] = (size_t)1920 * 1080 * 3 / 2, bytes[1] = (size_t)4 * ((640 + 1) / 2) * 512;
    FILE* f[2];
    uint8_t* frames[2];
    for (int i = 0; i < 2; ++i) {
        void* p = NULL;
        if (vt_alloc_pinned(bytes[i], &p) != VT_OK) return fail("vt_alloc_pinned"); /* group frames are pinned */
        frames[i] = (uint8_t*)p;
        f[i] = fopen(path[i], "rb");
        if (!f[i]) {
            perror(path[i]);
            return 1;
        }
    }
    for (long step = 0;; ++step) {
        if (fread(frames[0], 1, bytes[0], f[0]) != bytes[0] || fread(frames[1], 1, bytes[1], f[1]) != bytes[1]) break;
        for (int i = 0; i < 2; ++i) { /* this step's key of camera i (≙ draining its cmd_rx, src/pipeline.rs:84-88) */
            const size_t nk = strlen(keys[i]);
            const char key = (size_t)step < nk ? keys[i][step] : '.';
            int32_t cmd = 0, fast = 0;
            if (key != '.' && vt_command_from_key((uint8_t)key, &cmd, &fast) &&
                vt_context_handle_command(vt_probe_group_context(grp, i), cmd, fast) != VT_OK)
                return fail("vt_context_handle_command");
        }
        if (vt_probe_group_frame(grp, frames, bytes, NULL) != VT_OK) return fail("vt_probe_group_frame");
        if (step % 30 == 0) {
            for (int i = 0; i < 2; ++i) {
                const vt_context* c = vt_probe_group_context(grp, i);
                vt_bbox b;
                const int has = vt_context_current_bbox(c, &b);
                printf("step %ld camera %d: %-12s score %.3f", step, i, vt_context_state_name(c), (double)vt_context_current_score(c));
                if (has) printf(" box %d %d %d %d", b.x, b.y, b.width, b.height);
                printf("\n");
            }
        }
    }
    for (int i = 0; i < 2; ++i) {
        fclose(f[i]);
        vt_free_pinned(frames[i]);
    }
    vt_probe_group_destroy(grp);
    return 0;
}
