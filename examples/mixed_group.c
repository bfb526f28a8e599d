/* mixed_group.c — a box with two different cameras tracked as ONE stream group (≙ the visible pipeline of src/pipeline.rs:26-36,
 * 1920x1080 NV12, and the IR pipeline of src/pipeline_ir.rs:27-56, 640x512 YUY2, each with its own TrackerContext): both streams go
 * through one batched ViT forward per step (vt_tracker_update_streams), each read, uploaded and drawn into with its own geometry.
 *
 *   gcc -std=c99 -Iinclude examples/mixed_group.c -Lgstreamer_vit_tracker_b200 -lvittrack_b200 -o mixed_group
 *   ./mixed_group model.vtw visible.nv12 x y w h  ir.yuy2 x y w h
 *
 * visible.nv12: tightly packed 1920x1080 NV12 frames; ir.yuy2: packed 640x512 YUY2 frames.  Each box is the target in frame 0 of its
 * file.  Needs a B200: there is no CPU fallback. */
#include <stdio.h>
#include <stdlib.h>

#include "vt_tracker.h"

static int fail(const char* what) {
    fprintf(stderr, "%s: %s\n", what, vt_last_error());
    return 1;
}

int main(int argc, char** argv) {
    if (argc != 12) {
        fprintf(stderr, "usage: %s model.vtw visible.nv12 x y w h ir.yuy2 x y w h\n", argv[0]);
        return 2;
    }
    /* slot 0: the visible camera (the handle's own geometry); slot 1: the IR camera (a geometry of its own) */
    vt_config cfg;
    vt_config_default(&cfg);
    cfg.weights_path = argv[1];
    cfg.format = VT_FMT_NV12, cfg.width = 1920, cfg.height = 1080;
    cfg.max_targets = 2;   /* one target slot per stream */
    cfg.box_overlay = 1;   /* every stream's box is drawn into its own frame */
    cfg.upload_window = 1; /* only the search windows travel over PCIe */
    vt_stream_geometry ir;
    ir.format = VT_FMT_YUY2, ir.width = 640, ir.height = 512, ir.reserved = 0;

    vt_tracker* trk = NULL;
    if (vt_tracker_create(&cfg, &trk) != VT_OK) return fail("vt_tracker_create");
    if (vt_tracker_set_stream_geometry(trk, 1, &ir) != VT_OK) return fail("vt_tracker_set_stream_geometry");

    const char* path[2] = {argv[2], argv[7]};
    const size_t bytes[2] = {(size_t)1920 * 1080 * 3 / 2, (size_t)4 * ((640 + 1) / 2) * 512};
    vt_bbox box[2];
    FILE* f[2];
    uint8_t* frames[2];
    for (int i = 0; i < 2; ++i) {
        const char* const* a = (const char* const*)argv + 3 + 5 * i;
        box[i].x = atoi(a[0]), box[i].y = atoi(a[1]), box[i].width = atoi(a[2]), box[i].height = atoi(a[3]);
        void* p = NULL;
        if (vt_alloc_pinned(bytes[i], &p) != VT_OK) return fail("vt_alloc_pinned");
        frames[i] = (uint8_t*)p;
        f[i] = fopen(path[i], "rb");
        if (!f[i]) {
            perror(path[i]);
            return 1;
        }
    }
    vt_result res[2];
    for (long step = 0;; ++step) {
        if (fread(frames[0], 1, bytes[0], f[0]) != bytes[0] || fread(frames[1], 1, bytes[1], f[1]) != bytes[1]) break;
        if (step == 0) {
            for (int i = 0; i < 2; ++i)
                if (vt_tracker_init(trk, i, frames[i], bytes[i], box[i]) != VT_OK) return fail("vt_tracker_init");
            continue;
        }
        if (vt_tracker_update_streams(trk, frames, bytes, 2, res) != VT_OK) return fail("vt_tracker_update_streams");
        for (int i = 0; i < 2; ++i)
            printf("step %ld %s: %s score %.4f box (%d, %d, %d, %d)\n", step, i ? "ir     " : "visible", res[i].success ? "ok  " : "lost",
                   res[i].score, res[i].bbox.x, res[i].bbox.y, res[i].bbox.width, res[i].bbox.height);
    }
    for (int i = 0; i < 2; ++i) fclose(f[i]), vt_free_pinned(frames[i]);
    vt_tracker_destroy(trk);
    return 0;
}
