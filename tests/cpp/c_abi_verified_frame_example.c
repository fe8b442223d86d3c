/* c_abi_multi_box_example.c with pose verification, as INTEGRATION.md section 3c shows it: the detector trained and the
 * frame uploaded once, then ONE b200cv_match_frame_verified call for all YOLO boxes (one crop pass, one ICP launch for
 * every object, one scoring of every object's refined candidates), the best-supported candidate of each box returned with
 * its fit.  Every box here is of the same class, so the one detector and the one model serve them all.
 *
 * usage: c_abi_multi_box_example DIR leaf relative_sampling_step rows cols fx fy ppx ppy x y w h [x y w h ...]
 *   DIR/scene.f32  the frame, float32 x y z rows
 *   DIR/depth.f32  the depth image, rows x cols float32 metres (row-major)
 *   DIR/model.f32  the model, float32 x y z nx ny nz rows
 * prints one line per box: "box <i> <status> <votes> <clusters> <residual> <fit> <inliers> <visible> <rank>
 * <16 pose values, row-major>": the best candidate's fit and its rank among the pose clusters (0 = most voted) */
#include <stdio.h>
#include <stdlib.h>
#include "b200ppf.h"

#define MAX_BOXES 64

static float *read_f32(const char *dir, const char *name, size_t *count) {
    char path[4096];
    FILE *f;
    long bytes;
    float *buf;
    snprintf(path, sizeof(path), "%s/%s", dir, name);
    f = fopen(path, "rb");
    if (!f) return NULL;
    fseek(f, 0, SEEK_END);
    bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    buf = (float *)malloc(bytes > 0 ? (size_t)bytes : 1);
    *count = bytes > 0 ? (size_t)bytes / sizeof(float) : 0;
    if (buf && fread(buf, sizeof(float), *count, f) != *count) {
        free(buf);
        buf = NULL;
    }
    fclose(f);
    return buf;
}

int main(int argc, char **argv) {
    size_t n_scene = 0, n_depth = 0, n_model = 0, n_boxes, b;
    float *scene_xyz, *depth, *model_rows;
    float corners[12 * MAX_BOXES];
    b200cv_detector *detectors[MAX_BOXES];
    const b200ppf_cloud *models[MAX_BOXES];
    b200ppf_object_result results[MAX_BOXES];
    b200ppf_candidate candidates[MAX_BOXES * 5]; /* max(icp_poses, 1) slots per box, best first */
    b200ppf_verify_params verify;
    int status[MAX_BOXES];
    b200cv_object_params prm;
    b200ppf_ctx *ctx = NULL;
    b200cv_detector *det = NULL;
    b200ppf_cloud *frame = NULL, *model = NULL;
    int rows, cols, k, rc = 1;
    double fx, fy, ppx, ppy;
    if (argc < 14 || (argc - 10) % 4 != 0 || (size_t)(argc - 10) / 4 > MAX_BOXES) {
        fprintf(stderr, "usage: %s DIR leaf relative_sampling_step rows cols fx fy ppx ppy x y w h [x y w h ...] (at most %d boxes)\n",
                argv[0], MAX_BOXES);
        return 2;
    }
    n_boxes = (size_t)(argc - 10) / 4;
    rows = atoi(argv[4]);
    cols = atoi(argv[5]);
    fx = atof(argv[6]);
    fy = atof(argv[7]);
    ppx = atof(argv[8]);
    ppy = atof(argv[9]);
    scene_xyz = read_f32(argv[1], "scene.f32", &n_scene);
    depth = read_f32(argv[1], "depth.f32", &n_depth);
    model_rows = read_f32(argv[1], "model.f32", &n_model);
    if (!scene_xyz || !depth || !model_rows || n_depth != (size_t)rows * (size_t)cols) {
        fprintf(stderr, "cannot read the inputs under %s\n", argv[1]);
        goto done;
    }
    if (b200ppf_create(0, &ctx)) {
        fprintf(stderr, "%s\n", b200ppf_last_error(NULL));
        goto done;
    }
    if (b200cv_detector_create(ctx, atof(argv[3]), 0.05, 30, &det) || b200cv_detector_train(det, model_rows, n_model / 6, 6) ||
        b200ppf_cloud_upload(ctx, model_rows, n_model / 6, 6, 3, &model) || b200ppf_cloud_upload_xyz(ctx, scene_xyz, n_scene / 3, 3, &frame)) {
        fprintf(stderr, "%s\n", b200ppf_last_error(ctx));
        goto done;
    }
    for (b = 0; b < n_boxes; ++b) {
        const char *const *box = (const char *const *)argv + 10 + 4 * b;
        if (b200ppf_frustum_corners(depth, rows, cols, atoi(box[0]), atoi(box[1]), atoi(box[2]), atoi(box[3]), fx, fy, ppx, ppy,
                                    corners + 12 * b)) {
            fprintf(stderr, "box %u: %s\n", (unsigned)b, b200ppf_last_error(NULL));
            goto done;
        }
        detectors[b] = det;  /* the detector and the model of box b's YOLO class */
        models[b] = model;
    }
    b200cv_object_params_default(&prm);
    prm.leaf = (float)atof(argv[2]);
    b200ppf_verify_params_default(&verify); /* 1 cm, 30 degrees */
    if (b200cv_match_frame_verified(ctx, frame, n_boxes, corners, detectors, models, &prm, &verify, results, status, candidates)) {
        fprintf(stderr, "%s\n", b200ppf_last_error(ctx));
        goto done;
    }
    for (b = 0; b < n_boxes; ++b) {
        const b200ppf_object_result *r = &results[b];
        const b200ppf_candidate *best = &candidates[b * 5]; /* prm.icp_poses = 5 slots per box */
        const int ok = status[b] == 0;
        printf("box %u %d %u %u %.17g %.9g %u %u %u", (unsigned)b, status[b], ok ? r->votes : 0u, ok ? r->n_poses : 0u,
               ok ? r->residual : 0.0, (double)best->fit.fit, best->fit.inliers, best->fit.visible, best->rank);
        for (k = 0; k < 16; ++k) printf(" %.17g", ok ? r->pose[k] : 0.0);
        printf("\n");
    }
    rc = 0;
done:
    b200ppf_cloud_free(frame);
    b200ppf_cloud_free(model);
    b200cv_detector_free(det);
    b200ppf_destroy(ctx);
    free(scene_xyz);
    free(depth);
    free(model_rows);
    return rc;
}
