/* The per-box body of the reference's main() (src/YOLO_cropping_ppf_test.cpp:91-122) through the C ABI with the engine the
 * reference calls, PPF3DDetector::match_S2B, as INTEGRATION.md section 3c shows it: the detector trained and the frame
 * uploaded once, one b200cv_match_object call per YOLO box.  The twin of c_abi_frame_example.c (the PCL engine).
 *
 * usage: c_abi_cv_frame_example DIR leaf relative_sampling_step rows cols fx fy ppx ppy x y w h [x y w h ...]
 *   DIR/scene.f32  the frame, float32 x y z rows
 *   DIR/depth.f32  the depth image, rows x cols float32 metres (row-major)
 *   DIR/model.f32  the model, float32 x y z nx ny nz rows
 * prints one line per box: "box <i> <rc> <votes> <clusters> <residual> <16 pose values, row-major>" */
#include <stdio.h>
#include <stdlib.h>
#include "b200ppf.h"

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
    size_t n_scene = 0, n_depth = 0, n_model = 0;
    float *scene_xyz, *depth, *model_rows;
    b200ppf_ctx *ctx = NULL;
    b200cv_detector *det = NULL;
    b200ppf_cloud *frame = NULL, *model = NULL;
    int rows, cols, i, k, status = 1;
    double fx, fy, ppx, ppy;
    if (argc < 14 || (argc - 10) % 4 != 0) {
        fprintf(stderr, "usage: %s DIR leaf relative_sampling_step rows cols fx fy ppx ppy x y w h [x y w h ...]\n", argv[0]);
        return 2;
    }
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
    /* PPF3DDetector(relativeSamplingStep, 0.05) + trainModel (include/CloudProcessing.h:205-236); the full model also
     * serves the ICP (models[id]) */
    if (b200cv_detector_create(ctx, atof(argv[3]), 0.05, 30, &det) || b200cv_detector_train(det, model_rows, n_model / 6, 6) ||
        b200ppf_cloud_upload(ctx, model_rows, n_model / 6, 6, 3, &model) || b200ppf_cloud_upload_xyz(ctx, scene_xyz, n_scene / 3, 3, &frame)) {
        fprintf(stderr, "%s\n", b200ppf_last_error(ctx));
        goto done;
    }
    for (i = 10; i + 3 < argc; i += 4) {
        float corners[12];
        b200cv_object_params prm;
        b200ppf_object_result r;
        int rc;
        if (b200ppf_frustum_corners(depth, rows, cols, atoi(argv[i]), atoi(argv[i + 1]), atoi(argv[i + 2]), atoi(argv[i + 3]), fx, fy,
                                    ppx, ppy, corners))
            goto done;
        b200cv_object_params_default(&prm);
        prm.leaf = (float)atof(argv[2]);
        rc = b200cv_match_object(det, frame, corners, model, &prm, &r, NULL, NULL);
        printf("box %d %d %u %u %.17g", (i - 10) / 4, rc, rc ? 0u : r.votes, rc ? 0u : r.n_poses, rc ? 0.0 : r.residual);
        for (k = 0; k < 16; ++k) printf(" %.17g", rc ? 0.0 : r.pose[k]);
        printf("\n");
        if (rc) fprintf(stderr, "box %d: %s\n", (i - 10) / 4, b200ppf_last_error(ctx));
    }
    status = 0;
done:
    b200ppf_cloud_free(frame);
    b200ppf_cloud_free(model);
    b200cv_detector_free(det);
    b200ppf_destroy(ctx);
    free(scene_xyz);
    free(depth);
    free(model_rows);
    return status;
}
