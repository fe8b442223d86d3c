// scene_grid.cu — uniform grid over the scene cloud for the d/2 neighbourhood of the voting loop.
//
// PCL answers "which scene points lie within max_dist/2 of the reference point" with a FLANN
// kd-tree radius search ([PCL] registration/impl/ppf_registration.hpp, scene_search_tree_).  On the
// device the scene is bucketed into cubic cells of edge >= radius and stored cell-sorted
// (x fastest), so that the 27-cell neighbourhood of a reference point is 9 contiguous runs of
// float4 positions: the candidate sweep is a handful of coalesced loads instead of a pass over
// the whole scene.  Which points pass the radius predicate — and therefore every vote count —
// is unchanged; only the order in which they are met differs.
//
// Built per align() call (the scene changes every frame): cell ids -> stable radix sort ->
// cell_start by binary search -> gather.  All buffers come from the stream-ordered pool.
#include <algorithm>
#include <cmath>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

__global__ void grid_cell_ids_kernel(const float4 *__restrict__ pos, uint32_t n, GridParams g,
                                     uint32_t *__restrict__ cell_ids) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pos[i];
    cell_ids[i] = grid_cell_linear(g, grid_cell_coord(g, p.x, 0), grid_cell_coord(g, p.y, 1), grid_cell_coord(g, p.z, 2));
}

__global__ void grid_gather_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm,
                                   const uint32_t *__restrict__ order, uint32_t n, float4 *__restrict__ spos,
                                   float4 *__restrict__ snrm) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t o = order[i];
    spos[i] = pos[o];
    snrm[i] = nrm[o];
}

}  // namespace

void scene_grid_free(b200ppf_ctx *ctx, SceneGrid *g) {
    if (g->cell_start) cudaFreeAsync(g->cell_start, ctx->stream);
    if (g->pos) cudaFreeAsync(g->pos, ctx->stream);
    if (g->nrm) cudaFreeAsync(g->nrm, ctx->stream);
    if (g->orig) cudaFreeAsync(g->orig, ctx->stream);
    g->cell_start = nullptr;
    g->pos = g->nrm = nullptr;
    g->orig = nullptr;
}

uint32_t scene_grid_params(const float *bbox_min, const float *bbox_max, float radius, GridParams *gp, uint32_t max_cells) {
    GridParams &g = *gp;
    // cell edge: the search radius plus a margin that absorbs the rounding of the cell coordinate
    double cell = (radius > 0.0f ? (double)radius : 1e-3) * 1.001;
    double ext[3];
    for (int k = 0; k < 3; ++k) {
        ext[k] = std::max(0.0, (double)bbox_max[k] - (double)bbox_min[k]);
        if (!std::isfinite(ext[k]) || !std::isfinite((double)bbox_min[k])) return 0;  // no grid over a non-finite box
    }
    if (!std::isfinite(cell)) return 0;
    for (int guard = 0;; ++guard) {
        double cells = 1.0;
        for (int k = 0; k < 3; ++k) cells *= std::floor(ext[k] / cell) + 1.0;
        if (cells <= (double)max_cells) break;
        if (guard > 400) return 0;  // 1.26^400 exceeds any finite extent: unreachable for finite input
        cell *= 1.26;  // coarser cells stay correct (a superset of candidates), just less selective
    }
    for (int k = 0; k < 3; ++k) {
        g.origin[k] = bbox_min[k];
        g.dims[k] = (int)(std::floor(ext[k] / cell) + 1.0);
    }
    g.inv_cell = (float)(1.0 / cell);
    return (uint32_t)g.dims[0] * (uint32_t)g.dims[1] * (uint32_t)g.dims[2];
}

int scene_grid_build(b200ppf_ctx *ctx, const b200ppf_cloud *scene, float radius, SceneGrid *out) {
    *out = SceneGrid();
    const uint32_t n = (uint32_t)scene->n;
    GridParams &g = out->gp;
    out->n_cells = scene_grid_params(scene->bbox_min, scene->bbox_max, radius, &g);
    if (out->n_cells == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "scene grid: the cloud's bounding box or the search radius is not finite");

    // scratch leaves with the scope on every path; the grid's own arrays are the caller's to free (scene_grid_free,
    // also after a failure)
    StreamBuf<uint32_t> ids0(ctx), ids1(ctx), ord0(ctx), ord1(ctx);
    PPF_CUDA(ctx, ids0.alloc(n));
    PPF_CUDA(ctx, ids1.alloc(n));
    PPF_CUDA(ctx, ord0.alloc(n));
    PPF_CUDA(ctx, ord1.alloc(n));
    PPF_CUDA(ctx, cudaMallocAsync(&out->cell_start, ((size_t)out->n_cells + 1) * sizeof(uint32_t), ctx->stream));
    PPF_CUDA(ctx, cudaMallocAsync(&out->pos, std::max(1u, n) * sizeof(float4), ctx->stream));
    PPF_CUDA(ctx, cudaMallocAsync(&out->nrm, std::max(1u, n) * sizeof(float4), ctx->stream));
    const unsigned gb = (n + 255) / 256;
    bool in_alt = false;
    if (n) {
        PPF_LAUNCH(ctx, grid_cell_ids_kernel, gb, 256, 0, scene->pos, n, g, ids0.p);
        int rc = radix_sort_u32(ctx, ids0, ids1, ord0, ord1, nullptr, nullptr, n, out->n_cells - 1, /*v0_iota=*/true, &in_alt);
        if (rc) return rc;
    }
    const uint32_t *ids_sorted = in_alt ? ids1.p : ids0.p;
    const uint32_t *ord_sorted = in_alt ? ord1.p : ord0.p;
    if (int rc = lower_bounds(ctx, ids_sorted, n, nullptr, out->n_cells, 0, out->cell_start)) return rc;
    if (n) PPF_LAUNCH(ctx, grid_gather_kernel, gb, 256, 0, scene->pos, scene->nrm, ord_sorted, n, out->pos, out->nrm);
    out->orig = in_alt ? ord1.release() : ord0.release();  // sorted position -> original scene index
    return B200PPF_OK;
}

}  // namespace b200ppf
