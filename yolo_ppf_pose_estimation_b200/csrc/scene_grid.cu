// scene_grid.cu — uniform cell-sorted grids over clouds: the one builder behind the d/2 neighbourhood of the voting loop
// (K3), the k nearest neighbours of pre-processing and the nearest-neighbour test of pose verification.
//
// PCL answers "which scene points lie within max_dist/2 of the reference point" with a FLANN
// kd-tree radius search ([PCL] registration/impl/ppf_registration.hpp, scene_search_tree_).  On the
// device the scene is bucketed into cubic cells of edge >= radius and stored cell-sorted
// (x fastest), so that the 27-cell neighbourhood of a reference point is 9 contiguous runs of
// float4 positions: the candidate sweep is a handful of coalesced loads instead of a pass over
// the whole scene.  Which points pass the radius predicate — and therefore every vote count —
// is unchanged; only the order in which they are met differs.
//
// Built per call (the scene changes every frame), all scenes of a call in one pass: cell ids are scene-major (scene s owns
// the ids cell_base[s] ..), an end key (the largest id) is appended so that the sort never sees zero elements, one stable
// radix sort orders every scene by cell at once, one cell_start array (lower_bounds over the points alone) indexes them
// all, and one gather writes the cell-sorted copies with the point's index in its own scene in pos.w.  A one-scene build
// passes its scene to the kernels by value, so it uploads nothing.  All buffers come from the stream-ordered pool.
#include <algorithm>
#include <cmath>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

// the scene of concatenated point i: the last scene that starts at or before it (an empty scene never is that one); the
// one scene of a one-scene build comes by value
__device__ __forceinline__ GridScene scene_of(const GridScene *__restrict__ sc, uint32_t n_scenes, const GridScene &one, uint32_t i) {
    if (n_scenes == 1) return one;
    uint32_t lo = 0, hi = n_scenes;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (sc[mid].first <= i) lo = mid; else hi = mid;
    }
    return sc[lo];
}

__global__ void grid_cell_ids_kernel(const GridScene *__restrict__ sc, uint32_t n_scenes, GridScene one, uint32_t n_total,
                                     uint32_t end_id, uint32_t *__restrict__ ids) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_total) return;
    if (i == n_total) {
        ids[i] = end_id;
        return;
    }
    const GridScene s = scene_of(sc, n_scenes, one, i);
    const float4 p = s.pos[i - s.first];
    ids[i] = s.cell_base + grid_cell_linear(s.gp, grid_cell_coord(s.gp, p.x, 0), grid_cell_coord(s.gp, p.y, 1),
                                            grid_cell_coord(s.gp, p.z, 2));
}

__global__ void grid_gather_kernel(const GridScene *__restrict__ sc, uint32_t n_scenes, GridScene one,
                                   const uint32_t *__restrict__ order, uint32_t n_total, float4 *__restrict__ spos,
                                   float4 *__restrict__ snrm) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_total) return;
    const uint32_t i = order[j];
    const GridScene s = scene_of(sc, n_scenes, one, i);
    float4 p = s.pos[i - s.first];
    p.w = __uint_as_float(i - s.first);
    spos[j] = p;
    snrm[j] = s.nrm[i - s.first];
}

}  // namespace

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

int scene_grid_build(b200ppf_ctx *ctx, const b200ppf_cloud *const *clouds, uint32_t n_scenes, float cell_edge,
                     uint32_t cells_per_scene, uint32_t key_limit, bool device_table, SceneGrids *out) {
    std::vector<GridScene> &scenes = out->scenes;
    scenes.assign(n_scenes, GridScene{});
    out->n_cells = 0;
    uint32_t n = 0, n_cells = 0;
    for (uint32_t k = 0; k < n_scenes; ++k) {
        GridScene &s = scenes[k];
        const b200ppf_cloud *c = clouds[k];
        const uint32_t cells = cells_per_scene ? scene_grid_params(c->bbox_min, c->bbox_max, cell_edge, &s.gp, cells_per_scene) : 0;
        if (cells == 0) return B200PPF_OK;
        s.pos = c->pos;
        s.nrm = c->nrm;
        s.first = n;
        s.n = (uint32_t)c->n;
        s.cell_base = n_cells;
        n += s.n;
        n_cells += cells;
    }
    out->n_cells = n_cells;

    StreamBuf<uint32_t> ids0(ctx), ids1(ctx), ord0(ctx), ord1(ctx);
    PPF_CUDA(ctx, ids0.alloc((size_t)n + 1));
    PPF_CUDA(ctx, ids1.alloc((size_t)n + 1));
    PPF_CUDA(ctx, ord0.alloc((size_t)n + 1));
    PPF_CUDA(ctx, ord1.alloc((size_t)n + 1));
    PPF_CUDA(ctx, out->cell_start.alloc((size_t)n_cells + 1));
    PPF_CUDA(ctx, out->pos.alloc(n));
    PPF_CUDA(ctx, out->nrm.alloc(n));
    if (device_table || n_scenes > 1) {
        PPF_CUDA(ctx, out->table.alloc(n_scenes));
        PPF_CUDA(ctx, cudaMemcpyAsync(out->table, scenes.data(), n_scenes * sizeof(GridScene), cudaMemcpyHostToDevice, ctx->stream));
    }
    const GridScene *table = n_scenes == 1 ? nullptr : out->table.p;
    const GridScene &one = scenes[0];

    const uint32_t end_id = n_cells - 1;  // sorts behind every point of the last cell (the sort is stable)
    PPF_LAUNCH(ctx, grid_cell_ids_kernel, (n + 1 + 255) / 256, 256, 0, table, n_scenes, one, n, end_id, ids0.p);
    bool in_alt = false;
    if (int rc = radix_sort_u32(ctx, ids0, ids1, ord0, ord1, nullptr, nullptr, (size_t)n + 1, std::max(key_limit, end_id),
                                /*v0_iota=*/true, &in_alt))
        return rc;
    const uint32_t *ids_sorted = in_alt ? ids1.p : ids0.p, *ord_sorted = in_alt ? ord1.p : ord0.p;
    if (int rc = lower_bounds(ctx, ids_sorted, n, nullptr, n_cells, 0, out->cell_start)) return rc;
    PPF_LAUNCH(ctx, grid_gather_kernel, std::max(1u, (n + 255) / 256), 256, 0, table, n_scenes, one, ord_sorted, n, out->pos.p,
               out->nrm.p);
    return B200PPF_OK;
}

int scene_grid_build_one(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, float cell_edge, SceneGrids *out) {
    if (int rc = scene_grid_build(ctx, &cloud, 1, cell_edge, 1u << 22, 0, /*device_table=*/false, out)) return rc;
    if (out->n_cells == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "scene grid: the cloud's bounding box or the search radius is not finite");
    return B200PPF_OK;
}

}  // namespace b200ppf
