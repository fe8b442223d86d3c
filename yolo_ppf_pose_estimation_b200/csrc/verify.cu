// verify.cu — pose verification (b200ppf_score_poses): how much of a pose's visible model surface the scene supports.
//
// Every distinct scene of a call gets a uniform grid of cell edge >= inlier_dist, and all of them are built in one pass:
// cell ids are box-major (scene s owns the ids cell_base[s] .. cell_base[s+1]-1), so one stable radix sort of the
// concatenated points of all scenes over a fixed 24-bit key orders every scene by cell at once, and one cell_start array
// indexes them all.  A one-past-the-end key (the total cell count) is appended so that the sort never sees zero elements:
// the call's launches are the same whatever the number of jobs, poses or scene points.
//
// The score is one block per (pose, chunk of CHUNK model points): each thread moves its points (in double), tests
// visibility, and searches the 27 cells around the moved point for the nearest scene point within inlier_dist (exact
// squared distance in double, the lower original index on ties).  Counts are exact integers; the squared distances of the
// inliers are summed in double in a fixed order (thread, then a fixed shuffle tree, then warps, then chunks), so a pose's
// record does not depend on what else the call scores.
#include <algorithm>
#include <cmath>
#include <unordered_map>
#include <vector>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

constexpr int KEY_BITS = 24;
constexpr uint32_t MAX_CELLS_TOTAL = (1u << KEY_BITS) - 1;  // leaves the id MAX_CELLS_TOTAL for the end key
constexpr uint32_t PER_SCENE_CELLS = 1u << 22;
constexpr int THREADS = 256;
constexpr uint32_t CHUNK = 1024;  // model points per block

struct VScene {
    const float4 *pos, *nrm;
    uint32_t first, n;  // its points in the call's concatenation
    uint32_t cell_base;
    GridParams gp;
};

struct VPose {
    double R[9], t[3];
    const float4 *mpos, *mnrm;
    uint32_t n_model, scene;
};

struct Partial {
    uint32_t inliers, visible;
    double sum_d2;
};

// the scene of concatenated point i: the last scene that starts at or before it (an empty scene never is that one)
__device__ __forceinline__ uint32_t scene_of(const VScene *__restrict__ sc, uint32_t n_scenes, uint32_t i) {
    uint32_t lo = 0, hi = n_scenes;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (sc[mid].first <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// the cells c-1 .. c+1 around coordinate v's cell c, inside the grid; false when c lies more than one cell outside it
__device__ __forceinline__ bool cell_range(const GridParams &gp, double v, int axis, int *lo, int *hi) {
    const float f = floorf(((float)v - gp.origin[axis]) * gp.inv_cell);
    if (!(f >= -1.0f && f <= (float)gp.dims[axis])) return false;
    const int c = (int)f;
    *lo = max(c - 1, 0);
    *hi = min(c + 1, gp.dims[axis] - 1);
    return true;
}

__global__ void verify_cell_ids_kernel(const VScene *__restrict__ sc, uint32_t n_scenes, uint32_t n_total, uint32_t end_id,
                                       uint32_t *__restrict__ ids) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_total) return;
    if (i == n_total) {
        ids[i] = end_id;
        return;
    }
    const VScene &s = sc[scene_of(sc, n_scenes, i)];
    const float4 p = s.pos[i - s.first];
    ids[i] = s.cell_base + grid_cell_linear(s.gp, grid_cell_coord(s.gp, p.x, 0), grid_cell_coord(s.gp, p.y, 1),
                                            grid_cell_coord(s.gp, p.z, 2));
}

// cell-sorted copies of the points; w of a position holds the point's index in its own scene (the tie-break)
__global__ void verify_gather_kernel(const VScene *__restrict__ sc, uint32_t n_scenes, const uint32_t *__restrict__ order,
                                     uint32_t n_total, float4 *__restrict__ spos, float4 *__restrict__ snrm) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_total) return;
    const uint32_t i = order[j];
    const VScene &s = sc[scene_of(sc, n_scenes, i)];
    float4 p = s.pos[i - s.first];
    p.w = __uint_as_float(i - s.first);
    spos[j] = p;
    snrm[j] = s.nrm[i - s.first];
}

__global__ void __launch_bounds__(THREADS, 1)
verify_score_kernel(const VPose *__restrict__ poses, const VScene *__restrict__ scenes, const uint32_t *__restrict__ cell_start,
                    const float4 *__restrict__ spos, const float4 *__restrict__ snrm, double tau2, double cos_min, int use_normals,
                    uint32_t n_chunks, Partial *__restrict__ partials) {
    const VPose &P = poses[blockIdx.x];
    const uint32_t begin = blockIdx.y * CHUNK;
    if (begin >= P.n_model) return;  // a chunk past this pose's model: the finalisation never reads it
    const uint32_t end = min(P.n_model, begin + CHUNK);
    const VScene &S = scenes[P.scene];
    const GridParams gp = S.gp;
    uint32_t inliers = 0, visible = 0;
    double sum = 0.0;
    for (uint32_t i = begin + threadIdx.x; i < end; i += THREADS) {
        const float4 mp = P.mpos[i], mn = P.mnrm[i];
        const double px = P.R[0] * mp.x + P.R[1] * mp.y + P.R[2] * mp.z + P.t[0];
        const double py = P.R[3] * mp.x + P.R[4] * mp.y + P.R[5] * mp.z + P.t[1];
        const double pz = P.R[6] * mp.x + P.R[7] * mp.y + P.R[8] * mp.z + P.t[2];
        const double nx = P.R[0] * mn.x + P.R[1] * mn.y + P.R[2] * mn.z;
        const double ny = P.R[3] * mn.x + P.R[4] * mn.y + P.R[5] * mn.z;
        const double nz = P.R[6] * mn.x + P.R[7] * mn.y + P.R[8] * mn.z;
        const bool zero_normal = mn.x == 0.0f && mn.y == 0.0f && mn.z == 0.0f;
        if (!zero_normal && !(-(nx * px + ny * py + nz * pz) > 0.0)) continue;
        ++visible;
        if (S.n == 0) continue;
        // the cell of the moved point; a point more than one cell outside the grid has no scene point within reach
        int x0, x1, y0, y1, z0, z1;
        if (!cell_range(gp, px, 0, &x0, &x1) || !cell_range(gp, py, 1, &y0, &y1) || !cell_range(gp, pz, 2, &z0, &z1)) continue;
        double best = tau2;
        uint32_t best_idx = 0xFFFFFFFFu, best_j = 0;
        for (int z = z0; z <= z1; ++z)
            for (int y = y0; y <= y1; ++y) {
                const uint32_t row = S.cell_base + grid_cell_linear(gp, x0, y, z);
                const uint32_t j0 = cell_start[row], j1 = cell_start[row + (uint32_t)(x1 - x0) + 1];
                for (uint32_t j = j0; j < j1; ++j) {
                    const float4 q = spos[j];
                    const double dx = (double)q.x - px, dy = (double)q.y - py, dz = (double)q.z - pz;
                    const double d2 = dx * dx + dy * dy + dz * dz;
                    const uint32_t idx = __float_as_uint(q.w);
                    if (d2 < best || (d2 == best && idx < best_idx)) {
                        best = d2;
                        best_idx = idx;
                        best_j = j;
                    }
                }
            }
        if (best_idx == 0xFFFFFFFFu) continue;
        if (use_normals) {
            const float4 qn = snrm[best_j];
            if (!((double)qn.x * nx + (double)qn.y * ny + (double)qn.z * nz >= cos_min)) continue;
        }
        ++inliers;
        sum += best;
    }
    // fixed-order block reduction: a shuffle tree per warp, then the warps in order
    __shared__ Partial warp_part[THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        inliers += __shfl_down_sync(0xFFFFFFFFu, inliers, o);
        visible += __shfl_down_sync(0xFFFFFFFFu, visible, o);
        sum += __shfl_down_sync(0xFFFFFFFFu, sum, o);
    }
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = Partial{inliers, visible, sum};
    __syncthreads();
    if (threadIdx.x == 0) {
        Partial t = warp_part[0];
        for (int w = 1; w < THREADS / 32; ++w) {
            t.inliers += warp_part[w].inliers;
            t.visible += warp_part[w].visible;
            t.sum_d2 += warp_part[w].sum_d2;
        }
        partials[(size_t)blockIdx.x * n_chunks + blockIdx.y] = t;
    }
}

__global__ void verify_finish_kernel(const VPose *__restrict__ poses, uint32_t n_poses, const Partial *__restrict__ partials,
                                     uint32_t n_chunks, b200ppf_pose_fit *__restrict__ fits) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_poses) return;
    const uint32_t own = (poses[k].n_model + CHUNK - 1) / CHUNK;
    uint32_t inliers = 0, visible = 0;
    double sum = 0.0;
    for (uint32_t c = 0; c < own; ++c) {
        const Partial &p = partials[(size_t)k * n_chunks + c];
        inliers += p.inliers;
        visible += p.visible;
        sum += p.sum_d2;
    }
    b200ppf_pose_fit f;
    f.inliers = inliers;
    f.visible = visible;
    f.fit = visible ? (float)inliers / (float)visible : 0.0f;
    f.rms = inliers ? (float)sqrt(sum / (double)inliers) : 0.0f;
    fits[k] = f;
}

}  // namespace

int verify_score_poses(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_verify_params &params,
                       b200ppf_pose_fit *fits) {
    // the distinct scenes, in order of first appearance, and the poses, job-major
    std::unordered_map<const b200ppf_cloud *, uint32_t> scene_index;
    std::vector<VScene> scenes;
    std::vector<const b200ppf_cloud *> scene_clouds;
    std::vector<VPose> poses;
    uint64_t n_total = 0;
    uint32_t max_chunks = 1;
    for (size_t j = 0; j < n_jobs; ++j) {
        const b200ppf_icp_job &jb = jobs[j];
        if (jb.n_poses == 0) continue;
        auto it = scene_index.find(jb.scene);
        if (it == scene_index.end()) {
            it = scene_index.emplace(jb.scene, (uint32_t)scenes.size()).first;
            VScene s{};
            s.pos = jb.scene->pos;
            s.nrm = jb.scene->nrm;
            s.first = (uint32_t)n_total;
            s.n = (uint32_t)jb.scene->n;
            n_total += jb.scene->n;
            if (n_total >= 0xFFFFFFFFull - (1u << 20))
                return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: the scenes hold more than 2^32 points in all");
            scenes.push_back(s);
            scene_clouds.push_back(jb.scene);
        }
        if (jb.model->n > 0xFFFFFFFFull - CHUNK)
            return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: a model of more than 2^32 points");
        max_chunks = std::max(max_chunks, (uint32_t)((jb.model->n + CHUNK - 1) / CHUNK));
        for (size_t k = 0; k < jb.n_poses; ++k) {
            const double *T = jb.poses16 + 16 * k;
            VPose p{};
            for (int r = 0; r < 3; ++r) {
                for (int c = 0; c < 3; ++c) p.R[3 * r + c] = T[4 * r + c];
                p.t[r] = T[4 * r + 3];
            }
            p.mpos = jb.model->pos;
            p.mnrm = jb.model->nrm;
            p.n_model = (uint32_t)jb.model->n;
            p.scene = it->second;
            poses.push_back(p);
        }
    }
    if (poses.empty()) return B200PPF_OK;
    if (poses.size() > 0x7FFFFFFFull || max_chunks > 65535)
        return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: too many poses or model points");
    // the grids: cells of edge >= inlier_dist, the scenes sharing the 24-bit id space
    const uint32_t budget = std::min<uint32_t>(PER_SCENE_CELLS, MAX_CELLS_TOTAL / (uint32_t)scenes.size());
    uint32_t n_cells = 0;
    for (size_t k = 0; k < scenes.size(); ++k) {
        VScene &s = scenes[k];
        const b200ppf_cloud *c = scene_clouds[k];
        const uint32_t cells = budget ? scene_grid_params(c->bbox_min, c->bbox_max, params.inlier_dist, &s.gp, budget) : 0;
        if (cells == 0) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: no grid fits a scene (too many scenes, or a non-finite bounding box)");
        s.cell_base = n_cells;
        n_cells += cells;
    }
    const uint32_t n = (uint32_t)n_total, n_poses = (uint32_t)poses.size();

    StreamBuf<VScene> d_scenes(ctx);
    StreamBuf<VPose> d_poses(ctx);
    StreamBuf<uint32_t> ids0(ctx), ids1(ctx), ord0(ctx), ord1(ctx), cell_start(ctx);
    StreamBuf<float4> spos(ctx), snrm(ctx);
    StreamBuf<Partial> partials(ctx);
    StreamBuf<b200ppf_pose_fit> d_fits(ctx);
    PPF_CUDA(ctx, d_scenes.alloc(scenes.size()));
    PPF_CUDA(ctx, d_poses.alloc(poses.size()));
    PPF_CUDA(ctx, ids0.alloc(n + 1));
    PPF_CUDA(ctx, ids1.alloc(n + 1));
    PPF_CUDA(ctx, ord0.alloc(n + 1));
    PPF_CUDA(ctx, ord1.alloc(n + 1));
    PPF_CUDA(ctx, cell_start.alloc((size_t)n_cells + 1));
    PPF_CUDA(ctx, spos.alloc(n));
    PPF_CUDA(ctx, snrm.alloc(n));
    PPF_CUDA(ctx, partials.alloc((size_t)n_poses * max_chunks));
    PPF_CUDA(ctx, d_fits.alloc(n_poses));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_scenes, scenes.data(), scenes.size() * sizeof(VScene), cudaMemcpyHostToDevice, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_poses, poses.data(), poses.size() * sizeof(VPose), cudaMemcpyHostToDevice, ctx->stream));

    const uint32_t n_scenes = (uint32_t)scenes.size();
    PPF_LAUNCH(ctx, verify_cell_ids_kernel, (n + 1 + 255) / 256, 256, 0, d_scenes.p, n_scenes, n, n_cells, ids0.p);
    bool in_alt = false;
    if (int rc = radix_sort_u32(ctx, ids0, ids1, ord0, ord1, nullptr, nullptr, (size_t)n + 1, MAX_CELLS_TOTAL, /*v0_iota=*/true,
                                &in_alt))
        return rc;
    const uint32_t *ids_sorted = in_alt ? ids1.p : ids0.p, *ord_sorted = in_alt ? ord1.p : ord0.p;
    if (int rc = lower_bounds(ctx, ids_sorted, n + 1, nullptr, n_cells, 0, cell_start)) return rc;
    PPF_LAUNCH(ctx, verify_gather_kernel, std::max(1u, (n + 255) / 256), 256, 0, d_scenes.p, n_scenes, ord_sorted, n, spos.p, snrm.p);

    const double tau = (double)params.inlier_dist;
    const bool use_normals = !(params.normal_angle >= 3.14159265358979323846f);
    const double cos_min = use_normals ? std::cos((double)params.normal_angle) : -2.0;
    PPF_LAUNCH(ctx, verify_score_kernel, dim3(n_poses, max_chunks), THREADS, 0, d_poses.p, d_scenes.p, cell_start.p, spos.p, snrm.p,
               tau * tau, cos_min, use_normals ? 1 : 0, max_chunks, partials.p);
    PPF_LAUNCH(ctx, verify_finish_kernel, (n_poses + 127) / 128, 128, 0, d_poses.p, n_poses, partials.p, max_chunks, d_fits.p);
    PPF_CUDA(ctx, cudaMemcpyAsync(fits, d_fits, (size_t)n_poses * sizeof(b200ppf_pose_fit), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

}  // namespace b200ppf
