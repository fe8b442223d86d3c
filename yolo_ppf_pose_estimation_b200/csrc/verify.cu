// verify.cu — pose verification (b200ppf_score_poses): how much of a pose's visible model surface the scene supports.
//
// Every distinct scene of a call gets a uniform grid of cell edge >= inlier_dist, and all of them are built in one pass
// (scene_grid_build, scene_grid.cu): scene s owns the cell ids cell_base[s] ..., the sort runs over a fixed 24-bit key
// whatever the scenes, and an end key keeps it from ever seeing zero elements, so the call's launches are the same whatever
// the number of jobs, poses or scene points.  w of a cell-sorted position holds the point's index in its own scene.
//
// The score is one block per (pose, chunk of CHUNK model points): each thread moves its points (in double), tests
// visibility, and searches the 27 cells around the moved point for the nearest scene point within inlier_dist (exact
// squared distance in double, the lower original index on ties).  Counts are exact integers; the squared distances of the
// inliers are summed in double in a fixed order (thread, then a fixed shuffle tree, then warps, then chunks), so a pose's
// record does not depend on what else the call scores.
//
// The depth score (b200ppf_score_poses_depth) builds the same grids, then runs four kernels over the same (pose, chunk)
// blocks: project (each point's pixel, z' and flags into a scratch array, and each pose's splat rectangle folded with
// integer atomics), one host wait to lay the poses' z-buffers out in one slab, splat (a 64-bit atomicMin of z' over each
// in-view point's square: order-independent), score (the classification of the rule; only judged, consistent points run the
// nearest-neighbour search, the same device function) and the finish.
#include <algorithm>
#include <cmath>
#include <unordered_map>
#include <vector>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

// the scenes of a call share a fixed 24-bit id space, so the sort's passes do not depend on the jobs
constexpr uint32_t MAX_CELLS_TOTAL = (1u << 24) - 1;
constexpr uint32_t PER_SCENE_CELLS = 1u << 22;
constexpr int THREADS = 256;
constexpr uint32_t CHUNK = 1024;  // model points per block

struct VPose {
    double R[9], t[3];
    const float4 *mpos, *mnrm;
    uint32_t n_model, scene;
    uint64_t proj_first;  // the pose's first point in the projection scratch of a depth score
};

struct Partial {
    uint32_t inliers, visible;
    double sum_d2;
};

// the cells c-1 .. c+1 around coordinate v's cell c, inside the grid; false when c lies more than one cell outside it
__device__ __forceinline__ bool cell_range(const GridParams &gp, double v, int axis, int *lo, int *hi) {
    const float f = floorf(((float)v - gp.origin[axis]) * gp.inv_cell);
    if (!(f >= -1.0f && f <= (float)gp.dims[axis])) return false;
    const int c = (int)f;
    *lo = max(c - 1, 0);
    *hi = min(c + 1, gp.dims[axis] - 1);
    return true;
}

// model point i of pose P moved by it (p' = R p + t, n' = R n in double); true when it faces the camera (n'.(-p') > 0) or
// has a zero normal
__device__ __forceinline__ bool move_point(const VPose &P, uint32_t i, double p[3], double n[3]) {
    const float4 mp = P.mpos[i], mn = P.mnrm[i];
    p[0] = P.R[0] * mp.x + P.R[1] * mp.y + P.R[2] * mp.z + P.t[0];
    p[1] = P.R[3] * mp.x + P.R[4] * mp.y + P.R[5] * mp.z + P.t[1];
    p[2] = P.R[6] * mp.x + P.R[7] * mp.y + P.R[8] * mp.z + P.t[2];
    n[0] = P.R[0] * mn.x + P.R[1] * mn.y + P.R[2] * mn.z;
    n[1] = P.R[3] * mn.x + P.R[4] * mn.y + P.R[5] * mn.z;
    n[2] = P.R[6] * mn.x + P.R[7] * mn.y + P.R[8] * mn.z;
    const bool zero_normal = mn.x == 0.0f && mn.y == 0.0f && mn.z == 0.0f;
    return zero_normal || -(n[0] * p[0] + n[1] * p[1] + n[2] * p[2]) > 0.0;
}

// the nearest-neighbour test of a moved point: its nearest scene point (exact squared distance in double, the lower original
// index on ties) lies within inlier_dist and, with use_normals, that point's normal is within the normal angle of n.  *d2
// receives the squared distance of an inlier.
__device__ __forceinline__ bool nearest_inlier(const GridScene &S, const uint32_t *__restrict__ cell_start, const float4 *__restrict__ spos,
                                               const float4 *__restrict__ snrm, const double p[3], const double n[3], double tau2,
                                               double cos_min, int use_normals, double *d2) {
    if (S.n == 0) return false;
    const GridParams &gp = S.gp;
    // the cell of the moved point; a point more than one cell outside the grid has no scene point within reach
    int x0, x1, y0, y1, z0, z1;
    if (!cell_range(gp, p[0], 0, &x0, &x1) || !cell_range(gp, p[1], 1, &y0, &y1) || !cell_range(gp, p[2], 2, &z0, &z1)) return false;
    double best = tau2;
    uint32_t best_idx = 0xFFFFFFFFu, best_j = 0;
    for (int z = z0; z <= z1; ++z)
        for (int y = y0; y <= y1; ++y) {
            const uint32_t row = S.cell_base + grid_cell_linear(gp, x0, y, z);
            const uint32_t j0 = cell_start[row], j1 = cell_start[row + (uint32_t)(x1 - x0) + 1];
            for (uint32_t j = j0; j < j1; ++j) {
                const float4 q = spos[j];
                const double dx = (double)q.x - p[0], dy = (double)q.y - p[1], dz = (double)q.z - p[2];
                const double e2 = dx * dx + dy * dy + dz * dz;
                const uint32_t idx = __float_as_uint(q.w);
                if (e2 < best || (e2 == best && idx < best_idx)) {
                    best = e2;
                    best_idx = idx;
                    best_j = j;
                }
            }
        }
    if (best_idx == 0xFFFFFFFFu) return false;
    if (use_normals) {
        const float4 qn = snrm[best_j];
        if (!((double)qn.x * n[0] + (double)qn.y * n[1] + (double)qn.z * n[2] >= cos_min)) return false;
    }
    *d2 = best;
    return true;
}

__global__ void __launch_bounds__(THREADS, 1)
verify_score_kernel(const VPose *__restrict__ poses, const GridScene *__restrict__ scenes, const uint32_t *__restrict__ cell_start,
                    const float4 *__restrict__ spos, const float4 *__restrict__ snrm, double tau2, double cos_min, int use_normals,
                    uint32_t n_chunks, Partial *__restrict__ partials) {
    const VPose &P = poses[blockIdx.x];
    const uint32_t begin = blockIdx.y * CHUNK;
    if (begin >= P.n_model) return;  // a chunk past this pose's model: the finalisation never reads it
    const uint32_t end = min(P.n_model, begin + CHUNK);
    const GridScene &S = scenes[P.scene];
    uint32_t inliers = 0, visible = 0;
    double sum = 0.0;
    for (uint32_t i = begin + threadIdx.x; i < end; i += THREADS) {
        double p[3], n[3], d2;
        if (!move_point(P, i, p, n)) continue;
        ++visible;
        if (!nearest_inlier(S, cell_start, spos, snrm, p, n, tau2, cos_min, use_normals, &d2)) continue;
        ++inliers;
        sum += d2;
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

// ---- verification against the depth image ---------------------------------------------------------------------------
constexpr uint32_t FACING = 1u, IN_VIEW = 2u;

struct DepthView {
    const float *d;
    int rows, cols;
    double fx, fy, ppx, ppy;
};

// a model point after the projection: z', its pixel v * cols + u (when in view) and FACING | IN_VIEW
struct Proj {
    double z;
    uint32_t pix, flags;
};

// the z-buffer of a pose: the rectangle [u0, u0 + w) x [v0, v0 + h) of the image at off in the slab; w = 0 without one
struct ZRect {
    uint64_t off;
    int u0, v0, w, h;
};

struct DPartial {
    uint32_t inliers, judged, visible, self_occluded, occluded, violations, unknown;
    double sum_d2;
};

__device__ __forceinline__ bool depth_measured(float d) { return d > 0.0f && d < INFINITY; }  // NaN fails both

// the splat half-width of an in-view point at depth z: min(floor(fx tau / (2 z)), B200PPF_DEPTH_SPLAT_MAX)
__device__ __forceinline__ int splat_half(const DepthView &D, double tau, double z) {
    return (int)fmin(floor(D.fx * tau / (2.0 * z)), (double)B200PPF_DEPTH_SPLAT_MAX);
}

// one block per (pose, CHUNK model points): every point moved and projected into proj; the clipped splat squares of the
// block's in-view points folded into the pose's rectangle (lo = umin, vmin and hi = umax, vmax as 2 words per pose)
__global__ void __launch_bounds__(THREADS)
depth_project_kernel(const VPose *__restrict__ poses, uint32_t n_poses, DepthView D, double tau, uint32_t *__restrict__ rect,
                     Proj *__restrict__ proj) {
    const VPose &P = poses[blockIdx.x];
    const uint32_t begin = blockIdx.y * CHUNK;
    if (begin >= P.n_model) return;
    const uint32_t end = min(P.n_model, begin + CHUNK);
    uint32_t lo_u = 0xFFFFFFFFu, lo_v = 0xFFFFFFFFu, hi_u = 0u, hi_v = 0u;
    for (uint32_t i = begin + threadIdx.x; i < end; i += THREADS) {
        double p[3], n[3];
        uint32_t flags = move_point(P, i, p, n) ? FACING : 0u, pix = 0xFFFFFFFFu;
        if (p[2] > 0.0) {
            const double fu = D.fx * p[0] / p[2] + D.ppx + 0.5, fv = D.fy * p[1] / p[2] + D.ppy + 0.5;
            if (fu >= 0.0 && fu < (double)D.cols && fv >= 0.0 && fv < (double)D.rows) {  // floor() inside the image
                const int u = (int)fu, v = (int)fv, h = splat_half(D, tau, p[2]);
                flags |= IN_VIEW;
                pix = (uint32_t)v * (uint32_t)D.cols + (uint32_t)u;
                lo_u = min(lo_u, (uint32_t)max(u - h, 0));
                lo_v = min(lo_v, (uint32_t)max(v - h, 0));
                hi_u = max(hi_u, (uint32_t)min(u + h, D.cols - 1));
                hi_v = max(hi_v, (uint32_t)min(v + h, D.rows - 1));
            }
        }
        proj[P.proj_first + i] = Proj{p[2], pix, flags};
    }
    lo_u = __reduce_min_sync(0xFFFFFFFFu, lo_u);
    lo_v = __reduce_min_sync(0xFFFFFFFFu, lo_v);
    hi_u = __reduce_max_sync(0xFFFFFFFFu, hi_u);
    hi_v = __reduce_max_sync(0xFFFFFFFFu, hi_v);
    if ((threadIdx.x & 31) == 0 && lo_u != 0xFFFFFFFFu) {  // a warp with an in-view point
        atomicMin(rect + 2 * blockIdx.x, lo_u);
        atomicMin(rect + 2 * blockIdx.x + 1, lo_v);
        atomicMax(rect + 2 * (size_t)n_poses + 2 * blockIdx.x, hi_u);
        atomicMax(rect + 2 * (size_t)n_poses + 2 * blockIdx.x + 1, hi_v);
    }
}

// every in-view point writes z' into its clipped square of the pose's z-buffer; the smallest value stays (the bits of a
// positive double order as the values, so the 64-bit atomicMin is exact and order-independent)
__global__ void __launch_bounds__(THREADS)
depth_splat_kernel(const VPose *__restrict__ poses, const ZRect *__restrict__ zr, DepthView D, double tau, const Proj *__restrict__ proj,
                   unsigned long long *__restrict__ zbuf) {
    const VPose &P = poses[blockIdx.x];
    const uint32_t begin = blockIdx.y * CHUNK;
    if (begin >= P.n_model) return;
    const uint32_t end = min(P.n_model, begin + CHUNK);
    const ZRect Z = zr[blockIdx.x];
    for (uint32_t i = begin + threadIdx.x; i < end; i += THREADS) {
        const Proj q = proj[P.proj_first + i];
        if (!(q.flags & IN_VIEW)) continue;
        const int u = (int)(q.pix % (uint32_t)D.cols), v = (int)(q.pix / (uint32_t)D.cols), h = splat_half(D, tau, q.z);
        const unsigned long long bits = (unsigned long long)__double_as_longlong(q.z);
        const int u1 = min(u + h, D.cols - 1), v1 = min(v + h, D.rows - 1);
        for (int y = max(v - h, 0); y <= v1; ++y) {
            unsigned long long *row = zbuf + Z.off + (uint64_t)(y - Z.v0) * (uint64_t)Z.w;
            for (int x = max(u - h, 0); x <= u1; ++x) atomicMin(row + (x - Z.u0), bits);
        }
    }
}

// the classification of the rule (include/b200ppf.h) and the nearest-neighbour test of the judged, consistent points
__global__ void __launch_bounds__(THREADS, 1)
depth_score_kernel(const VPose *__restrict__ poses, const GridScene *__restrict__ scenes, const uint32_t *__restrict__ cell_start,
                   const float4 *__restrict__ spos, const float4 *__restrict__ snrm, const ZRect *__restrict__ zr, DepthView D,
                   double tau, double tau2, double cos_min, int use_normals, const Proj *__restrict__ proj,
                   const unsigned long long *__restrict__ zbuf, uint32_t n_chunks, DPartial *__restrict__ partials) {
    const VPose &P = poses[blockIdx.x];
    const uint32_t begin = blockIdx.y * CHUNK;
    if (begin >= P.n_model) return;
    const uint32_t end = min(P.n_model, begin + CHUNK);
    const GridScene &S = scenes[P.scene];
    const ZRect Z = zr[blockIdx.x];
    uint32_t c[7] = {0, 0, 0, 0, 0, 0, 0};  // inliers judged visible self_occluded occluded violations unknown
    double sum = 0.0;
    for (uint32_t i = begin + threadIdx.x; i < end; i += THREADS) {
        const Proj q = proj[P.proj_first + i];
        if (q.flags != (FACING | IN_VIEW)) continue;
        const int u = (int)(q.pix % (uint32_t)D.cols), v = (int)(q.pix / (uint32_t)D.cols);
        const double zb = __longlong_as_double((long long)zbuf[Z.off + (uint64_t)(v - Z.v0) * (uint64_t)Z.w + (uint64_t)(u - Z.u0)]);
        if (q.z > zb + tau) {
            ++c[3];
            continue;
        }
        ++c[2];
        const float dm = D.d[q.pix];
        if (!depth_measured(dm)) {
            ++c[6];
            continue;
        }
        const double d = (double)dm;
        if (q.z > d + tau) {
            ++c[4];
            continue;
        }
        ++c[1];
        if (q.z < d - tau) {
            ++c[5];
            continue;
        }
        double p[3], n[3], d2;
        move_point(P, i, p, n);
        if (!nearest_inlier(S, cell_start, spos, snrm, p, n, tau2, cos_min, use_normals, &d2)) continue;
        ++c[0];
        sum += d2;
    }
    // fixed-order block reduction, as verify_score_kernel's
    __shared__ DPartial warp_part[THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 7; ++k) c[k] += __shfl_down_sync(0xFFFFFFFFu, c[k], o);
        sum += __shfl_down_sync(0xFFFFFFFFu, sum, o);
    }
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = DPartial{c[0], c[1], c[2], c[3], c[4], c[5], c[6], sum};
    __syncthreads();
    if (threadIdx.x == 0) {
        DPartial t = warp_part[0];
        for (int w = 1; w < THREADS / 32; ++w) {
            const DPartial &s = warp_part[w];
            t.inliers += s.inliers, t.judged += s.judged, t.visible += s.visible, t.self_occluded += s.self_occluded;
            t.occluded += s.occluded, t.violations += s.violations, t.unknown += s.unknown, t.sum_d2 += s.sum_d2;
        }
        partials[(size_t)blockIdx.x * n_chunks + blockIdx.y] = t;
    }
}

__global__ void depth_finish_kernel(const VPose *__restrict__ poses, uint32_t n_poses, const DPartial *__restrict__ partials,
                                    uint32_t n_chunks, b200ppf_depth_fit *__restrict__ fits) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_poses) return;
    const uint32_t own = (poses[k].n_model + CHUNK - 1) / CHUNK;
    DPartial t{0, 0, 0, 0, 0, 0, 0, 0.0};
    for (uint32_t c = 0; c < own; ++c) {
        const DPartial &s = partials[(size_t)k * n_chunks + c];
        t.inliers += s.inliers, t.judged += s.judged, t.visible += s.visible, t.self_occluded += s.self_occluded;
        t.occluded += s.occluded, t.violations += s.violations, t.unknown += s.unknown, t.sum_d2 += s.sum_d2;
    }
    b200ppf_depth_fit f;
    f.inliers = t.inliers;
    f.judged = t.judged;
    f.visible = t.visible;
    f.self_occluded = t.self_occluded;
    f.occluded = t.occluded;
    f.violations = t.violations;
    f.unknown = t.unknown;
    f.fit = t.judged ? (float)t.inliers / (float)t.judged : 0.0f;
    f.rms = t.inliers ? (float)sqrt(t.sum_d2 / (double)t.inliers) : 0.0f;
    fits[k] = f;
}

}  // namespace

namespace {

// the scene grids of a call (one per distinct scene, all built in one pass) and its poses on the device
struct Grids {
    std::vector<VPose> poses;
    uint32_t max_chunks = 1;
    uint64_t n_points = 0;  // model points over all poses
    StreamBuf<VPose> d_poses;
    SceneGrids grids;
    explicit Grids(b200ppf_ctx *ctx) : d_poses(ctx), grids(ctx) {}
};

// the distinct scenes, in order of first appearance, and the poses, job-major; g->poses stays empty when there is nothing to
// score, and nothing runs then
int build_grids(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_verify_params &params, Grids *g) {
    std::unordered_map<const b200ppf_cloud *, uint32_t> scene_index;
    std::vector<const b200ppf_cloud *> scenes;
    std::vector<VPose> &poses = g->poses;
    uint64_t n_total = 0;
    uint32_t max_chunks = 1;
    for (size_t j = 0; j < n_jobs; ++j) {
        const b200ppf_icp_job &jb = jobs[j];
        if (jb.n_poses == 0) continue;
        auto it = scene_index.find(jb.scene);
        if (it == scene_index.end()) {
            it = scene_index.emplace(jb.scene, (uint32_t)scenes.size()).first;
            n_total += jb.scene->n;
            if (n_total >= 0xFFFFFFFFull - (1u << 20))
                return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: the scenes hold more than 2^32 points in all");
            scenes.push_back(jb.scene);
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
            p.proj_first = g->n_points;
            g->n_points += jb.model->n;
            poses.push_back(p);
        }
    }
    if (poses.empty()) return B200PPF_OK;
    if (poses.size() > 0x7FFFFFFFull || max_chunks > 65535)
        return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: too many poses or model points");
    g->max_chunks = max_chunks;
    // the grids: cells of edge >= inlier_dist, the scenes sharing the 24-bit id space
    const uint32_t budget = std::min<uint32_t>(PER_SCENE_CELLS, MAX_CELLS_TOTAL / (uint32_t)scenes.size());
    if (int rc = scene_grid_build(ctx, scenes.data(), (uint32_t)scenes.size(), params.inlier_dist, budget, MAX_CELLS_TOTAL,
                                  /*device_table=*/true, &g->grids))
        return rc;
    if (g->grids.n_cells == 0)
        return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "score poses: no grid fits a scene (too many scenes, or a non-finite bounding box)");
    PPF_CUDA(ctx, g->d_poses.alloc(poses.size()));
    PPF_CUDA(ctx, cudaMemcpyAsync(g->d_poses, poses.data(), poses.size() * sizeof(VPose), cudaMemcpyHostToDevice, ctx->stream));
    return B200PPF_OK;
}

struct NormalTest {
    double cos_min;
    int use_normals;
};

NormalTest normal_test(const b200ppf_verify_params &params) {
    const bool use_normals = !(params.normal_angle >= 3.14159265358979323846f);
    return NormalTest{use_normals ? std::cos((double)params.normal_angle) : -2.0, use_normals ? 1 : 0};
}

}  // namespace

int verify_score_poses(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_verify_params &params,
                       b200ppf_pose_fit *fits) {
    Grids g(ctx);
    if (int rc = build_grids(ctx, jobs, n_jobs, params, &g)) return rc;
    if (g.poses.empty()) return B200PPF_OK;
    const uint32_t n_poses = (uint32_t)g.poses.size();
    StreamBuf<Partial> partials(ctx);
    StreamBuf<b200ppf_pose_fit> d_fits(ctx);
    PPF_CUDA(ctx, partials.alloc((size_t)n_poses * g.max_chunks));
    PPF_CUDA(ctx, d_fits.alloc(n_poses));
    const double tau = (double)params.inlier_dist;
    const NormalTest nt = normal_test(params);
    PPF_LAUNCH(ctx, verify_score_kernel, dim3(n_poses, g.max_chunks), THREADS, 0, g.d_poses.p, g.grids.table.p, g.grids.cell_start.p,
               g.grids.pos.p, g.grids.nrm.p, tau * tau, nt.cos_min, nt.use_normals, g.max_chunks, partials.p);
    PPF_LAUNCH(ctx, verify_finish_kernel, (n_poses + 127) / 128, 128, 0, g.d_poses.p, n_poses, partials.p, g.max_chunks, d_fits.p);
    PPF_CUDA(ctx, cudaMemcpyAsync(fits, d_fits, (size_t)n_poses * sizeof(b200ppf_pose_fit), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int verify_score_poses_depth(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_depth_image *depth,
                             const b200ppf_verify_params &params, b200ppf_depth_fit *fits) {
    Grids g(ctx);
    if (int rc = build_grids(ctx, jobs, n_jobs, params, &g)) return rc;
    if (g.poses.empty()) return B200PPF_OK;
    const uint32_t n_poses = (uint32_t)g.poses.size();
    const DepthView D{depth->d, depth->rows, depth->cols, depth->K[0], depth->K[1], depth->K[2], depth->K[3]};
    const double tau = (double)params.inlier_dist;
    const NormalTest nt = normal_test(params);
    const dim3 grid(n_poses, g.max_chunks);

    // project every point and fold the splat rectangles
    StreamBuf<uint32_t> rect(ctx);
    StreamBuf<Proj> proj(ctx);
    PPF_CUDA(ctx, rect.alloc(4 * (size_t)n_poses));
    PPF_CUDA(ctx, proj.alloc(g.n_points));
    PPF_CUDA(ctx, cudaMemsetAsync(rect, 0xFF, 2 * (size_t)n_poses * sizeof(uint32_t), ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(rect + 2 * (size_t)n_poses, 0x00, 2 * (size_t)n_poses * sizeof(uint32_t), ctx->stream));
    PPF_LAUNCH(ctx, depth_project_kernel, grid, THREADS, 0, g.d_poses.p, n_poses, D, tau, rect.p, proj.p);
    // the call's one wait: the rectangles lay out the z-buffers
    std::vector<uint32_t> r(4 * (size_t)n_poses);
    PPF_CUDA(ctx, cudaMemcpyAsync(r.data(), rect, r.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<ZRect> zr(n_poses);
    uint64_t slab = 0;
    for (uint32_t k = 0; k < n_poses; ++k) {
        const uint32_t u0 = r[2 * k], v0 = r[2 * k + 1], u1 = r[2 * (size_t)n_poses + 2 * k], v1 = r[2 * (size_t)n_poses + 2 * k + 1];
        zr[k] = ZRect{slab, 0, 0, 0, 0};
        if (u0 > u1) continue;  // no point in view
        zr[k] = ZRect{slab, (int)u0, (int)v0, (int)(u1 - u0 + 1), (int)(v1 - v0 + 1)};
        slab += (uint64_t)zr[k].w * (uint64_t)zr[k].h;
    }
    StreamBuf<ZRect> d_zr(ctx);
    StreamBuf<unsigned long long> zbuf(ctx);
    StreamBuf<DPartial> partials(ctx);
    StreamBuf<b200ppf_depth_fit> d_fits(ctx);
    PPF_CUDA(ctx, d_zr.alloc(n_poses));
    PPF_CUDA(ctx, zbuf.alloc(slab));
    PPF_CUDA(ctx, partials.alloc((size_t)n_poses * g.max_chunks));
    PPF_CUDA(ctx, d_fits.alloc(n_poses));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_zr, zr.data(), zr.size() * sizeof(ZRect), cudaMemcpyHostToDevice, ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(zbuf, 0xFF, std::max<uint64_t>(slab, 1) * sizeof(unsigned long long), ctx->stream));  // above any positive double
    PPF_LAUNCH(ctx, depth_splat_kernel, grid, THREADS, 0, g.d_poses.p, d_zr.p, D, tau, proj.p, zbuf.p);
    PPF_LAUNCH(ctx, depth_score_kernel, grid, THREADS, 0, g.d_poses.p, g.grids.table.p, g.grids.cell_start.p, g.grids.pos.p,
               g.grids.nrm.p, d_zr.p, D, tau, tau * tau, nt.cos_min, nt.use_normals, proj.p, zbuf.p, g.max_chunks, partials.p);
    PPF_LAUNCH(ctx, depth_finish_kernel, (n_poses + 127) / 128, 128, 0, g.d_poses.p, n_poses, partials.p, g.max_chunks, d_fits.p);
    PPF_CUDA(ctx, cudaMemcpyAsync(fits, d_fits, (size_t)n_poses * sizeof(b200ppf_depth_fit), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

}  // namespace b200ppf
