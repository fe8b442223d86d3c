// prep.cu — scene pre-processing on the device ("next" rows, SURVEY.md §8f rank 2 and the crop of rank 4): the
// stages the reference runs between its YOLO boxes and the PPF engine, so that a frame goes full scene cloud ->
// N x 6 object cloud without leaving HBM.
//
//   P0 frustum crop       reference include/CloudProcessing.h:263-339  pcl::ConvexHull + pcl::CropHull (dim 3)
//                         on {four corner rays, origin}; include/Camera.h:50-61 back_projection_bbox
//   P1 voxel grid         reference include/CloudProcessing.h:359-377  pcl::VoxelGrid<PointXYZ>
//                         [PCL] filters/include/pcl/filters/impl/voxel_grid.hpp applyFilter
//   P2 k nearest          FLANN kd-tree behind StatisticalOutlierRemoval / NormalEstimationOMP
//      neighbours         [PCL] kdtree/include/pcl/kdtree/impl/kdtree_flann.hpp nearestKSearch
//   P3 outlier removal    reference :340-358  pcl::StatisticalOutlierRemoval<PointXYZ>(meanK = 50, thresh)
//                         [PCL] filters/include/pcl/filters/impl/statistical_outlier_removal.hpp
//   P4 normals+curvature  reference :378-401  pcl::NormalEstimationOMP<PointXYZ, Normal>, k = 30
//                         [PCL] features/normal_3d.h, common/impl/centroid.hpp, common/impl/eigen.hpp
//   P5 curvature edges    reference :402-427  EdgeExtraction (curvature > threshold)
//   P6 renormalise        reference :163-190  PointCloudXYZNormalToMat
//
// Data layout: the same float4 SoA cloud the PPF kernels read (pos = x y z 1, nrm = nx ny nz curvature; the PPF
// kernels never read nrm.w).  Neighbour search: the uniform cell-sorted grid of scene_grid.cu with a cell edge
// chosen from the point density; one thread per query point, queries taken in cell order so that a warp's
// candidates are the same few contiguous runs (L1-resident), rings of cells visited until the k-th distance is
// inside the searched block.  The k best are a sorted list of 64-bit (distance bits, index) words, which is also
// FLANN's output order (ties by index).  Everything order-dependent follows the CPU checker: voxel sums in
// original point order, covariance sums in neighbour order, un-fused float arithmetic (-fmad=false).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <new>
#include <string>
#include <vector>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

// ---- bounding box of a device cloud (PCL getMinMax3D) ---------------------------------------------------------
__device__ __forceinline__ uint32_t float_order(float f) {  // order-preserving float -> uint
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
inline float float_unorder(uint32_t u) {
    const uint32_t b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    float f;
    memcpy(&f, &b, 4);
    return f;
}

__global__ void __launch_bounds__(256) bbox_kernel(const float4 *__restrict__ pos, uint32_t n, uint32_t *__restrict__ mm) {
    uint32_t lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 p = pos[i];
        const uint32_t c[3] = {float_order(p.x), float_order(p.y), float_order(p.z)};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            lo[k] = min(lo[k], c[k]);
            hi[k] = max(hi[k], c[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        lo[k] = __reduce_min_sync(0xFFFFFFFFu, lo[k]);
        hi[k] = __reduce_max_sync(0xFFFFFFFFu, hi[k]);
    }
    __shared__ uint32_t sh[6][8];
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) sh[k][threadIdx.x >> 5] = lo[k], sh[3 + k][threadIdx.x >> 5] = hi[k];
    }
    __syncthreads();
    if (threadIdx.x < 6) {  // one atomic per block and bound
        uint32_t v = sh[threadIdx.x][0];
        for (int w = 1; w < 8; ++w) v = threadIdx.x < 3 ? min(v, sh[threadIdx.x][w]) : max(v, sh[threadIdx.x][w]);
        if (threadIdx.x < 3) atomicMin(mm + threadIdx.x, v);
        else atomicMax(mm + threadIdx.x, v);
    }
}

int cloud_bbox_from_device(b200ppf_ctx *ctx, b200ppf_cloud *c) {
    for (int k = 0; k < 3; ++k) c->bbox_min[k] = c->bbox_max[k] = 0.0f;
    if (c->n == 0) return B200PPF_OK;
    StreamBuf<uint32_t> mm(ctx);
    PPF_CUDA(ctx, mm.alloc(6));
    PPF_CUDA(ctx, cudaMemsetAsync(mm, 0xFF, 3 * sizeof(uint32_t), ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(mm + 3, 0x00, 3 * sizeof(uint32_t), ctx->stream));
    const unsigned grid = (unsigned)std::min<size_t>((c->n + 255) / 256, (size_t)ctx->sm_count * 8);
    PPF_LAUNCH(ctx, bbox_kernel, grid, 256, 0, c->pos, (uint32_t)c->n, mm);
    uint32_t h[6];
    PPF_CUDA(ctx, cudaMemcpyAsync(h, mm, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 3; ++k) {
        c->bbox_min[k] = float_unorder(h[k]);
        c->bbox_max[k] = float_unorder(h[3 + k]);
    }
    return B200PPF_OK;
}

// ---- P1: voxel grid -------------------------------------------------------------------------------------------
struct VoxelParams {
    float inv[3];
    int min_b[3];
    int mul[3];
};

__global__ void __launch_bounds__(256)
voxel_ids_kernel(const float4 *__restrict__ pos, uint32_t n, VoxelParams vp, uint32_t *__restrict__ ids) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pos[i];
    // ijk = static_cast<int>(std::floor(x * inverse_leaf_size_) - static_cast<float>(min_b_))
    const int ijk0 = (int)(floorf(p.x * vp.inv[0]) - (float)vp.min_b[0]);
    const int ijk1 = (int)(floorf(p.y * vp.inv[1]) - (float)vp.min_b[1]);
    const int ijk2 = (int)(floorf(p.z * vp.inv[2]) - (float)vp.min_b[2]);
    ids[i] = (uint32_t)(ijk0 * vp.mul[0] + ijk1 * vp.mul[1] + ijk2 * vp.mul[2]);
}

// starts[v] = first sorted position of voxel v; starts[n_voxels] = n
__global__ void __launch_bounds__(256)
voxel_starts_kernel(const uint32_t *__restrict__ head, const uint32_t *__restrict__ rank, uint32_t n, uint32_t n_voxels,
                    uint32_t *__restrict__ starts) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) starts[n_voxels] = n;
    if (i >= n) return;
    if (head[i]) starts[rank[i]] = i;
}

// one thread per voxel: sequential float sum in original point order (the sort is stable), then / count
__global__ void __launch_bounds__(128)
voxel_centroid_kernel(const float4 *__restrict__ pos, const uint32_t *__restrict__ order, const uint32_t *__restrict__ starts,
                      uint32_t n_voxels, float4 *__restrict__ out_pos, float4 *__restrict__ out_nrm) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_voxels) return;
    const uint32_t first = starts[v], last = starts[v + 1];
    float cx = 0.0f, cy = 0.0f, cz = 0.0f;
    for (uint32_t i = first; i < last; ++i) {
        const float4 p = pos[order[i]];
        cx += p.x;
        cy += p.y;
        cz += p.z;
    }
    const float cnt = (float)(last - first);
    out_pos[v] = make_float4(cx / cnt, cy / cnt, cz / cnt, 1.0f);
    out_nrm[v] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

__global__ void __launch_bounds__(256)
copy_cloud_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm, uint32_t n, float4 *__restrict__ out_pos,
                  float4 *__restrict__ out_nrm) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out_pos[i] = pos[i];
    out_nrm[i] = nrm[i];
}

// ---- P2: k nearest neighbours ---------------------------------------------------------------------------------
enum { KNN_EXPORT = 0, KNN_MEAN_DISTANCE = 1, KNN_NORMAL = 2 };

struct KnnArgs {
    const float4 *pos;    // cloud, original order
    const float4 *gpos;   // cloud, cell-sorted
    const uint32_t *cell_start;
    const uint32_t *orig;  // cell-sorted position -> original index
    GridParams gp;
    float cell;  // cell edge
    uint32_t n;
    int k;  // neighbours wanted (self included), <= CAP, <= n
    // outputs (by mode)
    uint32_t *out_idx;  // [n*k]
    float *out_d2;      // [n*k]
    float *out_dist;    // [n] mean distance to the k-1 nearest other points
    float4 *out_nrm;    // [n] nx ny nz curvature
    float vp[3];        // viewpoint
    int cov_mode;       // 0: sums shifted by the first neighbour (PCL >= 1.12), 1: raw sums
};

// the query below is __host__ __device__: b200ppf_debug_knn_host runs the very same code on the CPU (test hook,
// like b200ppf_debug_alpha_bins), so the traversal and the epilogues can be checked without a GPU
__host__ __device__ __forceinline__ uint32_t f32_bits(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
#endif
}
__host__ __device__ __forceinline__ float bits_f32(uint32_t u) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}
template <typename T>
__host__ __device__ __forceinline__ T ld_ro(const T *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// [PCL] common/impl/eigen.hpp computeRoots2
__host__ __device__ __forceinline__ void compute_roots2(float b, float c, float *roots) {
    roots[0] = 0.0f;
    float d = b * b - 4.0f * c;
    if (d < 0.0f) d = 0.0f;
    const float sd = sqrtf(d);
    roots[2] = 0.5f * (b + sd);
    roots[1] = 0.5f * (b - sd);
}

// [PCL] common/impl/eigen.hpp computeRoots (symmetric 3x3, eigenvalues ascending)
__host__ __device__ inline void compute_roots(const float *m, float *roots) {
    const float m00 = m[0], m01 = m[1], m02 = m[2], m11 = m[4], m12 = m[5], m22 = m[8];
    const float c0 = m00 * m11 * m22 + 2.0f * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 - m22 * m01 * m01;
    const float c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12;
    const float c2 = m00 + m11 + m22;
    if (fabsf(c0) < 1.1920929e-07f) {  // std::numeric_limits<float>::epsilon()
        compute_roots2(c2, c1, roots);
        return;
    }
    const float s_inv3 = (float)(1.0 / 3.0);
    const float s_sqrt3 = 1.7320508075688772f;  // sqrtf(3.0f)
    const float c2_over_3 = c2 * s_inv3;
    float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
    if (a_over_3 > 0.0f) a_over_3 = 0.0f;
    const float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
    float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
    if (q > 0.0f) q = 0.0f;
    const float rho = sqrtf(-a_over_3);
    const float theta = atan2f(sqrtf(-q), half_b) * s_inv3;
    const float cos_theta = cosf(theta);
    const float sin_theta = sinf(theta);
    roots[0] = c2_over_3 + 2.0f * rho * cos_theta;
    roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
    roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
    float t;
    if (roots[0] >= roots[1]) t = roots[0], roots[0] = roots[1], roots[1] = t;
    if (roots[1] >= roots[2]) {
        t = roots[1], roots[1] = roots[2], roots[2] = t;
        if (roots[0] >= roots[1]) t = roots[0], roots[0] = roots[1], roots[1] = t;
    }
    if (roots[0] <= 0.0f) compute_roots2(c2, c1, roots);
}

// [PCL] common/impl/eigen.hpp eigen33(mat, eigenvalue, eigenvector): the smallest eigenpair
__host__ __device__ inline void eigen33_smallest(const float *cov, float *eigenvalue, float *evec) {
    float scale = 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k) scale = fmaxf(scale, fabsf(cov[k]));
    if (scale <= 1.17549435e-38f) scale = 1.0f;  // std::numeric_limits<float>::min()
    float s[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) s[k] = cov[k] / scale;
    float roots[3];
    compute_roots(s, roots);
    *eigenvalue = roots[0] * scale;
    s[0] -= roots[0];
    s[4] -= roots[0];
    s[8] -= roots[0];
    float v[3][3];
    // rows 0x1, 0x2, 1x2
    v[0][0] = s[1] * s[5] - s[2] * s[4], v[0][1] = s[2] * s[3] - s[0] * s[5], v[0][2] = s[0] * s[4] - s[1] * s[3];
    v[1][0] = s[1] * s[8] - s[2] * s[7], v[1][1] = s[2] * s[6] - s[0] * s[8], v[1][2] = s[0] * s[7] - s[1] * s[6];
    v[2][0] = s[4] * s[8] - s[5] * s[7], v[2][1] = s[5] * s[6] - s[3] * s[8], v[2][2] = s[3] * s[7] - s[4] * s[6];
    float len[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) len[k] = sqrtf(v[k][0] * v[k][0] + v[k][1] * v[k][1] + v[k][2] * v[k][2]);
    int best = 0;
    if (len[1] > len[best]) best = 1;
    if (len[2] > len[best]) best = 2;
    const float l = best == 0 ? len[0] : (best == 1 ? len[1] : len[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) evec[k] = (best == 0 ? v[0][k] : (best == 1 ? v[1][k] : v[2][k])) / l;
}

// where a query keeps its k best: a per-thread array (local memory; the host build) or a column of the block's
// shared memory — slot i of thread t at word i*128 + t, so a warp's accesses to whatever slots its lanes are at
// fall into distinct bank pairs.  With 1 536 resident threads the local-memory arrays (k x 8 bytes each) overflow
// L1 and ncu showed them travelling to DRAM (2.5 GB per launch on the 1 Mi-point scene); shared memory keeps them
// on the SM at the price of occupancy.
constexpr int KNN_THREADS = 128;
template <int CAP>
struct LocalKeys {
    unsigned long long v[CAP];
    __host__ __device__ __forceinline__ unsigned long long &operator[](int i) { return v[i]; }
};
struct SharedKeys {
    unsigned long long *base;  // &smem[threadIdx.x]
    __device__ __forceinline__ unsigned long long &operator[](int i) { return base[i * KNN_THREADS]; }
};

// one query point (q = its cell-sorted position): the k nearest, then the epilogue of MODE
template <int MODE, typename Keys>
__host__ __device__ inline void knn_query(const KnnArgs &a, const uint32_t q, Keys &best) {
    const float4 pq = a.gpos[q];
    const int cx = grid_cell_coord(a.gp, pq.x, 0), cy = grid_cell_coord(a.gp, pq.y, 1), cz = grid_cell_coord(a.gp, pq.z, 2);
    const int dx = a.gp.dims[0], dy = a.gp.dims[1], dz = a.gp.dims[2];
    const int k = a.k;
    // the k best so far as (distance bits << 32 | original index) words: an unordered buffer while it fills, a
    // max-heap (largest at [0]) once it holds k — a better candidate replaces the root in O(log k) — and an
    // ascending array after the final heap sort
    int cnt = 0;
    auto sift_down = [&](int i, const int end, const unsigned long long v) {  // place v at or below i, heap = [0, end)
        for (;;) {
            int c = 2 * i + 1;
            if (c >= end) break;
            if (c + 1 < end && best[c + 1] > best[c]) ++c;
            if (best[c] <= v) break;
            best[i] = best[c];
            i = c;
        }
        best[i] = v;
    };

    // candidates of the sorted positions [s0, s1)
    auto scan_run = [&](uint32_t s0, uint32_t s1) {
        for (uint32_t s = s0; s < s1; ++s) {
            const float4 p = ld_ro(a.gpos + s);
            // FLANN L2_Simple: result += diff * diff over x, y, z
            const float ex = pq.x - p.x, ey = pq.y - p.y, ez = pq.z - p.z;
            float d2 = ex * ex;
            d2 += ey * ey;
            d2 += ez * ez;
            const unsigned long long key = ((unsigned long long)f32_bits(d2) << 32) | (unsigned long long)ld_ro(a.orig + s);
            if (cnt < k) {
                best[cnt++] = key;
                if (cnt == k)
                    for (int i = k / 2 - 1; i >= 0; --i) sift_down(i, k, best[i]);  // heapify
            } else if (key < best[0]) {
                sift_down(0, k, key);
            }
        }
    };

    int r_max = cx > dx - 1 - cx ? cx : dx - 1 - cx;
    r_max = cy > r_max ? cy : r_max;
    r_max = dy - 1 - cy > r_max ? dy - 1 - cy : r_max;
    r_max = cz > r_max ? cz : r_max;
    r_max = dz - 1 - cz > r_max ? dz - 1 - cz : r_max;
    for (int r = 0; r <= r_max; ++r) {
        // shell of cells at Chebyshev distance exactly r; rows along x are contiguous runs of sorted positions
        for (int oz = -r; oz <= r; ++oz) {
            const int z = cz + oz;
            if (z < 0 || z >= dz) continue;
            for (int oy = -r; oy <= r; ++oy) {
                const int y = cy + oy;
                if (y < 0 || y >= dy) continue;
                const uint32_t row = ((uint32_t)z * (uint32_t)dy + (uint32_t)y) * (uint32_t)dx;
                if (oz == -r || oz == r || oy == -r || oy == r) {
                    const int x0 = cx - r > 0 ? cx - r : 0, x1 = cx + r < dx - 1 ? cx + r : dx - 1;
                    scan_run(ld_ro(a.cell_start + row + x0), ld_ro(a.cell_start + row + x1 + 1));
                } else {  // interior row of the shell: only its two end cells (r >= 1 here)
                    if (cx - r >= 0) scan_run(ld_ro(a.cell_start + row + cx - r), ld_ro(a.cell_start + row + cx - r + 1));
                    if (cx + r < dx) scan_run(ld_ro(a.cell_start + row + cx + r), ld_ro(a.cell_start + row + cx + r + 1));
                }
            }
        }
        // every unvisited point is more than (r - margin) cells away along some axis; the margin absorbs the
        // float rounding of the cell coordinate
        if (cnt == k && r >= 1) {
            const float reach = ((float)r - 1e-3f) * a.cell;
            if (bits_f32((uint32_t)(best[0] >> 32)) <= reach * reach) break;
        }
    }

    // ascending order = FLANN's (distance, then index): heap sort in place
    if (cnt < k)
        for (int i = cnt / 2 - 1; i >= 0; --i) sift_down(i, cnt, best[i]);
    for (int end = cnt - 1; end > 0; --end) {
        const unsigned long long v = best[end];
        best[end] = best[0];
        sift_down(0, end, v);
    }

    const uint32_t me = a.orig[q];
    if (MODE == KNN_EXPORT) {
        for (int j = 0; j < k; ++j) {
            a.out_idx[(size_t)me * k + j] = j < cnt ? (uint32_t)best[j] : 0xFFFFFFFFu;
            a.out_d2[(size_t)me * k + j] = j < cnt ? bits_f32((uint32_t)(best[j] >> 32)) : INFINITY;
        }
    } else if (MODE == KNN_MEAN_DISTANCE) {
        // dist_sum += sqrt(nn_dists[k]) for k = 1 .. mean_k (0 is the query itself); (float)(dist_sum / mean_k)
        double dist_sum = 0.0;
        for (int j = 1; j < cnt; ++j) dist_sum += (double)sqrtf(bits_f32((uint32_t)(best[j] >> 32)));
        a.out_dist[me] = (float)(dist_sum / (double)(k - 1));
    } else {
        if (cnt < 3) {
            const float nan = bits_f32(0x7FC00000u);
            a.out_nrm[me] = make_float4(nan, nan, nan, nan);
            return;
        }
        // computeMeanAndCovarianceMatrix (float), neighbours in FLANN's order
        float Kx = 0.0f, Ky = 0.0f, Kz = 0.0f;
        if (a.cov_mode == 0) {
            const float4 p0 = a.pos[(uint32_t)best[0]];
            Kx = p0.x, Ky = p0.y, Kz = p0.z;
        }
        float accu[9] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
        for (int j = 0; j < cnt; ++j) {
            const float4 p = ld_ro(a.pos + (uint32_t)best[j]);
            const float x = p.x - Kx, y = p.y - Ky, z = p.z - Kz;
            accu[0] += x * x;
            accu[1] += x * y;
            accu[2] += x * z;
            accu[3] += y * y;
            accu[4] += y * z;
            accu[5] += z * z;
            accu[6] += x;
            accu[7] += y;
            accu[8] += z;
        }
        const float fcnt = (float)cnt;
#pragma unroll
        for (int t = 0; t < 9; ++t) accu[t] /= fcnt;
        float cov[9];
        cov[0] = accu[0] - accu[6] * accu[6];
        cov[1] = accu[1] - accu[6] * accu[7];
        cov[2] = accu[2] - accu[6] * accu[8];
        cov[4] = accu[3] - accu[7] * accu[7];
        cov[5] = accu[4] - accu[7] * accu[8];
        cov[8] = accu[5] - accu[8] * accu[8];
        cov[3] = cov[1], cov[6] = cov[2], cov[7] = cov[5];
        // solvePlaneParameters
        float ev, nv[3];
        eigen33_smallest(cov, &ev, nv);
        const float eig_sum = cov[0] + cov[4] + cov[8];
        float curvature = 0.0f;
        if (eig_sum != 0.0f) curvature = fabsf(ev / eig_sum);
        // flipNormalTowardsViewpoint
        const float vx = a.vp[0] - pq.x, vy = a.vp[1] - pq.y, vz = a.vp[2] - pq.z;
        const float cos_theta = vx * nv[0] + vy * nv[1] + vz * nv[2];
        if (cos_theta < 0.0f) nv[0] *= -1.0f, nv[1] *= -1.0f, nv[2] *= -1.0f;
        a.out_nrm[me] = make_float4(nv[0], nv[1], nv[2], curvature);
    }
}

template <int CAP, int MODE>
__global__ void __launch_bounds__(KNN_THREADS) knn_kernel(const KnnArgs a) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;  // cell-sorted position of the query
    if (q >= a.n) return;
    LocalKeys<CAP> best;
    knn_query<MODE>(a, q, best);
}

template <int MODE>
__global__ void __launch_bounds__(KNN_THREADS) knn_smem_kernel(const KnnArgs a) {
    extern __shared__ unsigned long long knn_keys[];  // [k][KNN_THREADS]
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.n) return;
    SharedKeys best{knn_keys + threadIdx.x};
    knn_query<MODE>(a, q, best);
}

template <int MODE>
int knn_launch(b200ppf_ctx *ctx, const KnnArgs &a) {
    const unsigned grid = (a.n + KNN_THREADS - 1) / KNN_THREADS;
    static const bool force_local = getenv("B200PPF_KNN_LOCAL") != nullptr;  // tuning switch: the local-memory variant
    if (!force_local) {
        const size_t smem = (size_t)a.k * KNN_THREADS * sizeof(unsigned long long);
        PPF_CUDA(ctx, cudaFuncSetAttribute(knn_smem_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * KNN_THREADS * 8));
        PPF_LAUNCH(ctx, knn_smem_kernel<MODE>, grid, KNN_THREADS, smem, a);
        return B200PPF_OK;
    }
    void (*kern)(const KnnArgs) = a.k <= 32 ? knn_kernel<32, MODE> : (a.k <= 64 ? knn_kernel<64, MODE> : knn_kernel<128, MODE>);
    PPF_LAUNCH(ctx, kern, grid, KNN_THREADS, 0, a);
    return B200PPF_OK;
}

// cell edge for the neighbour grid: about k/2 points per cell if the cloud were one surface spanning the two
// largest extents of its bounding box (a wrong guess costs time, not correctness)
float knn_cell_edge(const b200ppf_cloud *c, int k) {
    double e[3];
    for (int t = 0; t < 3; ++t) e[t] = std::max(0.0, (double)c->bbox_max[t] - (double)c->bbox_min[t]);
    std::sort(e, e + 3);
    const double area = e[2] * e[1];
    double h = area > 0.0 ? std::sqrt(0.5 * (double)k * area / (double)std::max<size_t>(1, c->n)) : 0.0;
    h = std::max(h, e[2] / 1024.0);
    if (!(h > 0.0)) h = 1e-3;
    return (float)h;
}

// grid + neighbour kernel of one mode over `cloud`
template <int MODE>
int knn_run(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, KnnArgs a) {
    SceneGrid grid;
    std::unique_ptr<SceneGrid, SceneGridFree> grid_owner(&grid, SceneGridFree{ctx});
    int rc = scene_grid_build(ctx, cloud, knn_cell_edge(cloud, a.k), &grid);
    if (rc != B200PPF_OK) return rc;
    a.pos = cloud->pos;
    a.gpos = grid.pos;
    a.cell_start = grid.cell_start;
    a.orig = grid.orig;
    a.gp = grid.gp;
    a.cell = 1.0f / grid.gp.inv_cell;
    a.n = (uint32_t)cloud->n;
    return knn_launch<MODE>(ctx, a);
}

// ---- P3: statistical outlier removal --------------------------------------------------------------------------
// per-block partial sums of d and d*d (float product, as PCL writes it) in double, fixed tree
__global__ void __launch_bounds__(256)
sor_partial_sums_kernel(const float *__restrict__ dist, uint32_t n, double *__restrict__ partial) {
    __shared__ double sh[2][8];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    double s = 0.0, ss = 0.0;
    if (i < n) {
        const float d = dist[i];
        s = (double)d;
        ss = (double)(d * d);
    }
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xFFFFFFFFu, s, o);
        ss += __shfl_down_sync(0xFFFFFFFFu, ss, o);
    }
    if ((threadIdx.x & 31) == 0) sh[0][threadIdx.x >> 5] = s, sh[1][threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0.0, tss = 0.0;
        for (int w = 0; w < 8; ++w) ts += sh[0][w], tss += sh[1][w];
        partial[2 * blockIdx.x] = ts;
        partial[2 * blockIdx.x + 1] = tss;
    }
}

__global__ void __launch_bounds__(256)
sor_flag_kernel(const float *__restrict__ dist, uint32_t n, double threshold, uint32_t *__restrict__ flags) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flags[i] = ((double)dist[i] > threshold) ? 0u : 1u;  // removed when distances[i] > distance_threshold
}

__global__ void __launch_bounds__(256)
curvature_flag_kernel(const float4 *__restrict__ nrm, uint32_t n, float threshold, uint32_t *__restrict__ flags) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flags[i] = (nrm[i].w > threshold) ? 1u : 0u;
}

__global__ void __launch_bounds__(256)
compact_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm, const uint32_t *__restrict__ flags,
               const uint32_t *__restrict__ rank, uint32_t n, float4 *__restrict__ out_pos, float4 *__restrict__ out_nrm,
               uint32_t *__restrict__ out_index) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flags[i]) return;
    const uint32_t r = rank[i];
    out_pos[r] = pos[i];
    out_nrm[r] = nrm[i];
    if (out_index) out_index[r] = i;
}

// keep the flagged points, in order -> new cloud (and, optionally, their indices on the host)
int compact_cloud(b200ppf_ctx *ctx, const b200ppf_cloud *in, const uint32_t *flags, b200ppf_cloud **out, uint32_t *kept_host) {
    const uint32_t n = (uint32_t)in->n;
    StreamBuf<uint32_t> rank(ctx), index(ctx);
    PPF_CUDA(ctx, rank.alloc(n));
    uint32_t m = 0;
    int rc = flag_scan_host(ctx, flags, n, rank, &m);
    if (rc != B200PPF_OK) return rc;
    CloudPtr c;
    if ((rc = cloud_alloc(ctx, m, &c)) != B200PPF_OK) return rc;
    if (kept_host && m) PPF_CUDA(ctx, index.alloc(m));
    if (n) PPF_LAUNCH(ctx, compact_kernel, (n + 255) / 256, 256, 0, in->pos, in->nrm, flags, rank, n, c->pos, c->nrm, index);
    if (index) PPF_CUDA(ctx, cudaMemcpyAsync(kept_host, index, (size_t)m * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if ((rc = cloud_bbox_from_device(ctx, c.get())) != B200PPF_OK) return rc;  // synchronises the stream
    *out = c.release();
    return B200PPF_OK;
}

// ---- P0: frustum crop ----------------------------------------------------------------------------------------
// the pyramid {apex = camera origin, four far corners} as five half-spaces n.p <= d (double)
struct PyramidPlanes {
    double n[5][3];
    double d[5];
};

// the one inside test of both crops, so that a point falls the same way for a box alone and in a frame of boxes
__device__ __forceinline__ bool pyramid_contains(const PyramidPlanes &pl, const float4 p) {
    const double x = p.x, y = p.y, z = p.z;
    bool in = true;
#pragma unroll
    for (int f = 0; f < 5; ++f) in = in && (pl.n[f][0] * x + pl.n[f][1] * y + pl.n[f][2] * z <= pl.d[f]);
    return in;
}

__global__ void __launch_bounds__(256)
pyramid_flag_kernel(const float4 *__restrict__ pos, uint32_t n, PyramidPlanes pl, uint32_t *__restrict__ flags) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flags[i] = pyramid_contains(pl, pos[i]) ? 1u : 0u;
}

// ---- P0 for up to 64 boxes: one tile of CROP_TILE points per block -------------------------------------------
constexpr int MAX_BOXES = 64;
constexpr int CROP_TILE = 1024;

// membership mask of every point, the tile's count per box (counts[b * n_tiles + tile]) and each box's bounding box
// (lo[3 * b ..], hi[3 * b ..] as order-preserving words): the bounds of a box's points are those of its cloud
__global__ void __launch_bounds__(CROP_TILE)
pyramids_mask_kernel(const float4 *__restrict__ pos, uint32_t n, const PyramidPlanes *__restrict__ planes, int n_boxes,
                     unsigned long long *__restrict__ mask, uint32_t *__restrict__ counts, uint32_t *__restrict__ lo,
                     uint32_t *__restrict__ hi) {
    __shared__ PyramidPlanes s_pl[MAX_BOXES];
    __shared__ uint32_t s_cnt[MAX_BOXES], s_lo[MAX_BOXES][3], s_hi[MAX_BOXES][3];
    for (int t = threadIdx.x; t < n_boxes * (int)(sizeof(PyramidPlanes) / sizeof(double)); t += CROP_TILE)
        reinterpret_cast<double *>(s_pl)[t] = reinterpret_cast<const double *>(planes)[t];
    for (int b = threadIdx.x; b < n_boxes; b += CROP_TILE) {
        s_cnt[b] = 0;
        for (int k = 0; k < 3; ++k) s_lo[b][k] = 0xFFFFFFFFu, s_hi[b][k] = 0u;
    }
    __syncthreads();
    const uint32_t i = blockIdx.x * CROP_TILE + threadIdx.x, lane = threadIdx.x & 31;
    const float4 p = i < n ? pos[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    unsigned long long m = 0;
    if (i < n)
        for (int b = 0; b < n_boxes; ++b)
            if (pyramid_contains(s_pl[b], p)) m |= 1ull << b;
    if (i < n) mask[i] = m;
    const uint32_t c[3] = {float_order(p.x), float_order(p.y), float_order(p.z)};
    for (int b = 0; b < n_boxes; ++b) {
        const bool in = (m >> b) & 1ull;
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, in);
        if (!bal) continue;  // warp-uniform
        for (int k = 0; k < 3; ++k) {
            const uint32_t l = __reduce_min_sync(0xFFFFFFFFu, in ? c[k] : 0xFFFFFFFFu);
            const uint32_t h = __reduce_max_sync(0xFFFFFFFFu, in ? c[k] : 0u);
            if (lane == 0) atomicMin(&s_lo[b][k], l), atomicMax(&s_hi[b][k], h);
        }
        if (lane == 0) atomicAdd(&s_cnt[b], (uint32_t)__popc(bal));
    }
    __syncthreads();
    for (int b = threadIdx.x; b < n_boxes; b += CROP_TILE) {
        counts[(size_t)b * gridDim.x + blockIdx.x] = s_cnt[b];
        if (s_cnt[b])
            for (int k = 0; k < 3; ++k) atomicMin(lo + 3 * b + k, s_lo[b][k]), atomicMax(hi + 3 * b + k, s_hi[b][k]);
    }
}

// every point into each of its boxes' clouds at (scanned tile offset + rank in the tile): input order, as compaction
// keeps it.  out[b] / out[n_boxes + b] are cloud b's pos / nrm arrays.
__global__ void __launch_bounds__(CROP_TILE)
pyramids_scatter_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm, uint32_t n,
                        const unsigned long long *__restrict__ mask, int n_boxes, const uint32_t *__restrict__ tile_off,
                        float4 *const *__restrict__ out) {
    __shared__ uint32_t s_warp[MAX_BOXES][32];  // box b: points of warps before w in this tile
    const uint32_t i = blockIdx.x * CROP_TILE + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long m = i < n ? mask[i] : 0ull;
    for (int b = 0; b < n_boxes; ++b) {
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, (m >> b) & 1ull);
        if (lane == 0) s_warp[b][warp] = (uint32_t)__popc(bal);
    }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < (uint32_t)n_boxes * 32; t += CROP_TILE) {  // one warp per box row: exclusive scan
        const uint32_t v = s_warp[t >> 5][lane];
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += u;
        }
        s_warp[t >> 5][lane] = incl - v;
    }
    __syncthreads();
    const float4 p = m ? pos[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f), q = m ? nrm[i] : p;
    for (int b = 0; b < n_boxes; ++b) {
        const bool in = (m >> b) & 1ull;
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, in);
        if (!in) continue;
        const uint32_t r = tile_off[(size_t)b * gridDim.x + blockIdx.x] + s_warp[b][warp] + __popc(bal & ((1u << lane) - 1u));
        out[b][r] = p;
        out[n_boxes + b][r] = q;
    }
}

// ---- P6 ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) renormalize_kernel(float4 *__restrict__ nrm, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 v = nrm[i];
    // double A = sqrt(nx*nx + ny*ny + nz*nz): float sum, float sqrt (the overload `using namespace std` selects),
    // widened; if (A > 0.00001) n /= static_cast<float>(A)
    const double A = (double)sqrtf(v.x * v.x + v.y * v.y + v.z * v.z);
    if (A > 0.00001) {
        const float fa = (float)A;
        v.x /= fa;
        v.y /= fa;
        v.z /= fa;
        nrm[i] = v;
    }
}

// ---- download: SoA -> caller's AoS rows through a device staging buffer ----------------------------------------
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm, uint32_t n, uint32_t stride, uint32_t noff,
                 uint32_t coff, float *__restrict__ rows) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pos[i], q = nrm[i];
    float *r = rows + (size_t)i * stride;
    for (uint32_t t = 0; t < stride; ++t) r[t] = 0.0f;
    r[0] = p.x, r[1] = p.y, r[2] = p.z;
    if (noff) r[noff] = q.x, r[noff + 1] = q.y, r[noff + 2] = q.z;
    if (coff) r[coff] = q.w;
}

struct EventTimer {  // prep_ms of the timings block
    b200ppf_ctx *ctx;
    explicit EventTimer(b200ppf_ctx *c) : ctx(c) { cudaEventRecord(ctx->ev[0], ctx->stream); }
    void stop() {
        cudaEventRecord(ctx->ev[1], ctx->stream);
        if (cudaEventSynchronize(ctx->ev[1]) == cudaSuccess) cudaEventElapsedTime(&ctx->timings.prep_ms, ctx->ev[0], ctx->ev[1]);
    }
};

}  // namespace

// ================================================================================================================
// host entry points (called from capi.cu)

int prep_upload_xyz(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride, b200ppf_cloud **out) {
    PPF_CUDA(ctx, grow_buffer(&ctx->stage, &ctx->stage_cap, std::max<size_t>(1, n), /*pinned=*/true));
    float4 *sp = ctx->stage;
    size_t m = 0;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (size_t i = 0; i < n; ++i) {
        const float *p = host + i * stride;
        if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) continue;  // PCL filters skip non-finite points
        sp[m++] = make_float4(p[0], p[1], p[2], 1.0f);
        for (int k = 0; k < 3; ++k) {
            lo[k] = std::min(lo[k], p[k]);
            hi[k] = std::max(hi[k], p[k]);
        }
    }
    CloudPtr c;
    int rc = cloud_alloc(ctx, m, &c);
    if (rc != B200PPF_OK) return rc;
    for (int k = 0; k < 3; ++k) {
        c->bbox_min[k] = m ? lo[k] : 0.0f;
        c->bbox_max[k] = m ? hi[k] : 0.0f;
    }
    if (m) PPF_CUDA(ctx, cudaMemcpyAsync(c->pos, sp, m * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    if (m) PPF_CUDA(ctx, cudaMemsetAsync(c->nrm, 0, m * sizeof(float4), ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the staging buffer is reused by the next upload
    *out = c.release();
    return B200PPF_OK;
}

int prep_download(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, float *host, size_t stride, size_t noff, size_t coff) {
    const size_t n = cloud->n;
    if (n == 0) return B200PPF_OK;
    StreamBuf<float> rows(ctx);
    PPF_CUDA(ctx, rows.alloc(n * stride));
    PPF_LAUNCH(ctx, pack_rows_kernel, (unsigned)((n + 255) / 256), 256, 0, cloud->pos, cloud->nrm, (uint32_t)n, (uint32_t)stride,
               (uint32_t)noff, (uint32_t)coff, rows);
    PPF_CUDA(ctx, cudaMemcpyAsync(host, rows, n * stride * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int prep_voxel_grid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *leaf3, b200ppf_cloud **out) {
    const uint32_t n = (uint32_t)in->n;
    EventTimer timer(ctx);
    if (n == 0) {
        CloudPtr c;
        int rc = cloud_alloc(ctx, 0, &c);
        timer.stop();
        *out = c.release();
        return rc;
    }
    VoxelParams vp;
    for (int k = 0; k < 3; ++k) vp.inv[k] = 1.0f / leaf3[k];  // inverse_leaf_size_ = Array4f::Ones() / leaf_size_
    // "Leaf size is too small for the input dataset. Integer indices would overflow." -> PCL returns the input
    int64_t d[3];
    for (int k = 0; k < 3; ++k) d[k] = (int64_t)((in->bbox_max[k] - in->bbox_min[k]) * vp.inv[k]) + 1;
    const bool overflow = d[0] * d[1] * d[2] > (int64_t)INT32_MAX;
    if (overflow) {
        CloudPtr c;
        int rc = cloud_alloc(ctx, n, &c);
        if (rc != B200PPF_OK) return rc;
        PPF_LAUNCH(ctx, copy_cloud_kernel, (n + 255) / 256, 256, 0, in->pos, in->nrm, n, c->pos, c->nrm);
        for (int k = 0; k < 3; ++k) c->bbox_min[k] = in->bbox_min[k], c->bbox_max[k] = in->bbox_max[k];
        timer.stop();
        ctx->error = "voxel grid: leaf size is too small for the input dataset, integer indices would overflow; input returned unchanged";
        *out = c.release();
        return B200PPF_OK;
    }
    int div_b[3];
    for (int k = 0; k < 3; ++k) {
        vp.min_b[k] = (int)floorf(in->bbox_min[k] * vp.inv[k]);
        const int max_b = (int)floorf(in->bbox_max[k] * vp.inv[k]);
        div_b[k] = max_b - vp.min_b[k] + 1;
    }
    vp.mul[0] = 1, vp.mul[1] = div_b[0], vp.mul[2] = div_b[0] * div_b[1];
    const uint64_t n_cells = (uint64_t)div_b[0] * (uint64_t)div_b[1] * (uint64_t)div_b[2];

    StreamBuf<uint32_t> ids0(ctx), ids1(ctx), ord0(ctx), ord1(ctx), head(ctx), rank(ctx), starts(ctx);
    PPF_CUDA(ctx, ids0.alloc(n));
    PPF_CUDA(ctx, ids1.alloc(n));
    PPF_CUDA(ctx, ord0.alloc(n));
    PPF_CUDA(ctx, ord1.alloc(n));
    PPF_CUDA(ctx, head.alloc(n));
    PPF_CUDA(ctx, rank.alloc(n));
    const unsigned gb = (n + 255) / 256;
    PPF_LAUNCH(ctx, voxel_ids_kernel, gb, 256, 0, in->pos, n, vp, ids0);
    bool in_alt = false;
    int rc = radix_sort_u32(ctx, ids0, ids1, ord0, ord1, nullptr, nullptr, n, n_cells - 1, /*v0_iota=*/true, &in_alt);
    if (rc != B200PPF_OK) return rc;
    const uint32_t *sorted_ids = in_alt ? ids1 : ids0, *order = in_alt ? ord1 : ord0;
    if ((rc = run_heads(ctx, sorted_ids, n, head)) != B200PPF_OK) return rc;
    uint32_t m = 0;
    if ((rc = flag_scan_host(ctx, head, n, rank, &m)) != B200PPF_OK) return rc;
    PPF_CUDA(ctx, starts.alloc((size_t)m + 1));
    CloudPtr c;
    if ((rc = cloud_alloc(ctx, m, &c)) != B200PPF_OK) return rc;
    PPF_LAUNCH(ctx, voxel_starts_kernel, gb, 256, 0, head, rank, n, m, starts);
    PPF_LAUNCH(ctx, voxel_centroid_kernel, (m + 127) / 128, 128, 0, in->pos, order, starts, m, c->pos, c->nrm);
    if ((rc = cloud_bbox_from_device(ctx, c.get())) != B200PPF_OK) return rc;
    timer.stop();
    *out = c.release();
    return B200PPF_OK;
}

int prep_knn(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, int k, uint32_t *idx_host, float *d2_host) {
    const size_t n = cloud->n;
    if (n == 0) return B200PPF_OK;
    KnnArgs a{};
    a.k = k;
    StreamBuf<uint32_t> out_idx(ctx);
    StreamBuf<float> out_d2(ctx);
    PPF_CUDA(ctx, out_idx.alloc(n * (size_t)k));
    PPF_CUDA(ctx, out_d2.alloc(n * (size_t)k));
    a.out_idx = out_idx;
    a.out_d2 = out_d2;
    EventTimer timer(ctx);
    int rc = knn_run<KNN_EXPORT>(ctx, cloud, a);
    timer.stop();
    if (rc != B200PPF_OK) return rc;
    if (idx_host) PPF_CUDA(ctx, cudaMemcpyAsync(idx_host, out_idx, n * (size_t)k * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (d2_host) PPF_CUDA(ctx, cudaMemcpyAsync(d2_host, out_d2, n * (size_t)k * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int prep_sor(b200ppf_ctx *ctx, const b200ppf_cloud *in, int mean_k, double stddev_mul, b200ppf_cloud **out, uint32_t *kept_host,
             float *distances_host, double *threshold_out) {
    const uint32_t n = (uint32_t)in->n;
    KnnArgs a{};
    a.k = mean_k + 1;
    StreamBuf<float> dist(ctx);
    StreamBuf<double> partial(ctx);
    StreamBuf<uint32_t> flags(ctx);
    const uint32_t nb = (n + 255) / 256;
    PPF_CUDA(ctx, dist.alloc(n));
    PPF_CUDA(ctx, partial.alloc((size_t)nb * 2));
    PPF_CUDA(ctx, flags.alloc(n));
    a.out_dist = dist;
    EventTimer timer(ctx);
    int rc = knn_run<KNN_MEAN_DISTANCE>(ctx, in, a);
    if (rc != B200PPF_OK) return rc;
    PPF_LAUNCH(ctx, sor_partial_sums_kernel, nb, 256, 0, dist, n, partial);
    std::vector<double> hp((size_t)nb * 2);
    PPF_CUDA(ctx, cudaMemcpyAsync(hp.data(), partial, hp.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (distances_host)
        PPF_CUDA(ctx, cudaMemcpyAsync(distances_host, dist, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    double sum = 0.0, sq_sum = 0.0;
    for (uint32_t b = 0; b < nb; ++b) sum += hp[2 * b], sq_sum += hp[2 * b + 1];
    // mean / variance / threshold exactly as PCL forms them (all points are valid here)
    const double mean = sum / (double)n;
    const double variance = (sq_sum - sum * sum / (double)n) / ((double)n - 1.0);
    const double stddev = sqrt(variance);
    const double thr = mean + stddev_mul * stddev;
    if (threshold_out) *threshold_out = thr;
    PPF_LAUNCH(ctx, sor_flag_kernel, nb, 256, 0, dist, n, thr, flags);
    rc = compact_cloud(ctx, in, flags, out, kept_host);
    timer.stop();
    return rc;
}

int prep_normals(b200ppf_ctx *ctx, b200ppf_cloud *cloud, int k, const float *viewpoint3, int cov_mode) {
    if (cloud->n == 0) return B200PPF_OK;
    KnnArgs a{};
    a.k = (int)std::min<size_t>((size_t)k, cloud->n);
    a.out_nrm = cloud->nrm;
    for (int t = 0; t < 3; ++t) a.vp[t] = viewpoint3 ? viewpoint3[t] : 0.0f;
    a.cov_mode = cov_mode;
    EventTimer timer(ctx);
    int rc = knn_run<KNN_NORMAL>(ctx, cloud, a);
    timer.stop();
    if (rc == B200PPF_OK) PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return rc;
}

int prep_curvature_edges(b200ppf_ctx *ctx, const b200ppf_cloud *in, float threshold, b200ppf_cloud **out) {
    const uint32_t n = (uint32_t)in->n;
    StreamBuf<uint32_t> flags(ctx);
    PPF_CUDA(ctx, flags.alloc(n));
    EventTimer timer(ctx);
    if (n) PPF_LAUNCH(ctx, curvature_flag_kernel, (n + 255) / 256, 256, 0, in->nrm, n, threshold, flags);
    int rc = compact_cloud(ctx, in, flags, out, nullptr);
    timer.stop();
    return rc;
}

// reference include/CloudProcessing.h:270-300 + include/Camera.h:50-61, restated: host arithmetic on four pixels
void prep_frustum_corners(const float *depth, int rows, int cols, int bx, int by, int bw, int bh, double fx, double fy,
                          double ppx, double ppy, float *corners12) {
    double left = bx - 30;  // the box grown by 30 pixels, clamped to the image
    if (left < 0) left = 0;
    double top = by - 30;
    if (top < 0) top = 0;
    double right = bx + bw + 30;
    if (right >= cols) right = cols - 1;
    double bottom = by + bh + 30;
    if (bottom >= rows) bottom = rows - 1;
    const int l = (int)left, t = (int)top, r = (int)right, b = (int)bottom;
    const float depth_avg = (depth[(size_t)t * cols + l] + depth[(size_t)t * cols + r] + depth[(size_t)b * cols + l] +
                             depth[(size_t)b * cols + r]) / 4;
    const int us[4] = {l, l, r, r}, vs[4] = {t, b, t, b};  // left_top, left_bot, right_top, right_bot
    for (int c = 0; c < 4; ++c) {
        // back_projection_bbox: point.x = (float)(u - ppx) * z / fx  (float product, double quotient, float store)
        corners12[3 * c + 0] = (float)((float)(us[c] - ppx) * depth_avg / fx);
        corners12[3 * c + 1] = (float)((float)(vs[c] - ppy) * depth_avg / fy);
        float z = depth_avg;
        z += 0.15;  // "left_top.z += 0.15": float += double
        corners12[3 * c + 2] = z;
    }
}

namespace {

// the five half-spaces of the pyramid {origin, four corners}; 0, or B200PPF_ERR_* with the reason in *why
int pyramid_planes(const float *corners12, PyramidPlanes *pl, const char **why) {
    double c[4][3], m[3] = {0, 0, 0};
    for (int i = 0; i < 4; ++i)
        for (int k = 0; k < 3; ++k) c[i][k] = corners12[3 * i + k], m[k] += 0.25 * corners12[3 * i + k];
    auto cross = [](const double *a, const double *b, double *o) {
        o[0] = a[1] * b[2] - a[2] * b[1];
        o[1] = a[2] * b[0] - a[0] * b[2];
        o[2] = a[0] * b[1] - a[1] * b[0];
    };
    auto dot = [](const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
    const int cyc[4] = {0, 1, 3, 2};  // left_top -> left_bot -> right_bot -> right_top
    for (int s = 0; s < 4; ++s) {  // side faces contain the apex (the origin): d = 0; the corners' centroid is inside
        cross(c[cyc[s]], c[cyc[(s + 1) & 3]], pl->n[s]);
        if (dot(pl->n[s], m) > 0)
            for (int k = 0; k < 3; ++k) pl->n[s][k] = -pl->n[s][k];
        pl->d[s] = 0.0;
    }
    double e1[3], e2[3];
    for (int k = 0; k < 3; ++k) e1[k] = c[1][k] - c[0][k], e2[k] = c[2][k] - c[0][k];
    cross(e1, e2, pl->n[4]);
    pl->d[4] = dot(pl->n[4], c[0]);
    if (pl->d[4] < 0) {  // the apex is inside
        for (int k = 0; k < 3; ++k) pl->n[4][k] = -pl->n[4][k];
        pl->d[4] = -pl->d[4];
    }
    const double nn = std::sqrt(dot(pl->n[4], pl->n[4]));
    if (!(nn > 0.0) || !(pl->d[4] > 0.0)) {
        *why = "the four corners do not span a base in front of the camera";
        return B200PPF_ERR_INVALID;
    }
    // the reference's corners share one z; a base that is not planar would make the hull a different solid
    if (std::fabs(dot(pl->n[4], c[3]) - pl->d[4]) > 1e-6 * nn * (std::fabs(c[3][0]) + std::fabs(c[3][1]) + std::fabs(c[3][2]) + 1.0)) {
        *why = "the four corners are not coplanar";
        return B200PPF_ERR_UNSUPPORTED;
    }
    return B200PPF_OK;
}

}  // namespace

int prep_crop_pyramid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, b200ppf_cloud **out, uint32_t *kept_host) {
    PyramidPlanes pl;
    const char *why = nullptr;
    if (int rc = pyramid_planes(corners12, &pl, &why)) return fail_msg(ctx, rc, (std::string("crop: ") + why).c_str());
    const uint32_t n = (uint32_t)in->n;
    StreamBuf<uint32_t> flags(ctx);
    PPF_CUDA(ctx, flags.alloc(n));
    EventTimer timer(ctx);
    if (n) PPF_LAUNCH(ctx, pyramid_flag_kernel, (n + 255) / 256, 256, 0, in->pos, n, pl, flags);
    int rc = compact_cloud(ctx, in, flags, out, kept_host);
    timer.stop();
    return rc;
}

int prep_crop_pyramids(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, size_t n_boxes, b200ppf_cloud **out) {
    std::vector<PyramidPlanes> pl(n_boxes);
    for (size_t b = 0; b < n_boxes; ++b) {
        const char *why = nullptr;
        if (int rc = pyramid_planes(corners12 + 12 * b, &pl[b], &why)) {
            char msg[160];
            snprintf(msg, sizeof(msg), "crop: box %zu: %s", b, why);
            return fail_msg(ctx, rc, msg);
        }
    }
    const uint32_t n = (uint32_t)in->n, K = (uint32_t)n_boxes, T = (n + CROP_TILE - 1) / CROP_TILE;
    // scratch: planes, masks, tile counts (box-major, scanned in place), and the words read back: K totals, 6K bounds
    StreamBuf<PyramidPlanes> d_pl(ctx);
    StreamBuf<unsigned long long> mask(ctx);
    StreamBuf<uint32_t> counts(ctx), back(ctx);
    StreamBuf<float4 *> d_out(ctx);
    PPF_CUDA(ctx, d_pl.alloc(K));
    PPF_CUDA(ctx, mask.alloc(n));
    PPF_CUDA(ctx, counts.alloc((size_t)K * T));
    PPF_CUDA(ctx, back.alloc(7 * (size_t)K));
    PPF_CUDA(ctx, d_out.alloc(2 * (size_t)K));
    uint32_t *d_tot = back, *d_lo = back + K, *d_hi = back + 4 * K;
    EventTimer timer(ctx);
    PPF_CUDA(ctx, cudaMemcpyAsync(d_pl, pl.data(), K * sizeof(PyramidPlanes), cudaMemcpyHostToDevice, ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(d_tot, 0, K * sizeof(uint32_t), ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(d_lo, 0xFF, 3 * K * sizeof(uint32_t), ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(d_hi, 0x00, 3 * K * sizeof(uint32_t), ctx->stream));
    if (n) {
        PPF_LAUNCH(ctx, pyramids_mask_kernel, T, CROP_TILE, 0, in->pos, n, d_pl, (int)K, mask, counts, d_lo, d_hi);
        if (int rc = scan_rows(ctx, counts, K, T, d_tot)) return rc;
    }
    std::vector<uint32_t> h(7 * (size_t)K);
    PPF_CUDA(ctx, cudaMemcpyAsync(h.data(), back, h.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the one wait: the clouds are sized by the counts
    std::vector<CloudPtr> c(K);
    std::vector<float4 *> ptrs(2 * (size_t)K);
    for (uint32_t b = 0; b < K; ++b) {
        if (int rc = cloud_alloc(ctx, h[b], &c[b])) return rc;
        for (int k = 0; k < 3; ++k) {  // cloud_bbox_from_device's values: exact bounds, zeros for an empty cloud
            c[b]->bbox_min[k] = h[b] ? float_unorder(h[K + 3 * b + k]) : 0.0f;
            c[b]->bbox_max[k] = h[b] ? float_unorder(h[4 * K + 3 * b + k]) : 0.0f;
        }
        ptrs[b] = c[b]->pos;
        ptrs[K + b] = c[b]->nrm;
    }
    if (n) {
        PPF_CUDA(ctx, cudaMemcpyAsync(d_out, ptrs.data(), ptrs.size() * sizeof(float4 *), cudaMemcpyHostToDevice, ctx->stream));
        PPF_LAUNCH(ctx, pyramids_scatter_kernel, T, CROP_TILE, 0, in->pos, in->nrm, n, mask, (int)K, counts, d_out);
    }
    timer.stop();
    for (uint32_t b = 0; b < K; ++b) out[b] = c[b].release();
    return B200PPF_OK;
}

int prep_renormalize(b200ppf_ctx *ctx, b200ppf_cloud *cloud) {
    const uint32_t n = (uint32_t)cloud->n;
    if (n) PPF_LAUNCH(ctx, renormalize_kernel, (n + 255) / 256, 256, 0, cloud->nrm, n);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

// Test hook: the neighbour query of the kernels (knn_query, __host__ __device__) run on the CPU over a grid built
// on the host with the same geometry (scene_grid_params / grid_cell_coord).  Not a product path: nothing in the
// library calls it; tests use it to check the traversal and the epilogues where there is no GPU.
int prep_debug_knn_host(const float *xyz, size_t n, size_t stride, int k, int mode, float cell_edge, const float *viewpoint3,
                        int cov_mode, uint32_t *idx, float *d2, float *mean_dist, float *normals4) {
    if (n == 0) return B200PPF_OK;
    std::vector<float4> pos(n), gpos(n), nrm(mode == KNN_NORMAL ? n : 0);
    b200ppf_cloud c;
    c.n = n;
    for (int t = 0; t < 3; ++t) c.bbox_min[t] = INFINITY, c.bbox_max[t] = -INFINITY;
    for (size_t i = 0; i < n; ++i) {
        const float *p = xyz + i * stride;
        pos[i] = make_float4(p[0], p[1], p[2], 1.0f);
        for (int t = 0; t < 3; ++t) {
            c.bbox_min[t] = std::min(c.bbox_min[t], p[t]);
            c.bbox_max[t] = std::max(c.bbox_max[t], p[t]);
        }
    }
    KnnArgs a{};
    a.k = k;
    const uint32_t n_cells = scene_grid_params(c.bbox_min, c.bbox_max, cell_edge > 0.0f ? cell_edge : knn_cell_edge(&c, k), &a.gp);
    std::vector<uint32_t> cell(n), start((size_t)n_cells + 1, 0u), orig(n);
    for (size_t i = 0; i < n; ++i) {
        cell[i] = grid_cell_linear(a.gp, grid_cell_coord(a.gp, pos[i].x, 0), grid_cell_coord(a.gp, pos[i].y, 1),
                                   grid_cell_coord(a.gp, pos[i].z, 2));
        start[cell[i] + 1]++;
    }
    for (uint32_t t = 0; t < n_cells; ++t) start[t + 1] += start[t];
    {
        std::vector<uint32_t> fill(start.begin(), start.end() - 1);
        for (size_t i = 0; i < n; ++i) {  // stable: original order inside a cell, like the radix sort
            const uint32_t s = fill[cell[i]]++;
            orig[s] = (uint32_t)i;
            gpos[s] = pos[i];
        }
    }
    a.pos = pos.data();
    a.gpos = gpos.data();
    a.cell_start = start.data();
    a.orig = orig.data();
    a.cell = 1.0f / a.gp.inv_cell;
    a.n = (uint32_t)n;
    a.out_idx = idx;
    a.out_d2 = d2;
    a.out_dist = mean_dist;
    a.out_nrm = nrm.data();
    for (int t = 0; t < 3; ++t) a.vp[t] = viewpoint3 ? viewpoint3[t] : 0.0f;
    a.cov_mode = cov_mode;
    LocalKeys<128> keys;
    for (uint32_t q = 0; q < (uint32_t)n; ++q) {
        if (mode == KNN_EXPORT) {
            knn_query<KNN_EXPORT>(a, q, keys);
        } else if (mode == KNN_MEAN_DISTANCE) {
            knn_query<KNN_MEAN_DISTANCE>(a, q, keys);
        } else {
            knn_query<KNN_NORMAL>(a, q, keys);
        }
    }
    if (mode == KNN_NORMAL)
        for (size_t i = 0; i < n; ++i) normals4[4 * i] = nrm[i].x, normals4[4 * i + 1] = nrm[i].y, normals4[4 * i + 2] = nrm[i].z, normals4[4 * i + 3] = nrm[i].w;
    return B200PPF_OK;
}

}  // namespace b200ppf
