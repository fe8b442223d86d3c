// k6_icp.cu — K6: ICP refinement of the top PPF poses ("next" row of the path, SURVEY.md §8f rank 1).
//
// Replaces, for the step that follows PPF matching in the reference
// (include/CloudProcessing.h:465-470 / :518-523: ICP icp(100, 0.005f, 2.5f, 8);
//  icp.registerModelToScene(models[id], pc_scene, resultsSub)), opencv_contrib's
// surface_matching/src/icp.cpp — the multi-resolution "picky" point-to-plane ICP (Birdal & Ilic):
//   both clouds centred on the mean of their centroids and scaled by n / mean distance to the origin;
//   coarse to fine over num_levels, level L on every round(n / round(n / 2^L))-th point of both clouds with
//   tolerance * (L+1)^2 and max_iterations / (L+1) iterations; pose <- PoseX * pose per level; the
//   normalisation is undone at the end.  The tests' CPU restatement of the same source is the checker.
//
// One persistent thread-block CLUSTER (8 CTAs x 1024 threads, one SM each) per pose hypothesis runs the whole
// refinement — every pyramid level and every iteration — in ONE launch: the reference refines its five best
// poses, and an iteration is far too small (<= 20 k points) to be worth a kernel launch, let alone several.
// Several jobs (models and scenes) share launches: every pose reads its clouds and scratch slices from a descriptor, and
// the poses whose models want the same cluster size run in one launch (b200ppf_icp_refine_batch).
// The samples are strided over the cluster; sums and histograms are combined through distributed shared
// memory (every CTA adds the eight partials in rank order, so all of them hold bit-identical state and take
// the same branches); cluster.sync() is the only inter-SM synchronisation.  FP64 is scarce on this part
// (measured: the double transforms dominate), which is what the eight SMs per pose are for.  Per iteration:
//   nearest scene sample of every moved model sample   uniform grid over the level's scene samples, growing
//                                                      shells, exact (ties: lowest index), float distances
//   robust threshold  median + scale * 1.4826 * MAD    two exact radix selects (4 x 8-bit shared histograms)
//   one model sample per scene sample                  64-bit atomicMin on (distance bits, model sample)
//   point-to-plane normal equations                    27 doubles reduced by shuffles + shared memory
//   6 x 6 minimum-norm solve                           first warp (elimination on lane 0 when the rank is full)
//   Euler -> pose, error, stop test                    thread 0, double precision
//   move the level's samples                           all threads
// Arithmetic follows the original operation for operation (float where cv::Mat is CV_32F, double elsewhere,
// -fmad=false), so the only differences are libm's double sin/cos and the order of the reductions.
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>
#include <utility>
#include <vector>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

namespace cg = cooperative_groups;

constexpr int ICP_THREADS = 1024;
constexpr int ICP_CLUSTER = 8;  // CTAs (SMs) per pose, at most
constexpr uint32_t ICP_BRUTE_MAX = 1024;  // levels with at most this many scene samples search them all from shared memory
constexpr int ICP_WARPS = ICP_THREADS / 32;
constexpr uint32_t ICP_CELLS_MAX = 1u << 16;  // grid cells per level (scanned by the CTA)
constexpr int NEQ = 29;                       // 21 (upper A) + 6 (b) + 1 (squared error) + 1 (matches)

// one pose of a launch: its clouds, and its slices of the call's scratch slab (sized by its own clouds)
struct IcpPose {
    const float4 *mpos, *mnrm;
    const float4 *spos, *snrm;
    uint32_t n_model, n_scene;
    uint32_t slot;               // index of the pose in the call's poses / residuals
    float *src_norm, *dst_norm;  // [n_model][6], [n_scene][6]  normalised clouds
    float *src_t;                // [n_model][6]  level samples under the level's start pose
    float *moved;                // [n_model][3]
    int *nn;                     // [n_model]  nearest scene sample of every level sample (kept between iterations)
    int *nn_prev;                // [n_model]  the same at the end of the previous (coarser) level
    float *d2;                   // [n_model]
    unsigned long long *winner;  // [n_scene]
    uint32_t *cell_start;        // [ICP_CELLS_MAX + 1]
    uint32_t *cell_fill;         // [ICP_CELLS_MAX]
    float4 *items;               // [n_scene]  cell-sorted level scene samples {x, y, z, sample index}
};

struct IcpArgs {
    const IcpPose *pose;  // [gridDim.y]: the cluster of blockIdx.y refines pose[blockIdx.y]
    int max_iterations, num_levels;
    float tolerance, rejection_scale;
    double *poses;       // [n_poses][16] in: start, out: refined
    double *residuals;   // [n_poses]
    unsigned long long *iterations;
};

struct GridDev {  // any exact nearest-neighbour structure gives the same matches: the grid itself is fp32
    float lo[3], cell, inv_cell;
    int dim[3];
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// sum K doubles per thread over the CTA; the totals land in out[0..K) (shared), visible after the call
template <int K>
__device__ void block_sum(const double *v, double *out, double (*scratch)[NEQ]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const double s = warp_sum(v[k]);
        if (lane == 0) scratch[w][k] = s;
    }
    __syncthreads();
    if (w == 0) {
        for (int k = 0; k < K; ++k) {
            const double s = warp_sum(lane < ICP_WARPS ? scratch[lane][k] : 0.0);
            if (lane == 0) out[k] = s;
        }
    }
    __syncthreads();
}

// the same over the cluster: every CTA adds the partials of all ranks in rank order -> identical totals everywhere
template <int K>
__device__ void cluster_sum(cg::cluster_group &cluster, const double *v, double *part, double *out, double (*scratch)[NEQ]) {
    block_sum<K>(v, part, scratch);
    cluster.sync();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (unsigned r = 0; r < cluster.num_blocks(); ++r) s += cluster.map_shared_rank(part, r)[threadIdx.x];
        out[threadIdx.x] = s;
    }
    cluster.sync();
}

__device__ __forceinline__ void transform_point(const double *P, const float *s, float *d, bool with_normal) {
    const double x = s[0], y = s[1], z = s[2];
    double w = P[12] * x + P[13] * y + P[14] * z + P[15];
    if (w == 0.0) w = 1.0;
    d[0] = (float)((P[0] * x + P[1] * y + P[2] * z + P[3]) / w);
    d[1] = (float)((P[4] * x + P[5] * y + P[6] * z + P[7]) / w);
    d[2] = (float)((P[8] * x + P[9] * y + P[10] * z + P[11]) / w);
    if (with_normal) {
        const double nx = s[3], ny = s[4], nz = s[5];
        double rx = P[0] * nx + P[1] * ny + P[2] * nz;
        double ry = P[4] * nx + P[5] * ny + P[6] * nz;
        double rz = P[8] * nx + P[9] * ny + P[10] * nz;
        const double len = sqrt(rx * rx + ry * ry + rz * rz);
        if (len > 1e-12) {
            rx /= len;
            ry /= len;
            rz /= len;
        }
        d[3] = (float)rx;
        d[4] = (float)ry;
        d[5] = (float)rz;
    }
}

__device__ __forceinline__ void mat4_mul(const double *a, const double *b, double *c) {
    for (int r = 0; r < 4; ++r)
        for (int k = 0; k < 4; ++k) {
            double s = 0.0;
            for (int q = 0; q < 4; ++q) s += a[r * 4 + q] * b[q * 4 + k];
            c[r * 4 + k] = s;
        }
}

// Minimum-norm least squares from the 6 x 6 Gram matrix (what cv::solve(DECOMP_SVD) returns for the n x 6 system): cyclic
// Jacobi rotations, eigenvalues below 1e-12 of the largest dropped.  With fewer than six surviving correspondences (the
// coarsest levels of a small cloud) an elimination would divide by rounding noise; this stays put in the directions the
// data do not constrain.  Operation for operation the solve the tests' CPU checker performs, run by one warp on shared
// memory.  The 15 index pairs of a sweep are taken as 5 rounds of 3 disjoint pairs (the same table as the checker's):
// lanes 0-5, 6-11 and 12-17 evaluate the three rotations of a round side by side — the divide / square-root chain of a
// rotation is five dependent double-precision operations, ~0.4 us, and a sweep is five of them instead of fifteen — and
// lane 6 u + k takes index k of rotation u's column updates and then of its row updates; the convergence sums are
// evaluated redundantly by every lane in the checker's order.
__constant__ int JACOBI_ROUNDS[5][3][2] = {{{0, 5}, {1, 4}, {2, 3}}, {{1, 5}, {0, 2}, {3, 4}}, {{2, 5}, {1, 3}, {0, 4}},
                                           {{3, 5}, {2, 4}, {0, 1}}, {{4, 5}, {0, 3}, {1, 2}}};

__device__ bool solve6_min_norm_warp(double *A, double *V, const double *b, double *x, int lane) {
    if (lane < 6)
        for (int k = 0; k < 6; ++k) V[lane * 6 + k] = k == lane ? 1.0 : 0.0;
    __syncwarp();
    const int u = lane < 18 ? lane / 6 : 0, k = lane % 6;  // lanes 18-31 shadow pair 0 and write nothing
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int p = 0; p < 6; ++p) {
            diag += fabs(A[p * 6 + p]);
            for (int q = p + 1; q < 6; ++q) off += fabs(A[p * 6 + q]);
        }
        if (!(off > 1e-300) || off <= 1e-18 * diag) break;  // warp-uniform
        for (int round = 0; round < 5; ++round) {
            const int p = JACOBI_ROUNDS[round][u][0], q = JACOBI_ROUNDS[round][u][1];
            const double apq = A[p * 6 + q];
            double c = 1.0, sn = 0.0;
            if (apq != 0.0) {
                const double theta = (A[q * 6 + q] - A[p * 6 + p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                c = 1.0 / sqrt(t * t + 1.0);
                sn = t * c;
            }
            __syncwarp();  // every lane has read its rotation's inputs
            if (lane < 18) {  // columns p, q of A and V, row k
                const double akp = A[k * 6 + p], akq = A[k * 6 + q];
                A[k * 6 + p] = c * akp - sn * akq;
                A[k * 6 + q] = sn * akp + c * akq;
                const double vkp = V[k * 6 + p], vkq = V[k * 6 + q];
                V[k * 6 + p] = c * vkp - sn * vkq;
                V[k * 6 + q] = sn * vkp + c * vkq;
            }
            __syncwarp();
            if (lane < 18) {  // rows p, q of A, column k
                const double apk = A[p * 6 + k], aqk = A[q * 6 + k];
                A[p * 6 + k] = c * apk - sn * aqk;
                A[q * 6 + k] = sn * apk + c * aqk;
            }
            __syncwarp();
        }
    }
    bool ok = true;
    if (lane == 0) {
        double lmax = 0.0;
        for (int k = 0; k < 6; ++k) lmax = fmax(lmax, A[k * 6 + k]);
        ok = lmax > 0.0;
        if (ok) {
            const double cut = 1e-12 * lmax;
            for (int r = 0; r < 6; ++r) x[r] = 0.0;
            for (int k = 0; k < 6; ++k) {
                const double l = A[k * 6 + k];
                if (!(l > cut)) continue;
                double proj = 0.0;
                for (int r = 0; r < 6; ++r) proj += V[r * 6 + k] * b[r];
                proj /= l;
                for (int r = 0; r < 6; ++r) x[r] += V[r * 6 + k] * proj;
            }
            for (int c = 0; c < 6; ++c)
                if (!isfinite(x[c])) ok = false;
        }
    }
    return __shfl_sync(0xFFFFFFFFu, ok ? 1 : 0, 0) != 0;
}

// Fast path (lane 0): the elimination of round 1 (partial pivoting) while every pivot is at least 1e-9 of the largest
// diagonal entry — then the system has full rank and the least-squares solution is the minimum-norm one; otherwise (fewer
// than six independent correspondences) the Jacobi form above.  Both implementations take the same branch on the same
// numbers.  Called by the whole first warp; A, V, b, x live in shared memory.
__device__ bool solve6_warp(double *A, double *V, const double *b, double *x, int lane) {
    int state = 0;  // 0: rank-deficient, 1: solved, 2: failed
    if (lane == 0) {
        double E[36], g[6], dmax = 0.0;
        for (int k = 0; k < 36; ++k) E[k] = A[k];
        for (int k = 0; k < 6; ++k) {
            g[k] = b[k];
            dmax = fmax(dmax, fabs(A[k * 6 + k]));
        }
        const double floor_pivot = 1e-9 * dmax;
        int perm[6] = {0, 1, 2, 3, 4, 5};
        bool full_rank = dmax > 0.0;
        for (int c = 0; c < 6 && full_rank; ++c) {
            int piv = c;
            for (int r = c + 1; r < 6; ++r)
                if (fabs(E[perm[r] * 6 + c]) > fabs(E[perm[piv] * 6 + c])) piv = r;
            const int t = perm[c];
            perm[c] = perm[piv];
            perm[piv] = t;
            const double d = E[perm[c] * 6 + c];
            if (!(fabs(d) > floor_pivot)) {
                full_rank = false;
                break;
            }
            for (int r = c + 1; r < 6; ++r) {
                const double f = E[perm[r] * 6 + c] / d;
                for (int k = c; k < 6; ++k) E[perm[r] * 6 + k] -= f * E[perm[c] * 6 + k];
                g[perm[r]] -= f * g[perm[c]];
            }
        }
        if (full_rank) {
            double xs[6];
            for (int c = 5; c >= 0; --c) {
                double sacc = g[perm[c]];
                for (int k = c + 1; k < 6; ++k) sacc -= E[perm[c] * 6 + k] * xs[k];
                xs[c] = sacc / E[perm[c] * 6 + c];
            }
            state = 1;
            for (int c = 0; c < 6; ++c) {
                x[c] = xs[c];
                if (!isfinite(xs[c])) state = 2;
            }
        }
    }
    state = __shfl_sync(0xFFFFFFFFu, state, 0);
    if (state == 0) return solve6_min_norm_warp(A, V, b, x, lane);
    return state == 1;
}

__device__ void pose_from_euler(const double *rpy, const double *t, double *P) {
    const double cx = cos(rpy[0]), sx = sin(rpy[0]);
    const double cy = cos(rpy[1]), sy = sin(rpy[1]);
    const double cz = cos(rpy[2]), sz = sin(rpy[2]);
    const double Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx};
    const double Ry[9] = {cy, 0, sy, 0, 1, 0, -sy, 0, cy};
    const double Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1};
    double T[9], R[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) T[r * 3 + c] = Ry[r * 3] * Rz[c] + Ry[r * 3 + 1] * Rz[3 + c] + Ry[r * 3 + 2] * Rz[6 + c];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r * 3 + c] = Rx[r * 3] * T[c] + Rx[r * 3 + 1] * T[3 + c] + Rx[r * 3 + 2] * T[6 + c];
    for (int k = 0; k < 16; ++k) P[k] = 0.0;
    P[15] = 1.0;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) P[r * 4 + c] = R[r * 3 + c];
        P[r * 4 + 3] = t[r];
    }
}

// k-th smallest (0-based) of the non-negative floats f(i) over this cluster's samples i = first, first + stride, ...
// 4 passes of 8-bit histograms: local shared histogram, summed over the cluster through distributed shared memory
template <class F>
__device__ float cluster_select(cg::cluster_group &cluster, uint32_t m, uint32_t first, uint32_t stride, uint32_t k, F f,
                                uint32_t *hist, uint32_t *hist_tot, uint32_t *s_sel /*[2]: prefix, k*/) {
    if (threadIdx.x == 0) {
        s_sel[0] = 0;
        s_sel[1] = k;
    }
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (uint32_t d = threadIdx.x; d < 256; d += ICP_THREADS) hist[d] = 0;
        __syncthreads();
        const uint32_t prefix = s_sel[0];
        for (uint32_t i = first; i < m; i += stride) {
            const uint32_t bits = __float_as_uint(f(i));
            if (shift == 24 || (bits >> (shift + 8)) == prefix) atomicAdd(&hist[(bits >> shift) & 255u], 1u);
        }
        cluster.sync();
        if (threadIdx.x < 256) {
            uint32_t t = 0;
            for (unsigned r = 0; r < cluster.num_blocks(); ++r) t += cluster.map_shared_rank(hist, r)[threadIdx.x];
            hist_tot[threadIdx.x] = t;
        }
        cluster.sync();
        if (threadIdx.x == 0) {
            uint32_t kk = s_sel[1], d = 0;
            while (d < 255 && hist_tot[d] <= kk) kk -= hist_tot[d++];
            s_sel[0] = (prefix << 8) | d;
            s_sel[1] = kk;
        }
        __syncthreads();
    }
    return __uint_as_float(s_sel[0]);
}

__device__ __forceinline__ int grid_coord(const GridDev &g, float v, int c) {
    const int k = (int)floorf((v - g.lo[c]) * g.inv_cell);
    return k < 0 ? 0 : (k >= g.dim[c] ? g.dim[c] - 1 : k);
}

__global__ void __launch_bounds__(ICP_THREADS, 1) icp_refine_kernel(const IcpArgs a) {
    __shared__ double s_red[ICP_WARPS][NEQ];
    __shared__ double s_part[NEQ], s_tot[NEQ];
    __shared__ double s_pose[16], s_posex[16], s_mean[3];
    __shared__ double s_A[36], s_V[36], s_b6[6], s_x6[6];  // the 6 x 6 solve of the first warp
    __shared__ float4 s_items[ICP_BRUTE_MAX];              // a small level's scene samples (x, y, z, index)
    __shared__ double s_scale, s_fold, s_fperc, s_fmin;
    __shared__ GridDev s_grid;
    __shared__ uint32_t s_hist[256], s_hist_tot[256], s_sel[2], s_carry;
    __shared__ int s_flag, s_iter;
    __shared__ float s_bb[ICP_WARPS][6];

    __shared__ IcpPose s_job;

    cg::cluster_group cluster = cg::this_cluster();
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t rank = cluster.block_rank(), csize = cluster.num_blocks();
    const uint32_t first = rank * ICP_THREADS + tid, stride = csize * ICP_THREADS;  // this thread's samples
    if (tid == 0) s_job = a.pose[blockIdx.y];
    __syncthreads();
    const uint32_t p = s_job.slot;
    const uint32_t n = s_job.n_model, nd = s_job.n_scene;
    const float4 *const mpos = s_job.mpos, *const mnrm = s_job.mnrm, *const spos = s_job.spos, *const snrm = s_job.snrm;
    float *src = s_job.src_norm, *dst = s_job.dst_norm;
    float *src_t = s_job.src_t, *moved = s_job.moved;
    int *nn = s_job.nn;
    int *nn_prev = s_job.nn_prev;
    float *d2 = s_job.d2;
    unsigned long long *winner = s_job.winner;
    uint32_t *cell_start = s_job.cell_start;
    uint32_t *cell_fill = s_job.cell_fill;
    float4 *items = s_job.items;
    double start_pose[16];
    for (int k = 0; k < 16; ++k) start_pose[k] = a.poses[(size_t)p * 16 + k];

    // ---- srcTemp = transformPCPose(model, start); centre both clouds, scale ------------------------------------
    double acc[NEQ];
    for (int k = 0; k < NEQ; ++k) acc[k] = 0.0;
    for (uint32_t i = first; i < n; i += stride) {
        const float4 q = mpos[i], r = mnrm[i];
        const float in[6] = {q.x, q.y, q.z, r.x, r.y, r.z};
        float out[6];
        transform_point(start_pose, in, out, true);
        for (int c = 0; c < 6; ++c) src[6 * (size_t)i + c] = out[c];
        acc[0] += out[0];
        acc[1] += out[1];
        acc[2] += out[2];
    }
    for (uint32_t i = first; i < nd; i += stride) {
        const float4 q = spos[i], r = snrm[i];
        dst[6 * (size_t)i] = q.x;
        dst[6 * (size_t)i + 1] = q.y;
        dst[6 * (size_t)i + 2] = q.z;
        dst[6 * (size_t)i + 3] = r.x;
        dst[6 * (size_t)i + 4] = r.y;
        dst[6 * (size_t)i + 5] = r.z;
        acc[3] += q.x;
        acc[4] += q.y;
        acc[5] += q.z;
    }
    cluster_sum<6>(cluster, acc, s_part, s_tot, s_red);
    if (tid == 0)
        for (int c = 0; c < 3; ++c) s_mean[c] = 0.5 * (s_tot[c] / (double)n + s_tot[3 + c] / (double)nd);
    __syncthreads();
    acc[0] = acc[1] = 0.0;
    for (uint32_t i = first; i < n; i += stride) {
        float *q = src + 6 * (size_t)i;
        for (int c = 0; c < 3; ++c) q[c] = (float)((double)q[c] - s_mean[c]);
        acc[0] += sqrt((double)q[0] * q[0] + (double)q[1] * q[1] + (double)q[2] * q[2]);
    }
    for (uint32_t i = first; i < nd; i += stride) {
        float *q = dst + 6 * (size_t)i;
        for (int c = 0; c < 3; ++c) q[c] = (float)((double)q[c] - s_mean[c]);
        acc[1] += sqrt((double)q[0] * q[0] + (double)q[1] * q[1] + (double)q[2] * q[2]);
    }
    cluster_sum<2>(cluster, acc, s_part, s_tot, s_red);
    if (tid == 0) {
        s_scale = (double)n / ((s_tot[0] + s_tot[1]) * 0.5);
        for (int k = 0; k < 16; ++k) s_pose[k] = (k % 5 == 0) ? 1.0 : 0.0;
        s_fmin = 0.0;
    }
    __syncthreads();
    const double scale = s_scale;
    for (uint32_t i = first; i < n; i += stride)
        for (int c = 0; c < 3; ++c) src[6 * (size_t)i + c] = (float)((double)src[6 * (size_t)i + c] * scale);
    for (uint32_t i = first; i < nd; i += stride)
        for (int c = 0; c < 3; ++c) dst[6 * (size_t)i + c] = (float)((double)dst[6 * (size_t)i + c] * scale);
    __threadfence();
    cluster.sync();

    double residual = 0.0;
    unsigned long long iterations = 0;
    int prev_step = 0;
    uint32_t prev_m = 0;
    for (int level = a.num_levels - 1; level >= 0; --level) {
        const double div = pow(2.0, (double)level);
        const int num_samples = (int)nearbyint((double)n / div);
        const double tol_p = (double)a.tolerance * (double)(level + 1) * (double)(level + 1);
        const int max_it = (int)nearbyint((double)a.max_iterations / (double)(level + 1));
        if (num_samples < 1) continue;
        const int step = max(1, (int)nearbyint((double)n / (double)num_samples));
        const uint32_t m = (n + step - 1) / step, md = (nd + step - 1) / step;
        if (m == 0 || md == 0) continue;

        // ---- level samples of the model under the pose so far; bounding box of the scene samples ---------------
        for (uint32_t i = first; i < m; i += stride) {
            float out[6];
            transform_point(s_pose, src + 6 * (size_t)i * step, out, true);
            for (int c = 0; c < 6; ++c) src_t[6 * (size_t)i + c] = out[c];
            for (int c = 0; c < 3; ++c) moved[3 * (size_t)i + c] = out[c];
            // seed of the nearest-neighbour search: the match of the closest sample of the previous, coarser
            // level (sample k there is sample k * prev_step / step here; likewise for the scene samples)
            int seed = -1;
            if (prev_step > 0) {
                const uint32_t ratio = (uint32_t)prev_step / (uint32_t)step;
                if (ratio >= 1 && (uint32_t)prev_step == ratio * (uint32_t)step) {
                    const uint32_t k = min(i / ratio, prev_m - 1);
                    const long long j = (long long)nn_prev[k] * ratio;
                    if (nn_prev[k] >= 0 && j < (long long)md) seed = (int)j;
                }
            }
            nn[i] = seed;
        }
        float lo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, hi[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
        for (uint32_t j = tid; j < md; j += ICP_THREADS)  // every CTA scans all scene samples: no exchange needed
            for (int c = 0; c < 3; ++c) {
                const float v = dst[6 * (size_t)j * step + c];
                lo[c] = fminf(lo[c], v);
                hi[c] = fmaxf(hi[c], v);
            }
        for (int c = 0; c < 3; ++c)
            for (int o = 16; o > 0; o >>= 1) {
                lo[c] = fminf(lo[c], __shfl_xor_sync(0xFFFFFFFFu, lo[c], o));
                hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xFFFFFFFFu, hi[c], o));
            }
        if (lane == 0)
            for (int c = 0; c < 3; ++c) {
                s_bb[warp][c] = lo[c];
                s_bb[warp][3 + c] = hi[c];
            }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < ICP_WARPS; ++w)
                for (int c = 0; c < 3; ++c) {
                    lo[c] = fminf(lo[c], s_bb[w][c]);
                    hi[c] = fmaxf(hi[c], s_bb[w][3 + c]);
                }
            // ~2 samples per cell, at most ICP_CELLS_MAX cells
            const float ex = fmaxf(hi[0] - lo[0], 1e-9f), ey = fmaxf(hi[1] - lo[1], 1e-9f), ez = fmaxf(hi[2] - lo[2], 1e-9f);
            float cell = cbrtf(ex * ey * ez / fmaxf(1.0f, fminf(0.5f * (float)md, (float)ICP_CELLS_MAX / 8.0f)));
            cell = fmaxf(cell, fmaxf(ex, fmaxf(ey, ez)) / 256.0f);
            for (;;) {
                s_grid.dim[0] = (int)floorf(ex / cell) + 1;
                s_grid.dim[1] = (int)floorf(ey / cell) + 1;
                s_grid.dim[2] = (int)floorf(ez / cell) + 1;
                if ((unsigned long long)s_grid.dim[0] * s_grid.dim[1] * s_grid.dim[2] <= ICP_CELLS_MAX) break;
                cell *= 1.26f;
            }
            s_grid.cell = cell;
            s_grid.inv_cell = 1.0f / cell;
            for (int c = 0; c < 3; ++c) s_grid.lo[c] = lo[c];
            for (int k = 0; k < 16; ++k) s_posex[k] = (k % 5 == 0) ? 1.0 : 0.0;
            s_fold = 9999999999.0;
            s_fperc = 0.0;
            s_fmin = 9999999999.0;
            s_iter = 0;
            s_carry = 0;
        }
        __syncthreads();
        const GridDev g = s_grid;
        const uint32_t cells = (uint32_t)g.dim[0] * g.dim[1] * g.dim[2];
        // A small level (the coarse levels of every cloud, every level of the reference's 681-point object) keeps its scene
        // samples in shared memory and tests them all: a few microseconds per iteration, where walking the grid rows around
        // a far-away previous match is a chain of ~700 dependent global loads (~0.2 ms per iteration, whatever the size).
        // The nearest sample, lowest index on ties, is the same either way.
        const bool brute = md <= ICP_BRUTE_MAX;
        if (brute) {
            for (uint32_t j = tid; j < md; j += ICP_THREADS) {
                const float *q = dst + 6 * (size_t)j * step;
                s_items[j] = make_float4(q[0], q[1], q[2], __uint_as_float(j));
            }
            __syncthreads();
        } else {
        // ---- counting sort of the scene samples by cell (counts and fill by the cluster, scan by rank 0) -----------
        for (uint32_t c = first; c < cells; c += stride) cell_fill[c] = 0;
        __threadfence();
        cluster.sync();
        for (uint32_t j = first; j < md; j += stride) {
            const float *q = dst + 6 * (size_t)j * step;
            const uint32_t c = ((uint32_t)grid_coord(g, q[2], 2) * g.dim[1] + grid_coord(g, q[1], 1)) * g.dim[0] +
                               grid_coord(g, q[0], 0);
            atomicAdd(&cell_fill[c], 1u);
        }
        __threadfence();
        cluster.sync();
        if (rank == 0) {
            for (uint32_t base = 0; base < cells; base += ICP_THREADS) {  // exclusive scan, 1024 cells per round
                const uint32_t c = base + tid;
                const uint32_t v = c < cells ? cell_fill[c] : 0u;
                uint32_t incl = v;
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if ((int)lane >= o) incl += t;
                }
                if (lane == 31) s_hist[warp] = incl;
                __syncthreads();
                if (warp == 0) {
                    uint32_t w = s_hist[lane], wi = w;
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, o);
                        if ((int)lane >= o) wi += t;
                    }
                    s_hist[lane] = wi - w;
                    if (lane == 31) s_hist[32] = wi;
                }
                __syncthreads();
                const uint32_t excl = s_carry + s_hist[warp] + incl - v;
                if (c < cells) {
                    cell_start[c] = excl;
                    cell_fill[c] = excl;
                }
                __syncthreads();
                if (tid == 0) s_carry += s_hist[32];
                __syncthreads();
            }
            if (tid == 0) cell_start[cells] = md;
        }
        __threadfence();
        cluster.sync();
        for (uint32_t j = first; j < md; j += stride) {
            const float *q = dst + 6 * (size_t)j * step;
            const uint32_t c = ((uint32_t)grid_coord(g, q[2], 2) * g.dim[1] + grid_coord(g, q[1], 1)) * g.dim[0] +
                               grid_coord(g, q[0], 0);
            items[atomicAdd(&cell_fill[c], 1u)] = make_float4(q[0], q[1], q[2], __uint_as_float(j));
        }
        __threadfence();
        cluster.sync();
        }

        // ---- iterations --------------------------------------------------------------------------------------------
        for (;;) {
            if (tid == 0)
                s_flag = (!(s_fperc < (1.0 + tol_p) && s_fperc > (1.0 - tol_p)) && s_iter < max_it) ? 1 : 0;
            __syncthreads();
            if (!s_flag) break;
            // nearest scene sample of every moved model sample
            const int max_r = max(g.dim[0], max(g.dim[1], g.dim[2]));
            for (uint32_t i = first; i < m; i += stride) {
                const float qx = moved[3 * (size_t)i], qy = moved[3 * (size_t)i + 1], qz = moved[3 * (size_t)i + 2];
                const int cx = grid_coord(g, qx, 0), cy = grid_coord(g, qy, 1), cz = grid_coord(g, qz, 2);
                int best = nn[i];
                float best_d2 = 3.402823466e38f;
                if (brute) {
                    best = -1;
                    for (uint32_t sidx = 0; sidx < md; ++sidx) {
                        const float4 q = s_items[sidx];
                        const float dx = qx - q.x, dy = qy - q.y, dz = qz - q.z;
                        const float dd = dx * dx + dy * dy + dz * dz;
                        const int j = (int)__float_as_uint(q.w);
                        if (dd < best_d2 || (dd == best_d2 && j < best)) {
                            best_d2 = dd;
                            best = j;
                        }
                    }
                } else if (best >= 0) {
                    // Seeded search: the previous iteration's (or level's) match bounds the distance, and only the
                    // cells that intersect the ball of that radius are visited — rows (z, y) and the x range inside
                    // a row are pruned with the current best, which only shrinks.  A sample whose true neighbour
                    // is 15 cells away costs ~700 mostly empty row steps instead of 30 000 distance tests.
                    {
                        const float *q = dst + 6 * (size_t)best * step;
                        const float dx = qx - q[0], dy = qy - q[1], dz = qz - q[2];
                        best_d2 = dx * dx + dy * dy + dz * dz;
                    }
                    const float slack = 1e-3f * g.cell;
                    const float r0 = sqrtf(best_d2) * 1.001f + slack;
                    const int z0 = grid_coord(g, qz - r0, 2), z1 = grid_coord(g, qz + r0, 2);
                    const int y0 = grid_coord(g, qy - r0, 1), y1 = grid_coord(g, qy + r0, 1);
                    const int ny = y1 - y0 + 1, nrows = (z1 - z0 + 1) * ny;
                    int row = 0;
                    uint32_t sidx = 0, e = 0;
                    for (;;) {
                        if (sidx < e) {
                            const float4 q = items[sidx++];
                            const float dx = qx - q.x, dy = qy - q.y, dz = qz - q.z;
                            const float dd = dx * dx + dy * dy + dz * dz;
                            const int j = (int)__float_as_uint(q.w);
                            if (dd < best_d2 || (dd == best_d2 && j < best)) {
                                best_d2 = dd;
                                best = j;
                            }
                        } else {
                            if (row >= nrows) break;
                            const int z = z0 + row / ny, y = y0 + row % ny;
                            ++row;
                            // lower bounds of the distance from the query to slab z / row y (a sliver of a cell
                            // of slack: the cell of a sample comes from floor((v - lo) * inv_cell) in fp32)
                            const float zl = g.lo[2] + (float)z * g.cell, yl = g.lo[1] + (float)y * g.cell;
                            const float gz = fmaxf(0.0f, fmaxf(zl - qz, qz - (zl + g.cell)) - slack) * 0.999f;
                            const float gy = fmaxf(0.0f, fmaxf(yl - qy, qy - (yl + g.cell)) - slack) * 0.999f;
                            const float rem = best_d2 - gz * gz - gy * gy;
                            if (rem < 0.0f) continue;
                            const float reach = sqrtf(rem) * 1.001f + slack;
                            const uint32_t base = ((uint32_t)z * g.dim[1] + y) * g.dim[0];
                            sidx = cell_start[base + grid_coord(g, qx - reach, 0)];
                            e = cell_start[base + grid_coord(g, qx + reach, 0) + 1];
                        }
                    }
                } else
                // Unseeded (the coarsest level): cubes of growing radius.  The cells x0..x1 of one (z, y) row are one
                // contiguous run of the cell-sorted samples, so a cube is (2r+1)^2 plain loops — every lane of
                // the warp walks the same loop nest (the shell-by-shell form left 2 of 32 lanes active).  A
                // larger cube re-tests the inner one; with ~2 samples per cell almost every query ends at r = 1.
                for (int r = 1; r <= max_r; ++r) {
                    const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dim[2] - 1);
                    const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dim[1] - 1);
                    const int x0 = max(cx - r, 0), x1 = min(cx + r, g.dim[0] - 1);
                    // one flat loop over the concatenated runs: an iteration either tests a sample or steps to
                    // the next row, so lanes whose rows are empty do not idle while others walk theirs
                    const int ny = y1 - y0 + 1, nrows = (z1 - z0 + 1) * ny;
                    int row = 0;
                    uint32_t sidx = 0, e = 0;
                    for (;;) {
                        if (sidx < e) {
                            const float4 q = items[sidx++];
                            const float dx = qx - q.x, dy = qy - q.y, dz = qz - q.z;
                            const float dd = dx * dx + dy * dy + dz * dz;
                            const int j = (int)__float_as_uint(q.w);
                            if (dd < best_d2 || (dd == best_d2 && j < best)) {
                                best_d2 = dd;
                                best = j;
                            }
                        } else {
                            if (row >= nrows) break;
                            const int z = z0 + row / ny, y = y0 + row % ny;
                            const uint32_t base = ((uint32_t)z * g.dim[1] + y) * g.dim[0];
                            sidx = cell_start[base + x0];
                            e = cell_start[base + x1 + 1];
                            ++row;
                        }
                    }
                    // every sample outside the cube is more than r cells away along one axis (slack: fp32 grid)
                    const float reach = (float)r * g.cell * 0.999f;
                    if (best >= 0 && best_d2 <= reach * reach) break;
                }
                nn[i] = best;
                d2[i] = best_d2;
            }
            for (uint32_t j = first; j < md; j += stride) winner[j] = ~0ull;
            __threadfence();
            // robust rejection threshold on the squared distances (the selects synchronise the cluster)
            float thr = 3.402823466e38f;
            if (a.rejection_scale > 0.0f) {
                const uint32_t k = (m - 1) / 2;
                const float med = cluster_select(cluster, m, first, stride, k, [&](uint32_t i) { return d2[i]; }, s_hist,
                                                 s_hist_tot, s_sel);
                const float mad = cluster_select(
                    cluster, m, first, stride, k, [&](uint32_t i) { return (float)fabs((double)d2[i] - (double)med); },
                    s_hist, s_hist_tot, s_sel);
                const float sdev = 1.48257968f * mad;
                thr = a.rejection_scale * sdev + med;
            } else {
                cluster.sync();
            }
            // of several model samples on one scene sample the closest survives (lowest index on ties)
            for (uint32_t i = first; i < m; i += stride)
                if (a.rejection_scale <= 0.0f || d2[i] < thr)
                    atomicMin(&winner[nn[i]], ((unsigned long long)__float_as_uint(d2[i]) << 32) | i);
            __threadfence();
            cluster.sync();
            // point-to-plane normal equations over the surviving pairs
            for (int k = 0; k < NEQ; ++k) acc[k] = 0.0;
            for (uint32_t j = first; j < md; j += stride) {
                const unsigned long long wv = winner[j];
                if (wv == ~0ull) continue;
                const float *s = src_t + 6 * (size_t)(uint32_t)wv;
                const float *d = dst + 6 * (size_t)j * step;
                const double sp[3] = {s[0], s[1], s[2]}, dp[3] = {d[0], d[1], d[2]}, nr[3] = {d[3], d[4], d[5]};
                const double row[6] = {sp[1] * nr[2] - sp[2] * nr[1], sp[2] * nr[0] - sp[0] * nr[2],
                                       sp[0] * nr[1] - sp[1] * nr[0], nr[0], nr[1], nr[2]};
                const double rhs = (dp[0] - sp[0]) * nr[0] + (dp[1] - sp[1]) * nr[1] + (dp[2] - sp[2]) * nr[2];
                int q = 0;
                for (int r = 0; r < 6; ++r)
                    for (int c = r; c < 6; ++c) acc[q++] += row[r] * row[c];
                for (int r = 0; r < 6; ++r) acc[21 + r] += row[r] * rhs;
                for (int c = 0; c < 6; ++c) {
                    const double e = (double)s[c] - (double)d[c];
                    acc[27] += e * e;
                }
                acc[28] += 1.0;
            }
            cluster_sum<NEQ>(cluster, acc, s_part, s_tot, s_red);
            if (tid < 32) {  // the first warp solves; lane 0 does the scalar parts
                if (tid == 0) {
                    int q = 0;
                    for (int r = 0; r < 6; ++r)
                        for (int c = r; c < 6; ++c) {
                            s_A[r * 6 + c] = s_tot[q];
                            s_A[c * 6 + r] = s_tot[q];
                            ++q;
                        }
                    for (int r = 0; r < 6; ++r) s_b6[r] = s_tot[21 + r];
                }
                __syncwarp();
                bool ok = s_tot[28] > 0.0;
                if (ok) ok = solve6_warp(s_A, s_V, s_b6, s_x6, (int)tid);
                __syncwarp();
                if (tid == 0) {
                    if (ok) {
                        pose_from_euler(s_x6, s_x6 + 3, s_posex);
                        const double fval = sqrt(s_tot[27]) / (double)m;
                        s_fperc = fval / s_fold;
                        s_fold = fval;
                        if (fval < s_fmin) s_fmin = fval;
                        ++s_iter;
                    }
                    s_flag = ok ? 1 : 0;
                }
            }
            __syncthreads();
            if (!s_flag) break;
            ++iterations;
            for (uint32_t i = first; i < m; i += stride) {
                float out[3];
                transform_point(s_posex, src_t + 6 * (size_t)i, out, false);
                for (int c = 0; c < 3; ++c) moved[3 * (size_t)i + c] = out[c];
            }
            __syncthreads();
        }
        if (tid == 0) {
            double np[16];
            mat4_mul(s_posex, s_pose, np);
            for (int k = 0; k < 16; ++k) s_pose[k] = np[k];
        }
        residual = s_fmin;
        for (uint32_t i = first; i < m; i += stride) nn_prev[i] = nn[i];
        prev_step = step;
        prev_m = m;
        __threadfence();
        cluster.sync();
    }
    if (tid == 0 && rank == 0) {
        // undo the normalisation, then Pose3D::appendPose: refined = delta * start
        double delta[16], out[16];
        for (int k = 0; k < 16; ++k) delta[k] = s_pose[k];
        for (int r = 0; r < 3; ++r) {
            const double rm = delta[r * 4] * s_mean[0] + delta[r * 4 + 1] * s_mean[1] + delta[r * 4 + 2] * s_mean[2];
            delta[r * 4 + 3] = delta[r * 4 + 3] / s_scale + s_mean[r] - rm;
        }
        mat4_mul(delta, start_pose, out);
        for (int k = 0; k < 16; ++k) a.poses[(size_t)p * 16 + k] = out[k];
        if (a.residuals) a.residuals[p] = residual;
        if (a.iterations) atomicAdd(a.iterations, iterations);
    }
}

// CTAs per pose cluster for a model of n points.  An iteration is a chain of ~20 cluster-wide synchronisations around little
// arithmetic, so the cluster is only as large as the model needs: one CTA per 1 024 model points, at most ICP_CLUSTER (the
// reference's 543-point bottle runs in a single CTA, whose cluster barrier is a block barrier).  The cluster size fixes the
// order of the reductions, so a pose gives the same bits whatever else shares its launch.
int icp_cluster_size(size_t n_model) {
    int csize = 1;
    while (csize < ICP_CLUSTER && (size_t)csize * ICP_THREADS < n_model) csize *= 2;
    if (const char *e = getenv("B200PPF_ICP_CLUSTER")) csize = std::max(1, std::min(ICP_CLUSTER, atoi(e)));
    return csize;
}

}  // namespace

int k6_icp_refine_batch(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, int max_iterations, float tolerance,
                        float rejection_scale, int num_levels, uint64_t *iterations_host) {
    char msg[160];
    auto bad = [&](int code, size_t j, const char *what) {  // the single call's messages name no job
        if (n_jobs == 1) snprintf(msg, sizeof(msg), "icp: %s", what);
        else snprintf(msg, sizeof(msg), "icp: job %zu: %s", j, what);
        return fail_msg(ctx, code, msg);
    };
    size_t P = 0;
    for (size_t j = 0; j < n_jobs; ++j) {
        if (jobs[j].n_poses == 0) continue;
        if (jobs[j].n_poses > 65535) return bad(B200PPF_ERR_UNSUPPORTED, j, "more than 65535 poses per call");
        if (jobs[j].model->n == 0 || jobs[j].scene->n == 0) return bad(B200PPF_ERR_INVALID, j, "empty cloud");
        P += jobs[j].n_poses;
    }
    if (P == 0) return B200PPF_OK;
    if (max_iterations < 1 || num_levels < 1 || num_levels > 30 || !(tolerance >= 0.0f))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "icp: bad parameters");
    // one launch per cluster size, sizes ascending; within a launch the poses keep job order
    std::vector<std::pair<int, size_t>> order;  // (cluster size, job)
    for (size_t j = 0; j < n_jobs; ++j)
        if (jobs[j].n_poses) order.push_back({icp_cluster_size(jobs[j].model->n), j});
    std::stable_sort(order.begin(), order.end(), [](const auto &x, const auto &y) { return x.first < y.first; });
    for (size_t g = 0, e = 0; g < order.size(); g = e) {
        size_t poses = 0;
        for (e = g; e < order.size() && order[e].first == order[g].first; ++e) poses += jobs[order[e].second].n_poses;
        if (poses > 65535) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "icp: more than 65535 poses of one cluster size per call");
    }
    // one slab for all scratch: the call's poses, residuals, iteration counter and descriptors, then each pose's slices
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off += (bytes + 255) & ~(size_t)255;
        return o;
    };
    const size_t o_poses = take(P * 16 * sizeof(double)), o_res = take(P * sizeof(double)), o_it = take(sizeof(unsigned long long));
    const size_t o_desc = take(P * sizeof(IcpPose));
    std::vector<size_t> job_first(n_jobs, 0), pose_off(P);  // first slot of each job; scratch offset of each slot
    struct Slices {
        size_t src, dst, srct, moved, nn, nnp, d2, win, cs, cf, items;
    };
    auto slices = [&](size_t n, size_t nd) {
        Slices s;
        s.src = take(n * 6 * sizeof(float)), s.dst = take(nd * 6 * sizeof(float));
        s.srct = take(n * 6 * sizeof(float)), s.moved = take(n * 3 * sizeof(float));
        s.nn = take(n * sizeof(int)), s.nnp = take(n * sizeof(int)), s.d2 = take(n * sizeof(float));
        s.win = take(nd * sizeof(unsigned long long));
        s.cs = take((ICP_CELLS_MAX + 1) * sizeof(uint32_t)), s.cf = take(ICP_CELLS_MAX * sizeof(uint32_t));
        s.items = take(nd * sizeof(float4));
        return s;
    };
    std::vector<Slices> sl(P);
    for (size_t j = 0, slot = 0; j < n_jobs; ++j) {
        job_first[j] = slot;
        for (size_t k = 0; k < jobs[j].n_poses; ++k, ++slot) sl[slot] = slices(jobs[j].model->n, jobs[j].scene->n);
    }
    StreamBuf<unsigned char> slab(ctx);
    PPF_CUDA(ctx, slab.alloc(off));
    std::vector<IcpPose> desc;  // launch order
    std::vector<double> poses(P * 16), residuals(P);
    desc.reserve(P);
    for (const auto &o : order) {
        const b200ppf_icp_job &jb = jobs[o.second];
        for (size_t k = 0; k < jb.n_poses; ++k) {
            const size_t slot = job_first[o.second] + k;
            const Slices &s = sl[slot];
            IcpPose d;
            d.mpos = jb.model->pos, d.mnrm = jb.model->nrm;
            d.spos = jb.scene->pos, d.snrm = jb.scene->nrm;
            d.n_model = (uint32_t)jb.model->n, d.n_scene = (uint32_t)jb.scene->n;
            d.slot = (uint32_t)slot;
            d.src_norm = reinterpret_cast<float *>(slab + s.src), d.dst_norm = reinterpret_cast<float *>(slab + s.dst);
            d.src_t = reinterpret_cast<float *>(slab + s.srct), d.moved = reinterpret_cast<float *>(slab + s.moved);
            d.nn = reinterpret_cast<int *>(slab + s.nn), d.nn_prev = reinterpret_cast<int *>(slab + s.nnp);
            d.d2 = reinterpret_cast<float *>(slab + s.d2);
            d.winner = reinterpret_cast<unsigned long long *>(slab + s.win);
            d.cell_start = reinterpret_cast<uint32_t *>(slab + s.cs), d.cell_fill = reinterpret_cast<uint32_t *>(slab + s.cf);
            d.items = reinterpret_cast<float4 *>(slab + s.items);
            desc.push_back(d);
        }
    }
    for (size_t j = 0; j < n_jobs; ++j)
        if (jobs[j].n_poses) memcpy(poses.data() + 16 * job_first[j], jobs[j].poses16, jobs[j].n_poses * 16 * sizeof(double));
    IcpArgs a;
    a.max_iterations = max_iterations;
    a.num_levels = num_levels;
    a.tolerance = tolerance;
    a.rejection_scale = rejection_scale;
    a.poses = reinterpret_cast<double *>(slab + o_poses);
    a.residuals = reinterpret_cast<double *>(slab + o_res);
    a.iterations = reinterpret_cast<unsigned long long *>(slab + o_it);
    IcpPose *d_desc = reinterpret_cast<IcpPose *>(slab + o_desc);
    PPF_CUDA(ctx, cudaMemcpyAsync(a.poses, poses.data(), P * 16 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_desc, desc.data(), P * sizeof(IcpPose), cudaMemcpyHostToDevice, ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(a.iterations, 0, sizeof(unsigned long long), ctx->stream));
    cudaEventRecord(ctx->ev[0], ctx->stream);
    for (size_t g = 0, e = 0, first = 0; g < order.size(); g = e) {
        // one cluster per pose: grid (csize, poses of this size), cluster dimension (csize, 1, 1)
        const int csize = order[g].first;
        size_t count = 0;
        for (e = g; e < order.size() && order[e].first == csize; ++e) count += jobs[order[e].second].n_poses;
        a.pose = d_desc + first;
        first += count;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)csize, (unsigned)count, 1);
        cfg.blockDim = dim3(ICP_THREADS, 1, 1);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = ctx->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)csize;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        PPF_CUDA(ctx, cudaLaunchKernelEx(&cfg, icp_refine_kernel, a));
        ctx->launches++;
    }
    cudaEventRecord(ctx->ev[1], ctx->stream);
    PPF_CUDA(ctx, cudaMemcpyAsync(poses.data(), a.poses, P * 16 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(residuals.data(), a.residuals, P * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long it = 0;
    PPF_CUDA(ctx, cudaMemcpyAsync(&it, a.iterations, sizeof(it), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->timings.icp_ms, ctx->ev[0], ctx->ev[1]);
    for (size_t j = 0; j < n_jobs; ++j) {
        if (!jobs[j].n_poses) continue;
        memcpy(jobs[j].poses16, poses.data() + 16 * job_first[j], jobs[j].n_poses * 16 * sizeof(double));
        if (jobs[j].residuals) memcpy(jobs[j].residuals, residuals.data() + job_first[j], jobs[j].n_poses * sizeof(double));
    }
    if (iterations_host) *iterations_host = it;
    return B200PPF_OK;
}

int k6_icp_refine(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_cloud *scene, int max_iterations,
                  float tolerance, float rejection_scale, int num_levels, double *poses16_host, size_t n_poses,
                  double *residuals_host, uint64_t *iterations_host) {
    const b200ppf_icp_job job = {model, scene, poses16_host, n_poses, residuals_host};
    return k6_icp_refine_batch(ctx, &job, 1, max_iterations, tolerance, rejection_scale, num_levels, iterations_host);
}

}  // namespace b200ppf
