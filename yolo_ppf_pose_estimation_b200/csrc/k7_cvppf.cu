// k7_cvppf.cu — the engine the reference actually calls: cv::ppf_match_3d::PPF3DDetector on the device.
//
// Replaces opencv_contrib modules/surface_matching/src/ppf_match_3d.cpp (trainModel, match, clusterPoses),
// ppf_helpers.cpp (samplePCByQuantization, computeBboxStd), c_utils.hpp (computeTransformRT, aaToR, TAngle3Normalized),
// hash_murmur86.hpp and t_hash_int.cpp as the reference drives them: include/CloudProcessing.h:205-236 (constructor,
// trainModel), :442 (match), :495 (match_S2B, fork-only: inferred, see b200ppf.h).  SURVEY.md Appendix B.
//
// It is a second engine, not a front-end of the PCL one: double-precision features (atan2 of cross / dot), keys hashed
// with MurmurHash3_x86_32 into a power-of-two table whose buckets mix colliding keys, no radius cut (every sampled scene
// point is paired with every reference point), alpha binned over 4*pi, clustering on the scalar rotation angles.
//   sample   cell index per point (float arithmetic as upstream writes it) -> stable radix sort -> one thread per
//            occupied cell averages its points in input order in double, normal renormalised;
//   train    one thread per ordered model pair: features, hash, alpha_m -> radix sort by bucket -> CSR over the
//            2^k buckets (the chained hash table: same bucket contents, collisions included);
//   match    one CTA per reference point (persistent over the references): lanes compute pair features, the warp walks
//            each lane's bucket together, votes are L2 reductions into the CTA's own M x numAngles accumulator, the peak is
//            the first maximum in (model point, alpha index) order, the pose Tsg^-1 Rx(alpha) Tmg is assembled in double;
//   cluster  one CTA: the per-reference poses (a few hundred to a few thousand: the engine subsamples the scene) are ranked
//            by votes, assigned greedily — each pose against all cluster leaders at once — and averaged (cv_cluster_kernel).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "ppf_common.cuh"

struct b200cv_detector {
    b200ppf_ctx *ctx = nullptr;
    double sampling_step_relative = 0.05, distance_step_relative = 0.05, num_angles_arg = 30;
    double angle_step = 0, distance_step = 0;
    double position_threshold = 0, rotation_threshold = 0;
    size_t m = 0;                 // sampled model points
    size_t table_size = 0;        // power of two >= 16
    size_t n_nodes = 0;           // m * (m - 1)
    float *d_model = nullptr;     // m x 6
    float *d_alpha = nullptr;     // m * m, index i * m + j (upstream's ppf matrix, fifth column)
    uint32_t *d_offsets = nullptr;  // table_size + 1
    uint32_t *d_nodes = nullptr;    // ppfInd = i * m + j, grouped by bucket, ascending inside a bucket
    std::vector<float> h_model;
    // last match
    std::vector<b200cv_pose> raw;   // per reference point, before clustering
    std::vector<float> h_scene;     // sampled scene of the last match (m x 6)
    float *d_scene = nullptr, *d_second = nullptr;
    size_t n_scene = 0, n_second = 0;
    bool second_is_scene = true;
};

namespace b200ppf {

namespace {

constexpr double CV_EPS = 1.192092896e-07;  // EPS of c_utils.hpp
constexpr double PI_D = 3.14159265358979323846;

struct D3 {
    double x, y, z;
};
__host__ __device__ __forceinline__ D3 d3(double x, double y, double z) { return D3{x, y, z}; }
__host__ __device__ __forceinline__ D3 ld6(const float *p) { return D3{(double)p[0], (double)p[1], (double)p[2]}; }
__host__ __device__ __forceinline__ double ddot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__host__ __device__ __forceinline__ D3 dcross(D3 a, D3 b) { return D3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
__host__ __device__ __forceinline__ double dnorm(D3 a) { return sqrt(ddot(a, a)); }

struct M33 {
    double m[9];
};
__host__ __device__ __forceinline__ D3 mmul(const M33 &R, D3 v) {
    return D3{R.m[0] * v.x + R.m[1] * v.y + R.m[2] * v.z, R.m[3] * v.x + R.m[4] * v.y + R.m[5] * v.z,
              R.m[6] * v.x + R.m[7] * v.y + R.m[8] * v.z};
}

// c_utils.hpp aaToR
__host__ __device__ __forceinline__ void aa_to_r(D3 axis, double angle, M33 &R) {
    const double sinA = sin(angle), cosA = cos(angle), cos1A = 1.0 - cosA;
    const double a[3] = {axis.x, axis.y, axis.z};
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            double v = (i == j) ? cosA : 0.0;
            if (i != j) v += (((i + 1) % 3 == j) ? -1.0 : 1.0) * sinA * a[3 - i - j];
            v += cos1A * a[i] * a[j];
            R.m[3 * i + j] = v;
        }
}

// c_utils.hpp computeTransformRT
__host__ __device__ __forceinline__ void transform_rt(D3 p1, D3 n1, M33 &R, D3 &t) {
    const double angle = acos(n1.x);
    D3 axis = d3(0.0, n1.z, -n1.y);
    if (n1.y == 0 && n1.z == 0) {
        axis.y = 1;
        axis.z = 0;
    } else {
        const double nn = dnorm(axis);
        if (nn > CV_EPS) axis = d3(axis.x / nn, axis.y / nn, axis.z / nn);
    }
    aa_to_r(axis, angle, R);
    const D3 rp = mmul(R, p1);
    t = d3(-rp.x, -rp.y, -rp.z);
}

__host__ __device__ __forceinline__ double angle3(D3 a, D3 b) { return atan2(dnorm(dcross(a, b)), ddot(a, b)); }

// PPF3DDetector::computePPFFeatures
__host__ __device__ __forceinline__ void cv_features(D3 p1, D3 n1, D3 p2, D3 n2, double *f) {
    f[0] = f[1] = f[2] = f[3] = 0.0;
    D3 d = d3(p2.x - p1.x, p2.y - p1.y, p2.z - p1.z);
    f[3] = dnorm(d);
    if (f[3] <= CV_EPS) return;
    const double inv = 1.0 / f[3];
    d = d3(d.x * inv, d.y * inv, d.z * inv);
    f[0] = angle3(n1, d);
    f[1] = angle3(n2, d);
    f[2] = angle3(n1, n2);
}

__host__ __device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
// MurmurHash3_x86_32 of four 32-bit words, seed 42 (hashPPF)
__host__ __device__ __forceinline__ uint32_t hash_ppf(const double *f, double angle_step, double distance_step) {
    const int32_t key[4] = {(int32_t)(f[0] / angle_step), (int32_t)(f[1] / angle_step), (int32_t)(f[2] / angle_step),
                            (int32_t)(f[3] / distance_step)};
    uint32_t h1 = 42u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t k1 = (uint32_t)key[i];
        k1 *= 0xcc9e2d51u;
        k1 = rotl32(k1, 15);
        k1 *= 0x1b873593u;
        h1 ^= k1;
        h1 = rotl32(h1, 13);
        h1 = h1 * 5 + 0xe6546b64u;
    }
    h1 ^= 16u;
    h1 ^= h1 >> 16;
    h1 *= 0x85ebca6bu;
    h1 ^= h1 >> 13;
    h1 *= 0xc2b2ae35u;
    h1 ^= h1 >> 16;
    return h1;
}

// PPF3DDetector::computeAlpha
__host__ __device__ __forceinline__ double cv_alpha(const M33 &R, D3 t, D3 p2, bool *is_nan) {
    const D3 rp = mmul(R, p2);
    const D3 mpt = d3(t.x + rp.x, t.y + rp.y, t.z + rp.z);
    double alpha = atan2(-mpt.z, mpt.y);
    *is_nan = alpha != alpha;
    if (*is_nan) return 0.0;
    if (sin(alpha) * mpt.z < 0.0) alpha = -alpha;
    return -alpha;
}

// ---- samplePCByQuantization ------------------------------------------------------------------------------------
struct SampleRange {
    float lo[3], ext[3];
    int ns;
};

// where samplePCByQuantization reads its points from: the same kernels serve both, so a device cloud and its downloaded
// rows go through identical arithmetic
struct RowPoints {  // host input uploaded as is: rows of `stride` floats [x y z nx ny nz ...]
    const float *pc;
    uint32_t stride;
    __device__ __forceinline__ void xyz(uint32_t i, float p[3]) const {
        const float *r = pc + (size_t)i * stride;
        p[0] = r[0], p[1] = r[1], p[2] = r[2];
    }
    __device__ __forceinline__ void row(uint32_t i, float p[6]) const {
        const float *r = pc + (size_t)i * stride;
#pragma unroll
        for (int k = 0; k < 6; ++k) p[k] = r[k];
    }
};
struct CloudPoints {  // b200ppf_cloud: x y z in pos, the normal in nrm.xyz; nrm.w holds the curvature and is never read
    const float4 *pos, *nrm;
    __device__ __forceinline__ void xyz(uint32_t i, float p[3]) const {
        const float4 v = pos[i];
        p[0] = v.x, p[1] = v.y, p[2] = v.z;
    }
    __device__ __forceinline__ void row(uint32_t i, float p[6]) const {
        xyz(i, p);
        const float4 q = nrm[i];
        p[3] = q.x, p[4] = q.y, p[5] = q.z;
    }
};

template <class Points>
__global__ void cv_cell_index_kernel(const Points pts, uint32_t n, SampleRange r, uint32_t *__restrict__ cell) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float p[3];
    pts.xyz(i, p);
    // (int)((float)numSamplesDim * (x - xrange[0]) / xr), index = xc * ns * ns + yc * ns + zc — upstream's stride, under which a
    // coordinate on the upper bound (cell ns) lands in a neighbouring cell's list
    const int xc = (int)((float)r.ns * (p[0] - r.lo[0]) / r.ext[0]);
    const int yc = (int)((float)r.ns * (p[1] - r.lo[1]) / r.ext[1]);
    const int zc = (int)((float)r.ns * (p[2] - r.lo[2]) / r.ext[2]);
    cell[i] = (uint32_t)(xc * r.ns * r.ns + yc * r.ns + zc);
}

// one thread per occupied cell: the cell's points averaged in input order, in double
template <class Points>
__global__ void cv_cell_average_kernel(const Points pts, const uint32_t *__restrict__ order, const uint32_t *__restrict__ head,
                                       const uint32_t *__restrict__ rank, uint32_t n, float *__restrict__ out6) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !head[i]) return;
    double a[6] = {0, 0, 0, 0, 0, 0};
    uint32_t q = i, cnt = 0;
    do {
        float p[6];
        pts.row(order[q], p);
#pragma unroll
        for (int k = 0; k < 6; ++k) a[k] += (double)p[k];
        ++cnt;
        ++q;
    } while (q < n && !head[q]);
#pragma unroll
    for (int k = 0; k < 6; ++k) a[k] /= (double)cnt;
    const double nn = sqrt(a[3] * a[3] + a[4] * a[4] + a[5] * a[5]);
    float *o = out6 + (size_t)rank[i] * 6;
    o[0] = (float)a[0];
    o[1] = (float)a[1];
    o[2] = (float)a[2];
    o[3] = o[4] = o[5] = 0.0f;
    if (nn > CV_EPS) {
        o[3] = (float)(a[3] / nn);
        o[4] = (float)(a[4] / nn);
        o[5] = (float)(a[5] / nn);
    }
}

// ---- trainModel ------------------------------------------------------------------------------------------------
constexpr uint32_t CV_INVALID = 0xFFFFFFFFu;

__global__ void __launch_bounds__(256)
cv_train_pairs_kernel(const float *__restrict__ model, uint32_t m, double angle_step, double distance_step, uint32_t mask,
                      uint32_t *__restrict__ keys, float *__restrict__ alpha_m) {
    __shared__ M33 sR;
    __shared__ D3 st, sp, sn;
    const uint32_t i = blockIdx.y;
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (threadIdx.x == 0) {
        sp = ld6(model + 6 * (size_t)i);
        sn = ld6(model + 6 * (size_t)i + 3);
        transform_rt(sp, sn, sR, st);
    }
    __syncthreads();
    if (j >= m) return;
    const size_t idx = (size_t)i * m + j;
    if (i == j) {
        keys[idx] = CV_INVALID;
        alpha_m[idx] = 0.0f;
        return;
    }
    const D3 p2 = ld6(model + 6 * (size_t)j), n2 = ld6(model + 6 * (size_t)j + 3);
    double f[4];
    cv_features(sp, sn, p2, n2, f);
    const uint32_t h = hash_ppf(f, angle_step, distance_step);
    bool is_nan;
    const double alpha = cv_alpha(sR, st, p2, &is_nan);
    alpha_m[idx] = (float)alpha;
    keys[idx] = h & mask;  // hash % table size (a power of two)
}

// ---- match -----------------------------------------------------------------------------------------------------
struct CvVoteArgs {
    const float *scene;    // sampled scene, ns x 6: the reference points
    const float *second;   // the points a reference point is paired with (the scene itself, or the sampled edge cloud)
    uint32_t ns, n2, step, refs;
    int skip_same_index;   // match(): i == j is skipped
    const float *model;
    uint32_t m;
    const float *alpha_m;
    const uint32_t *offsets, *nodes;
    uint32_t mask;
    double angle_step, distance_step;
    int num_angles;
    uint32_t *acc;         // gridDim.x accumulators of m * num_angles words, zero on entry and on exit
    b200cv_pose *poses;    // refs records
    uint32_t *acc_dump;    // debug: accumulator of reference `dump_ref`
    uint32_t dump_ref;
};

constexpr int CV_VOTE_THREADS = 256;

__global__ void __launch_bounds__(CV_VOTE_THREADS)
cv_vote_kernel(const CvVoteArgs a) {
    __shared__ M33 sR;
    __shared__ D3 st, sp, sn;
    __shared__ unsigned long long s_best[CV_VOTE_THREADS / 32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t acc_len = (size_t)a.m * a.num_angles;
    uint32_t *acc = a.acc + (size_t)blockIdx.x * acc_len;
    for (uint32_t r = blockIdx.x; r < a.refs; r += gridDim.x) {
        const uint32_t i = r * a.step;
        __syncthreads();
        if (threadIdx.x == 0) {
            sp = ld6(a.scene + 6 * (size_t)i);
            sn = ld6(a.scene + 6 * (size_t)i + 3);
            transform_rt(sp, sn, sR, st);
        }
        __syncthreads();
        // lanes compute pair features; the warp then walks each lane's bucket together
        for (uint32_t j0 = warp * 32; j0 < a.n2; j0 += CV_VOTE_THREADS) {
            const uint32_t j = j0 + lane;
            uint32_t b = 0, e = 0;
            double alpha_scene = 0.0;
            if (j < a.n2 && !(a.skip_same_index && j == i)) {
                const D3 p2 = ld6(a.second + 6 * (size_t)j), n2 = ld6(a.second + 6 * (size_t)j + 3);
                double f[4];
                cv_features(sp, sn, p2, n2, f);
                const uint32_t h = hash_ppf(f, a.angle_step, a.distance_step) & a.mask;
                bool is_nan;
                alpha_scene = cv_alpha(sR, st, p2, &is_nan);
                if (!is_nan) {
                    b = a.offsets[h];
                    e = a.offsets[h + 1];
                }
            }
            uint32_t pending = __ballot_sync(0xFFFFFFFFu, e > b);
            while (pending) {
                const int src = __ffs(pending) - 1;
                pending &= pending - 1;
                const uint32_t sb = __shfl_sync(0xFFFFFFFFu, b, src), se = __shfl_sync(0xFFFFFFFFu, e, src);
                const double as = __shfl_sync(0xFFFFFFFFu, alpha_scene, src);
                for (uint32_t p = sb + lane; p < se; p += 32) {
                    const uint32_t node = a.nodes[p];
                    const double alpha = (double)a.alpha_m[node] - as;
                    const int alpha_index = (int)((double)a.num_angles * (alpha + 2 * PI_D) / (4 * PI_D));
                    const size_t cell = (size_t)(node / a.m) * a.num_angles + (size_t)alpha_index;
                    if (cell < acc_len) atomicAdd(acc + cell, 1u);  // alpha == +2*pi exactly would index one past the row
                }
            }
        }
        __threadfence_block();
        __syncthreads();
        // first maximum in (model point, alpha index) order == max of (votes, ~flat); the accumulator is cleared on the way
        unsigned long long best = 0;
        for (size_t c = threadIdx.x; c < acc_len; c += CV_VOTE_THREADS) {
            const uint32_t v = __ldcg(acc + c);
            if (a.acc_dump && r == a.dump_ref) a.acc_dump[c] = v;
            if (v) {
                best = max(best, ((unsigned long long)v << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)c));
                acc[c] = 0;
            }
        }
        for (int o = 16; o > 0; o >>= 1) best = max(best, (unsigned long long)__shfl_xor_sync(0xFFFFFFFFu, best, o));
        if (lane == 0) s_best[warp] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < CV_VOTE_THREADS / 32; ++w) best = max(best, s_best[w]);
            const uint32_t max_votes = (uint32_t)(best >> 32);
            const uint32_t flat = max_votes ? 0xFFFFFFFFu - (uint32_t)(best & 0xFFFFFFFFu) : 0u;
            const uint32_t ref_max = flat / (uint32_t)a.num_angles, alpha_max = flat % (uint32_t)a.num_angles;
            // pose = TsgInv * Rx(alpha) * Tmg, 4x4 row-major products as upstream multiplies them
            M33 RInv;
#pragma unroll
            for (int x = 0; x < 3; ++x)
#pragma unroll
                for (int y = 0; y < 3; ++y) RInv.m[3 * x + y] = sR.m[3 * y + x];
            const D3 rt = mmul(RInv, st);
            double TsgInv[16], Tmg[16], Talpha[16], tmp[16];
            auto rt_to_pose = [](const M33 &R, D3 t, double *mm) {
                for (int x = 0; x < 3; ++x)
                    for (int y = 0; y < 3; ++y) mm[4 * x + y] = R.m[3 * x + y];
                mm[3] = t.x, mm[7] = t.y, mm[11] = t.z;
                mm[12] = mm[13] = mm[14] = 0.0;
                mm[15] = 1.0;
            };
            auto mul44 = [](const double *x, const double *y, double *o) {
                for (int rr = 0; rr < 4; ++rr)
                    for (int cc = 0; cc < 4; ++cc) {
                        double s = 0;
                        for (int k = 0; k < 4; ++k) s += x[4 * rr + k] * y[4 * k + cc];
                        o[4 * rr + cc] = s;
                    }
            };
            rt_to_pose(RInv, d3(-rt.x, -rt.y, -rt.z), TsgInv);
            M33 Rmg;
            D3 tmg;
            transform_rt(ld6(a.model + 6 * (size_t)ref_max), ld6(a.model + 6 * (size_t)ref_max + 3), Rmg, tmg);
            rt_to_pose(Rmg, tmg, Tmg);
            const double alpha = ((double)alpha_max * (4 * PI_D)) / a.num_angles - 2 * PI_D;
            M33 Rx;
            Rx.m[0] = 1, Rx.m[1] = 0, Rx.m[2] = 0, Rx.m[3] = 0, Rx.m[4] = cos(alpha), Rx.m[5] = -sin(alpha), Rx.m[6] = 0,
            Rx.m[7] = sin(alpha), Rx.m[8] = cos(alpha);  // getUnitXRotation
            rt_to_pose(Rx, d3(0, 0, 0), Talpha);
            b200cv_pose P;
            mul44(Talpha, Tmg, tmp);
            mul44(TsgInv, tmp, P.pose);
            P.alpha = alpha;
            P.residual = 0.0;
            P.model_index = ref_max;
            P.num_votes = max_votes;
            // Pose3D::updatePose: angle from the trace, translation, quaternion (w x y z)
            const double trace = P.pose[0] + P.pose[5] + P.pose[10];
            if (fabs(trace - 3) <= CV_EPS) P.angle = 0;
            else if (fabs(trace + 1) <= CV_EPS) P.angle = PI_D;
            else P.angle = acos((trace - 1) / 2);
            P.t[0] = P.pose[3], P.t[1] = P.pose[7], P.t[2] = P.pose[11];
            {
                const double *R = P.pose;
                const double r00 = R[0], r01 = R[1], r02 = R[2], r10 = R[4], r11 = R[5], r12 = R[6], r20 = R[8], r21 = R[9], r22 = R[10];
                const double tr = r00 + r11 + r22;
                double *q = P.q;
                if (tr > 0.0) {
                    const double s = sqrt(tr + 1.0) * 2.0;
                    q[0] = 0.25 * s, q[1] = (r21 - r12) / s, q[2] = (r02 - r20) / s, q[3] = (r10 - r01) / s;
                } else if (r00 > r11 && r00 > r22) {
                    const double s = sqrt(1.0 + r00 - r11 - r22) * 2.0;
                    q[0] = (r21 - r12) / s, q[1] = 0.25 * s, q[2] = (r01 + r10) / s, q[3] = (r02 + r20) / s;
                } else if (r11 > r22) {
                    const double s = sqrt(1.0 + r11 - r00 - r22) * 2.0;
                    q[0] = (r02 - r20) / s, q[1] = (r01 + r10) / s, q[2] = 0.25 * s, q[3] = (r12 + r21) / s;
                } else {
                    const double s = sqrt(1.0 + r22 - r00 - r11) * 2.0;
                    q[0] = (r10 - r01) / s, q[1] = (r02 + r20) / s, q[2] = (r12 + r21) / s, q[3] = 0.25 * s;
                }
            }
            P.alpha_index = alpha_max;
            P.reference_index = r;
            a.poses[r] = P;
        }
    }
}

// computeBboxStd over rows of `stride` floats
void bbox6(const float *pc, size_t n, size_t stride, float r[6]) {
    for (int k = 0; k < 3; ++k) r[2 * k] = r[2 * k + 1] = n ? pc[k] : 0.f;
    for (size_t i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) {
            r[2 * k] = std::min(r[2 * k], pc[stride * i + k]);
            r[2 * k + 1] = std::max(r[2 * k + 1], pc[stride * i + k]);
        }
}

// samplePCByQuantization over the box `range` -> device rows of 6 floats (cudaMalloc: the caller frees them) and their count
template <class Points>
int cv_sample_points(b200ppf_ctx *ctx, const Points &pts, size_t n, const float range[6], float sample_step, float **d_out,
                     size_t *n_out) {
    *d_out = nullptr;
    *n_out = 0;
    if (n == 0) return B200PPF_OK;
    if (n >= 0x7FFFFFFFull) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "cv sample: too many points");
    SampleRange r;
    r.ns = (int)(1.0 / sample_step);
    if (r.ns < 1 || r.ns > 1000) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv sample: the relative step must lie in [0.001, 1]");
    for (int k = 0; k < 3; ++k) {
        r.lo[k] = range[2 * k];
        r.ext[k] = range[2 * k + 1] - range[2 * k];
        if (!(r.ext[k] > 0.0f) || !std::isfinite(r.ext[k]))
            return fail_msg(ctx, B200PPF_ERR_INVALID, "cv sample: the cloud's bounding box is flat or not finite (upstream divides by its extent)");
    }
    const uint32_t nn = (uint32_t)n;
    StreamBuf<uint32_t> cell0(ctx), cell1(ctx), ord0(ctx), ord1(ctx), head(ctx), rank(ctx);
    PPF_CUDA(ctx, cell0.alloc(n));
    PPF_CUDA(ctx, cell1.alloc(n));
    PPF_CUDA(ctx, ord0.alloc(n));
    PPF_CUDA(ctx, ord1.alloc(n));
    PPF_CUDA(ctx, head.alloc(n));
    PPF_CUDA(ctx, rank.alloc(n));
    const unsigned g = (nn + 255) / 256;
    PPF_LAUNCH(ctx, cv_cell_index_kernel<Points>, g, 256, 0, pts, nn, r, cell0.p);
    const uint64_t n_cells = (uint64_t)(r.ns + 1) * (r.ns + 1) * (r.ns + 1);
    bool in_alt = false;
    int rc = radix_sort_u32(ctx, cell0, cell1, ord0, ord1, nullptr, nullptr, n, n_cells - 1, /*v0_iota=*/true, &in_alt);
    if (rc) return rc;
    const uint32_t *cs = in_alt ? cell1.p : cell0.p, *os = in_alt ? ord1.p : ord0.p;
    if ((rc = run_heads(ctx, cs, nn, head))) return rc;
    uint32_t cells = 0;
    if ((rc = flag_scan_host(ctx, head, nn, rank, &cells))) return rc;
    float *out = nullptr;
    PPF_CUDA(ctx, cudaMalloc(&out, std::max<size_t>(1, cells) * 6 * sizeof(float)));
    std::unique_ptr<float, cudaError_t (*)(void *)> owner(out, cudaFree);
    cv_cell_average_kernel<Points><<<g, 256, 0, ctx->stream>>>(pts, os, head.p, rank.p, nn, out);
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess)
        return fail_msg(ctx, B200PPF_ERR_CUDA, "cv sample: kernel failed");
    *d_out = owner.release();
    *n_out = cells;
    return B200PPF_OK;
}

// samplePCByQuantization of a host cloud: its rows uploaded as they are
int cv_sample(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride, const float range[6], float sample_step, float **d_out,
              size_t *n_out) {
    *d_out = nullptr;
    *n_out = 0;
    if (n == 0) return B200PPF_OK;
    StreamBuf<float> d_pc(ctx);
    PPF_CUDA(ctx, d_pc.alloc(n * stride));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_pc, host, n * stride * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    return cv_sample_points(ctx, RowPoints{d_pc.p, (uint32_t)stride}, n, range, sample_step, d_out, n_out);
}

// samplePCByQuantization of a device cloud over its own bounding box: bbox_min / bbox_max are the exact, order-free
// min / max of pos that every producer of a cloud sets (the host upload, cloud_bbox_from_device after the device
// stages), so the result equals that of the cloud's downloaded rows bit for bit
int cv_sample_cloud(b200ppf_ctx *ctx, const b200ppf_cloud *c, float sample_step, float **d_out, size_t *n_out) {
    const float range[6] = {c->bbox_min[0], c->bbox_max[0], c->bbox_min[1], c->bbox_max[1], c->bbox_min[2], c->bbox_max[2]};
    return cv_sample_points(ctx, CloudPoints{c->pos, c->nrm}, c->n, range, sample_step, d_out, n_out);
}

void cv_free_match(b200cv_detector *d) {
    if (d->d_scene) cudaFree(d->d_scene);
    if (d->d_second && !d->second_is_scene) cudaFree(d->d_second);
    d->d_scene = d->d_second = nullptr;
    d->n_scene = d->n_second = 0;
    d->second_is_scene = true;
}

void cv_free_model(b200cv_detector *d) {
    if (d->d_model) cudaFree(d->d_model);
    if (d->d_alpha) cudaFree(d->d_alpha);
    if (d->d_offsets) cudaFree(d->d_offsets);
    if (d->d_nodes) cudaFree(d->d_nodes);
    d->d_model = d->d_alpha = nullptr;
    d->d_offsets = d->d_nodes = nullptr;
    d->m = d->table_size = d->n_nodes = 0;
}

// the voting launch of match / match_S2B over the detector's sampled clouds
int cv_vote(b200cv_detector *d, uint32_t step, uint32_t refs, uint32_t *acc_dump_host, uint32_t dump_ref, StreamBuf<b200cv_pose> &poses) {
    b200ppf_ctx *ctx = d->ctx;
    const int num_angles = (int)std::floor(2 * PI_D / d->angle_step);
    const size_t acc_len = d->m * (size_t)num_angles;
    const unsigned grid = (unsigned)std::min<size_t>(refs, (size_t)ctx->sm_count * 2);
    StreamBuf<uint32_t> acc(ctx), dump(ctx);
    PPF_CUDA(ctx, acc.alloc(acc_len * grid));
    PPF_CUDA(ctx, cudaMemsetAsync(acc, 0, acc_len * grid * sizeof(uint32_t), ctx->stream));
    PPF_CUDA(ctx, poses.alloc(refs));
    if (acc_dump_host) {
        PPF_CUDA(ctx, dump.alloc(acc_len));
        PPF_CUDA(ctx, cudaMemsetAsync(dump, 0, acc_len * sizeof(uint32_t), ctx->stream));
    }
    CvVoteArgs a;
    a.scene = d->d_scene;
    a.second = d->d_second;
    a.ns = (uint32_t)d->n_scene;
    a.n2 = (uint32_t)d->n_second;
    a.step = step;
    a.refs = refs;
    a.skip_same_index = d->second_is_scene ? 1 : 0;
    a.model = d->d_model;
    a.m = (uint32_t)d->m;
    a.alpha_m = d->d_alpha;
    a.offsets = d->d_offsets;
    a.nodes = d->d_nodes;
    a.mask = (uint32_t)(d->table_size - 1);
    a.angle_step = d->angle_step;
    a.distance_step = d->distance_step;
    a.num_angles = num_angles;
    a.acc = acc;
    a.poses = poses;
    a.acc_dump = acc_dump_host ? dump.p : nullptr;
    a.dump_ref = dump_ref;
    cudaEventRecord(ctx->ev[0], ctx->stream);
    PPF_LAUNCH(ctx, cv_vote_kernel, grid, CV_VOTE_THREADS, 0, a);
    cudaEventRecord(ctx->ev[1], ctx->stream);
    d->raw.resize(refs);
    PPF_CUDA(ctx, cudaMemcpyAsync(d->raw.data(), poses, refs * sizeof(b200cv_pose), cudaMemcpyDeviceToHost, ctx->stream));
    if (acc_dump_host)
        PPF_CUDA(ctx, cudaMemcpyAsync(acc_dump_host, dump, acc_len * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->timings.vote_ms, ctx->ev[0], ctx->ev[1]);
    return B200PPF_OK;
}

// PPF3DDetector::clusterPoses on the per-reference poses: sorted by votes (ties: reference order), each pose joins the
// first cluster whose FIRST pose matches (|angle difference| < rotation threshold and |t difference| < position
// threshold), clusters sorted by their vote sums, plain average of quaternions and translations.
// One CTA: the engine produces a few hundred to a few thousand poses per match, and upstream's greedy loop is sequential
// in the poses — each step tests the pose against all cluster leaders in parallel and takes the lowest matching cluster.
// Both sorts are rank counts (stable: ties keep reference / creation order); the sums of a cluster run over its members
// in the order they joined, as upstream's loop adds them.
constexpr int CV_CLUSTER_THREADS = 1024;
struct CvClusterArgs {
    const b200cv_pose *poses;  // per reference point
    uint32_t n;
    double position_threshold, rotation_threshold;
    uint32_t *order;           // [n] sorted position -> pose
    uint32_t *member_of;       // [n] sorted position -> cluster (creation index)
    double4 *lead;             // [n] cluster -> (t, angle) of its first pose
    uint32_t *lead_pose;       // [n] cluster -> its first pose
    uint32_t *size;            // [n] members per cluster
    unsigned long long *votes; // [n] vote sum per cluster
    uint32_t *corder;          // [n] output position -> cluster
    b200cv_pose *out;          // [n] clusters, best first
    uint32_t *n_clusters;
};

__global__ void __launch_bounds__(CV_CLUSTER_THREADS) cv_cluster_kernel(const CvClusterArgs a) {
    __shared__ uint32_t s_first, s_ncl;
    const uint32_t tid = threadIdx.x, n = a.n;
    // poses by votes, descending; ties in reference order
    for (uint32_t i = tid; i < n; i += CV_CLUSTER_THREADS) {
        const uint32_t v = a.poses[i].num_votes;
        uint32_t rank = 0;
        for (uint32_t j = 0; j < n; ++j) {
            const uint32_t w = a.poses[j].num_votes;
            rank += (w > v || (w == v && j < i)) ? 1u : 0u;
        }
        a.order[rank] = i;
    }
    if (tid == 0) {
        s_first = 0xFFFFFFFFu;
        s_ncl = 0;
    }
    __syncthreads();
    // the greedy assignment
    for (uint32_t k = 0; k < n; ++k) {
        const uint32_t pi = a.order[k];
        const b200cv_pose &p = a.poses[pi];
        const double px = p.t[0], py = p.t[1], pz = p.t[2], pa = p.angle;
        const uint32_t ncl = s_ncl;
        for (uint32_t c = tid; c < ncl; c += CV_CLUSTER_THREADS) {
            const double4 l = a.lead[c];
            const double dx = l.x - px, dy = l.y - py, dz = l.z - pz;
            const double dn = sqrt(dx * dx + dy * dy + dz * dz);
            const double phi = fabs(pa - l.w);
            if (phi < a.rotation_threshold && dn < a.position_threshold) atomicMin(&s_first, c);
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t c = s_first;
            if (c == 0xFFFFFFFFu) {
                c = ncl;
                a.lead[c] = make_double4(px, py, pz, pa);
                a.lead_pose[c] = pi;
                a.size[c] = 0;
                a.votes[c] = 0;
                s_ncl = ncl + 1;
            }
            a.member_of[k] = c;
            a.size[c] += 1;
            a.votes[c] += p.num_votes;
            s_first = 0xFFFFFFFFu;
        }
        __syncthreads();
    }
    const uint32_t ncl = s_ncl;
    if (tid == 0) *a.n_clusters = ncl;
    // clusters by vote sum, descending; ties in creation order
    for (uint32_t c = tid; c < ncl; c += CV_CLUSTER_THREADS) {
        const unsigned long long v = a.votes[c];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < ncl; ++j) {
            const unsigned long long w = a.votes[j];
            rank += (w > v || (w == v && j < c)) ? 1u : 0u;
        }
        a.corder[rank] = c;
    }
    __syncthreads();
    // averages (updatePoseQuat: the averaged quaternion normalised, then the rotation matrix)
    for (uint32_t o = tid; o < ncl; o += CV_CLUSTER_THREADS) {
        const uint32_t c = a.corder[o];
        double q[4] = {0, 0, 0, 0}, t[3] = {0, 0, 0};
        for (uint32_t k = 0; k < n; ++k) {
            if (a.member_of[k] != c) continue;
            const b200cv_pose &m = a.poses[a.order[k]];
            for (int e = 0; e < 4; ++e) q[e] += m.q[e];
            for (int e = 0; e < 3; ++e) t[e] += m.t[e];
        }
        const double inv = 1.0 / (double)a.size[c];
        for (int e = 0; e < 4; ++e) q[e] *= inv;
        for (int e = 0; e < 3; ++e) t[e] *= inv;
        b200cv_pose P;
        for (int e = 0; e < 16; ++e) P.pose[e] = 0.0;
        const double nq = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
        if (nq > 0)
            for (int e = 0; e < 4; ++e) q[e] /= nq;
        const double w = q[0], x = q[1], y = q[2], z = q[3];
        double *R = P.pose;
        R[0] = 1 - 2 * (y * y + z * z), R[1] = 2 * (x * y - z * w), R[2] = 2 * (x * z + y * w);
        R[4] = 2 * (x * y + z * w), R[5] = 1 - 2 * (x * x + z * z), R[6] = 2 * (y * z - x * w);
        R[8] = 2 * (x * z - y * w), R[9] = 2 * (y * z + x * w), R[10] = 1 - 2 * (x * x + y * y);
        R[3] = t[0], R[7] = t[1], R[11] = t[2], R[15] = 1.0;
        const double trace = R[0] + R[5] + R[10];
        if (fabs(trace - 3) <= CV_EPS) P.angle = 0;
        else if (fabs(trace + 1) <= CV_EPS) P.angle = PI_D;
        else P.angle = acos((trace - 1) / 2);
        for (int e = 0; e < 3; ++e) P.t[e] = t[e];
        for (int e = 0; e < 4; ++e) P.q[e] = q[e];
        const unsigned long long vs = a.votes[c];
        P.num_votes = vs > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)vs;
        const b200cv_pose &first = a.poses[a.lead_pose[c]];
        P.model_index = first.model_index;
        P.alpha = first.alpha;
        P.residual = 0.0;
        P.alpha_index = first.alpha_index;
        P.reference_index = first.reference_index;
        a.out[o] = P;
    }
}

int cv_cluster(b200cv_detector *d, const b200cv_pose *d_poses, uint32_t refs, b200cv_pose *results, size_t cap, size_t *n_clusters) {
    b200ppf_ctx *ctx = d->ctx;
    StreamBuf<uint32_t> order(ctx), member_of(ctx), lead_pose(ctx), size(ctx), corder(ctx), ncl(ctx);
    StreamBuf<double4> lead(ctx);
    StreamBuf<unsigned long long> votes(ctx);
    StreamBuf<b200cv_pose> out(ctx);
    PPF_CUDA(ctx, order.alloc(refs));
    PPF_CUDA(ctx, member_of.alloc(refs));
    PPF_CUDA(ctx, lead_pose.alloc(refs));
    PPF_CUDA(ctx, size.alloc(refs));
    PPF_CUDA(ctx, corder.alloc(refs));
    PPF_CUDA(ctx, ncl.alloc(1));
    PPF_CUDA(ctx, lead.alloc(refs));
    PPF_CUDA(ctx, votes.alloc(refs));
    PPF_CUDA(ctx, out.alloc(refs));
    CvClusterArgs a;
    a.poses = d_poses;
    a.n = refs;
    a.position_threshold = d->position_threshold;
    a.rotation_threshold = d->rotation_threshold;
    a.order = order;
    a.member_of = member_of;
    a.lead = lead;
    a.lead_pose = lead_pose;
    a.size = size;
    a.votes = votes;
    a.corder = corder;
    a.out = out;
    a.n_clusters = ncl;
    cudaEventRecord(ctx->ev[2], ctx->stream);
    PPF_LAUNCH(ctx, cv_cluster_kernel, 1, CV_CLUSTER_THREADS, 0, a);
    cudaEventRecord(ctx->ev[3], ctx->stream);
    uint32_t h_ncl = 0;
    PPF_CUDA(ctx, cudaMemcpyAsync(&h_ncl, ncl.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t take = std::min<size_t>(h_ncl, cap);
    if (take) {
        PPF_CUDA(ctx, cudaMemcpyAsync(results, out.p, take * sizeof(b200cv_pose), cudaMemcpyDeviceToHost, ctx->stream));
        PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    cudaEventElapsedTime(&ctx->timings.cluster_ms, ctx->ev[2], ctx->ev[3]);
    *n_clusters = h_ncl;
    return B200PPF_OK;
}

}  // namespace

b200ppf_ctx *cv_detector_context(const b200cv_detector *d) { return d->ctx; }
bool cv_detector_trained(const b200cv_detector *d) { return d->d_offsets != nullptr; }

}  // namespace b200ppf

using namespace b200ppf;

extern "C" {

int b200cv_detector_create(b200ppf_ctx *ctx, double relative_sampling_step, double relative_distance_step, double num_angles,
                           b200cv_detector **out) {
    if (!ctx || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv detector: null argument");
    *out = nullptr;
    if (!(relative_sampling_step > 0) || !(relative_distance_step > 0) || !(num_angles >= 1))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cv detector: steps and the number of angles must be positive");
    b200cv_detector *d = new (std::nothrow) b200cv_detector();
    if (!d) return fail_msg(ctx, B200PPF_ERR_NOMEM, "cv detector: out of host memory");
    d->ctx = ctx;
    d->sampling_step_relative = relative_sampling_step;
    d->distance_step_relative = relative_distance_step;
    d->num_angles_arg = num_angles;
    // setSearchParams() defaults: position threshold = relative sampling step, rotation threshold = 2 pi / numAngles
    d->position_threshold = relative_sampling_step;
    d->rotation_threshold = (360.0 / num_angles) / 180.0 * PI_D;
    *out = d;
    return B200PPF_OK;
}

void b200cv_detector_free(b200cv_detector *d) {
    if (!d) return;
    DeviceGuard guard(d->ctx->device);
    cudaStreamSynchronize(d->ctx->stream);
    cv_free_match(d);
    cv_free_model(d);
    delete d;
}

int b200cv_detector_set_search_params(b200cv_detector *d, double position_threshold, double rotation_threshold) {
    if (!d) return fail_msg(nullptr, B200PPF_ERR_INVALID, "cv detector: null handle");
    if (position_threshold >= 0) d->position_threshold = position_threshold;
    if (rotation_threshold >= 0) d->rotation_threshold = rotation_threshold;
    return B200PPF_OK;
}

int b200cv_detector_train(b200cv_detector *d, const float *model, size_t n, size_t stride) {
    if (!d || !model) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_INVALID, "cv train: null argument");
    b200ppf_ctx *ctx = d->ctx;
    if (stride < 6 || n == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv train: the model is N x 6 [x y z nx ny nz], N >= 1");
    DeviceGuard guard(ctx->device);
    cv_free_model(d);
    float r[6];
    bbox6(model, n, stride, r);
    const float dx = r[1] - r[0], dy = r[3] - r[2], dz = r[5] - r[4];
    const float diameter = std::sqrt(dx * dx + dy * dy + dz * dz);
    const float distance_step = (float)(diameter * d->sampling_step_relative);  // upstream: diameter * sampling_step_relative
    int rc = cv_sample(ctx, model, n, stride, r, (float)d->sampling_step_relative, &d->d_model, &d->m);
    if (rc) return rc;
    const size_t m = d->m;
    // the table addresses its m^2 pair slots and its power-of-two bucket count with 32-bit words: m^2 <= 2^31 keeps both in
    // range (46341^2 > 2^31 would round the bucket count up to 2^32); refused before any of the O(m^2) buffers is allocated
    if (m < 2 || m > 46340) {
        cv_free_model(d);
        return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "cv train: 2 .. 46340 sampled model points (m^2 pair slots in 32-bit offsets)");
    }
    d->h_model.resize(m * 6);
    PPF_CUDA(ctx, cudaMemcpyAsync(d->h_model.data(), d->d_model, m * 6 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    d->angle_step = (360.0 / d->num_angles_arg) * PI_D / 180.0;
    d->distance_step = distance_step;
    size_t pow2 = 16;  // hashtableCreate: at least 16, else the next power of two
    while (pow2 < m * m) pow2 <<= 1;
    d->table_size = pow2;
    const size_t count = m * m;
    StreamBuf<uint32_t> k0(ctx), k1(ctx), i0(ctx), i1(ctx);
    PPF_CUDA(ctx, k0.alloc(count));
    PPF_CUDA(ctx, k1.alloc(count));
    PPF_CUDA(ctx, i0.alloc(count));
    PPF_CUDA(ctx, i1.alloc(count));
    PPF_CUDA(ctx, cudaMalloc(&d->d_alpha, count * sizeof(float)));
    PPF_CUDA(ctx, cudaMalloc(&d->d_offsets, (pow2 + 1) * sizeof(uint32_t)));
    cudaEventRecord(ctx->ev[0], ctx->stream);
    dim3 grid((unsigned)((m + 255) / 256), (unsigned)m);
    PPF_LAUNCH(ctx, cv_train_pairs_kernel, grid, 256, 0, d->d_model, (uint32_t)m, d->angle_step, (double)distance_step,
               (uint32_t)(pow2 - 1), k0.p, d->d_alpha);
    cudaEventRecord(ctx->ev[1], ctx->stream);
    // all 32 key bits: the diagonal's CV_INVALID keys have to end up behind every bucket
    bool in_alt = false;
    rc = radix_sort_u32(ctx, k0, k1, i0, i1, nullptr, nullptr, count, 0xFFFFFFFFu, /*v0_iota=*/true, &in_alt);
    if (rc) return rc;
    cudaEventRecord(ctx->ev[2], ctx->stream);
    const uint32_t *ks = in_alt ? k1.p : k0.p, *is = in_alt ? i1.p : i0.p;
    // keys == CV_INVALID (the diagonal) sort behind every bucket
    if ((rc = lower_bounds(ctx, ks, (uint32_t)count, nullptr, (uint32_t)pow2, 0, d->d_offsets))) return rc;
    d->n_nodes = m * (m - 1);
    PPF_CUDA(ctx, cudaMalloc(&d->d_nodes, std::max<size_t>(1, d->n_nodes) * sizeof(uint32_t)));
    PPF_CUDA(ctx, cudaMemcpyAsync(d->d_nodes, is, d->n_nodes * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    cudaEventRecord(ctx->ev[3], ctx->stream);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->timings.keys_ms, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->timings.sort_ms, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&ctx->timings.csr_ms, ctx->ev[2], ctx->ev[3]);
    return B200PPF_OK;
}

int b200cv_detector_get_info(const b200cv_detector *d, b200cv_info *info) {
    if (!d || !info) return fail_msg(nullptr, B200PPF_ERR_INVALID, "cv info: null argument");
    info->n_sampled = d->m;
    info->table_size = d->table_size;
    info->n_nodes = d->n_nodes;
    info->angle_step = d->angle_step;
    info->distance_step = d->distance_step;
    info->num_angles = d->angle_step > 0 ? (int)std::floor(2 * PI_D / d->angle_step) : 0;
    info->position_threshold = d->position_threshold;
    info->rotation_threshold = d->rotation_threshold;
    info->n_scene_sampled = d->n_scene;
    info->n_second_sampled = d->n_second;
    return B200PPF_OK;
}

int b200cv_detector_model_points(const b200cv_detector *d, float *out6) {
    if (!d || !out6) return fail_msg(nullptr, B200PPF_ERR_INVALID, "cv model points: null argument");
    memcpy(out6, d->h_model.data(), d->h_model.size() * sizeof(float));
    return B200PPF_OK;
}

int b200cv_detector_scene_points(const b200cv_detector *d, float *out6) {
    if (!d || !out6) return fail_msg(nullptr, B200PPF_ERR_INVALID, "cv scene points: null argument");
    memcpy(out6, d->h_scene.data(), d->h_scene.size() * sizeof(float));
    return B200PPF_OK;
}

int b200cv_detector_bucket(b200cv_detector *d, size_t bucket, uint32_t *ppf_ind, size_t cap, size_t *n_found) {
    if (!d || !n_found || (cap && !ppf_ind)) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_INVALID, "cv bucket: null argument");
    *n_found = 0;
    if (!d->d_offsets || bucket >= d->table_size) return B200PPF_OK;
    b200ppf_ctx *ctx = d->ctx;
    DeviceGuard guard(ctx->device);
    uint32_t off[2];
    PPF_CUDA(ctx, cudaMemcpyAsync(off, d->d_offsets + bucket, sizeof(off), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_found = off[1] - off[0];
    const size_t take = std::min<size_t>(cap, *n_found);
    if (take) {
        PPF_CUDA(ctx, cudaMemcpyAsync(ppf_ind, d->d_nodes + off[0], take * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return B200PPF_OK;
}

int b200cv_detector_table_export(b200cv_detector *d, uint32_t *offsets, uint32_t *nodes, float *alpha_m) {
    if (!d || !d->d_offsets) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_STATE, "cv export: the detector is not trained");
    b200ppf_ctx *ctx = d->ctx;
    DeviceGuard guard(ctx->device);
    if (offsets) PPF_CUDA(ctx, cudaMemcpyAsync(offsets, d->d_offsets, (d->table_size + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (nodes) PPF_CUDA(ctx, cudaMemcpyAsync(nodes, d->d_nodes, d->n_nodes * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (alpha_m) PPF_CUDA(ctx, cudaMemcpyAsync(alpha_m, d->d_alpha, d->m * d->m * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

// the checks every match makes; *step = the reference stride of relativeSceneSampleStep
static int cv_match_begin(b200cv_detector *d, b200cv_pose *results, size_t cap, size_t *n_results, double relative_scene_sample_step,
                          double relative_scene_distance, int *step) {
    if (!d || !n_results || (cap && !results)) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_INVALID, "cv match: null argument");
    *n_results = 0;
    b200ppf_ctx *ctx = d->ctx;
    if (!d->d_offsets) return fail_msg(ctx, B200PPF_ERR_STATE, "cv match: the detector is not trained");
    if (!(relative_scene_sample_step > 0) || !(relative_scene_distance > 0))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match: the scene steps must be positive");
    *step = (int)(1.0 / relative_scene_sample_step);
    if (*step < 1) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match: relativeSceneSampleStep must not exceed 1");
    return B200PPF_OK;
}

// everything after sampling, whichever input the sampled clouds came from: the last-match state (sampled scene on the
// host, per-reference poses), voting, clustering
static int cv_match_sampled(b200cv_detector *d, int step, b200cv_pose *results, size_t cap, size_t *n_results, uint32_t *acc_dump,
                            size_t dump_ref) {
    b200ppf_ctx *ctx = d->ctx;
    d->h_scene.resize(d->n_scene * 6);
    PPF_CUDA(ctx, cudaMemcpyAsync(d->h_scene.data(), d->d_scene, d->n_scene * 6 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    const size_t refs = (d->n_scene + step - 1) / step;
    d->raw.clear();
    if (refs == 0) return B200PPF_OK;
    StreamBuf<b200cv_pose> d_poses(ctx);  // per reference point, clustered on the device
    int rc = cv_vote(d, (uint32_t)step, (uint32_t)refs, acc_dump, (uint32_t)dump_ref, d_poses);
    if (rc) return rc;
    size_t ncl = 0;
    rc = cv_cluster(d, d_poses, (uint32_t)refs, results, cap, &ncl);
    if (rc) return rc;
    *n_results = ncl;
    return B200PPF_OK;
}

static int cv_match_impl(b200cv_detector *d, const float *scene, size_t n, size_t stride, const float *edge, size_t n_edge,
                         size_t edge_stride, double relative_scene_sample_step, double relative_scene_distance,
                         b200cv_pose *results, size_t cap, size_t *n_results, uint32_t *acc_dump, size_t dump_ref) {
    if (!scene) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_INVALID, "cv match: null argument");
    int step = 0;
    int rc = cv_match_begin(d, results, cap, n_results, relative_scene_sample_step, relative_scene_distance, &step);
    if (rc) return rc;
    b200ppf_ctx *ctx = d->ctx;
    if (stride < 6 || (edge && edge_stride < 6) || n == 0)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match: clouds are N x 6 [x y z nx ny nz]");
    DeviceGuard guard(ctx->device);
    cv_free_match(d);
    float r[6];
    bbox6(scene, n, stride, r);
    rc = cv_sample(ctx, scene, n, stride, r, (float)relative_scene_distance, &d->d_scene, &d->n_scene);
    if (rc) return rc;
    d->second_is_scene = edge == nullptr;
    if (edge) {
        float re[6];
        bbox6(edge, n_edge, edge_stride, re);
        rc = cv_sample(ctx, edge, n_edge, edge_stride, re, (float)relative_scene_distance, &d->d_second, &d->n_second);
        if (rc) return rc;
    } else {
        d->d_second = d->d_scene;
        d->n_second = d->n_scene;
    }
    return cv_match_sampled(d, step, results, cap, n_results, acc_dump, dump_ref);
}

int b200cv_detector_match_cloud(b200cv_detector *d, const b200ppf_cloud *scene, const b200ppf_cloud *edge,
                                double relative_scene_sample_step, double relative_scene_distance, b200cv_pose *results, size_t cap,
                                size_t *n_results) {
    int step = 0;
    int rc = cv_match_begin(d, results, cap, n_results, relative_scene_sample_step, relative_scene_distance, &step);
    if (rc) return rc;
    b200ppf_ctx *ctx = d->ctx;
    if (!scene) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match cloud: null scene");
    if (scene->ctx != ctx || (edge && edge->ctx != ctx))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match cloud: the clouds belong to another context than the detector");
    if (scene->n == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match cloud: empty scene cloud");
    if (edge && edge->n == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match_S2B: empty edge cloud");
    DeviceGuard guard(ctx->device);
    cv_free_match(d);
    rc = cv_sample_cloud(ctx, scene, (float)relative_scene_distance, &d->d_scene, &d->n_scene);
    if (rc) return rc;
    d->second_is_scene = edge == nullptr;
    if (edge) {
        rc = cv_sample_cloud(ctx, edge, (float)relative_scene_distance, &d->d_second, &d->n_second);
        if (rc) return rc;
    } else {
        d->d_second = d->d_scene;
        d->n_second = d->n_scene;
    }
    return cv_match_sampled(d, step, results, cap, n_results, nullptr, 0);
}

int b200cv_detector_match(b200cv_detector *d, const float *scene, size_t n, size_t stride, double relative_scene_sample_step,
                          double relative_scene_distance, b200cv_pose *results, size_t cap, size_t *n_results) {
    return cv_match_impl(d, scene, n, stride, nullptr, 0, 0, relative_scene_sample_step, relative_scene_distance, results, cap,
                         n_results, nullptr, 0);
}

int b200cv_detector_match_s2b(b200cv_detector *d, const float *scene, size_t n, size_t stride, const float *edge, size_t n_edge,
                              size_t edge_stride, double relative_scene_sample_step, double relative_scene_distance,
                              b200cv_pose *results, size_t cap, size_t *n_results) {
    if (!edge || n_edge == 0) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_INVALID, "cv match_S2B: empty edge cloud");
    return cv_match_impl(d, scene, n, stride, edge, n_edge, edge_stride, relative_scene_sample_step, relative_scene_distance, results,
                         cap, n_results, nullptr, 0);
}

int b200cv_detector_raw_poses(const b200cv_detector *d, b200cv_pose *raw, size_t cap, size_t *n) {
    if (!d || !n) return fail_msg(nullptr, B200PPF_ERR_INVALID, "cv raw poses: null argument");
    *n = d->raw.size();
    for (size_t k = 0; k < d->raw.size() && k < cap; ++k) raw[k] = d->raw[k];
    return B200PPF_OK;
}

int b200cv_detector_debug_accumulator(b200cv_detector *d, const float *scene, size_t n, size_t stride, const float *edge,
                                      size_t n_edge, size_t edge_stride, double relative_scene_sample_step,
                                      double relative_scene_distance, size_t reference, uint32_t *acc) {
    if (!acc) return fail_msg(d ? d->ctx : nullptr, B200PPF_ERR_INVALID, "cv accumulator: null output");
    b200cv_pose one;
    size_t k = 0;
    return cv_match_impl(d, scene, n, stride, edge, n_edge, edge_stride, relative_scene_sample_step, relative_scene_distance, &one, 1,
                         &k, acc, reference);
}

}  // extern "C"
