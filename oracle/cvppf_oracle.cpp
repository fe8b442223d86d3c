/*
 * cvppf_oracle.cpp — CPU restatement of the PPF engine the reference actually calls:
 * cv::ppf_match_3d::PPF3DDetector (opencv_contrib modules/surface_matching/src/ppf_match_3d.cpp, ppf_helpers.cpp,
 * c_utils.hpp, pose_3d.cpp, t_hash_int.cpp, hash_murmur86.hpp), reference call sites include/CloudProcessing.h:205,
 * :217, :234-236 (constructor, trainModel), :442 (match), :495 (match_S2B, fork-only).
 *
 * TEST INFRASTRUCTURE ONLY, and the checker of a row that is NOT BUILT on the device yet (SURVEY.md §8f rank 4,
 * DESIGN.md §8-9): written first, as the round order asks, so that the table and voting kernels of that row have
 * something to be compared with.
 *
 * PARITY UNPINNED, twice over: opencv_contrib is neither vendored in the reference nor installed here (the
 * reference even builds against a private fork), and the file is restated from memory of the upstream source plus
 * SURVEY.md Appendix B.  Known soft spots, in decreasing order of effect on results:
 *   - the hash: upstream selects hashMurmurx64 (MurmurHash3_x64_128) on 64-bit builds and hashMurmurx86
 *     (MurmurHash3_x86_32) otherwise; this file uses the 32-bit variant (seed 42).  Which model pairs share a
 *     bucket by accident (different keys, equal hash modulo the table size) therefore differs from a 64-bit
 *     OpenCV build; with N^2 nodes in >= N^2 buckets such collisions are a handful per table.
 *   - std::sort in clusterPoses is not stable; ties (equal votes) are ordered by reference index here.
 *   - the rotation -> quaternion conversion used for the cluster average is the textbook branch-on-largest form;
 *     upstream's dcmToQuat may choose the opposite sign of q for some rotations, which matters only when a cluster
 *     averages poses on both sides of such a branch.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <vector>

#ifdef _OPENMP
#include <omp.h>
#endif

#include "ppf_oracle.h"

namespace {

constexpr double CV_EPS = 1.192092896e-07;  // EPS of c_utils.hpp (FLT_EPSILON)
constexpr double PI = 3.14159265358979323846;

struct V3 {
    double x, y, z;
};
inline V3 sub(const V3 &a, const V3 &b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline double dot(const V3 &a, const V3 &b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(const V3 &a, const V3 &b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline double norm(const V3 &a) { return std::sqrt(dot(a, a)); }
inline V3 ld(const float *p) { return {(double)p[0], (double)p[1], (double)p[2]}; }

struct M33 {
    double m[9];
};
inline V3 mul(const M33 &R, const V3 &v) {
    return {R.m[0] * v.x + R.m[1] * v.y + R.m[2] * v.z, R.m[3] * v.x + R.m[4] * v.y + R.m[5] * v.z,
            R.m[6] * v.x + R.m[7] * v.y + R.m[8] * v.z};
}

/* c_utils.hpp aaToR: R = cosA * I + sinA * [axis]x + (1 - cosA) * axis axis^T, element by element as upstream */
inline void aa_to_r(const V3 &axis, double angle, M33 &R) {
    const double sinA = std::sin(angle), cosA = std::cos(angle), cos1A = 1.0 - cosA;
    const double a[3] = {axis.x, axis.y, axis.z};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double v = (i == j) ? cosA : 0.0;
            if (i != j) v += (((i + 1) % 3 == j) ? -1.0 : 1.0) * sinA * a[3 - i - j];
            v += cos1A * a[i] * a[j];
            R.m[3 * i + j] = v;
        }
}

/* c_utils.hpp computeTransformRT: rotation taking n1 onto the x axis (axis n1 x e_x), t = -R p1 */
inline void compute_transform_rt(const V3 &p1, const V3 &n1, M33 &R, V3 &t) {
    const double angle = std::acos(n1.x);
    V3 axis{0.0, n1.z, -n1.y};
    if (n1.y == 0 && n1.z == 0) {
        axis.y = 1;
        axis.z = 0;
    } else {
        const double nn = norm(axis);
        if (nn > CV_EPS) axis = {axis.x / nn, axis.y / nn, axis.z / nn};
    }
    aa_to_r(axis, angle, R);
    const V3 rp = mul(R, p1);
    t = {-rp.x, -rp.y, -rp.z};
}

/* c_utils.hpp TAngle3Normalized */
inline double angle3(const V3 &a, const V3 &b) { return std::atan2(norm(cross(a, b)), dot(a, b)); }

/* PPF3DDetector::computePPFFeatures: (angle(n1,d), angle(n2,d), angle(n1,n2), |d|); f stays 0 when |d| <= EPS */
inline void ppf_features(const V3 &p1, const V3 &n1, const V3 &p2, const V3 &n2, double f[4]) {
    f[0] = f[1] = f[2] = f[3] = 0.0;
    V3 d = sub(p2, p1);
    f[3] = norm(d);
    if (f[3] <= CV_EPS) return;
    const double inv = 1.0 / f[3];
    d = {d.x * inv, d.y * inv, d.z * inv};
    f[0] = angle3(n1, d);
    f[1] = angle3(n2, d);
    f[2] = angle3(n1, n2);
}

/* MurmurHash3_x86_32 (hash_murmur86.hpp hashMurmurx86) */
inline uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
inline uint32_t murmur3_x86_32(const void *key, int len, uint32_t seed) {
    const uint8_t *data = static_cast<const uint8_t *>(key);
    const int nblocks = len / 4;
    uint32_t h1 = seed;
    const uint32_t c1 = 0xcc9e2d51u, c2 = 0x1b873593u;
    for (int i = 0; i < nblocks; ++i) {
        uint32_t k1;
        std::memcpy(&k1, data + 4 * i, 4);
        k1 *= c1;
        k1 = rotl32(k1, 15);
        k1 *= c2;
        h1 ^= k1;
        h1 = rotl32(h1, 13);
        h1 = h1 * 5 + 0xe6546b64u;
    }
    const uint8_t *tail = data + nblocks * 4;
    uint32_t k1 = 0;
    switch (len & 3) {
        case 3: k1 ^= (uint32_t)tail[2] << 16; /* fallthrough */
        case 2: k1 ^= (uint32_t)tail[1] << 8;  /* fallthrough */
        case 1:
            k1 ^= tail[0];
            k1 *= c1;
            k1 = rotl32(k1, 15);
            k1 *= c2;
            h1 ^= k1;
    }
    h1 ^= (uint32_t)len;
    h1 ^= h1 >> 16;
    h1 *= 0x85ebca6bu;
    h1 ^= h1 >> 13;
    h1 *= 0xc2b2ae35u;
    h1 ^= h1 >> 16;
    return h1;
}

/* hashPPF: the four features truncated to ints by their steps, hashed with seed 42 */
inline uint32_t hash_ppf(const double f[4], double angle_step, double distance_step) {
    const int32_t key[4] = {(int32_t)(f[0] / angle_step), (int32_t)(f[1] / angle_step), (int32_t)(f[2] / angle_step),
                            (int32_t)(f[3] / distance_step)};
    return murmur3_x86_32(key, 16, 42u);
}

/* PPF3DDetector::computeAlpha: planar angle of p2 in the frame that puts (p1, n1) at the origin / x axis */
inline double planar_alpha(const M33 &R, const V3 &t, const V3 &p2, bool *is_nan) {
    const V3 rp = mul(R, p2);
    const V3 mpt{t.x + rp.x, t.y + rp.y, t.z + rp.z};
    double alpha = std::atan2(-mpt.z, mpt.y);
    *is_nan = alpha != alpha;
    if (*is_nan) return 0.0;
    if (std::sin(alpha) * mpt.z < 0.0) alpha = -alpha;
    return -alpha;
}

struct Pose {
    double m[16];  // row-major 4x4
    double angle;  // rotation angle, as Pose3D::updatePose forms it
    double t[3];
    double q[4];  // w x y z
    double alpha;
    uint32_t model_index;
    uint32_t votes;
    uint32_t order;  // reference order, the tie-break of the vote sort
};

inline void rotation_to_quat(const double *R /*row-major 3x3, stride 4*/, double q[4]) {
    const double r00 = R[0], r01 = R[1], r02 = R[2], r10 = R[4], r11 = R[5], r12 = R[6], r20 = R[8], r21 = R[9], r22 = R[10];
    const double tr = r00 + r11 + r22;
    if (tr > 0.0) {
        const double s = std::sqrt(tr + 1.0) * 2.0;
        q[0] = 0.25 * s, q[1] = (r21 - r12) / s, q[2] = (r02 - r20) / s, q[3] = (r10 - r01) / s;
    } else if (r00 > r11 && r00 > r22) {
        const double s = std::sqrt(1.0 + r00 - r11 - r22) * 2.0;
        q[0] = (r21 - r12) / s, q[1] = 0.25 * s, q[2] = (r01 + r10) / s, q[3] = (r02 + r20) / s;
    } else if (r11 > r22) {
        const double s = std::sqrt(1.0 + r11 - r00 - r22) * 2.0;
        q[0] = (r02 - r20) / s, q[1] = (r01 + r10) / s, q[2] = 0.25 * s, q[3] = (r12 + r21) / s;
    } else {
        const double s = std::sqrt(1.0 + r22 - r00 - r11) * 2.0;
        q[0] = (r10 - r01) / s, q[1] = (r02 + r20) / s, q[2] = (r12 + r21) / s, q[3] = 0.25 * s;
    }
}

inline void quat_to_rotation(const double qin[4], double *R /*stride 4*/) {
    double q[4] = {qin[0], qin[1], qin[2], qin[3]};
    const double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n > 0)
        for (double &v : q) v /= n;
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    R[0] = 1 - 2 * (y * y + z * z), R[1] = 2 * (x * y - z * w), R[2] = 2 * (x * z + y * w);
    R[4] = 2 * (x * y + z * w), R[5] = 1 - 2 * (x * x + z * z), R[6] = 2 * (y * z - x * w);
    R[8] = 2 * (x * z - y * w), R[9] = 2 * (y * z + x * w), R[10] = 1 - 2 * (x * x + y * y);
}

/* Pose3D::updatePose(Matx44d): angle from the trace (0 / pi at the ends), t, q */
inline void pose_update(Pose &p) {
    const double trace = p.m[0] + p.m[5] + p.m[10];
    if (std::fabs(trace - 3) <= CV_EPS) p.angle = 0;
    else if (std::fabs(trace + 1) <= CV_EPS) p.angle = PI;
    else p.angle = std::acos((trace - 1) / 2);
    p.t[0] = p.m[3], p.t[1] = p.m[7], p.t[2] = p.m[11];
    rotation_to_quat(p.m, p.q);
}

inline void rt_to_pose(const M33 &R, const V3 &t, double *m) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) m[4 * r + c] = R.m[3 * r + c];
    m[3] = t.x, m[7] = t.y, m[11] = t.z;
    m[12] = m[13] = m[14] = 0.0;
    m[15] = 1.0;
}
inline void mat44_mul(const double *a, const double *b, double *o) {
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            for (int k = 0; k < 4; ++k) s += a[4 * r + k] * b[4 * k + c];
            o[4 * r + c] = s;
        }
}

/* ppf_helpers.cpp samplePCByQuantization (weightByCenter = 0): cells of 1/sampleStep per axis over the bounding box,
 * positions and normals of a cell averaged in double in point order, normals renormalised.  The cell index uses
 * stride numSamplesDim although a coordinate at the upper bound lands in cell numSamplesDim — upstream's quirk,
 * kept: such points merge into a neighbouring cell's list. */
std::vector<float> sample_by_quantization(const float *pc, size_t n, const float range[6], float sample_step) {
    const int ns = (int)(1.0 / sample_step);
    const float xr = range[1] - range[0], yr = range[3] - range[2], zr = range[5] - range[4];
    std::vector<std::vector<uint32_t>> map((size_t)(ns + 1) * (ns + 1) * (ns + 1));
    for (size_t i = 0; i < n; ++i) {
        const float *p = pc + 6 * i;
        const int xc = (int)((float)ns * (p[0] - range[0]) / xr);
        const int yc = (int)((float)ns * (p[1] - range[2]) / yr);
        const int zc = (int)((float)ns * (p[2] - range[4]) / zr);
        const int index = xc * ns * ns + yc * ns + zc;
        map[(size_t)index].push_back((uint32_t)i);
    }
    std::vector<float> out;
    for (const auto &cell : map) {
        if (cell.empty()) continue;
        double a[6] = {0, 0, 0, 0, 0, 0};
        for (uint32_t i : cell)
            for (int k = 0; k < 6; ++k) a[k] += (double)pc[6 * (size_t)i + k];
        for (double &v : a) v /= (double)cell.size();
        const double nn = std::sqrt(a[3] * a[3] + a[4] * a[4] + a[5] * a[5]);
        float row[6] = {(float)a[0], (float)a[1], (float)a[2], 0.f, 0.f, 0.f};  // Mat(numPoints, cols, CV_32F) is not zeroed upstream
        if (nn > CV_EPS) row[3] = (float)(a[3] / nn), row[4] = (float)(a[4] / nn), row[5] = (float)(a[5] / nn);
        out.insert(out.end(), row, row + 6);
    }
    return out;
}

void bbox6(const float *pc, size_t n, float r[6]) {  // computeBboxStd
    for (int k = 0; k < 3; ++k) r[2 * k] = r[2 * k + 1] = n ? pc[k] : 0.f;
    for (size_t i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) {
            r[2 * k] = std::min(r[2 * k], pc[6 * i + k]);
            r[2 * k + 1] = std::max(r[2 * k + 1], pc[6 * i + k]);
        }
}

}  // namespace

struct oracle_cv_detector {
    double sampling_step_relative, distance_step_relative, num_angles_arg;
    double angle_step = 0, distance_step = 0;
    double position_threshold, rotation_threshold;
    std::vector<float> sampled;   // M x 6
    std::vector<float> alpha_m;   // M*M, index i*M + j (the fifth column of upstream's ppf matrix)
    size_t table_size = 0;        // power of two >= 16
    std::vector<std::vector<std::pair<uint32_t, uint32_t>>> buckets;  // chains of (i, ppfInd)
    size_t m() const { return sampled.size() / 6; }
};

extern "C" {

/* PPF3DDetector(relativeSamplingStep, relativeDistanceStep = 0.05, numAngles = 30) + setSearchParams() defaults:
 * position_threshold = relativeSamplingStep, rotation_threshold = 2 pi / numAngles (SURVEY.md Appendix B) */
oracle_cv_detector *oracle_cv_create(double relative_sampling_step, double relative_distance_step, double num_angles) {
    auto *d = new oracle_cv_detector();
    d->sampling_step_relative = relative_sampling_step;
    d->distance_step_relative = relative_distance_step;
    d->num_angles_arg = num_angles;
    d->position_threshold = relative_sampling_step;
    d->rotation_threshold = (360.0 / num_angles) / 180.0 * PI;
    return d;
}
void oracle_cv_destroy(oracle_cv_detector *d) { delete d; }
void oracle_cv_set_search_params(oracle_cv_detector *d, double position_threshold, double rotation_threshold) {
    if (position_threshold >= 0) d->position_threshold = position_threshold;
    if (rotation_threshold >= 0) d->rotation_threshold = rotation_threshold;
}

/* samplePCByQuantization over the cloud's own bounding box; out holds up to n rows of 6 floats; returns the count */
size_t oracle_cv_sample(const float *pc, size_t n, float sample_step, float *out) {
    float r[6];
    bbox6(pc, n, r);
    const std::vector<float> s = sample_by_quantization(pc, n, r, sample_step);
    std::memcpy(out, s.data(), s.size() * sizeof(float));
    return s.size() / 6;
}

/* the hash alone (known-answer tests) */
uint32_t oracle_cv_murmur(const void *key, int len, uint32_t seed) { return murmur3_x86_32(key, len, seed); }

/* one pair: f[4] = computePPFFeatures, returns hashPPF */
uint32_t oracle_cv_pair(const float *p1n1, const float *p2n2, double angle_step, double distance_step, double *f) {
    ppf_features(ld(p1n1), ld(p1n1 + 3), ld(p2n2), ld(p2n2 + 3), f);
    return hash_ppf(f, angle_step, distance_step);
}

/* PPF3DDetector::trainModel: returns the number of sampled model points */
size_t oracle_cv_train(oracle_cv_detector *d, const float *model, size_t n) {
    float r[6];
    bbox6(model, n, r);
    const float dx = r[1] - r[0], dy = r[3] - r[2], dz = r[5] - r[4];
    const float diameter = std::sqrt(dx * dx + dy * dy + dz * dz);
    const float distance_step = (float)(diameter * d->sampling_step_relative);
    d->sampled = sample_by_quantization(model, n, r, (float)d->sampling_step_relative);
    const size_t m = d->m();
    d->angle_step = (360.0 / d->num_angles_arg) * PI / 180.0;
    d->distance_step = distance_step;
    size_t size = m * m;
    size_t pow2 = 16;  // hashtableCreate: at least 16, else the next power of two
    while (pow2 < size) pow2 <<= 1;
    d->table_size = pow2;
    d->buckets.assign(pow2, {});
    d->alpha_m.assign(m * m, 0.f);
    for (size_t i = 0; i < m; ++i) {
        const V3 p1 = ld(&d->sampled[6 * i]), n1 = ld(&d->sampled[6 * i + 3]);
        M33 R;
        V3 t;
        compute_transform_rt(p1, n1, R, t);
        for (size_t j = 0; j < m; ++j) {
            if (i == j) continue;
            const V3 p2 = ld(&d->sampled[6 * j]), n2 = ld(&d->sampled[6 * j + 3]);
            double f[4];
            ppf_features(p1, n1, p2, n2, f);
            const uint32_t h = hash_ppf(f, d->angle_step, distance_step);
            bool is_nan;
            const double alpha = planar_alpha(R, t, p2, &is_nan);
            const uint32_t ppf_ind = (uint32_t)(i * m + j);
            d->alpha_m[ppf_ind] = (float)alpha;
            // hash % size; hashtableInsertHashed prepends to the chain — the order inside a chain does not reach the
            // votes, so the cheaper append is used
            d->buckets[h & (pow2 - 1)].push_back({(uint32_t)i, ppf_ind});
        }
    }
    return m;
}

size_t oracle_cv_model_points(const oracle_cv_detector *d, float *out6) {
    if (out6) std::memcpy(out6, d->sampled.data(), d->sampled.size() * sizeof(float));
    return d->m();
}

/* PPF3DDetector::match: scene sampled with relative_scene_distance, every (int)(1/relative_scene_sample_step)-th
 * sampled point a reference, all other sampled points paired with it, votes per (model point, alpha index over
 * 4 pi), first maximum, pose = Tsg^-1 Rx(alpha) Tmg; then clusterPoses.  out_poses: up to cap rows of 16 doubles,
 * out_votes their cluster votes.  raw (optional, capacity = number of reference points): the per-reference poses
 * before clustering as (votes, model index, alpha index).  Returns the number of clusters. */
size_t oracle_cv_match(const oracle_cv_detector *d, const float *scene, size_t n, double relative_scene_sample_step,
                       double relative_scene_distance, double *out_poses, uint32_t *out_votes, size_t cap, uint32_t *raw3,
                       size_t *n_refs, int n_threads) {
    return oracle_cv_match_s2b(d, scene, n, nullptr, 0, relative_scene_sample_step, relative_scene_distance, out_poses, out_votes,
                               cap, raw3, n_refs, n_threads);
}

/* match_S2B(scene, edge, ...) of the reference's private fork (include/CloudProcessing.h:495) — source unavailable.
 * INFERRED from the name (Choi et al., surface-to-boundary pairs) and from its inputs (the object cloud and the
 * curvature-edge cloud EdgeExtraction makes of it): reference points are taken from the sampled surface cloud exactly
 * as in match(); the points they are paired with are the sampled EDGE cloud (sampled over its own bounding box with
 * the same relative distance) instead of the surface cloud itself.  edge == nullptr is match(). */
size_t oracle_cv_match_s2b(const oracle_cv_detector *d, const float *scene, size_t n, const float *edge, size_t n_edge,
                           double relative_scene_sample_step, double relative_scene_distance, double *out_poses,
                           uint32_t *out_votes, size_t cap, uint32_t *raw3, size_t *n_refs, int n_threads) {
    const size_t m = d->m();
    const int num_angles = (int)std::floor(2 * PI / d->angle_step);
    const int step = (int)(1.0 / relative_scene_sample_step);
    float r[6];
    bbox6(scene, n, r);
    const std::vector<float> sampled = sample_by_quantization(scene, n, r, (float)relative_scene_distance);
    const size_t ns = sampled.size() / 6;
    std::vector<float> sampled_edge;
    if (edge) {
        float re[6];
        bbox6(edge, n_edge, re);
        sampled_edge = sample_by_quantization(edge, n_edge, re, (float)relative_scene_distance);
    }
    const std::vector<float> &second = edge ? sampled_edge : sampled;  // the points a reference point is paired with
    const size_t n2 = second.size() / 6;
    const size_t refs = step > 0 ? (ns + step - 1) / step : 0;
    if (n_refs) *n_refs = refs;
    std::vector<Pose> poses(refs);
    if (n_threads < 1) n_threads = 1;
#pragma omp parallel for num_threads(n_threads) schedule(dynamic, 1)
    for (long long rr = 0; rr < (long long)refs; ++rr) {
        const size_t i = (size_t)rr * step;
        std::vector<uint32_t> acc((size_t)num_angles * m, 0u);
        const V3 p1 = ld(&sampled[6 * i]), n1 = ld(&sampled[6 * i + 3]);
        M33 Rsg;
        V3 tsg;
        compute_transform_rt(p1, n1, Rsg, tsg);
        for (size_t j = 0; j < n2; ++j) {
            if (!edge && i == j) continue;
            const V3 p2 = ld(&second[6 * j]), nrm2 = ld(&second[6 * j + 3]);
            double f[4];
            ppf_features(p1, n1, p2, nrm2, f);
            const uint32_t h = hash_ppf(f, d->angle_step, (float)d->distance_step);
            bool is_nan;
            const double alpha_scene = planar_alpha(Rsg, tsg, p2, &is_nan);
            if (is_nan) continue;
            for (const auto &node : d->buckets[h & (d->table_size - 1)]) {
                const double alpha = (double)d->alpha_m[node.second] - alpha_scene;
                const int alpha_index = (int)(num_angles * (alpha + 2 * PI) / (4 * PI));
                const size_t a = (size_t)node.first * num_angles + (size_t)alpha_index;
                if (a < acc.size()) acc[a]++;  // alpha = +2 pi exactly would index one past the row, as upstream does
            }
        }
        uint32_t max_votes = 0, ref_max = 0, alpha_max = 0;
        for (size_t k = 0; k < m; ++k)
            for (int j = 0; j < num_angles; ++j) {
                const uint32_t v = acc[k * num_angles + j];
                if (v > max_votes) max_votes = v, ref_max = (uint32_t)k, alpha_max = (uint32_t)j;
            }
        // TsgInv
        M33 RInv;
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) RInv.m[3 * a + b] = Rsg.m[3 * b + a];
        const V3 rt = mul(RInv, tsg);
        double TsgInv[16], Tmg[16], Talpha[16], tmp[16];
        rt_to_pose(RInv, V3{-rt.x, -rt.y, -rt.z}, TsgInv);
        M33 Rmg;
        V3 tmg;
        compute_transform_rt(ld(&d->sampled[6 * (size_t)ref_max]), ld(&d->sampled[6 * (size_t)ref_max + 3]), Rmg, tmg);
        rt_to_pose(Rmg, tmg, Tmg);
        const double alpha = ((double)alpha_max * (4 * PI)) / num_angles - 2 * PI;
        const M33 Rx{{1, 0, 0, 0, std::cos(alpha), -std::sin(alpha), 0, std::sin(alpha), std::cos(alpha)}};  // getUnitXRotation
        rt_to_pose(Rx, V3{0, 0, 0}, Talpha);
        Pose &P = poses[(size_t)rr];
        mat44_mul(Talpha, Tmg, tmp);
        mat44_mul(TsgInv, tmp, P.m);
        P.alpha = alpha;
        P.model_index = ref_max;
        P.votes = max_votes;
        P.order = (uint32_t)rr;
        pose_update(P);
        if (raw3) raw3[3 * rr] = max_votes, raw3[3 * rr + 1] = ref_max, raw3[3 * rr + 2] = alpha_max;
    }

    /* clusterPoses: sort by votes (ties: reference order), greedy assignment to the first cluster whose FIRST pose
     * matches (matchPose: |angle difference| < rotation_threshold and |t difference| < position_threshold), clusters
     * sorted by their vote sums, plain average of quaternions and translations */
    std::vector<uint32_t> order(refs);
    for (size_t k = 0; k < refs; ++k) order[k] = (uint32_t)k;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return poses[a].votes > poses[b].votes; });
    std::vector<std::vector<uint32_t>> clusters;
    std::vector<uint64_t> cluster_votes;
    for (uint32_t k : order) {
        const Pose &p = poses[k];
        bool assigned = false;
        for (size_t c = 0; c < clusters.size() && !assigned; ++c) {
            const Pose &centre = poses[clusters[c][0]];
            const double dv[3] = {centre.t[0] - p.t[0], centre.t[1] - p.t[1], centre.t[2] - p.t[2]};
            const double dn = std::sqrt(dv[0] * dv[0] + dv[1] * dv[1] + dv[2] * dv[2]);
            const double phi = std::fabs(p.angle - centre.angle);
            if (phi < d->rotation_threshold && dn < d->position_threshold) {
                clusters[c].push_back(k);
                cluster_votes[c] += p.votes;
                assigned = true;
            }
        }
        if (!assigned) {
            clusters.push_back({k});
            cluster_votes.push_back(p.votes);
        }
    }
    std::vector<uint32_t> corder(clusters.size());
    for (size_t c = 0; c < clusters.size(); ++c) corder[c] = (uint32_t)c;
    std::stable_sort(corder.begin(), corder.end(), [&](uint32_t a, uint32_t b) { return cluster_votes[a] > cluster_votes[b]; });
    const size_t n_out = std::min(cap, clusters.size());
    for (size_t o = 0; o < n_out; ++o) {
        const auto &cl = clusters[corder[o]];
        double q[4] = {0, 0, 0, 0}, t[3] = {0, 0, 0};
        for (uint32_t k : cl) {
            for (int e = 0; e < 4; ++e) q[e] += poses[k].q[e];
            for (int e = 0; e < 3; ++e) t[e] += poses[k].t[e];
        }
        const double inv = 1.0 / (double)cl.size();
        for (double &v : q) v *= inv;
        for (double &v : t) v *= inv;
        double *M = out_poses + 16 * o;
        std::memset(M, 0, 16 * sizeof(double));
        quat_to_rotation(q, M);  // updatePoseQuat normalises the averaged quaternion
        M[3] = t[0], M[7] = t[1], M[11] = t[2], M[15] = 1.0;
        out_votes[o] = (uint32_t)std::min<uint64_t>(cluster_votes[corder[o]], 0xFFFFFFFFull);
    }
    return clusters.size();
}

size_t oracle_cv_table_size(const oracle_cv_detector *d) { return d->table_size; }

/* the whole table as a CSR over the buckets: offsets (table_size + 1), nodes (ppfInd, ascending inside a bucket) */
void oracle_cv_table_export(const oracle_cv_detector *d, uint32_t *offsets, uint32_t *nodes) {
    size_t at = 0;
    for (size_t b = 0; b < d->buckets.size(); ++b) {
        offsets[b] = (uint32_t)at;
        const size_t first = at;
        for (const auto &node : d->buckets[b]) nodes[at++] = node.second;
        std::sort(nodes + first, nodes + at);
    }
    offsets[d->buckets.size()] = (uint32_t)at;
}

/* columns of an accumulator: numAngles = floor(2 pi / angle_step), as match() sizes it (one fewer than asked for 13, 25, ...) */
int oracle_cv_num_angles(const oracle_cv_detector *d) { return (int)std::floor(2 * PI / d->angle_step); }

size_t oracle_cv_bucket(const oracle_cv_detector *d, size_t bucket, uint32_t *ppf_ind, size_t cap) {
    if (bucket >= d->buckets.size()) return 0;
    std::vector<uint32_t> v;
    for (const auto &node : d->buckets[bucket]) v.push_back(node.second);
    std::sort(v.begin(), v.end());
    for (size_t k = 0; k < v.size() && k < cap; ++k) ppf_ind[k] = v[k];
    return v.size();
}

/* the voting loop of one reference point (index into the SAMPLED scene), accumulator only */
size_t oracle_cv_accumulator(const oracle_cv_detector *d, const float *scene, size_t n, const float *edge, size_t n_edge,
                             double relative_scene_distance, size_t i, uint32_t *acc) {
    const size_t m = d->m();
    const int num_angles = (int)std::floor(2 * PI / d->angle_step);
    float r[6];
    bbox6(scene, n, r);
    const std::vector<float> sampled = sample_by_quantization(scene, n, r, (float)relative_scene_distance);
    std::vector<float> sampled_edge;
    if (edge) {
        float re[6];
        bbox6(edge, n_edge, re);
        sampled_edge = sample_by_quantization(edge, n_edge, re, (float)relative_scene_distance);
    }
    const std::vector<float> &second = edge ? sampled_edge : sampled;
    const size_t ns = sampled.size() / 6, n2 = second.size() / 6;
    std::memset(acc, 0, m * (size_t)num_angles * sizeof(uint32_t));
    if (i >= ns) return 0;
    const V3 p1 = ld(&sampled[6 * i]), n1 = ld(&sampled[6 * i + 3]);
    M33 Rsg;
    V3 tsg;
    compute_transform_rt(p1, n1, Rsg, tsg);
    size_t votes = 0;
    for (size_t j = 0; j < n2; ++j) {
        if (!edge && i == j) continue;
        const V3 p2 = ld(&second[6 * j]), nrm2 = ld(&second[6 * j + 3]);
        double f[4];
        ppf_features(p1, n1, p2, nrm2, f);
        const uint32_t h = hash_ppf(f, d->angle_step, (float)d->distance_step);
        bool is_nan;
        const double alpha_scene = planar_alpha(Rsg, tsg, p2, &is_nan);
        if (is_nan) continue;
        for (const auto &node : d->buckets[h & (d->table_size - 1)]) {
            const double alpha = (double)d->alpha_m[node.second] - alpha_scene;
            const int alpha_index = (int)(num_angles * (alpha + 2 * PI) / (4 * PI));
            const size_t a = (size_t)node.first * num_angles + (size_t)alpha_index;
            if (a < m * (size_t)num_angles) acc[a]++, ++votes;
        }
    }
    return votes;
}

}  // extern "C"
