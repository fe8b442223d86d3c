// ppf_common.cuh — host-side objects behind the opaque handles of include/b200ppf.h
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <array>
#include <memory>
#include <string>
#include <vector>

#include "../../include/b200ppf.h"
#include "ppf_math.cuh"

namespace b200ppf {

static_assert(sizeof(b200ppf_hypothesis) == 64, "hypothesis record is the 64-byte all-gather unit");
static_assert(sizeof(b200ppf_signature) == 20, "pcl::PPFSignature is 20 bytes");

// smallest accumulator budget we plan slices against (bytes of dynamic shared memory)
constexpr size_t kSmemPerBlockMax = 227 * 1024;
// readable words behind the last table entry (the voting kernel loads whole batches of 8 x 32)
constexpr size_t ENTRY_PAD = 256;

}  // namespace b200ppf

struct b200ppf_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    int feature_mode = B200PPF_FEATURE_PCL_PFH;
    int alpha_mode = B200PPF_ALPHA_MODE_A;
    int nalpha_rule = B200PPF_NALPHA_CEIL;
    int sm_count = 148;
    size_t smem_optin = 0;
    std::string error;
    b200ppf_timings timings{};
    uint64_t launches = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_vote[4] = {nullptr, nullptr, nullptr, nullptr};  // last vote: start / grid built / voted / poses done
    bool vote_timed = false;
    // vote scratch (grown on demand, kept across calls)
    unsigned long long *d_stats = nullptr;  // [4]
    unsigned long long *d_peaks = nullptr;  // packed (votes<<32 | ~flat) per reference
    size_t peaks_cap = 0;
    uint32_t *d_vote_queue = nullptr;  // task counter of one-GPU vote launches on folding tables
    uint32_t *d_fold = nullptr;        // fold codes and groups of folding vote launches, one slot per CTA
    size_t fold_cap = 0;
    b200ppf_hypothesis *d_hyps = nullptr;  // staging for host-output votes
    size_t hyps_cap = 0;
    // cluster scratch of the last cluster call
    uint32_t *d_assign = nullptr;  // cluster creation index per hypothesis (input order)
    size_t assign_n = 0;    // hypotheses of the last cluster call
    size_t assign_cap = 0;  // capacity of d_assign
    uint32_t n_clusters = 0;
    // grow-only pinned staging buffer of cloud uploads
    float4 *stage = nullptr;
    size_t stage_cap = 0;
};

struct b200ppf_cloud {
    b200ppf_ctx *ctx = nullptr;
    size_t n = 0;
    float4 *pos = nullptr;  // x y z 1
    float4 *nrm = nullptr;  // nx ny nz 0
    float bbox_min[3] = {0, 0, 0}, bbox_max[3] = {0, 0, 0};  // exact min / max of pos: every producer of a cloud sets them
};

struct b200ppf_depth_image {
    b200ppf_ctx *ctx = nullptr;
    int rows = 0, cols = 0;
    double K[4] = {0, 0, 0, 0};  // fx fy ppx ppy
    float *d = nullptr;          // rows x cols, row-major
};

struct b200ppf_features {
    b200ppf_ctx *ctx = nullptr;
    size_t count = 0;              // n*n
    b200ppf_signature *d = nullptr;  // row-major [i*n+j]
};

struct b200ppf_table {
    b200ppf_ctx *ctx = nullptr;
    b200ppf_table_info info{};
    b200ppf::KeyParams kp{};
    b200ppf::BinParams bp{};
    uint32_t *offsets = nullptr;      // [n_slices*key_space + 1] bucket bounds
    uint32_t *sub_offsets = nullptr;  // [(n_slices*key_space << cells_log2) + 1] phase-cell bounds (phase-sorted tables)
    uint32_t *entry_w = nullptr;      // hot word per entry (ppf_math.cuh hot_word; plain row byte offset otherwise)
    uint32_t *entry_am = nullptr;     // alpha_m as fixed-point turns (per-entry path)
    float *entry_alpha = nullptr;  // alpha_m as PCL's float (guard-band votes, alpha_m_ export)
    uint32_t *entry_idx = nullptr;  // i*n + j per entry (API queries, alpha_m_ export)
    // phase-sorted tables: the entries of a cell that share (model row, bin of alpha_m) cast the same vote for every
    // scene pair whose phase lies in another cell — they are merged into one word with a count
    uint32_t *merged_w = nullptr;      // (count << 24) | hot word, bank-ordered inside each cell
    uint32_t *msub_offsets = nullptr;  // phase-cell bounds in merged_w, same indexing as sub_offsets
    size_t n_merged = 0;
    int feature_mode = 0;
};

namespace b200ppf {

#define PPF_CUDA(ctx, expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            char _b[512];                                                                     \
            snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
                     __FILE__, __LINE__);                                                     \
            return ::b200ppf::fail_msg(ctx, _e == cudaErrorMemoryAllocation ? B200PPF_ERR_NOMEM \
                                                                             : B200PPF_ERR_CUDA, \
                                       _b);                                                   \
        }                                                                                     \
    } while (0)

int fail_msg(b200ppf_ctx *ctx, int code, const char *msg);

// launch bookkeeping: every kernel launch of the library goes through this macro
#define PPF_LAUNCH(ctx, kernel, grid, block, smem, ...)                            \
    do {                                                                           \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);           \
        (ctx)->launches++;                                                         \
        PPF_CUDA(ctx, cudaGetLastError());                                         \
    } while (0)

// stream-ordered scratch buffer, returned to the pool when it leaves scope — also on the early error returns
template <typename T>
struct StreamBuf {
    b200ppf_ctx *ctx;
    T *p = nullptr;
    explicit StreamBuf(b200ppf_ctx *c) : ctx(c) {}
    StreamBuf(const StreamBuf &) = delete;
    StreamBuf &operator=(const StreamBuf &) = delete;
    ~StreamBuf() {
        if (p) cudaFreeAsync(p, ctx->stream);
    }
    cudaError_t alloc(size_t count) { return cudaMallocAsync(&p, (count ? count : 1) * sizeof(T), ctx->stream); }
    T *release() {
        T *r = p;
        p = nullptr;
        return r;
    }
    operator T *() const { return p; }
};

// a context buffer kept across calls and grown on demand (cudaMalloc, or pinned host memory): its contents are not
// kept, and after a failed allocation the pointer is null and the capacity 0
template <typename T>
cudaError_t grow_buffer(T **p, size_t *cap, size_t count, bool pinned = false) {
    if (*cap >= count) return cudaSuccess;
    if (*p) pinned ? cudaFreeHost(*p) : cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    const cudaError_t e = pinned ? cudaMallocHost(reinterpret_cast<void **>(p), count * sizeof(T)) : cudaMalloc(p, count * sizeof(T));
    if (e == cudaSuccess) *cap = count;
    return e;
}

// makes `dev` the current device for the scope
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// a handle owned through its C ABI free function, e.g. a cloud under construction until it is released to the caller
template <auto Free>
struct FreeWith {
    template <typename T>
    void operator()(T *p) const { Free(p); }
};
using CloudPtr = std::unique_ptr<b200ppf_cloud, FreeWith<b200ppf_cloud_free>>;
using TablePtr = std::unique_ptr<b200ppf_table, FreeWith<b200ppf_table_free>>;

// a cloud of n points whose arrays are allocated (pos | nrm in one stream-ordered allocation) but not filled
int cloud_alloc(b200ppf_ctx *ctx, size_t n, CloudPtr *out);

// one device array of a table: where its pointer lives, its length in 32-bit words and the readable zero words behind it
struct TableArray {
    uint32_t **slot;
    size_t words, pad;
    bool used;  // whether the table has this array at all
};
// the eight arrays of a table in file order, as its info, kp, bp and n_merged size them
std::array<TableArray, 8> table_arrays(b200ppf_table *t);
// allocates one array from the stream-ordered pool (at least one word) and zeroes its pad
cudaError_t table_array_alloc(cudaStream_t stream, const TableArray &a);

// ---- stage entry points implemented in the k*.cu files (host functions) ----------------------
int k1_features_compute(b200ppf_ctx *ctx, const b200ppf_cloud *model, b200ppf_signature *out);
int k2_build(b200ppf_ctx *ctx, const b200ppf_features *f, const b200ppf_cloud *model, float angle_step,
             float dist_step, b200ppf_table **out);
// partitions each phase cell's unmerged entries by sub-phase block (k2_table.cu), after a build and after a load, on the
// tables whose vote kernel folds (the one that walks own cells in blocks); the vote counts do not depend on it.
// B200PPF_NO_OWN_BLOCKS (debug) leaves the entries in sorted order.
int k2_order_own_blocks(b200ppf_ctx *ctx, b200ppf_table *t);
// bits of q in the fold codes of the table's vote launches (k3_vote.cu); 0: the table does not fold
uint32_t k3_fold_qbits(const b200ppf_table *t);
int k2_query_key(b200ppf_ctx *ctx, const b200ppf_table *t, const int32_t *d4, uint64_t *pairs, size_t cap,
                 size_t *n_found);
int k2_alpha_m(b200ppf_ctx *ctx, const b200ppf_table *t, float *host);
constexpr int MAX_PEERS = 16;
// completion signal of a vote (b200ppf_group): flag word `slot` of every target's flag array := value
struct VoteSignal {
    uint32_t *flags[MAX_PEERS];
    uint32_t slot, value;
    uint32_t *done_counter;
};
int k3_vote(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t, const b200ppf_cloud *scene,
            size_t ref_first, size_t ref_step, size_t ref_count, b200ppf_hypothesis *const *targets, int n_targets,
            size_t slot_first, size_t slot_step, const VoteSignal *signal = nullptr);
int k3_group_wait(b200ppf_ctx *ctx, const uint32_t *flags, int world, uint32_t value);
// one work queue shared by the ranks of a group (k3_vote.cu): counter in rank 0's memory, peaks merged into every rank's array
struct VoteQueue {
    uint32_t *counter;
    unsigned long long *peer_peaks[MAX_PEERS];
    uint32_t *flags[MAX_PEERS];
    int n_peers;
    uint32_t slot, value;
    uint32_t *done_counter;
};
int k3_vote_shared(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t ref_rate, size_t n_ref,
                   const VoteQueue *queue);
int k3_poses(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t, const b200ppf_cloud *scene, size_t ref_rate,
             size_t n_ref, const unsigned long long *peaks, b200ppf_hypothesis *out_records);
int k3_debug_pairs(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t s_r,
                   uint8_t *in_radius, int32_t *d4, float *alpha_s);
int k3_debug_accumulator(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t s_r,
                         uint32_t *acc);
int k3_debug_alpha_bins(b200ppf_ctx *ctx, float angle_step, int alpha_mode, int nalpha_rule, const float *alpha_m,
                         const float *alpha_s, size_t n, uint32_t *fast, uint32_t *exact);
BinParams make_bin_params(float angle_step, int alpha_mode, int nalpha_rule);
uint32_t num_alpha_bins(float angle_step, int nalpha_rule);
int microbench_atoms(b200ppf_ctx *ctx, int pattern, double *atoms_per_sec);
int k4_cluster(b200ppf_ctx *ctx, const b200ppf_hypothesis *hyps_device, size_t n, float pos_thr, float rot_thr,
               float *poses16, uint32_t *votes, size_t *n_out);
int k5_transform(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, const float *pose16, float *out_host,
                 size_t out_stride_floats);
int k6_icp_refine(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_cloud *scene, int max_iterations,
                  float tolerance, float rejection_scale, int num_levels, double *poses16_host, size_t n_poses,
                  double *residuals_host, uint64_t *iterations_host);
// the same for several (model, scene, poses) jobs: one launch per distinct cluster size, every pose as the single call
int k6_icp_refine_batch(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, int max_iterations, float tolerance,
                        float rejection_scale, int num_levels, uint64_t *iterations_host);
// the pose scores of b200ppf_score_poses (verify.cu) for checked arguments: fits of the jobs' poses, job-major
int verify_score_poses(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_verify_params &params,
                       b200ppf_pose_fit *fits);
// the same jobs scored against a depth image (b200ppf_score_poses_depth) for checked arguments
int verify_score_poses_depth(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_depth_image *depth,
                             const b200ppf_verify_params &params, b200ppf_depth_fit *fits);

// the context of an OpenCV-engine detector and whether it holds a trained model (k7_cvppf.cu)
b200ppf_ctx *cv_detector_context(const b200cv_detector *d);
bool cv_detector_trained(const b200cv_detector *d);

// scene pre-processing (prep.cu): voxel grid, k nearest neighbours, outlier removal, normals, curvature edges
int prep_upload_xyz(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride, b200ppf_cloud **out);
int prep_download(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, float *host, size_t stride, size_t noff, size_t coff);
int prep_voxel_grid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *leaf3, b200ppf_cloud **out);
int prep_knn(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, int k, uint32_t *idx_host, float *d2_host);
int prep_sor(b200ppf_ctx *ctx, const b200ppf_cloud *in, int mean_k, double stddev_mul, b200ppf_cloud **out, uint32_t *kept_host,
             float *distances_host, double *threshold_out);
int prep_normals(b200ppf_ctx *ctx, b200ppf_cloud *cloud, int k, const float *viewpoint3, int cov_mode);
int prep_curvature_edges(b200ppf_ctx *ctx, const b200ppf_cloud *in, float threshold, b200ppf_cloud **out);
int prep_renormalize(b200ppf_ctx *ctx, b200ppf_cloud *cloud);
void prep_frustum_corners(const float *depth, int rows, int cols, int bx, int by, int bw, int bh, double fx, double fy,
                          double ppx, double ppy, float *corners12);
int prep_crop_pyramid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, b200ppf_cloud **out, uint32_t *kept_host);
// the crop for n_boxes pyramids in one pass over the frame; out[b] as prep_crop_pyramid(corners12 + 12 * b) makes it
int prep_crop_pyramids(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, size_t n_boxes, b200ppf_cloud **out);
// the measured pixels of a depth image back-projected, in row-major pixel order (b200ppf_cloud_from_depth)
int prep_cloud_from_depth(b200ppf_ctx *ctx, const b200ppf_depth_image *d, b200ppf_cloud **out);
int prep_debug_knn_host(const float *xyz, size_t n, size_t stride, int k, int mode, float cell_edge, const float *viewpoint3,
                        int cov_mode, uint32_t *idx, float *d2, float *mean_dist, float *normals4);

// uniform grid over the scene (scene_grid.cu): cells of edge >= search radius, x fastest
struct GridParams {
    float origin[3];
    float inv_cell;
    int dims[3];
};

__host__ __device__ __forceinline__ int grid_cell_coord(const GridParams &g, float v, int axis) {
    int c = (int)floorf((v - g.origin[axis]) * g.inv_cell);
    return c < 0 ? 0 : (c >= g.dims[axis] ? g.dims[axis] - 1 : c);
}

__host__ __device__ __forceinline__ uint32_t grid_cell_linear(const GridParams &g, int x, int y, int z) {
    return ((uint32_t)z * (uint32_t)g.dims[1] + (uint32_t)y) * (uint32_t)g.dims[0] + (uint32_t)x;
}

// one scene of a grid build: its cloud's points, where they sit in the concatenation of the build's scenes, and its cells
// (the ids cell_base .. cell_base + cells - 1 of the shared id space)
struct GridScene {
    const float4 *pos, *nrm;
    uint32_t first, n;
    uint32_t cell_base;
    GridParams gp;
};

// the cell-sorted grids of one build (scene_grid_build): scene k is scenes[k] (on the device in table when asked for), its
// cells' points are pos / nrm [cell_start[cell_base + c], cell_start[cell_base + c + 1]), in input order inside a cell,
// and w of a position holds the bits of the point's index in its own scene (no arithmetic on it)
struct SceneGrids {
    std::vector<GridScene> scenes;
    uint32_t n_cells = 0;  // over all scenes
    StreamBuf<GridScene> table;
    StreamBuf<uint32_t> cell_start;  // [n_cells + 1]
    StreamBuf<float4> pos, nrm;
    explicit SceneGrids(b200ppf_ctx *ctx) : table(ctx), cell_start(ctx), pos(ctx), nrm(ctx) {}
};

// grid geometry for a bounding box and a cell edge (host), coarsened until it has at most max_cells cells; returns the
// number of cells (0 for a non-finite box or edge)
uint32_t scene_grid_params(const float *bbox_min, const float *bbox_max, float radius, GridParams *gp, uint32_t max_cells = 1u << 22);
// the grids of n_scenes clouds in one pass: cells of edge >= cell_edge, at most cells_per_scene per scene; the sort orders
// the bits of max(key_limit, total cells).  With device_table the scene table is uploaded for the caller's kernels.  When
// no grid fits a scene (a non-finite box or edge, or no cells to give) out->n_cells is 0, nothing runs, and the error is
// the caller's to report.
int scene_grid_build(b200ppf_ctx *ctx, const b200ppf_cloud *const *clouds, uint32_t n_scenes, float cell_edge,
                     uint32_t cells_per_scene, uint32_t key_limit, bool device_table, SceneGrids *out);
// the grid of one cloud (at most 2^22 cells, the sort over its own cells, no device table); B200PPF_ERR_INVALID when no
// grid fits it
int scene_grid_build_one(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, float cell_edge, SceneGrids *out);

// ---- sorted-key primitives (sort_scan.cu), all on the context stream ----------------------------------------------
// hand-written LSD radix sort: keys ascending, stable, two 32-bit payload streams.
// All buffers are device pointers of n elements; *_alt are the ping-pong partners.  On return
// *result_in_alt tells which set holds the sorted data.  max_key = the largest key the caller can produce: the sort
// orders its bits (at least one 8-bit pass, at most four).
// v0_iota: treat v0 as the identity permutation on entry (its contents are never read).
int radix_sort_u32(b200ppf_ctx *ctx, uint32_t *keys, uint32_t *keys_alt, uint32_t *v0, uint32_t *v0_alt,
                   uint32_t *v1, uint32_t *v1_alt, size_t n, uint64_t max_key, bool v0_iota, bool *result_in_alt);
// offsets[k] (k = 0 .. n_keys) = the first i with sorted[i] >= k << shift, the target taken in 64 bits (2^32 and above
// lie past every key); the length of sorted is *n_dev when n_dev is non-null (a list whose length only the device
// knows), else n.  One launch.
int lower_bounds(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, const uint32_t *n_dev, uint32_t n_keys, uint32_t shift,
                 uint32_t *offsets);
// exclusive scan of flags: rank[k] = the flags equal to 1 before k (written for every k < n), *total_dev = all of them.
// Three launches, no host wait; n == 0 zeroes the total and launches nothing.
int flag_scan(b200ppf_ctx *ctx, const uint32_t *flags, uint32_t n, uint32_t *rank, uint32_t *total_dev);
// the same with the total on the host: one more copy and one stream wait
int flag_scan_host(b200ppf_ctx *ctx, const uint32_t *flags, uint32_t n, uint32_t *rank, uint32_t *total_host);
// in place: each of the n_rows rows of data (row_len words, row-major) becomes its exclusive scan, totals[r] its sum.
// One launch.
int scan_rows(b200ppf_ctx *ctx, uint32_t *data, uint32_t n_rows, uint32_t row_len, uint32_t *totals);
// head[i] = 1 where a run of equal keys starts in sorted[0 .. n), else 0.  One launch.
int run_heads(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, uint32_t *head);

}  // namespace b200ppf
