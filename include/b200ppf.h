/*
 * b200ppf.h — C ABI of libb200ppf.so, the B200 (sm_100a) Point-Pair-Feature pose engine.
 *
 * This is the drop-in boundary for the PPF path that EmilyJrxx/YOLO_PPF_Pose_Estimation
 * drives after its YOLO crop (reference include/CloudProcessing.h:222-261 train,
 * :106-121 load, :428-533 match, fed by :163-190; called from
 * src/YOLO_cropping_ppf_test.cpp:113-127).  BASELINE.json fixes the operator surface to
 * PCL's:  pcl::PPFEstimation<PointNormal,PointNormal,PPFSignature>::compute,
 * pcl::PPFHashMapSearch::setInputFeatureCloud / nearestNeighborSearch and
 * pcl::PPFRegistration::setInputSource / setInputTarget / setSearchMethod / align.
 * PCL is not vendored in the reference; "[PCL] file" citations below name the upstream
 * file each entry point replaces (restated in SURVEY.md Appendix A).  The header-only
 * PCL-shaped C++ shim over this ABI is include/pcl_compat/.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative B200PPF_ERR_*;
 *     b200ppf_last_error() gives the message.  Nothing throws or aborts across the ABI
 *     (PCL's own convention on this path is PCL_ERROR + early return).
 *   - there is NO CPU fallback: b200ppf_create fails when no sm_100 device is usable.
 *   - a context is bound to one CUDA device and owns one stream; use one context per
 *     thread / per GPU (one process per GPU under torchrun).  Calls are synchronous unless
 *     the name ends in _device (asynchronous on the context stream, results stay in HBM).
 *   - host clouds are float32 AoS with a caller-given stride: pcl::PointNormal is
 *     stride 12 / normal offset 4; the reference's N x 6 cv::Mat is stride 6 / offset 3.
 */
#ifndef B200PPF_H
#define B200PPF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200PPF_VERSION 100

#define B200PPF_OK 0
#define B200PPF_ERR_INVALID (-1)     /* bad argument */
#define B200PPF_ERR_CUDA (-2)        /* CUDA runtime / kernel failure */
#define B200PPF_ERR_NOMEM (-3)       /* device or host allocation failed */
#define B200PPF_ERR_STATE (-4)       /* object used before it is ready / size mismatch */
#define B200PPF_ERR_UNSUPPORTED (-5) /* e.g. discretisation too fine for 32-bit keys */
#define B200PPF_ERR_IO (-6)          /* table file missing, truncated, corrupt or of another version */

/* feature functor: PCL_PFH is what PCL's PPF classes execute ([PCL] features/src/pfh.cpp
 * computePairFeatures); DROST_* are the textbook tuple ([PCL] features/src/ppf.cpp
 * computePPFPairFeature as cosines, or as angles). */
#define B200PPF_FEATURE_PCL_PFH 0
#define B200PPF_FEATURE_DROST_COS 1
#define B200PPF_FEATURE_DROST_ANGLE 2
/* alpha binning of the voting loop: A = PCL >= 1.12, B = PCL 1.8-1.11 legacy */
#define B200PPF_ALPHA_MODE_A 0
#define B200PPF_ALPHA_MODE_B 1
/* How many alpha columns the accumulator of the voting loop has, and what becomes of a vote whose bin lies past
 * the last one.  PCL sizes the rows with 2*pi / angle_step; for its float 12 degrees that quotient is
 * 30 - 1.3e-6, so the choice of rounding decides whether the 30th bin exists:
 *   CEIL        ceil(2*pi/step) columns — current PCL; every bin the binning formula can produce has a column
 *               (default; in the one-in-a-billion case of a quotient that is an exact integer the bin equal to the
 *               column count is clamped rather than written out of bounds);
 *   FLOOR_DROP  floor(2*pi/step) columns — PCL 1.8 .. 1.11; a vote for bin 29 increments the word behind the
 *               row's std::vector storage (inside glibc's 120-byte chunk for a 116-byte row) and is never read: lost;
 *   FLOOR_CLAMP floor columns, the vote joins the last column — what round 1 of this library did; kept as a switch.
 * The rule is read when a table is built and travels with the table (and its file). */
#define B200PPF_NALPHA_CEIL 0
#define B200PPF_NALPHA_FLOOR_DROP 1
#define B200PPF_NALPHA_FLOOR_CLAMP 2

typedef struct b200ppf_ctx b200ppf_ctx;
typedef struct b200ppf_cloud b200ppf_cloud;       /* device point+normal cloud (float4 SoA) */
typedef struct b200ppf_features b200ppf_features; /* device PointCloud<PPFSignature>, N*N   */
typedef struct b200ppf_table b200ppf_table;       /* device CSR table = PPFHashMapSearch    */

/* pcl::PPFSignature ([PCL] common/include/pcl/impl/point_types.hpp): 20 bytes */
typedef struct b200ppf_signature {
    float f1, f2, f3, f4, alpha_m;
} b200ppf_signature;

/* PPFRegistration::PoseWithVotes plus the peak it came from: 64 bytes, the record the
 * voting kernel emits per scene reference point and the unit of the multi-GPU all-gather */
typedef struct b200ppf_hypothesis {
    float pose[12]; /* 3x4 row-major, model -> scene */
    uint32_t votes;
    uint32_t model_index; /* i* */
    uint32_t alpha_bin;   /* j* */
    uint32_t scene_index; /* s_r */
} b200ppf_hypothesis;

typedef struct b200ppf_table_info {
    uint64_t n_model;     /* model points */
    uint64_t n_entries;   /* valid ordered pairs stored */
    uint64_t n_keys;      /* distinct keys (non-empty buckets of the multimap) */
    uint64_t key_space;   /* dense packed-key range per slice */
    uint32_t n_slices;    /* model-row slices (accumulator tiles), 1 for small models */
    uint32_t slice_rows;  /* model rows per slice */
    uint32_t n_alpha;     /* accumulator columns: ceil or floor of 2*pi/angle_step (nalpha_rule) */
    uint32_t key_bits;    /* bits sorted */
    int32_t lo[4];        /* lower bound of each quantised component */
    int32_t size[4];      /* extent of each quantised component */
    float angle_step, dist_step;
    float max_dist;       /* getModelDiameter() */
    uint32_t phase_cells; /* alpha_m phase cells per bucket (1: buckets are not subdivided) */
    uint32_t nalpha_rule; /* B200PPF_NALPHA_* the table was built under */
    uint32_t reserved;
    uint64_t n_merged;    /* words of the merged-vote array the voting kernel walks (<= n_entries; 0: no phase cells) */
} b200ppf_table_info;

/* per-stage device times of the last call on this context, milliseconds (CUDA events) */
typedef struct b200ppf_timings {
    float upload_ms, features_ms, keys_ms, sort_ms, csr_ms, grid_ms, vote_ms, pose_ms, cluster_ms,
        transform_ms, icp_ms, prep_ms;
} b200ppf_timings;

/* ---- context ---------------------------------------------------------------------------- */
int b200ppf_create(int device, b200ppf_ctx **out);
void b200ppf_destroy(b200ppf_ctx *ctx);
const char *b200ppf_last_error(const b200ppf_ctx *ctx); /* ctx may be NULL: global message */
int b200ppf_version(void);
int b200ppf_set_feature_mode(b200ppf_ctx *ctx, int feature_mode);
int b200ppf_set_alpha_mode(b200ppf_ctx *ctx, int alpha_mode);
int b200ppf_set_nalpha_rule(b200ppf_ctx *ctx, int nalpha_rule); /* B200PPF_NALPHA_*; default CEIL */
int b200ppf_get_device(const b200ppf_ctx *ctx);
void *b200ppf_get_stream(const b200ppf_ctx *ctx); /* cudaStream_t */
int b200ppf_synchronize(b200ppf_ctx *ctx);
int b200ppf_get_timings(b200ppf_ctx *ctx, b200ppf_timings *out);
/* number of kernels this context has launched so far */
uint64_t b200ppf_launch_count(const b200ppf_ctx *ctx);

/* ---- clouds: replaces setInputCloud/setInputNormals/setInputSource/setInputTarget ------- */
/* host may be pageable or pinned; points with a NaN coordinate or normal are dropped
 * (SURVEY.md A.8 rule 5) and *out keeps the surviving order. */
int b200ppf_cloud_upload(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride_floats,
                         size_t normal_offset_floats, b200ppf_cloud **out);
size_t b200ppf_cloud_size(const b200ppf_cloud *cloud);
void b200ppf_cloud_free(b200ppf_cloud *cloud);

/* ---- K1: [PCL] features/include/pcl/features/impl/ppf.hpp PPFEstimation::computeFeature -- */
int b200ppf_features_compute(b200ppf_ctx *ctx, const b200ppf_cloud *model, b200ppf_features **out);
int b200ppf_features_upload(b200ppf_ctx *ctx, const b200ppf_signature *host, size_t count,
                            b200ppf_features **out);
int b200ppf_features_download(b200ppf_ctx *ctx, const b200ppf_features *f, size_t first,
                              size_t count, b200ppf_signature *host);
size_t b200ppf_features_count(const b200ppf_features *f);
void b200ppf_features_free(b200ppf_features *f);

/* ---- K2: [PCL] registration/src/ppf_registration.cpp PPFHashMapSearch ------------------- */
/* setInputFeatureCloud: n = sqrt(count) model points. */
int b200ppf_table_build(b200ppf_ctx *ctx, const b200ppf_features *f, float angle_step,
                        float dist_step, b200ppf_table **out);
/* K1+K2 fused: the same table straight from the model cloud, no N*N*20-byte feature cloud */
int b200ppf_table_build_from_cloud(b200ppf_ctx *ctx, const b200ppf_cloud *model, float angle_step,
                                   float dist_step, b200ppf_table **out);
int b200ppf_table_get_info(const b200ppf_table *t, b200ppf_table_info *info);
/* nearestNeighborSearch: up to cap (i,j) pairs in canonical order (i asc, j asc);
 * *n_found receives the full bucket length. */
int b200ppf_table_query(b200ppf_ctx *ctx, const b200ppf_table *t, float f1, float f2, float f3,
                        float f4, uint64_t *pairs, size_t cap, size_t *n_found);
int b200ppf_table_query_key(b200ppf_ctx *ctx, const b200ppf_table *t, const int32_t *d4,
                            uint64_t *pairs, size_t cap, size_t *n_found);
/* the public alpha_m_[i][j] member, row-major n*n floats (NaN where the pair is invalid) */
int b200ppf_table_alpha_m(b200ppf_ctx *ctx, const b200ppf_table *t, float *host);
/* raw CSR export (parity tests, serialisation): offsets has n_slices*key_space+1 entries;
 * the three entry arrays have n_entries elements, in canonical (i, j) order inside every bucket.
 * Any pointer may be NULL. */
int b200ppf_table_export(b200ppf_ctx *ctx, const b200ppf_table *t, uint32_t *offsets,
                         uint32_t *entry_i, uint32_t *entry_j, float *entry_alpha_m);
/* a copy of a table on another context's device (device-to-device; NVLink between peers) */
int b200ppf_table_clone(b200ppf_ctx *dst, const b200ppf_table *src, b200ppf_table **out);
void b200ppf_table_free(b200ppf_table *t);

/* Trained-model persistence.  The reference never trains at run time: it deserialises a detector it
 * trained offline (include/CloudProcessing.h:242-258 detector.write(FileStorage) -> XML, :106-121
 * detector.read(fsload.root()), CLI argument 6 of src/YOLO_cropping_ppf_test.cpp:48,117).  save writes
 * the device table — parameters, bucket and phase-cell offsets, entry arrays — to one little-endian
 * binary file with a magic, a format version and a 64-bit checksum; load rebuilds it on ctx's device
 * without re-running K1/K2 and fails with B200PPF_ERR_IO on a missing, truncated, corrupt or
 * other-version file and with B200PPF_ERR_STATE when the file's feature / alpha mode differs from ctx's.
 * Beyond the checksum, load re-derives everything the voting kernel takes on trust (monotone offsets that stay
 * inside their buckets, key space = product of the key ranges, binning parameters as a function of the angle
 * step, every entry's pair index, slice, fixed-point alpha_m and hot word) and refuses a file that disagrees. */
int b200ppf_table_save(b200ppf_ctx *ctx, const b200ppf_table *t, const char *path);
int b200ppf_table_load(b200ppf_ctx *ctx, const char *path, b200ppf_table **out);

/* ---- K3: [PCL] registration/impl/ppf_registration.hpp computeTransformation, voting loop - */
/* One hypothesis per scene reference point ref_first + k*ref_step, k < ref_count (the slice a
 * rank owns when reference points are sharded across GPUs). */
int b200ppf_vote(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                 const b200ppf_cloud *scene, size_t ref_first, size_t ref_step, size_t ref_count,
                 b200ppf_hypothesis *hyps_host);
int b200ppf_vote_device(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                        const b200ppf_cloud *scene, size_t ref_first, size_t ref_step,
                        size_t ref_count, b200ppf_hypothesis *hyps_device);
/* Several GPUs (one process / context per GPU): the exchange of the 64-byte records — the one collective on
 * the path (north_star: "an NCCL allgather ... collects the pose hypotheses for clustering") — fused into the
 * vote epilogue.  The pose kernel writes record k of this rank into slot slot_first + k*slot_step of EVERY
 * buffer in peer_buffers (its own and the peers' buffers mapped through CUDA IPC, i.e. NVLink peer stores), so
 * with slot_first = rank, slot_step = world every GPU ends up with the complete array in reference order.  A
 * barrier across ranks (any: NCCL, MPI) must separate this call from the clustering that reads the buffer.
 *   hyp_buffer_create   cudaMalloc'd buffer of n_records + its 64-byte IPC handle (send it to the peers)
 *   hyp_buffer_open     map a peer's buffer from its handle (another process, same node)
 *   hyp_buffer_download records first .. first+count-1 to the host (after the context stream has drained)
 *   hyp_buffer_release  unmap (opened_from_handle = 1) or free (0) */
int b200ppf_hyp_buffer_create(b200ppf_ctx *ctx, size_t n_records, b200ppf_hypothesis **buffer,
                              unsigned char ipc_handle[64]);
int b200ppf_hyp_buffer_open(b200ppf_ctx *ctx, const unsigned char ipc_handle[64], b200ppf_hypothesis **buffer);
int b200ppf_hyp_buffer_download(b200ppf_ctx *ctx, const b200ppf_hypothesis *buffer, size_t first, size_t count,
                                b200ppf_hypothesis *host);
int b200ppf_hyp_buffer_release(b200ppf_ctx *ctx, b200ppf_hypothesis *buffer, int opened_from_handle);
int b200ppf_vote_scatter_device(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                                const b200ppf_cloud *scene, size_t ref_first, size_t ref_step,
                                size_t ref_count, b200ppf_hypothesis *const *peer_buffers, int n_peers,
                                size_t slot_first, size_t slot_step);
/* ---- several GPUs behind the ABI --------------------------------------------------------------------------------
 * PPFRegistration::align with the scene reference points spread over G GPUs (SURVEY.md §8e).  Every rank holds a replica
 * of the table and the scene; the persistent CTAs of all ranks draw (reference point, slice) tasks from ONE queue — a
 * counter in rank 0's memory, system-scope atomics over NVLink — so the ranks finish together whatever the scene's cost
 * distribution; every task's 8-byte peak is merged into every rank's peak array by a system-scope atomicMax, and a
 * per-step flag, raised by each rank's last CTA and awaited by a one-thread kernel on every rank's stream, separates
 * voting from pose assembly and clustering: no host synchronisation and no collective call on the path.
 *   b200ppf_group_*   one process per GPU (torchrun / MPI): create -> exchange the B200PPF_GROUP_HANDLE_BYTES blobs of
 *                     all ranks by any means (rank order) -> connect -> register per frame.  Every rank returns the
 *                     same poses (clustering is deterministic and runs on every rank's own complete copy).
 *   b200ppf_multi_*   one process driving G GPUs (what the PCL-shaped shim uses when B200PPF_DEVICES lists several):
 *                     train / load and scene upload replicate, register runs the G ranks from the calling thread. */
typedef struct b200ppf_group b200ppf_group;
typedef struct b200ppf_multi b200ppf_multi;
#define B200PPF_GROUP_HANDLE_BYTES 192
int b200ppf_group_create(b200ppf_ctx *ctx, int rank, int world, size_t n_records, b200ppf_group **out,
                         unsigned char handles[B200PPF_GROUP_HANDLE_BYTES]);
int b200ppf_group_connect(b200ppf_group *group, const unsigned char *all_handles /* world * B200PPF_GROUP_HANDLE_BYTES */);
void b200ppf_group_destroy(b200ppf_group *group);
/* vote: asynchronous; cluster: waits on the device for all ranks' flags, assembles the poses of all reference points
 * from this rank's complete peak array, returns this rank's clustered poses (model / table / scene as given to vote) */
int b200ppf_group_vote(b200ppf_group *group, const b200ppf_cloud *model, const b200ppf_table *table,
                       const b200ppf_cloud *scene, size_t ref_rate);
int b200ppf_group_cluster(b200ppf_group *group, const b200ppf_cloud *model, const b200ppf_table *table,
                          const b200ppf_cloud *scene, size_t ref_rate, float pos_thr, float rot_thr, float *final16,
                          float *poses16, uint32_t *votes, size_t *n_out);
int b200ppf_group_register(b200ppf_group *group, const b200ppf_cloud *model, const b200ppf_table *table,
                           const b200ppf_cloud *scene, size_t ref_rate, float pos_thr, float rot_thr, float *final16,
                           float *poses16, uint32_t *votes, size_t *n_out);
/* device pointer to the complete record set of the last step (reference order) */
const b200ppf_hypothesis *b200ppf_group_records(const b200ppf_group *group);

int b200ppf_multi_create(const int *devices, int n_devices, b200ppf_multi **out);
void b200ppf_multi_destroy(b200ppf_multi *multi);
int b200ppf_multi_size(const b200ppf_multi *multi);
b200ppf_ctx *b200ppf_multi_context(b200ppf_multi *multi, int g);
const b200ppf_table *b200ppf_multi_table(const b200ppf_multi *multi, int g);
const char *b200ppf_multi_last_error(const b200ppf_multi *multi);
int b200ppf_multi_train(b200ppf_multi *multi, const float *model_host, size_t n, size_t stride_floats,
                        size_t normal_offset_floats, float angle_step, float dist_step);
int b200ppf_multi_adopt(b200ppf_multi *multi, const float *model_host, size_t n, size_t stride_floats,
                        size_t normal_offset_floats, const b200ppf_table *table);
int b200ppf_multi_load(b200ppf_multi *multi, const float *model_host, size_t n, size_t stride_floats,
                       size_t normal_offset_floats, const char *table_path);
int b200ppf_multi_scene(b200ppf_multi *multi, const float *scene_host, size_t n, size_t stride_floats,
                        size_t normal_offset_floats);
int b200ppf_multi_register(b200ppf_multi *multi, size_t ref_rate, float pos_thr, float rot_thr, float *final16,
                           float *poses16, uint32_t *votes, size_t *n_out);

/* counters of the last vote on this context: pairs examined, pairs in radius (the metric's
 * "pairs voted"), non-empty bucket lookups, votes cast */
int b200ppf_vote_stats(b200ppf_ctx *ctx, uint64_t *stats4);
/* parity hooks: what the device computed for one reference point */
int b200ppf_vote_debug_pairs(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene,
                             size_t s_r, uint8_t *in_radius, int32_t *d4, float *alpha_s);
int b200ppf_vote_debug_accumulator(b200ppf_ctx *ctx, const b200ppf_table *t,
                                   const b200ppf_cloud *scene, size_t s_r, uint32_t *acc);

/* parity hook for the voting loop's alpha binning: evaluates the hot-loop form (fast) and the
 * literal PCL form (exact) for n (alpha_m, alpha_s) pairs — on the device when ctx is given, with
 * the host build of the same inline functions when ctx is NULL. */
int b200ppf_debug_alpha_bins(b200ppf_ctx *ctx, float angle_step, int alpha_mode, int nalpha_rule, const float *alpha_m,
                             const float *alpha_s, size_t n, uint32_t *fast, uint32_t *exact);

/* Parity hooks of the sorted-key primitives every stage that sorts keys shares (radix sort, bucket offsets, flag scan,
 * row scan, run heads).  They exist for the parity tests only; no product entry point routes through them.  Each one
 * mirrors its primitive's arguments with host arrays: every array is copied to the device whole, the words past the
 * documented range (up to *_cap) included, the primitive runs once on the context stream, every array it may write is
 * copied back whole, and the call waits for the stream.  The primitive's kernels are the only launches the call adds to
 * b200ppf_launch_count.  B200PPF_ERR_INVALID, before the context is looked at: a NULL array the call needs, a cap below
 * the range the primitive writes.
 *   radix_sort     keys / v0 / v1 ascending by key, stable; a NULL pair (v0, v0_alt) or (v1, v1_alt) is no such payload,
 *                  half a pair is an error.  max_key: the largest key (the pass count follows from its bits, one to four
 *                  8-bit passes); v0_iota: v0 is the identity 0..n-1 on entry and its contents are never read.
 *                  *result_in_alt = 1 when the sorted data is in the *_alt arrays.  n < 2^32 - 4096.
 *   lower_bounds   offsets[k] = first i < len with sorted[i] >= k << shift, k = 0 .. n_keys (shift < 32); len is n for
 *                  dev_len < 0, else dev_len (<= n), read from device memory as a compacted list's length is.
 *   flag_scan      rank[k] = the flags equal to 1 before k, k < n; *total = all of them: from the device total of
 *                  flag_scan (*total's value on entry is its initial device value) or, host_total != 0, flag_scan_host.
 *   scan_rows      each of the n_rows >= 1 rows of data (row_len words, row-major) in place to its exclusive scan,
 *                  totals[r] its sum.
 *   run_heads      head[i] = 1 where a run of equal keys of sorted[0 .. n) starts, else 0. */
int b200ppf_debug_radix_sort(b200ppf_ctx *ctx, uint32_t *keys, uint32_t *keys_alt, uint32_t *v0, uint32_t *v0_alt, uint32_t *v1,
                             uint32_t *v1_alt, size_t n, uint64_t max_key, int v0_iota, int *result_in_alt);
int b200ppf_debug_lower_bounds(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, int64_t dev_len, uint32_t n_keys,
                               uint32_t shift, uint32_t *offsets, size_t offsets_cap);
int b200ppf_debug_flag_scan(b200ppf_ctx *ctx, const uint32_t *flags, uint32_t n, uint32_t *rank, size_t rank_cap, int host_total,
                            uint32_t *total);
int b200ppf_debug_scan_rows(b200ppf_ctx *ctx, uint32_t *data, uint32_t n_rows, uint32_t row_len, size_t data_cap, uint32_t *totals,
                            size_t totals_cap);
int b200ppf_debug_run_heads(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, uint32_t *head, size_t head_cap);

/* roofline denominator the HBM/tensor peaks do not cover: measured rate of shared-memory reductions
 * (one per vote).  pattern 0 = conflict-free, 1 = random words (address from an LCG), 2 = one word,
 * 3 / 4 = exactly 2 / 4 lanes per bank; 5 / 6 / 7 = the voting loop's own shape (one coalesced 4-byte gather
 * from an L2-resident table per reduction, eight in flight per lane) with conflict-free / random / 2-per-bank
 * addresses.  +8 selects the 1024-thread x 1 CTA per SM shape instead of 512 x 2. */
int b200ppf_microbench_atoms(b200ppf_ctx *ctx, int pattern, double *atoms_per_sec);

/* ---- K4: [PCL] ppf_registration.hpp clusterPoses / posesWithinErrorBounds ---------------- */
int b200ppf_cluster(b200ppf_ctx *ctx, const b200ppf_hypothesis *hyps_host, size_t n, float pos_thr,
                    float rot_thr, float *poses16, uint32_t *votes, size_t *n_out);
int b200ppf_cluster_device(b200ppf_ctx *ctx, const b200ppf_hypothesis *hyps_device, size_t n,
                           float pos_thr, float rot_thr, float *poses16, uint32_t *votes,
                           size_t *n_out);
/* cluster creation index of every hypothesis of the last cluster call (input order) */
int b200ppf_cluster_assignment(b200ppf_ctx *ctx, uint32_t *assignment, size_t n,
                               size_t *n_clusters);

/* ---- K5: tail of computeTransformation, pcl::transformPointCloud (xyz only) -------------- */
int b200ppf_transform(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, const float *pose16,
                      float *out_host, size_t out_stride_floats);

/* ---- K6 ("next" row): ICP refinement of the best poses ---------------------------------------
 * The step the reference runs right after matching: include/CloudProcessing.h:465-470 / :518-523,
 *     ICP icp(100, 0.005f, 2.5f, 8);  icp.registerModelToScene(models[id], pc_scene, resultsSub);
 * (opencv_contrib surface_matching/src/icp.cpp: multi-resolution "picky" point-to-plane ICP).
 * poses16: n_poses row-major 4x4 doubles, model -> scene, refined in place (Pose3D::appendPose);
 * residuals (n_poses) and iterations (total over poses) may be NULL.  params NULL = the reference's
 * (100, 0.005, 2.5, 8).  All poses are refined concurrently, one thread-block cluster each, in a single launch.
 * The point-to-plane system is solved as upstream's cv::solve(DECOMP_SVD) solves it — least squares of minimum norm —
 * so levels that keep fewer correspondences than unknowns (a 543-point model has 4 samples at level 7) move the pose
 * only where the data constrain it. */
typedef struct b200ppf_icp_params {
    int max_iterations;    /* ICP(iterations = 100, ...) */
    float tolerance;       /* 0.005 */
    float rejection_scale; /* 2.5; <= 0 disables the robust rejection */
    int num_levels;        /* 8 */
} b200ppf_icp_params;
int b200ppf_icp_refine(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_cloud *scene,
                       const b200ppf_icp_params *params, double *poses16, size_t n_poses,
                       double *residuals, uint64_t *iterations);
/* Several ICP problems in one call: job k refines jobs[k].n_poses poses of jobs[k].model against jobs[k].scene, exactly
 * as b200ppf_icp_refine would (the same bits).  A pose's cluster size depends on its model only (one CTA per 1 024 model
 * points, at most 8), so the poses are grouped by it: one launch per distinct size, at most four, and one launch when
 * every model has the same size (the objects of a frame: 5 poses each of K objects refine side by side).  params and
 * iterations (the total over all poses) as for b200ppf_icp_refine; a job of 0 poses is skipped.  The clouds must belong
 * to ctx. */
typedef struct b200ppf_icp_job {
    const b200ppf_cloud *model, *scene;
    double *poses16;   /* n_poses row-major 4x4, refined in place */
    size_t n_poses;
    double *residuals; /* n_poses, may be NULL */
} b200ppf_icp_job;
int b200ppf_icp_refine_batch(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs,
                             const b200ppf_icp_params *params, uint64_t *iterations);

/* ---- scene pre-processing ("next" row): the stages between the YOLO crop and the PPF engine -------------
 * What the reference runs on every cropped object before matching (src/YOLO_cropping_ppf_test.cpp:96-103,
 * :120-121), each a PCL operator on the host there and a device stage here, chained without leaving HBM:
 *     SceneCropping(K)             include/CloudProcessing.h:263-339  pcl::ConvexHull + pcl::CropHull
 *     Subsampling(leaf)            include/CloudProcessing.h:359-377  pcl::VoxelGrid<PointXYZ>
 *     OutlierProcessing(50, thr)   include/CloudProcessing.h:340-358  pcl::StatisticalOutlierRemoval<PointXYZ>
 *     NormalEstimation(30)         include/CloudProcessing.h:378-401  pcl::NormalEstimationOMP<PointXYZ, Normal>
 *     EdgeExtraction(0.03)         include/CloudProcessing.h:402-427  curvature > threshold
 *     PointCloudXYZNormalToMat     include/CloudProcessing.h:163-190  normals re-normalised, N x 6 rows
 * A cloud made by upload_xyz has zero normals; normal_estimation fills normals and curvature in place.
 * Results that PCL leaves unspecified are fixed as: a voxel's points are summed in input order; neighbours at
 * equal distance are ordered by index. */
int b200ppf_cloud_upload_xyz(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride_floats, b200ppf_cloud **out);
/* rows of stride_floats floats: x y z at 0..2, the normal at normal_offset_floats and the curvature at
 * curvature_offset_floats (each >= 3, or 0 to leave it out); every other float of a row is written as 0 */
int b200ppf_cloud_download(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, float *host, size_t stride_floats,
                           size_t normal_offset_floats, size_t curvature_offset_floats);
/* SceneCropping, per YOLO box (include/CloudProcessing.h:263-339): the box grown by 30 pixels and clamped, the mean
 * depth at its four corners, the four corner rays at that depth (include/Camera.h:50-61 back_projection_bbox) pushed
 * 0.15 m further -> corners12 = left_top, left_bot, right_top, right_bot.  Host arithmetic on four pixels of the
 * row-major float depth image (metres); no context needed. */
int b200ppf_frustum_corners(const float *depth, int rows, int cols, int box_x, int box_y, int box_w, int box_h, double fx,
                            double fy, double ppx, double ppy, float corners12[12]);
/* The crop itself: the reference builds pcl::ConvexHull of {the four corners, the origin} and keeps what
 * pcl::CropHull (dim 3) finds inside — the points of the pyramid, here five half-space tests per point in double
 * (a point within rounding of a face may fall either way, as with PCL's ray casting).  The corners must be
 * coplanar (the reference's share one z).  Kept points keep their order and normals; kept_indices_host (capacity
 * n) is optional. */
int b200ppf_crop_pyramid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float corners12[12], b200ppf_cloud **out,
                         uint32_t *kept_indices_host);
/* SceneCropping for every box of a frame at once: out[b] is what b200ppf_crop_pyramid(in, corners12 + 12 * b) makes, bit
 * for bit (the same points in the same order, the same bounding box).  A point inside several pyramids goes to each of
 * them; a box that keeps nothing gives an empty cloud.  1 <= n_boxes <= 64.  One pass over the frame and a launch count
 * that does not grow with n_boxes.  Every box is checked before anything runs: a bad one fails the whole call, with
 * the code b200ppf_crop_pyramid gives it and its index in the message, and nothing is allocated. */
int b200ppf_crop_pyramids(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, size_t n_boxes,
                          b200ppf_cloud **out);
/* [PCL] filters/impl/voxel_grid.hpp VoxelGrid::applyFilter: one centroid per occupied leaf, in ascending leaf
 * index (x fastest).  A leaf so small that the index overflows an int returns a copy of the input, as PCL does
 * (b200ppf_last_error then holds PCL's warning). */
int b200ppf_voxel_grid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float leaf3[3], b200ppf_cloud **out);
/* parity hook: the k nearest neighbours of every point (itself included), rows of k sorted by (squared
 * distance, index); idx_host / d2_host are n*k, either may be NULL.  k <= min(n, 128). */
int b200ppf_knn(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, int k, uint32_t *idx_host, float *d2_host);
/* [PCL] filters/impl/statistical_outlier_removal.hpp applyFilterIndices (negative = false): drops the points
 * whose mean distance to their mean_k nearest neighbours exceeds mean + stddev_mul * stddev over the cloud.
 * Needs n > mean_k (PCL reads past its neighbour list otherwise) and mean_k <= 127.  Optional outputs: the kept
 * indices (capacity n), the per-point mean distances (n) and the threshold. */
int b200ppf_statistical_outlier_removal(b200ppf_ctx *ctx, const b200ppf_cloud *in, int mean_k, double stddev_mul,
                                        b200ppf_cloud **out, uint32_t *kept_indices_host, float *distances_host,
                                        double *threshold);
/* [PCL] features/impl/normal_3d_omp.hpp computeFeature with setKSearch(k): normal = eigenvector of the smallest
 * eigenvalue of the neighbourhood covariance (pcl::eigen33), flipped towards viewpoint3 (NULL = the origin,
 * PCL's default), curvature = lambda_0 / trace.  covariance_mode 0 = PCL >= 1.12 (sums shifted by the first
 * neighbour), 1 = PCL 1.8-1.11 (raw sums).  k <= 128. */
#define B200PPF_COVARIANCE_SHIFTED 0
#define B200PPF_COVARIANCE_RAW 1
int b200ppf_normal_estimation(b200ppf_ctx *ctx, b200ppf_cloud *cloud, int k, const float viewpoint3[3],
                              int covariance_mode);
/* EdgeExtraction: the points whose curvature exceeds the threshold, in order, with their normals */
int b200ppf_curvature_edges(b200ppf_ctx *ctx, const b200ppf_cloud *in, float curvature_threshold, b200ppf_cloud **out);
/* PointCloudXYZNormalToMat: n /= (float)sqrt(nx*nx + ny*ny + nz*nz) where that length exceeds 1e-5, in place */
int b200ppf_normalize_normals(b200ppf_ctx *ctx, b200ppf_cloud *cloud);

/* test hook (no context, no GPU): the neighbour query of the device kernels — the same __host__ __device__
 * function — run on the CPU over a host-built grid of cell edge cell_edge (0 = the library's choice).
 * mode 0: idx / d2 (n*k) as b200ppf_knn; 1: mean_dist (n) = mean distance to the k-1 nearest other points, as
 * the outlier removal forms it; 2: normals4 (n*4) = nx ny nz curvature, as normal_estimation forms them.
 * Like b200ppf_debug_alpha_bins with a NULL context this exists for the parity tests only; no product entry
 * point routes through it. */
int b200ppf_debug_knn_host(const float *xyz, size_t n, size_t stride_floats, int k, int mode, float cell_edge,
                           const float viewpoint3[3], int covariance_mode, uint32_t *idx, float *d2, float *mean_dist,
                           float *normals4);

/* ---- PPFRegistration::align in one call: vote + cluster, final16 = results.front() -------- */
int b200ppf_register(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                     const b200ppf_cloud *scene, size_t ref_rate, float pos_thr, float rot_thr,
                     float *final16, float *poses16, uint32_t *votes, size_t *n_out);

/* ---- YOLO boxes, start to finish: the match calls ---------------------------------------------------------------------
 * What src/YOLO_cropping_ppf_test.cpp:91-122 does per detected object, on device handles, nothing copied to the host
 * between the stages.  Every match call, per-object or frame, with either engine, runs this one chain:
 *   SceneCropping of all the call's boxes in one pass (b200ppf_crop_pyramids), then per box, one box after another:
 *   Subsampling(leaf) -> OutlierProcessing(mean_k, stddev_mul) -> NormalEstimation(normal_k) ->
 *   EdgeExtraction(edge_curvature) -> PointCloudXYZNormalToMat -> the engine's match; then ONE b200ppf_icp_refine_batch
 *   over the best poses of every box that got a pose (include/CloudProcessing.h:508-530: top N, ICP(100, 0.005, 2.5, 8))
 *   -> resultsSub[0] per box.
 * The engines: b200ppf_match_object / b200ppf_match_frame match with PPFRegistration::align (PCL arithmetic, the
 * thresholds below); b200cv_match_object / b200cv_match_frame with cv::ppf_match_3d::PPF3DDetector, the engine the
 * reference calls (below).  scene is the full frame (xyz; b200ppf_cloud_upload_xyz), corners12 comes from
 * b200ppf_frustum_corners (12 floats per box), model / table from the training calls above.
 * A per-object call is the frame call (below) on one box, plus object_out / edges_out (optional): when the box succeeds
 * they receive the pre-processed object cloud and its curvature edges (NULL if none were extracted); free them with
 * b200ppf_cloud_free.  It returns the frame call's own error if there is one, else the box's status.  Its result is the
 * frame's results[0]; crop_ms, icp_ms and total_wall_ms are then the box's own.
 * The edges are extracted only when edge_curvature > 0, and then: by a frame call always; by b200ppf_match_object when
 * edges_out asks for them; by b200cv_match_object under use_edges or when edges_out asks for them.
 * What the PCL engine is NOT: the reference's Matching_S2B feeds the edge cloud to its detector's match_S2B; the PCL
 * matching votes on the object cloud only, so it never needs the edges.  Its pose is PPFRegistration::align's, not
 * PPF3DDetector's.  PCL's clusterPoses returns at most three poses, so at most three are refined (icp_poses > 3 is
 * clamped); sor_stddev_mul has no default in the reference (argv[5]): 1.0 is this library's. */
typedef struct b200ppf_object_params {
    float leaf;             /* Subsampling leaf size (CLI argument 4 of the reference) */
    int sor_mean_k;         /* 50 */
    double sor_stddev_mul;  /* CLI argument 5 */
    int normal_k;           /* 30 */
    float edge_curvature;   /* 0.03; <= 0 skips the edge extraction */
    uint32_t ref_rate;      /* every ref_rate-th object point votes: 20 = the reference's 1 / 0.05 */
    float pos_thr, rot_thr; /* pose clustering: PCL's 0.01 m, 20 degrees (radians here) */
    int icp_poses;          /* best poses refined by ICP: 5 in the reference; clamped to the 3 that PCL's clustering returns; 0 = none */
    b200ppf_icp_params icp; /* (100, 0.005, 2.5, 8) */
} b200ppf_object_params;
typedef struct b200ppf_object_result {
    double pose[16];  /* row-major 4x4, model -> scene: the best pose, after ICP when icp_poses > 0 */
    double residual;  /* its ICP residual (0 without ICP) */
    uint32_t votes;   /* votes of its pose cluster */
    uint32_t n_poses; /* pose clusters the matching returned */
    uint32_t n_cropped, n_sampled, n_filtered, n_edges; /* object size after the crop, voxel grid, outlier removal; edges */
    /* device time per stage (CUDA events) and host wall time of the whole call, milliseconds */
    float crop_ms, voxel_ms, outlier_ms, normals_ms, edges_ms, match_ms, icp_ms, total_wall_ms;
} b200ppf_object_result;
void b200ppf_object_params_default(b200ppf_object_params *params);
int b200ppf_match_object(b200ppf_ctx *ctx, const b200ppf_cloud *scene, const float corners12[12],
                         const b200ppf_cloud *model, const b200ppf_table *table, const b200ppf_object_params *params,
                         b200ppf_object_result *result, b200ppf_cloud **object_out, b200ppf_cloud **edges_out);

/* ---- the engine the reference actually calls: cv::ppf_match_3d::PPF3DDetector ---------------------------------------
 * include/CloudProcessing.h:205,217,234 construct PPF3DDetector(relativeSamplingStep, relativeDistanceStep), :236 trains it
 * (trainModel), :442 matches (match(scene, results, relativeSceneSampleStep, relativeSceneDistance)) and :495 calls the
 * fork-only match_S2B(scene, edge, results, ...).  opencv_contrib surface_matching (ppf_match_3d.cpp, ppf_helpers.cpp,
 * c_utils.hpp, hash_murmur86.hpp, t_hash_int.cpp, pose_3d.cpp) restated for the device in csrc/k7_cvppf.cu; the
 * OpenCV-shaped class over these entry points is include/opencv_compat/opencv2/surface_matching/ppf_match_3d.hpp.
 * Clouds are host rows of stride_floats >= 6 floats [x y z nx ny nz] (the reference's N x 6 CV_32F cv::Mat).
 * match_S2B: the fork's source is not available; by its name (surface-to-boundary pairs, Choi et al.) and its inputs (the
 * object cloud and the curvature-edge cloud EdgeExtraction makes of it) it is taken to be match() with the reference
 * points drawn from the sampled surface cloud and paired with the sampled EDGE cloud instead of the surface cloud. */
typedef struct b200cv_detector b200cv_detector;
/* cv::ppf_match_3d::Pose3D: pose, alpha, residual, modelIndex, numVotes, angle, t, q (w x y z) + the peak it came from */
typedef struct b200cv_pose {
    double pose[16]; /* row-major 4x4, model -> scene */
    double alpha, residual, angle;
    double t[3];
    double q[4];
    uint32_t model_index, num_votes;
    uint32_t alpha_index, reference_index;
} b200cv_pose;
typedef struct b200cv_info {
    uint64_t n_sampled;  /* model points after samplePCByQuantization */
    uint64_t table_size; /* buckets of the hash table: the power of two >= n_sampled^2 (>= 16) */
    uint64_t n_nodes;    /* n_sampled * (n_sampled - 1) */
    uint64_t n_scene_sampled, n_second_sampled; /* last match: sampled scene points, points they were paired with */
    double angle_step, distance_step;
    double position_threshold, rotation_threshold;
    int32_t num_angles;
    int32_t reserved;
} b200cv_info;
int b200cv_detector_create(b200ppf_ctx *ctx, double relative_sampling_step, double relative_distance_step,
                           double num_angles, b200cv_detector **out);
void b200cv_detector_free(b200cv_detector *d);
/* setSearchParams(positionThreshold, rotationThreshold): a negative value keeps the default */
int b200cv_detector_set_search_params(b200cv_detector *d, double position_threshold, double rotation_threshold);
/* trainModel.  The model must sample to 2 .. 46340 points: the table's m^2 pair slots and its power-of-two bucket count
 * are 32-bit, so m^2 <= 2^31.  A larger sampled model is refused with B200PPF_ERR_UNSUPPORTED right after sampling,
 * before any table memory is allocated, and leaves the detector untrained (it can be trained again). */
int b200cv_detector_train(b200cv_detector *d, const float *model, size_t n, size_t stride_floats);
int b200cv_detector_get_info(const b200cv_detector *d, b200cv_info *info);
int b200cv_detector_model_points(const b200cv_detector *d, float *out6);  /* n_sampled x 6 */
int b200cv_detector_scene_points(const b200cv_detector *d, float *out6);  /* last match: n_scene_sampled x 6 */
/* results: the pose clusters, best first (at most cap are written, *n_results receives the number of clusters) */
int b200cv_detector_match(b200cv_detector *d, const float *scene, size_t n, size_t stride_floats,
                          double relative_scene_sample_step, double relative_scene_distance, b200cv_pose *results,
                          size_t cap, size_t *n_results);
int b200cv_detector_match_s2b(b200cv_detector *d, const float *scene, size_t n, size_t stride_floats, const float *edge,
                              size_t n_edge, size_t edge_stride_floats, double relative_scene_sample_step,
                              double relative_scene_distance, b200cv_pose *results, size_t cap, size_t *n_results);
/* match / match_S2B on device clouds of the detector's context (b200ppf_cloud: the normals, not the curvature, are read):
 * edge == NULL -> match, else match_S2B.  The same results, bit for bit, as the host calls on the clouds'
 * b200ppf_cloud_download rows; the last-match queries below report this call. */
int b200cv_detector_match_cloud(b200cv_detector *d, const b200ppf_cloud *scene, const b200ppf_cloud *edge,
                                double relative_scene_sample_step, double relative_scene_distance, b200cv_pose *results,
                                size_t cap, size_t *n_results);
/* parity hooks: one bucket of the table (ppfInd = i * n_sampled + j, ascending), the whole table, the per-reference poses
 * of the last match before clustering, the accumulator (n_sampled * num_angles words) of one reference point */
int b200cv_detector_bucket(b200cv_detector *d, size_t bucket, uint32_t *ppf_ind, size_t cap, size_t *n_found);
int b200cv_detector_table_export(b200cv_detector *d, uint32_t *offsets, uint32_t *nodes, float *alpha_m);
int b200cv_detector_raw_poses(const b200cv_detector *d, b200cv_pose *raw, size_t cap, size_t *n);
int b200cv_detector_debug_accumulator(b200cv_detector *d, const float *scene, size_t n, size_t stride_floats,
                                      const float *edge, size_t n_edge, size_t edge_stride_floats,
                                      double relative_scene_sample_step, double relative_scene_distance, size_t reference,
                                      uint32_t *acc);

/* ---- the match calls with the engine the reference calls -------------------------------------------------------------
 * The chain of b200ppf_match_object above, with the match step Matching_S2B (include/CloudProcessing.h:481-495:
 * match_S2B(object, edges, results, 0.05, 0.05); use_edges = 0 runs Matching, :428-442, whose step is 1/14) and ICP of
 * the first icp_poses pose clusters against model (the reference's models[id]: the full model, not the detector's
 * sampled one; :508-530).  d is trained (b200cv_detector_train); scene and model are clouds of d's context.  result:
 * pose / residual / votes of resultsSub[0], the number of pose clusters (n_poses), the stage sizes and device times;
 * match_ms covers scene sampling, voting and clustering.  Errors: an untrained detector, an empty crop or edge cloud and
 * a match without a pose cluster are B200PPF_ERR_STATE (the reference exits there, :502-507); clouds of another
 * context, and use_edges with edge_curvature <= 0, are B200PPF_ERR_INVALID. */
typedef struct b200cv_object_params {
    float leaf;                         /* Subsampling leaf size (CLI argument 4 of the reference) */
    int sor_mean_k;                     /* 50 */
    double sor_stddev_mul;              /* CLI argument 5; 1.0 here */
    int normal_k;                       /* 30 */
    float edge_curvature;               /* 0.03 */
    int use_edges;                      /* 1: Matching_S2B (default, what main() calls), 0: Matching */
    double relative_scene_sample_step;  /* 0.05 (:481); Matching uses 1/14 (:428) */
    double relative_scene_distance;     /* 0.05 */
    int icp_poses;                      /* 5 (:508), clamped to the clusters returned; 0 = no ICP */
    b200ppf_icp_params icp;             /* (100, 0.005, 2.5, 8) */
} b200cv_object_params;
void b200cv_object_params_default(b200cv_object_params *params);
int b200cv_match_object(b200cv_detector *d, const b200ppf_cloud *scene, const float corners12[12], const b200ppf_cloud *model,
                        const b200cv_object_params *params, b200ppf_object_result *result, b200ppf_cloud **object_out,
                        b200ppf_cloud **edges_out);

/* ---- every YOLO box of a frame in one call ---------------------------------------------------------------------------
 * The chain above for the whole list of boxes CloudProcessor(scene, depth, boxes, ids, idx) holds (corners12: n_boxes x
 * 12 floats).  Box b uses detectors[b] / tables[b] and models[b] (the class of its YOLO id); one detector, table or model
 * may serve several boxes.
 *   results[b]  pose, residual, votes, n_poses and the stage sizes are those b200cv_match_object / b200ppf_match_object
 *               give for that box, bit for bit (n_edges too when they extract the edges).  crop_ms, icp_ms and
 *               total_wall_ms are the frame's: the one crop, the one ICP and the whole call, repeated in every result; the
 *               other times are the box's own.
 *   status[b]   0, or the code the per-object call would have returned for that box: B200PPF_ERR_STATE for an empty crop,
 *               an object without edge points under use_edges, or a match without a pose cluster.  The reference exits
 *               there; a failed box here leaves the others to finish.  b200ppf_last_error names the last failure.
 * The return value is for the call itself: B200PPF_ERR_INVALID for NULL arrays, n_boxes of 0 or over 64, a cloud,
 * detector or table of another context and use_edges with edge_curvature <= 0; the crop's codes for a bad box;
 * B200PPF_ERR_STATE for an untrained detector; CUDA and memory failures.  Every intermediate cloud is freed then.
 * A detector's last-match queries (b200cv_detector_get_info, _scene_points, _raw_poses) report the last box it matched. */
int b200cv_match_frame(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                       b200cv_detector *const *detectors, const b200ppf_cloud *const *models,
                       const b200cv_object_params *params, b200ppf_object_result *results, int *status);
int b200ppf_match_frame(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                        const b200ppf_cloud *const *models, const b200ppf_table *const *tables,
                        const b200ppf_object_params *params, b200ppf_object_result *results, int *status);

/* ---- pose verification: how much of a pose's visible model surface the scene supports ---------------------------------
 * The last stage of a PPF pipeline (Drost et al. 2010; Vidal et al. 2018): every candidate pose is scored against the
 * points it should explain.  For a model cloud, a scene cloud and a pose T = [R t] (model -> scene), model point p with
 * normal n moves to p' = R p + t, n' = R n.  It is VISIBLE when n'.(-p') > 0 (the camera sits at the origin; a zero normal
 * counts as visible), and a visible point is an INLIER when its nearest scene point q (exact; the lowest index among
 * equally near points) lies within inlier_dist and q's normal has n_q.n' >= cos(normal_angle).  Per pose:
 *   inliers, visible   exact counts
 *   fit                inliers / visible (float), 0 when nothing is visible
 *   rms                root mean square distance of the inliers to their nearest scene points, 0 without inliers
 * A pose's record has the same bits alone or in any batch, and on every run. */
typedef struct b200ppf_verify_params {
    float inlier_dist;  /* metres, > 0; default 0.01 (the reference's leaf) */
    float normal_angle; /* radians, >= 0; default 30 degrees; >= pi: the distance alone decides */
} b200ppf_verify_params;
void b200ppf_verify_params_default(b200ppf_verify_params *params);
typedef struct b200ppf_pose_fit {
    uint32_t inliers, visible;
    float fit; /* inliers / visible; 0 when visible == 0 */
    float rms; /* root mean square of the inliers' distances; 0 without inliers */
} b200ppf_pose_fit;
/* Scores the poses of ICP jobs (the b200ppf_icp_refine_batch block: poses16 are read only, residuals are ignored) against
 * their scenes: fits receives the sum of the jobs' n_poses records, job-major.  params NULL = the defaults.  One grid per
 * distinct scene of the call, all built in one pass, and a launch count that does not grow with the jobs or the poses.
 * An empty scene gives 0 inliers.  B200PPF_ERR_INVALID, before anything is allocated: NULL arrays, a cloud of another
 * context, a non-finite pose, inlier_dist not finite and positive, normal_angle negative or NaN. */
int b200ppf_score_poses(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_verify_params *params,
                        b200ppf_pose_fit *fits);

/* The frame calls above, with every candidate pose of every box scored against the box's object cloud and the best one
 * returned.  The same chain runs (the crop, the per-box pre-processing and matching, the one batched ICP), then ONE
 * b200ppf_score_poses over the candidates of every box that reached the matching, each against models[b] and the box's
 * pre-processed object cloud (what the ICP registered to).  A box's candidates are the poses the call refines: its top
 * icp_poses clusters (clamped as for the unverified call), or with icp_poses = 0 its top cluster alone, unrefined.
 *   results[b]   pose, residual and votes are those of the candidate with the highest fit (ties: the lower rank); every
 *                other field is the unverified call's, bit for bit, but the frame-wide crop_ms, icp_ms and total_wall_ms
 *                (which now includes the scoring).
 *   candidates   NULL, or n_boxes x max(icp_poses, 1) records: box b's from b * max(icp_poses, 1), sorted by fit
 *                descending, ties by rank ascending.  Unused slots and the slots of a failed box are zero with
 *                rank = UINT32_MAX.  An application rejects a box's pose whose fit is too low (INTEGRATION.md §3c).
 *   status, return codes   as the unverified call's, and B200PPF_ERR_INVALID for bad verify values (NULL = the
 *                defaults), checked before the crop runs. */
typedef struct b200ppf_candidate {
    double pose[16];  /* row-major 4x4, model -> scene, after ICP when icp_poses > 0 */
    double residual;  /* its ICP residual (0 without ICP) */
    uint32_t votes;   /* votes of its pose cluster */
    uint32_t rank;    /* its position among the clusters, 0 = most voted; UINT32_MAX = unused slot */
    b200ppf_pose_fit fit;
} b200ppf_candidate;
int b200cv_match_frame_verified(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                                b200cv_detector *const *detectors, const b200ppf_cloud *const *models,
                                const b200cv_object_params *params, const b200ppf_verify_params *verify,
                                b200ppf_object_result *results, int *status, b200ppf_candidate *candidates);
int b200ppf_match_frame_verified(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                                 const b200ppf_cloud *const *models, const b200ppf_table *const *tables,
                                 const b200ppf_object_params *params, const b200ppf_verify_params *verify,
                                 b200ppf_object_result *results, int *status, b200ppf_candidate *candidates);

#ifdef __cplusplus
}
#endif
#endif /* B200PPF_H */
