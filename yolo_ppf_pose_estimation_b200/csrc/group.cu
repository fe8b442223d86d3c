// group.cu — PPFRegistration::align over several GPUs behind the C ABI.
//
// Scene reference points are independent units (SURVEY.md §8e); every rank holds its own replica of the model table
// and the scene.  The ranks share ONE work queue: a counter in rank 0's memory from which the persistent CTAs of every
// GPU draw (reference point, accumulator slice) tasks with system-scope atomics over NVLink — whichever GPU is free
// takes the next task, so the ranks finish together whatever the cost distribution of the scene (a static interleaving
// left 6 % imbalance at 8 GPUs).  The ONE exchange on the path is fused into the vote kernel: a task's peak — 8 bytes,
// (votes, ~flat index) — is merged into EVERY rank's peak array by a system-scope 64-bit atomicMax (the same merge that
// combines the slices of one reference point on one GPU).  When a rank's CTAs find the queue empty, its last CTA raises
// the rank's flag in every rank's flag array; a one-thread kernel on each rank's stream waits for all G flags, then the
// rank assembles all poses from its complete peak array and clusters.  No host synchronisation, no NCCL call, no
// staging copy between voting and clustering.
//
// Two ways to form a group, same code underneath:
//   * one process per GPU (torchrun, MPI): b200ppf_group_create -> exchange the 192-byte handle blobs by any means
//     (they are CUDA IPC handles) -> b200ppf_group_connect;
//   * one process driving several GPUs: b200ppf_multi_create makes G contexts + groups and connects them with
//     plain peer pointers; b200ppf_multi_register runs the G ranks from one host thread (every call is asynchronous
//     until the final read-back of rank 0's poses).
// Two sets of peak arrays, flags and queue counters alternate between steps, so a rank may be one step ahead of a peer that
// still clusters; a set is cleared by its owner one step before it is used (see b200ppf_group_vote).
#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "ppf_common.cuh"

struct b200ppf_group {
    b200ppf_ctx *ctx = nullptr;
    int rank = 0, world = 1;
    size_t n_records = 0;                      // capacity of every buffer (reference slots)
    unsigned long long *own[2] = {nullptr, nullptr};  // peak arrays, written by every rank's vote kernel
    uint32_t *own_flags = nullptr;             // [2][MAX_PEERS] step counters written by the peers, done counter at [32],
                                               // queue counters at [40], [41] (rank 0's are the ones in use)
    b200ppf_hypothesis *records = nullptr;     // this rank's hypothesis records of the last step (local)
    unsigned long long *peer[2][b200ppf::MAX_PEERS] = {};
    uint32_t *peer_flags[b200ppf::MAX_PEERS] = {};
    bool opened[b200ppf::MAX_PEERS] = {};      // mapped through an IPC handle (to be closed), not a local pointer
    bool connected = false;
    uint32_t step = 0;
};

struct b200ppf_multi {
    std::vector<b200ppf_ctx *> ctx;
    std::vector<b200ppf_group *> group;
    std::vector<b200ppf_cloud *> model, scene;
    std::vector<b200ppf_table *> table;
    std::string error;
};

using namespace b200ppf;

namespace {

constexpr size_t FLAG_WORDS = 2 * MAX_PEERS + 16;  // two flag sets, the done counter, two queue counters
constexpr size_t DONE_WORD = 2 * MAX_PEERS, QUEUE_WORD = 2 * MAX_PEERS + 8;

int group_alloc(b200ppf_ctx *ctx, int rank, int world, size_t n_records, b200ppf_group **out) {
    if (!ctx || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "group: null argument");
    *out = nullptr;
    if (world < 1 || world > MAX_PEERS || rank < 0 || rank >= world) return fail_msg(ctx, B200PPF_ERR_INVALID, "group: 1 <= world <= 16, 0 <= rank < world");
    b200ppf_group *g = new (std::nothrow) b200ppf_group();
    if (!g) return fail_msg(ctx, B200PPF_ERR_NOMEM, "group: out of host memory");
    g->ctx = ctx;
    g->rank = rank;
    g->world = world;
    g->n_records = std::max<size_t>(1, n_records);
    DeviceGuard guard(ctx->device);
    cudaError_t e = cudaSuccess;
    for (int s = 0; s < 2 && e == cudaSuccess; ++s) {  // cudaMalloc: exportable through CUDA IPC
        e = cudaMalloc(&g->own[s], g->n_records * sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaMemset(g->own[s], 0, g->n_records * sizeof(unsigned long long));
    }
    if (e == cudaSuccess) e = cudaMalloc(&g->records, g->n_records * sizeof(b200ppf_hypothesis));
    if (e == cudaSuccess) e = cudaMalloc(&g->own_flags, FLAG_WORDS * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(g->own_flags, 0, FLAG_WORDS * sizeof(uint32_t));
    if (e != cudaSuccess) {
        b200ppf_group_destroy(g);
        return fail_msg(ctx, B200PPF_ERR_NOMEM, "group: device allocation failed");
    }
    for (int s = 0; s < 2; ++s) g->peer[s][rank] = g->own[s];
    g->peer_flags[rank] = g->own_flags;
    g->connected = world == 1;
    *out = g;
    return B200PPF_OK;
}

}  // namespace

extern "C" {

int b200ppf_group_create(b200ppf_ctx *ctx, int rank, int world, size_t n_records, b200ppf_group **out,
                         unsigned char handles[B200PPF_GROUP_HANDLE_BYTES]) {
    int rc = group_alloc(ctx, rank, world, n_records, out);
    if (rc) return rc;
    if (handles) {
        static_assert(B200PPF_GROUP_HANDLE_BYTES == 3 * sizeof(cudaIpcMemHandle_t), "three IPC handles travel as one blob");
        DeviceGuard guard(ctx->device);
        b200ppf_group *g = *out;
        void *bufs[3] = {g->own[0], g->own[1], g->own_flags};
        for (int k = 0; k < 3; ++k) {
            cudaIpcMemHandle_t h;
            if (cudaIpcGetMemHandle(&h, bufs[k]) != cudaSuccess) {
                cudaGetLastError();
                b200ppf_group_destroy(g);
                *out = nullptr;
                return fail_msg(ctx, B200PPF_ERR_CUDA, "group: cudaIpcGetMemHandle failed");
            }
            memcpy(handles + k * sizeof(h), &h, sizeof(h));
        }
    }
    return B200PPF_OK;
}

int b200ppf_group_connect(b200ppf_group *g, const unsigned char *all_handles) {
    if (!g || !all_handles) return fail_msg(g ? g->ctx : nullptr, B200PPF_ERR_INVALID, "group connect: null argument");
    DeviceGuard guard(g->ctx->device);
    for (int r = 0; r < g->world; ++r) {
        if (r == g->rank) continue;
        void *p[3] = {nullptr, nullptr, nullptr};
        for (int k = 0; k < 3; ++k) {
            cudaIpcMemHandle_t h;
            memcpy(&h, all_handles + ((size_t)r * 3 + k) * sizeof(h), sizeof(h));
            if (cudaIpcOpenMemHandle(&p[k], h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                return fail_msg(g->ctx, B200PPF_ERR_CUDA, "group connect: cudaIpcOpenMemHandle failed (ranks must share one node with peer access)");
            }
        }
        g->peer[0][r] = static_cast<unsigned long long *>(p[0]);
        g->peer[1][r] = static_cast<unsigned long long *>(p[1]);
        g->peer_flags[r] = static_cast<uint32_t *>(p[2]);
        g->opened[r] = true;
    }
    g->connected = true;
    return B200PPF_OK;
}

void b200ppf_group_destroy(b200ppf_group *g) {
    if (!g) return;
    DeviceGuard guard(g->ctx->device);
    cudaStreamSynchronize(g->ctx->stream);
    for (int r = 0; r < g->world; ++r)
        if (g->opened[r]) {
            cudaIpcCloseMemHandle(g->peer[0][r]);
            cudaIpcCloseMemHandle(g->peer[1][r]);
            cudaIpcCloseMemHandle(g->peer_flags[r]);
        }
    for (int s = 0; s < 2; ++s)
        if (g->own[s]) cudaFree(g->own[s]);
    if (g->own_flags) cudaFree(g->own_flags);
    if (g->records) cudaFree(g->records);
    delete g;
}

/* the asynchronous half: this rank's persistent CTAs on the shared queue; peaks merged into every rank's array; flag raised */
int b200ppf_group_vote(b200ppf_group *g, const b200ppf_cloud *model, const b200ppf_table *table, const b200ppf_cloud *scene,
                       size_t ref_rate) {
    if (!g || !scene || !table) return fail_msg(g ? g->ctx : nullptr, B200PPF_ERR_INVALID, "group vote: null argument");
    (void)model;
    b200ppf_ctx *ctx = g->ctx;
    if (!g->connected) return fail_msg(ctx, B200PPF_ERR_STATE, "group vote: the group is not connected yet");
    if (ref_rate == 0) ref_rate = 1;
    const size_t n_ref = (scene->n + ref_rate - 1) / ref_rate;
    if (n_ref == 0) return fail_msg(ctx, B200PPF_ERR_STATE, "group vote: empty scene");
    if (n_ref > g->n_records) return fail_msg(ctx, B200PPF_ERR_INVALID, "group vote: more reference points than the group's buffers hold");
    DeviceGuard guard(ctx->device);
    const int set = (int)(g->step & 1u);
    g->step += 1;
    // Clear the OTHER set for the next step now: its last users finished before they raised the flags this rank waited for
    // at the end of the previous step, and its next users cannot start before this rank raises the flag of THIS step, which
    // the kernel launched below does when it ends (stream order).  The very first step finds both sets cleared by create.
    PPF_CUDA(ctx, cudaMemsetAsync(g->own[1 - set], 0, g->n_records * sizeof(unsigned long long), ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(g->own_flags + QUEUE_WORD + (1 - set), 0, sizeof(uint32_t), ctx->stream));
    VoteQueue q;
    q.counter = g->peer_flags[0] + QUEUE_WORD + set;  // rank 0 owns the queue
    q.n_peers = g->world;
    for (int r = 0; r < MAX_PEERS; ++r) {
        q.peer_peaks[r] = r < g->world ? g->peer[set][r] : nullptr;
        q.flags[r] = r < g->world ? g->peer_flags[r] + set * MAX_PEERS : nullptr;
    }
    q.slot = (uint32_t)g->rank;
    q.value = g->step;
    q.done_counter = g->own_flags + DONE_WORD;
    return k3_vote_shared(ctx, table, scene, ref_rate, n_ref, &q);
}

/* the second half: wait (on the device) for every rank's flag, assemble all poses from this rank's complete peak array,
 * cluster */
int b200ppf_group_cluster(b200ppf_group *g, const b200ppf_cloud *model, const b200ppf_table *table, const b200ppf_cloud *scene,
                          size_t ref_rate, float pos_thr, float rot_thr, float *final16, float *poses16, uint32_t *votes,
                          size_t *n_out) {
    if (!g || !poses16 || !votes || !n_out || !model || !table || !scene)
        return fail_msg(g ? g->ctx : nullptr, B200PPF_ERR_INVALID, "group cluster: null argument");
    b200ppf_ctx *ctx = g->ctx;
    if (g->step == 0) return fail_msg(ctx, B200PPF_ERR_STATE, "group cluster: no vote has been issued");
    if (ref_rate == 0) ref_rate = 1;
    const size_t n_ref = (scene->n + ref_rate - 1) / ref_rate;
    DeviceGuard guard(ctx->device);
    const int set = (int)((g->step - 1) & 1u);
    int rc = k3_group_wait(ctx, g->own_flags + set * MAX_PEERS, g->world, g->step);
    if (rc) return rc;
    rc = k3_poses(ctx, model, table, scene, ref_rate, n_ref, g->own[set], g->records);
    if (rc) return rc;
    rc = k4_cluster(ctx, g->records, n_ref, pos_thr, rot_thr, poses16, votes, n_out);
    if (rc) return rc;
    if (*n_out && final16) memcpy(final16, poses16, 16 * sizeof(float));
    return B200PPF_OK;
}

int b200ppf_group_register(b200ppf_group *g, const b200ppf_cloud *model, const b200ppf_table *table, const b200ppf_cloud *scene,
                           size_t ref_rate, float pos_thr, float rot_thr, float *final16, float *poses16, uint32_t *votes,
                           size_t *n_out) {
    int rc = b200ppf_group_vote(g, model, table, scene, ref_rate);
    if (rc) return rc;
    return b200ppf_group_cluster(g, model, table, scene, ref_rate, pos_thr, rot_thr, final16, poses16, votes, n_out);
}

const b200ppf_hypothesis *b200ppf_group_records(const b200ppf_group *g) { return g && g->step ? g->records : nullptr; }

/* ---- one process, several GPUs ------------------------------------------------------------------------------------ */

int b200ppf_multi_create(const int *devices, int n_devices, b200ppf_multi **out) {
    if (!out || !devices) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi: null argument");
    *out = nullptr;
    if (n_devices < 1 || n_devices > MAX_PEERS) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi: 1 .. 16 devices");
    b200ppf_multi *m = new (std::nothrow) b200ppf_multi();
    if (!m) return fail_msg(nullptr, B200PPF_ERR_NOMEM, "multi: out of host memory");
    for (int g = 0; g < n_devices; ++g) {
        b200ppf_ctx *c = nullptr;
        int rc = b200ppf_create(devices[g], &c);
        if (rc) {
            b200ppf_multi_destroy(m);
            return rc;
        }
        m->ctx.push_back(c);
    }
    // every device may store into every other device's buffers
    for (int a = 0; a < n_devices; ++a) {
        DeviceGuard guard(devices[a]);
        for (int b = 0; b < n_devices; ++b) {
            if (a == b || devices[a] == devices[b]) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, devices[a], devices[b]);
            if (!can) {
                b200ppf_multi_destroy(m);
                return fail_msg(nullptr, B200PPF_ERR_UNSUPPORTED, "multi: the devices have no peer access to one another");
            }
            cudaError_t e = cudaDeviceEnablePeerAccess(devices[b], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                b200ppf_multi_destroy(m);
                return fail_msg(nullptr, B200PPF_ERR_CUDA, "multi: cudaDeviceEnablePeerAccess failed");
            }
            cudaGetLastError();
        }
    }
    m->model.assign(n_devices, nullptr);
    m->scene.assign(n_devices, nullptr);
    m->table.assign(n_devices, nullptr);
    *out = m;
    return B200PPF_OK;
}

void b200ppf_multi_destroy(b200ppf_multi *m) {
    if (!m) return;
    for (b200ppf_group *g : m->group) b200ppf_group_destroy(g);
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        if (g < m->table.size() && m->table[g]) b200ppf_table_free(m->table[g]);
        if (g < m->model.size() && m->model[g]) b200ppf_cloud_free(m->model[g]);
        if (g < m->scene.size() && m->scene[g]) b200ppf_cloud_free(m->scene[g]);
    }
    for (b200ppf_ctx *c : m->ctx) b200ppf_destroy(c);
    delete m;
}

int b200ppf_multi_size(const b200ppf_multi *m) { return m ? (int)m->ctx.size() : 0; }
b200ppf_ctx *b200ppf_multi_context(b200ppf_multi *m, int g) { return m && g >= 0 && g < (int)m->ctx.size() ? m->ctx[g] : nullptr; }
const b200ppf_table *b200ppf_multi_table(const b200ppf_multi *m, int g) { return m && g >= 0 && g < (int)m->table.size() ? m->table[g] : nullptr; }
const char *b200ppf_multi_last_error(const b200ppf_multi *m) { return m ? m->error.c_str() : ""; }

namespace {
int multi_fail(b200ppf_multi *m, int g, int rc) {
    m->error = b200ppf_last_error(m->ctx[g]);
    return rc;
}
}  // namespace

/* TrainDetector on every device: the model cloud is uploaded and its table built G times (redundant builds need no
 * communication and take milliseconds; SURVEY.md §8e) */
int b200ppf_multi_train(b200ppf_multi *m, const float *model_host, size_t n, size_t stride, size_t noff, float angle_step,
                        float dist_step) {
    if (!m) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi: null handle");
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        if (m->table[g]) b200ppf_table_free(m->table[g]);
        if (m->model[g]) b200ppf_cloud_free(m->model[g]);
        m->table[g] = nullptr;
        m->model[g] = nullptr;
        int rc = b200ppf_cloud_upload(m->ctx[g], model_host, n, stride, noff, &m->model[g]);
        if (rc) return multi_fail(m, (int)g, rc);
    }
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        int rc = b200ppf_table_build_from_cloud(m->ctx[g], m->model[g], angle_step, dist_step, &m->table[g]);
        if (rc) return multi_fail(m, (int)g, rc);
    }
    return B200PPF_OK;
}

/* setInputSource + setSearchMethod with a table that already exists on some device: the model cloud goes to every
 * device, the table is copied device to device (NVLink) */
int b200ppf_multi_adopt(b200ppf_multi *m, const float *model_host, size_t n, size_t stride, size_t noff, const b200ppf_table *table) {
    if (!m || !table) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi: null argument");
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        if (m->table[g]) b200ppf_table_free(m->table[g]);
        if (m->model[g]) b200ppf_cloud_free(m->model[g]);
        m->table[g] = nullptr;
        m->model[g] = nullptr;
        int rc = b200ppf_cloud_upload(m->ctx[g], model_host, n, stride, noff, &m->model[g]);
        if (!rc) rc = b200ppf_table_clone(m->ctx[g], table, &m->table[g]);
        if (rc) return multi_fail(m, (int)g, rc);
    }
    return B200PPF_OK;
}

/* LoadTrainedDetector on every device */
int b200ppf_multi_load(b200ppf_multi *m, const float *model_host, size_t n, size_t stride, size_t noff, const char *table_path) {
    if (!m) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi: null handle");
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        if (m->table[g]) b200ppf_table_free(m->table[g]);
        if (m->model[g]) b200ppf_cloud_free(m->model[g]);
        m->table[g] = nullptr;
        m->model[g] = nullptr;
        int rc = b200ppf_cloud_upload(m->ctx[g], model_host, n, stride, noff, &m->model[g]);
        if (!rc) rc = b200ppf_table_load(m->ctx[g], table_path, &m->table[g]);
        if (rc) return multi_fail(m, (int)g, rc);
    }
    return B200PPF_OK;
}

/* setInputTarget: the scene replicated on every device */
int b200ppf_multi_scene(b200ppf_multi *m, const float *scene_host, size_t n, size_t stride, size_t noff) {
    if (!m) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi: null handle");
    for (size_t g = 0; g < m->ctx.size(); ++g) {
        if (m->scene[g]) b200ppf_cloud_free(m->scene[g]);
        m->scene[g] = nullptr;
        int rc = b200ppf_cloud_upload(m->ctx[g], scene_host, n, stride, noff, &m->scene[g]);
        if (rc) return multi_fail(m, (int)g, rc);
    }
    return B200PPF_OK;
}

/* align: every device votes on its interleaved share of the reference points (all launches are asynchronous, issued
 * from this thread), device 0 clusters the complete record set and its poses are returned */
int b200ppf_multi_register(b200ppf_multi *m, size_t ref_rate, float pos_thr, float rot_thr, float *final16, float *poses16,
                           uint32_t *votes, size_t *n_out) {
    if (!m || !poses16 || !votes || !n_out) return fail_msg(nullptr, B200PPF_ERR_INVALID, "multi register: null argument");
    *n_out = 0;
    const int G = (int)m->ctx.size();
    for (int g = 0; g < G; ++g)
        if (!m->model[g] || !m->table[g] || !m->scene[g]) {
            m->error = "multi register: train / load and scene upload come first";
            return B200PPF_ERR_STATE;
        }
    if (ref_rate == 0) ref_rate = 1;
    const size_t n_ref = (m->scene[0]->n + ref_rate - 1) / ref_rate;
    if (m->group.empty() || m->group[0]->n_records < n_ref) {
        for (b200ppf_group *g : m->group) b200ppf_group_destroy(g);
        m->group.clear();
        for (int g = 0; g < G; ++g) {
            b200ppf_group *grp = nullptr;
            int rc = group_alloc(m->ctx[g], g, G, n_ref + n_ref / 4, &grp);
            if (rc) return multi_fail(m, g, rc);
            m->group.push_back(grp);
        }
        for (int a = 0; a < G; ++a) {  // same process: the peers' pointers are usable as they are
            for (int b = 0; b < G; ++b) {
                m->group[a]->peer[0][b] = m->group[b]->own[0];
                m->group[a]->peer[1][b] = m->group[b]->own[1];
                m->group[a]->peer_flags[b] = m->group[b]->own_flags;
            }
            m->group[a]->connected = true;
        }
    }
    for (int g = 0; g < G; ++g) {
        int rc = b200ppf_group_vote(m->group[g], m->model[g], m->table[g], m->scene[g], ref_rate);
        if (rc) return multi_fail(m, g, rc);
    }
    int rc = b200ppf_group_cluster(m->group[0], m->model[0], m->table[0], m->scene[0], ref_rate, pos_thr, rot_thr, final16, poses16,
                                   votes, n_out);
    if (rc) return multi_fail(m, 0, rc);
    // the other devices only have to drain before their buffers are reused two steps from now; keep the steps aligned
    for (int g = 1; g < G; ++g) {
        DeviceGuard guard(m->ctx[g]->device);
        const int set = (int)((m->group[g]->step - 1) & 1u);
        rc = k3_group_wait(m->ctx[g], m->group[g]->own_flags + set * MAX_PEERS, G, m->group[g]->step);
        if (rc) return multi_fail(m, g, rc);
    }
    return B200PPF_OK;
}

}  // extern "C"
