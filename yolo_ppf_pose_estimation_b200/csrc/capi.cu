// capi.cu — the extern "C" surface declared in include/b200ppf.h.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include "ppf_common.cuh"

namespace b200ppf {

static std::mutex g_err_mutex;
static std::string g_error;

int fail_msg(b200ppf_ctx *ctx, int code, const char *msg) {
    if (ctx) ctx->error = msg;
    std::lock_guard<std::mutex> lock(g_err_mutex);
    g_error = msg;
    return code;
}

int cloud_alloc(b200ppf_ctx *ctx, size_t n, CloudPtr *out) {
    CloudPtr c(new (std::nothrow) b200ppf_cloud());
    if (!c) return fail_msg(ctx, B200PPF_ERR_NOMEM, "cloud: out of host memory");
    c->ctx = ctx;
    c->n = n;
    PPF_CUDA(ctx, cudaMallocAsync(&c->pos, std::max<size_t>(1, 2 * n) * sizeof(float4), ctx->stream));
    c->nrm = c->pos + n;
    *out = std::move(c);
    return B200PPF_OK;
}

std::array<TableArray, 8> table_arrays(b200ppf_table *t) {
    const uint64_t total_keys = (uint64_t)t->info.key_space * t->info.n_slices;
    const bool cells = t->bp.cells_log2 != 0, merged = cells && t->info.n_entries != 0;
    const size_t n_sub = cells ? (size_t)(total_keys << t->bp.cells_log2) + 1 : 0, ne = t->info.n_entries;
    return {{{&t->offsets, (size_t)total_keys + 1, 0, true},
             {&t->sub_offsets, n_sub, 0, cells},
             {&t->entry_w, ne, ENTRY_PAD, true},
             {&t->entry_am, ne, ENTRY_PAD, true},
             {reinterpret_cast<uint32_t **>(&t->entry_alpha), ne, 0, true},
             {&t->entry_idx, ne, 0, true},
             {&t->merged_w, merged ? t->n_merged : 0, ENTRY_PAD, merged},
             {&t->msub_offsets, merged ? n_sub : 0, 0, merged}}};
}

cudaError_t table_array_alloc(cudaStream_t stream, const TableArray &a) {
    cudaError_t e = cudaMallocAsync(a.slot, std::max<size_t>(1, a.words + a.pad) * sizeof(uint32_t), stream);
    if (e == cudaSuccess && a.pad) e = cudaMemsetAsync(*a.slot + a.words, 0, a.pad * sizeof(uint32_t), stream);
    return e;
}

}  // namespace b200ppf

using namespace b200ppf;

#define CHECK_CTX(ctx)                                   \
    if (!(ctx)) return fail_msg(nullptr, B200PPF_ERR_INVALID, "null context"); \
    DeviceGuard _guard((ctx)->device)

// the reference's ICP(100, 0.005f, 2.5f, 8): the default of both ICP calls and of both per-object parameter blocks
constexpr b200ppf_icp_params ICP_DEFAULT = {100, 0.005f, 2.5f, 8};

namespace {

// params (NULL = the defaults) -> *out, or B200PPF_ERR_INVALID
int verify_params(b200ppf_ctx *ctx, const b200ppf_verify_params *params, b200ppf_verify_params *out) {
    b200ppf_verify_params_default(out);
    if (params) *out = *params;
    if (!(std::isfinite(out->inlier_dist) && out->inlier_dist > 0.0f))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "verify: inlier_dist must be finite and positive");
    if (!(out->normal_angle >= 0.0f)) return fail_msg(ctx, B200PPF_ERR_INVALID, "verify: normal_angle must be >= 0");
    return B200PPF_OK;
}

// the parity hooks' copies: a host array of n words into a new stream-ordered buffer (none for a NULL array), and back
int to_device(b200ppf_ctx *ctx, StreamBuf<uint32_t> &d, const uint32_t *host, size_t n) {
    if (!host) return B200PPF_OK;
    PPF_CUDA(ctx, d.alloc(n));
    if (n) PPF_CUDA(ctx, cudaMemcpyAsync(d, host, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    return B200PPF_OK;
}

int to_host(b200ppf_ctx *ctx, uint32_t *host, const StreamBuf<uint32_t> &d, size_t n) {
    if (host && n) PPF_CUDA(ctx, cudaMemcpyAsync(host, d, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    return B200PPF_OK;
}

}  // namespace

extern "C" {

int b200ppf_version(void) { return B200PPF_VERSION; }

int b200ppf_create(int device, b200ppf_ctx **out) {
    if (!out) return fail_msg(nullptr, B200PPF_ERR_INVALID, "b200ppf_create: null output pointer");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail_msg(nullptr, B200PPF_ERR_CUDA,
                        "b200ppf_create: no CUDA device is visible; this library has no CPU fallback");
    }
    if (device < 0 || device >= count) return fail_msg(nullptr, B200PPF_ERR_INVALID, "b200ppf_create: device index out of range");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return fail_msg(nullptr, B200PPF_ERR_CUDA, "b200ppf_create: cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return fail_msg(nullptr, B200PPF_ERR_UNSUPPORTED,
                        "b200ppf_create: kernels are built for sm_100a (Blackwell B200) only");
    b200ppf_ctx *ctx = new (std::nothrow) b200ppf_ctx();
    if (!ctx) return fail_msg(nullptr, B200PPF_ERR_NOMEM, "b200ppf_create: out of host memory");
    ctx->device = device;
    DeviceGuard guard(device);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return fail_msg(nullptr, B200PPF_ERR_CUDA, "b200ppf_create: cudaStreamCreate failed");
    }
    for (auto &ev : ctx->ev) cudaEventCreate(&ev);
    for (auto &ev : ctx->ev_vote) cudaEventCreate(&ev);
    {   // keep freed scratch and table arrays in the device's stream-ordered pool instead of returning them to the driver
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
    }
    *out = ctx;
    return B200PPF_OK;
}

void b200ppf_destroy(b200ppf_ctx *ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->d_stats) cudaFree(ctx->d_stats);
    if (ctx->d_peaks) cudaFree(ctx->d_peaks);
    if (ctx->d_vote_queue) cudaFree(ctx->d_vote_queue);
    if (ctx->d_fold) cudaFree(ctx->d_fold);
    if (ctx->d_hyps) cudaFree(ctx->d_hyps);
    if (ctx->d_assign) cudaFree(ctx->d_assign);
    if (ctx->stage) cudaFreeHost(ctx->stage);
    for (auto &ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto &ev : ctx->ev_vote)
        if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *b200ppf_last_error(const b200ppf_ctx *ctx) {
    if (ctx) return ctx->error.c_str();
    std::lock_guard<std::mutex> lock(g_err_mutex);
    static thread_local std::string copy;
    copy = g_error;
    return copy.c_str();
}

int b200ppf_set_feature_mode(b200ppf_ctx *ctx, int mode) {
    if (!ctx) return fail_msg(nullptr, B200PPF_ERR_INVALID, "null context");
    if (mode < 0 || mode > 2) return fail_msg(ctx, B200PPF_ERR_INVALID, "unknown feature mode");
    ctx->feature_mode = mode;
    return B200PPF_OK;
}

int b200ppf_set_alpha_mode(b200ppf_ctx *ctx, int mode) {
    if (!ctx) return fail_msg(nullptr, B200PPF_ERR_INVALID, "null context");
    if (mode < 0 || mode > 1) return fail_msg(ctx, B200PPF_ERR_INVALID, "unknown alpha mode");
    ctx->alpha_mode = mode;
    return B200PPF_OK;
}

int b200ppf_set_nalpha_rule(b200ppf_ctx *ctx, int rule) {
    if (!ctx) return fail_msg(nullptr, B200PPF_ERR_INVALID, "null context");
    if (rule < 0 || rule > 2) return fail_msg(ctx, B200PPF_ERR_INVALID, "unknown alpha-column rule");
    ctx->nalpha_rule = rule;
    return B200PPF_OK;
}

int b200ppf_get_device(const b200ppf_ctx *ctx) { return ctx ? ctx->device : -1; }
void *b200ppf_get_stream(const b200ppf_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
uint64_t b200ppf_launch_count(const b200ppf_ctx *ctx) { return ctx ? ctx->launches : 0; }

int b200ppf_synchronize(b200ppf_ctx *ctx) {
    CHECK_CTX(ctx);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_get_timings(b200ppf_ctx *ctx, b200ppf_timings *out) {
    if (!ctx || !out) return fail_msg(nullptr, B200PPF_ERR_INVALID, "null argument");
    if (ctx->vote_timed) {  // the vote is asynchronous: resolve its events on demand
        DeviceGuard guard(ctx->device);
        if (cudaEventSynchronize(ctx->ev_vote[3]) == cudaSuccess) {
            cudaEventElapsedTime(&ctx->timings.grid_ms, ctx->ev_vote[0], ctx->ev_vote[1]);
            cudaEventElapsedTime(&ctx->timings.vote_ms, ctx->ev_vote[1], ctx->ev_vote[2]);
            cudaEventElapsedTime(&ctx->timings.pose_ms, ctx->ev_vote[2], ctx->ev_vote[3]);
        }
    }
    *out = ctx->timings;
    return B200PPF_OK;
}

/* ---- clouds ------------------------------------------------------------------------------- */

int b200ppf_cloud_upload(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride, size_t noff,
                         b200ppf_cloud **out) {
    CHECK_CTX(ctx);
    if (!out) return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud upload: null output pointer");
    *out = nullptr;
    if (n && !host) return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud upload: null host pointer");
    if (stride < 6 || noff < 3 || noff + 3 > stride)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud upload: stride/normal offset do not describe [x y z .. nx ny nz]");
    // AoS -> float4 SoA staging in the context's grow-only pinned buffer, dropping non-finite points
    PPF_CUDA(ctx, grow_buffer(&ctx->stage, &ctx->stage_cap, std::max<size_t>(1, 2 * n), /*pinned=*/true));
    float4 *stage = ctx->stage;
    size_t m = 0;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    float4 *sp = stage, *sn = stage + n;
    for (size_t i = 0; i < n; ++i) {
        const float *p = host + i * stride, *q = p + noff;
        // non-finite rows are dropped: NaN (SURVEY.md A.8 rule 5) and +-Inf alike (depth-derived clouds carry both;
        // an infinite coordinate would make the bounding box, and every grid sized from it, meaningless)
        if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2]) || !std::isfinite(q[0]) ||
            !std::isfinite(q[1]) || !std::isfinite(q[2]))
            continue;
        sp[m] = make_float4(p[0], p[1], p[2], 1.0f);
        sn[m] = make_float4(q[0], q[1], q[2], 0.0f);
        for (int k = 0; k < 3; ++k) {
            lo[k] = std::min(lo[k], p[k]);
            hi[k] = std::max(hi[k], p[k]);
        }
        ++m;
    }
    CloudPtr c;
    int rc = cloud_alloc(ctx, m, &c);
    if (rc) return rc;
    for (int k = 0; k < 3; ++k) {
        c->bbox_min[k] = m ? lo[k] : 0.0f;
        c->bbox_max[k] = m ? hi[k] : 0.0f;
    }
    cudaEventRecord(ctx->ev[0], ctx->stream);
    if (m) PPF_CUDA(ctx, cudaMemcpyAsync(c->pos, sp, m * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    if (m) PPF_CUDA(ctx, cudaMemcpyAsync(c->nrm, sn, m * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    cudaEventRecord(ctx->ev[1], ctx->stream);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the staging buffer is reused by the next upload
    cudaEventElapsedTime(&ctx->timings.upload_ms, ctx->ev[0], ctx->ev[1]);
    *out = c.release();
    return B200PPF_OK;
}

size_t b200ppf_cloud_size(const b200ppf_cloud *cloud) { return cloud ? cloud->n : 0; }

void b200ppf_cloud_free(b200ppf_cloud *c) {
    if (!c) return;
    DeviceGuard guard(c->ctx ? c->ctx->device : 0);
    if (c->pos) {  // pos | nrm share one stream-ordered allocation
        if (c->ctx) cudaFreeAsync(c->pos, c->ctx->stream);
        else cudaFree(c->pos);
    }
    delete c;
}

/* ---- K1 ----------------------------------------------------------------------------------- */

int b200ppf_features_compute(b200ppf_ctx *ctx, const b200ppf_cloud *model, b200ppf_features **out) {
    CHECK_CTX(ctx);
    if (!model || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "features compute: null argument");
    *out = nullptr;
    if (model->n > 65535) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "features compute: more than 65535 model points");
    b200ppf_features *f = new (std::nothrow) b200ppf_features();
    if (!f) return fail_msg(ctx, B200PPF_ERR_NOMEM, "features compute: out of host memory");
    f->ctx = ctx;
    f->count = model->n * model->n;
    cudaError_t e = cudaMalloc(&f->d, std::max<size_t>(1, f->count) * sizeof(b200ppf_signature));
    if (e != cudaSuccess) {
        delete f;
        return fail_msg(ctx, B200PPF_ERR_NOMEM, "features compute: device allocation of the N*N*20-byte feature cloud failed");
    }
    cudaEventRecord(ctx->ev[0], ctx->stream);
    int rc = k1_features_compute(ctx, model, f->d);
    cudaEventRecord(ctx->ev[1], ctx->stream);
    if (rc == B200PPF_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess)
        rc = fail_msg(ctx, B200PPF_ERR_CUDA, "features compute: kernel failed");
    if (rc != B200PPF_OK) {
        b200ppf_features_free(f);
        return rc;
    }
    cudaEventElapsedTime(&ctx->timings.features_ms, ctx->ev[0], ctx->ev[1]);
    *out = f;
    return B200PPF_OK;
}

int b200ppf_features_upload(b200ppf_ctx *ctx, const b200ppf_signature *host, size_t count, b200ppf_features **out) {
    CHECK_CTX(ctx);
    if (!out || (count && !host)) return fail_msg(ctx, B200PPF_ERR_INVALID, "features upload: null argument");
    *out = nullptr;
    b200ppf_features *f = new (std::nothrow) b200ppf_features();
    if (!f) return fail_msg(ctx, B200PPF_ERR_NOMEM, "features upload: out of host memory");
    f->ctx = ctx;
    f->count = count;
    cudaError_t e = cudaMalloc(&f->d, std::max<size_t>(1, count) * sizeof(b200ppf_signature));
    if (e == cudaSuccess && count)
        e = cudaMemcpyAsync(f->d, host, count * sizeof(b200ppf_signature), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        b200ppf_features_free(f);
        return fail_msg(ctx, e == cudaErrorMemoryAllocation ? B200PPF_ERR_NOMEM : B200PPF_ERR_CUDA, cudaGetErrorString(e));
    }
    *out = f;
    return B200PPF_OK;
}

int b200ppf_features_download(b200ppf_ctx *ctx, const b200ppf_features *f, size_t first, size_t count,
                              b200ppf_signature *host) {
    CHECK_CTX(ctx);
    if (!f || (count && !host)) return fail_msg(ctx, B200PPF_ERR_INVALID, "features download: null argument");
    if (first > f->count || count > f->count - first)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "features download: range exceeds the feature cloud");
    if (count) {
        PPF_CUDA(ctx, cudaMemcpyAsync(host, f->d + first, count * sizeof(b200ppf_signature), cudaMemcpyDeviceToHost,
                                      ctx->stream));
        PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return B200PPF_OK;
}

size_t b200ppf_features_count(const b200ppf_features *f) { return f ? f->count : 0; }

void b200ppf_features_free(b200ppf_features *f) {
    if (!f) return;
    DeviceGuard guard(f->ctx ? f->ctx->device : 0);
    if (f->d) cudaFree(f->d);
    delete f;
}

/* ---- K2 ----------------------------------------------------------------------------------- */

int b200ppf_table_build(b200ppf_ctx *ctx, const b200ppf_features *f, float angle_step, float dist_step,
                        b200ppf_table **out) {
    CHECK_CTX(ctx);
    if (!f || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: null argument");
    *out = nullptr;
    return k2_build(ctx, f, nullptr, angle_step, dist_step, out);
}

int b200ppf_table_build_from_cloud(b200ppf_ctx *ctx, const b200ppf_cloud *model, float angle_step, float dist_step,
                                   b200ppf_table **out) {
    CHECK_CTX(ctx);
    if (!model || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: null argument");
    *out = nullptr;
    return k2_build(ctx, nullptr, model, angle_step, dist_step, out);
}

int b200ppf_table_get_info(const b200ppf_table *t, b200ppf_table_info *info) {
    if (!t || !info) return fail_msg(nullptr, B200PPF_ERR_INVALID, "table info: null argument");
    *info = t->info;
    return B200PPF_OK;
}

int b200ppf_table_query_key(b200ppf_ctx *ctx, const b200ppf_table *t, const int32_t *d4, uint64_t *pairs, size_t cap,
                            size_t *n_found) {
    CHECK_CTX(ctx);
    if (!t || !d4 || !n_found || (cap && !pairs)) return fail_msg(ctx, B200PPF_ERR_INVALID, "table query: null argument");
    return k2_query_key(ctx, t, d4, pairs, cap, n_found);
}

int b200ppf_table_query(b200ppf_ctx *ctx, const b200ppf_table *t, float f1, float f2, float f3, float f4,
                        uint64_t *pairs, size_t cap, size_t *n_found) {
    CHECK_CTX(ctx);
    if (!t || !n_found || (cap && !pairs)) return fail_msg(ctx, B200PPF_ERR_INVALID, "table query: null argument");
    *n_found = 0;
    const float f[4] = {f1, f2, f3, f4};
    if (std::isnan(f1) || std::isnan(f2) || std::isnan(f3) || std::isnan(f4)) return B200PPF_OK;
    int d[4];
    quantise(t->kp, f, d);  // same IEEE divide + floor as the device
    return k2_query_key(ctx, t, d, pairs, cap, n_found);
}

int b200ppf_table_alpha_m(b200ppf_ctx *ctx, const b200ppf_table *t, float *host) {
    CHECK_CTX(ctx);
    if (!t || !host) return fail_msg(ctx, B200PPF_ERR_INVALID, "alpha_m export: null argument");
    return k2_alpha_m(ctx, t, host);
}

int b200ppf_table_export(b200ppf_ctx *ctx, const b200ppf_table *t, uint32_t *offsets, uint32_t *entry_i,
                         uint32_t *entry_j, float *entry_alpha_m) {
    CHECK_CTX(ctx);
    if (!t) return fail_msg(ctx, B200PPF_ERR_INVALID, "table export: null table");
    const size_t total = (size_t)t->info.key_space * t->info.n_slices + 1, ne = t->info.n_entries;
    if (offsets) PPF_CUDA(ctx, cudaMemcpyAsync(offsets, t->offsets, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<uint32_t> idx;
    std::vector<float> ent;
    if ((entry_i || entry_j) && ne) {
        idx.resize(ne);
        PPF_CUDA(ctx, cudaMemcpyAsync(idx.data(), t->entry_idx, ne * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (entry_alpha_m && ne) {
        ent.resize(ne);
        PPF_CUDA(ctx, cudaMemcpyAsync(ent.data(), t->entry_alpha, ne * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    }
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const uint32_t n = (uint32_t)t->info.n_model;
    if (t->info.phase_cells > 1 && ne) {
        // buckets are stored in (phase cell, i, j) order: report them in the canonical (i, j) order
        std::vector<uint32_t> off(total), all_idx(ne);
        PPF_CUDA(ctx, cudaMemcpyAsync(off.data(), t->offsets, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        PPF_CUDA(ctx, cudaMemcpyAsync(all_idx.data(), t->entry_idx, ne * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        std::vector<std::pair<uint32_t, uint32_t>> order;
        for (size_t k = 0; k + 1 < total; ++k) {
            const uint32_t b = off[k], e = off[k + 1];
            if (e - b < 2) continue;
            order.resize(e - b);
            for (uint32_t p = b; p < e; ++p) order[p - b] = std::make_pair(all_idx[p], p);
            std::sort(order.begin(), order.end());
            for (uint32_t p = b; p < e; ++p) {
                if (!idx.empty()) idx[p] = order[p - b].first;
                if (entry_alpha_m) entry_alpha_m[p] = ent[order[p - b].second];
            }
            if (entry_alpha_m)
                for (uint32_t p = b; p < e; ++p) ent[p] = entry_alpha_m[p];
        }
    }
    for (size_t e = 0; e < idx.size(); ++e) {
        if (entry_i) entry_i[e] = idx[e] / n;
        if (entry_j) entry_j[e] = idx[e] % n;
    }
    for (size_t e = 0; e < ent.size(); ++e) entry_alpha_m[e] = ent[e];
    return B200PPF_OK;
}

/* ---- table file ------------------------------------------------------------------------------- */
namespace {

constexpr uint64_t TABLE_MAGIC = 0x4C42543030325042ull;  // "BP200TBL" little-endian
constexpr uint32_t TABLE_FORMAT = 4;                      // 4: sub-phase byte above the hot word (3: alpha-column rule, bin-major hot words)

struct TableFileHeader {
    uint64_t magic;
    uint32_t format, header_bytes;
    uint32_t feature_mode, alpha_mode;
    uint64_t n_offsets, n_sub_offsets, n_entries;  // array lengths in 32-bit words (entries: without the padding)
    uint64_t n_merged;                              // merged-vote words (its cell bounds have n_sub_offsets words)
    uint64_t checksum;                              // over info, kp, bp and the six arrays, in file order
    b200ppf_table_info info;
    b200ppf::KeyParams kp;
    b200ppf::BinParams bp;
};

// 64-bit multiplicative checksum over 8-byte words (tail bytes zero-extended)
uint64_t mix_bytes(uint64_t h, const void *data, size_t bytes) {
    const unsigned char *p = static_cast<const unsigned char *>(data);
    size_t k = 0;
    for (; k + 8 <= bytes; k += 8) {
        uint64_t w;
        memcpy(&w, p + k, 8);
        h = (h ^ w) * 0x9E3779B97F4A7C15ull;
        h ^= h >> 29;
    }
    if (k < bytes) {
        uint64_t w = 0;
        memcpy(&w, p + k, bytes - k);
        h = (h ^ w) * 0x9E3779B97F4A7C15ull;
        h ^= h >> 29;
    }
    return h;
}

struct FileCloser {
    FILE *f;
    ~FileCloser() {
        if (f) fclose(f);
    }
};

// Everything the voting kernel takes on trust from a table, re-derived from the file's own parameters and entries:
// a file that passes cannot make the kernel read outside its arrays or add outside its accumulator slice, whoever
// wrote it (the checksum only catches accidents).  Returns nullptr or what is wrong.
const char *validate_table_file(const TableFileHeader &h, const std::vector<std::vector<uint32_t>> &a) {
    const b200ppf_table_info &info = h.info;
    const b200ppf::KeyParams &kp = h.kp;
    if (info.n_model < 1) return "no model points";
    if (!(info.angle_step > 0.0f) || !(info.dist_step > 0.0f) || kp.angle_step != info.angle_step || kp.dist_step != info.dist_step)
        return "discretisation steps";
    if (h.feature_mode > 2 || h.alpha_mode > 1 || info.nalpha_rule > 2) return "unknown mode";
    unsigned __int128 ks = 1;
    for (int k = 0; k < 4; ++k) {
        if (kp.size[k] < 1 || kp.size[k] != info.size[k] || kp.lo[k] != info.lo[k]) return "key ranges";
        ks *= (unsigned __int128)(uint32_t)kp.size[k];
    }
    if (ks != (unsigned __int128)info.key_space || kp.key_space != info.key_space) return "key space is not the product of the key ranges";
    if (info.n_slices < 1 || info.slice_rows < 1 || (uint64_t)info.n_slices * info.slice_rows < info.n_model ||
        (uint64_t)(info.n_slices - 1) * info.slice_rows >= info.n_model)
        return "accumulator slices do not tile the model rows";
    // the binning parameters are a function of (angle step, alpha mode, column rule); only the number of phase
    // cells may be lower than that function's choice (large key spaces halve it)
    b200ppf::BinParams ref = b200ppf::make_bin_params(info.angle_step, (int)h.alpha_mode, (int)info.nalpha_rule);
    if (h.bp.cells_log2 > ref.cells_log2) return "phase cells";
    ref.cells_log2 = h.bp.cells_log2;
    if (ref.cells_log2 == 0) ref.bulk = 0;
    if (memcmp(&ref, &h.bp, sizeof(ref)) != 0) return "binning parameters do not follow from the angle step";
    if (info.n_alpha != ref.n_alpha || info.phase_cells != (1u << ref.cells_log2)) return "alpha columns";
    const std::vector<uint32_t> &off = a[0], &sub = a[1], &ew = a[2], &eam = a[3], &ealpha = a[4], &eidx = a[5];
    const uint64_t ne = h.n_entries, total_keys = (uint64_t)info.key_space * info.n_slices;
    if (off.empty() || off[0] != 0 || off.back() != ne) return "bucket offsets do not cover the entries";
    for (size_t k = 0; k + 1 < off.size(); ++k)
        if (off[k] > off[k + 1]) return "bucket offsets decrease";
    if (!sub.empty()) {
        if (sub.back() != ne) return "phase-cell offsets do not cover the entries";
        for (size_t k = 0; k + 1 < sub.size(); ++k)
            if (sub[k] > sub[k + 1]) return "phase-cell offsets decrease";
        for (uint64_t k = 0; k <= total_keys; ++k)
            if (sub[k << ref.cells_log2] != off[k]) return "phase-cell offsets leave their bucket";
    }
    const uint64_t n = info.n_model, nn = n * n;
    if (kp.slice_rows != info.slice_rows || kp.n_slices != info.n_slices || kp.row_pitch != (info.slice_rows + 31u) / 32u * 32u)
        return "slice geometry";
    for (uint32_t slice = 0; slice < info.n_slices; ++slice) {
        const uint64_t p0 = off[(uint64_t)slice * info.key_space], p1 = off[(uint64_t)(slice + 1) * info.key_space];
        const uint64_t row0 = (uint64_t)slice * info.slice_rows, rows = std::min<uint64_t>(info.slice_rows, n - row0);
        for (uint64_t p = p0; p < p1; ++p) {
            if (eidx[p] >= nn) return "entry pair index out of range";
            const uint64_t i = eidx[p] / n;
            if (i < row0 || i >= row0 + rows) return "entry filed under another accumulator slice";
            float alpha;
            memcpy(&alpha, &ealpha[p], sizeof(float));
            if (!(alpha >= -3.14159274f && alpha <= 3.14159274f)) return "entry alpha_m outside [-pi, pi]";
            const uint32_t a_fix = b200ppf::alpha_to_fix(alpha), local = (uint32_t)(i - row0);
            if (eam[p] != a_fix) return "entry fixed-point alpha_m does not match its float";
            if (ew[p] != (ref.bulk ? b200ppf::entry_word(ref, kp.row_pitch, local, alpha) : 4u * local))
                return "entry hot word does not match its pair";
        }
    }
    // merged votes: cell bounds monotone inside the array; every word a 4-aligned offset inside the accumulator slice
    // with a count >= 1; the counts of a cell add up to the cell's entries (the votes cast are those of the entries)
    const std::vector<uint32_t> &mw = a[6], &msub = a[7];
    if (!mw.empty() || !msub.empty()) {
        if (msub.size() != sub.size() || msub.empty() || msub[0] != 0 || msub.back() != mw.size()) return "merged cell offsets";
        const uint32_t acc_bytes = ref.acc_cols * kp.row_pitch * 4u;
        for (size_t c = 0; c + 1 < msub.size(); ++c) {
            if (msub[c] > msub[c + 1]) return "merged cell offsets decrease";
            uint64_t votes = 0;
            for (uint64_t p = msub[c]; p < msub[c + 1]; ++p) {
                const uint32_t off = mw[p] & 0xFFFFFFu, cnt = mw[p] >> 24;
                if (cnt == 0 || (off & 3u) || off >= acc_bytes) return "merged vote word outside the accumulator slice";
                votes += cnt;
            }
            if (votes != (uint64_t)sub[c + 1] - sub[c]) return "merged vote counts do not add up to the cell's entries";
        }
    }
    return nullptr;
}

}  // namespace

int b200ppf_table_save(b200ppf_ctx *ctx, const b200ppf_table *t, const char *path) {
    CHECK_CTX(ctx);
    if (!t || !path) return fail_msg(ctx, B200PPF_ERR_INVALID, "table save: null argument");
    DeviceGuard guard(ctx->device);
    TableFileHeader h;
    memset(&h, 0, sizeof(h));
    h.magic = TABLE_MAGIC;
    h.format = TABLE_FORMAT;
    h.header_bytes = (uint32_t)sizeof(h);
    h.feature_mode = (uint32_t)t->feature_mode;
    h.alpha_mode = (uint32_t)t->bp.mode;
    h.info = t->info;
    h.kp = t->kp;
    h.bp = t->bp;
    const std::array<TableArray, 8> arrs = table_arrays(const_cast<b200ppf_table *>(t));  // read only
    h.n_offsets = arrs[0].words;
    h.n_sub_offsets = arrs[1].words;
    h.n_entries = t->info.n_entries;
    h.n_merged = arrs[6].words;
    std::vector<std::vector<uint32_t>> host(arrs.size());
    for (size_t a = 0; a < arrs.size(); ++a) {
        host[a].resize(arrs[a].words);
        if (arrs[a].words)
            PPF_CUDA(ctx, cudaMemcpyAsync(host[a].data(), *arrs[a].slot, arrs[a].words * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                          ctx->stream));
    }
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // the parameter block (info, kp, bp: everything behind the checksum field) and then the six arrays
    uint64_t sum = mix_bytes(0x42323030u, reinterpret_cast<const char *>(&h) + offsetof(TableFileHeader, info),
                             sizeof(h) - offsetof(TableFileHeader, info));
    for (const std::vector<uint32_t> &a : host) sum = mix_bytes(sum, a.data(), a.size() * sizeof(uint32_t));
    h.checksum = sum;
    FileCloser fc{fopen(path, "wb")};
    if (!fc.f) return fail_msg(ctx, B200PPF_ERR_IO, "table save: cannot open the file for writing");
    bool ok = fwrite(&h, sizeof(h), 1, fc.f) == 1;
    for (size_t a = 0; a < host.size() && ok; ++a)
        if (!host[a].empty()) ok = fwrite(host[a].data(), sizeof(uint32_t), host[a].size(), fc.f) == host[a].size();
    ok = ok && fflush(fc.f) == 0;
    if (!ok) return fail_msg(ctx, B200PPF_ERR_IO, "table save: short write");
    return B200PPF_OK;
}

int b200ppf_table_load(b200ppf_ctx *ctx, const char *path, b200ppf_table **out) {
    CHECK_CTX(ctx);
    if (!path || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "table load: null argument");
    *out = nullptr;
    DeviceGuard guard(ctx->device);
    FileCloser fc{fopen(path, "rb")};
    if (!fc.f) return fail_msg(ctx, B200PPF_ERR_IO, "table load: cannot open the file");
    TableFileHeader h;
    if (fread(&h, sizeof(h), 1, fc.f) != 1) return fail_msg(ctx, B200PPF_ERR_IO, "table load: truncated header");
    if (h.magic != TABLE_MAGIC) return fail_msg(ctx, B200PPF_ERR_IO, "table load: not a b200ppf table file");
    if (h.format != TABLE_FORMAT || h.header_bytes != sizeof(h))
        return fail_msg(ctx, B200PPF_ERR_IO, "table load: file written by another format version");
    if ((int)h.feature_mode != ctx->feature_mode || (int)h.alpha_mode != ctx->alpha_mode)
        return fail_msg(ctx, B200PPF_ERR_STATE, "table load: the file's feature / alpha mode differs from the context's");
    const uint64_t total_keys = (uint64_t)h.info.key_space * h.info.n_slices;
    const bool sane = h.n_offsets == total_keys + 1 && total_keys < (1ull << 31) && h.bp.cells_log2 <= 8 &&
                      (total_keys << h.bp.cells_log2) < (1ull << 31) &&
                      h.n_sub_offsets == (h.bp.cells_log2 ? (total_keys << h.bp.cells_log2) + 1 : 0) &&
                      h.n_entries == h.info.n_entries && h.n_entries <= 0xFFFFFFFFull && h.info.n_model >= 1 &&
                      h.info.n_model <= 65535 && h.n_entries <= h.info.n_model * h.info.n_model &&
                      h.info.n_alpha >= 1 && h.bp.n_alpha == h.info.n_alpha &&
                      h.kp.slice_rows == h.info.slice_rows && h.kp.n_slices == h.info.n_slices;
    if (!sane) return fail_msg(ctx, B200PPF_ERR_IO, "table load: inconsistent header");
    const bool has_merged = h.bp.cells_log2 != 0 && h.n_entries != 0;
    if (h.n_merged > h.n_entries || (has_merged ? h.n_merged == 0 : h.n_merged != 0) || h.info.n_merged != h.n_merged)
        return fail_msg(ctx, B200PPF_ERR_IO, "table load: inconsistent header");
    TablePtr t(new (std::nothrow) b200ppf_table());
    if (!t) return fail_msg(ctx, B200PPF_ERR_NOMEM, "table load: out of host memory");
    t->ctx = ctx;
    t->info = h.info;
    t->kp = h.kp;
    t->bp = h.bp;
    t->feature_mode = (int)h.feature_mode;
    t->n_merged = h.n_merged;
    // the header is consistent: these are the lengths it states
    const std::array<TableArray, 8> arrs = table_arrays(t.get());
    std::vector<std::vector<uint32_t>> host(arrs.size());
    // the parameter block (info, kp, bp: everything behind the checksum field) and then the six arrays
    uint64_t sum = mix_bytes(0x42323030u, reinterpret_cast<const char *>(&h) + offsetof(TableFileHeader, info),
                             sizeof(h) - offsetof(TableFileHeader, info));
    for (size_t a = 0; a < arrs.size(); ++a) {
        const size_t words = arrs[a].words;
        host[a].resize(words);
        if (words && fread(host[a].data(), sizeof(uint32_t), words, fc.f) != words)
            return fail_msg(ctx, B200PPF_ERR_IO, "table load: truncated file");
        sum = mix_bytes(sum, host[a].data(), host[a].size() * sizeof(uint32_t));
    }
    if (fgetc(fc.f) != EOF) return fail_msg(ctx, B200PPF_ERR_IO, "table load: trailing bytes");
    if (sum != h.checksum) return fail_msg(ctx, B200PPF_ERR_IO, "table load: checksum mismatch (corrupt file)");
    if (const char *why = validate_table_file(h, host)) {
        char msg[200];
        snprintf(msg, sizeof(msg), "table load: invalid table (%s)", why);
        return fail_msg(ctx, B200PPF_ERR_IO, msg);
    }

    for (size_t a = 0; a < arrs.size(); ++a) {
        if (!arrs[a].used) continue;
        PPF_CUDA(ctx, table_array_alloc(ctx->stream, arrs[a]));
        if (arrs[a].words)
            PPF_CUDA(ctx, cudaMemcpyAsync(*arrs[a].slot, host[a].data(), arrs[a].words * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                          ctx->stream));
    }
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return fail_msg(ctx, B200PPF_ERR_CUDA, "table load: upload failed");
    *out = t.release();
    return B200PPF_OK;
}

int b200ppf_table_clone(b200ppf_ctx *dst, const b200ppf_table *src, b200ppf_table **out) {
    CHECK_CTX(dst);
    if (!src || !out) return fail_msg(dst, B200PPF_ERR_INVALID, "table clone: null argument");
    *out = nullptr;
    if (src->ctx) cudaStreamSynchronize(src->ctx->stream);  // the source table's build has finished (device guard is dst's)
    TablePtr t(new (std::nothrow) b200ppf_table());
    if (!t) return fail_msg(dst, B200PPF_ERR_NOMEM, "table clone: out of host memory");
    t->ctx = dst;
    t->info = src->info;
    t->kp = src->kp;
    t->bp = src->bp;
    t->feature_mode = src->feature_mode;
    t->n_merged = src->n_merged;
    const int src_dev = src->ctx ? src->ctx->device : dst->device;
    const std::array<TableArray, 8> from = table_arrays(const_cast<b200ppf_table *>(src)), to = table_arrays(t.get());  // src: read only
    for (size_t a = 0; a < to.size(); ++a) {
        if (!to[a].used) continue;
        PPF_CUDA(dst, table_array_alloc(dst->stream, to[a]));
        if (to[a].words)
            PPF_CUDA(dst, cudaMemcpyPeerAsync(*to[a].slot, dst->device, *from[a].slot, src_dev, to[a].words * sizeof(uint32_t),
                                              dst->stream));
    }
    if (cudaStreamSynchronize(dst->stream) != cudaSuccess) return fail_msg(dst, B200PPF_ERR_CUDA, "table clone: copy failed");
    *out = t.release();
    return B200PPF_OK;
}

void b200ppf_table_free(b200ppf_table *t) {
    if (!t) return;
    DeviceGuard guard(t->ctx ? t->ctx->device : 0);
    // the arrays come from the device's stream-ordered pool (k2_build, load, clone): they go back to it, so that the
    // next build re-uses the memory instead of asking the driver for gigabytes again
    for (const TableArray &a : table_arrays(t)) {
        if (!*a.slot) continue;
        if (t->ctx) cudaFreeAsync(*a.slot, t->ctx->stream);
        else cudaFree(*a.slot);
    }
    delete t;
}

/* ---- K3 ----------------------------------------------------------------------------------- */

int b200ppf_vote_device(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                        const b200ppf_cloud *scene, size_t ref_first, size_t ref_step, size_t ref_count,
                        b200ppf_hypothesis *hyps_device) {
    CHECK_CTX(ctx);
    if (ref_count && !hyps_device) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote: null output pointer");
    return k3_vote(ctx, model, t, scene, ref_first, ref_step, ref_count, &hyps_device, 1, 0, 1);
}

/* ---- multi-GPU exchange fused into the vote epilogue -------------------------------------------- */
int b200ppf_vote_scatter_device(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                                const b200ppf_cloud *scene, size_t ref_first, size_t ref_step, size_t ref_count,
                                b200ppf_hypothesis *const *peer_buffers, int n_peers, size_t slot_first,
                                size_t slot_step) {
    CHECK_CTX(ctx);
    if (!peer_buffers || n_peers < 1) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote scatter: no output buffers");
    for (int g = 0; g < n_peers; ++g)
        if (!peer_buffers[g]) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote scatter: null peer buffer");
    if (slot_step == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote scatter: slot step must be >= 1");
    return k3_vote(ctx, model, t, scene, ref_first, ref_step, ref_count, peer_buffers, n_peers, slot_first, slot_step);
}

int b200ppf_hyp_buffer_create(b200ppf_ctx *ctx, size_t n_records, b200ppf_hypothesis **buffer,
                              unsigned char ipc_handle[64]) {
    CHECK_CTX(ctx);
    if (!buffer) return fail_msg(ctx, B200PPF_ERR_INVALID, "hypothesis buffer: null argument");
    *buffer = nullptr;
    DeviceGuard guard(ctx->device);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle travels as 64 bytes");
    b200ppf_hypothesis *p = nullptr;
    PPF_CUDA(ctx, cudaMalloc(&p, std::max<size_t>(1, n_records) * sizeof(b200ppf_hypothesis)));  // cudaMalloc: IPC-exportable
    std::unique_ptr<b200ppf_hypothesis, cudaError_t (*)(void *)> owner(p, cudaFree);
    PPF_CUDA(ctx, cudaMemset(p, 0, std::max<size_t>(1, n_records) * sizeof(b200ppf_hypothesis)));
    if (ipc_handle) {
        cudaIpcMemHandle_t h;
        cudaError_t e = cudaIpcGetMemHandle(&h, p);
        if (e != cudaSuccess) return fail_msg(ctx, B200PPF_ERR_CUDA, cudaGetErrorString(e));
        memcpy(ipc_handle, &h, 64);
    }
    *buffer = owner.release();
    return B200PPF_OK;
}

int b200ppf_hyp_buffer_open(b200ppf_ctx *ctx, const unsigned char ipc_handle[64], b200ppf_hypothesis **buffer) {
    CHECK_CTX(ctx);
    if (!ipc_handle || !buffer) return fail_msg(ctx, B200PPF_ERR_INVALID, "hypothesis buffer: null argument");
    *buffer = nullptr;
    DeviceGuard guard(ctx->device);
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, 64);
    void *p = nullptr;
    PPF_CUDA(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *buffer = static_cast<b200ppf_hypothesis *>(p);
    return B200PPF_OK;
}

int b200ppf_hyp_buffer_download(b200ppf_ctx *ctx, const b200ppf_hypothesis *buffer, size_t first, size_t count,
                                b200ppf_hypothesis *host) {
    CHECK_CTX(ctx);
    if (!buffer || (count && !host)) return fail_msg(ctx, B200PPF_ERR_INVALID, "hypothesis buffer: null argument");
    DeviceGuard guard(ctx->device);
    if (count)
        PPF_CUDA(ctx, cudaMemcpyAsync(host, buffer + first, count * sizeof(b200ppf_hypothesis), cudaMemcpyDeviceToHost,
                                      ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_hyp_buffer_release(b200ppf_ctx *ctx, b200ppf_hypothesis *buffer, int opened_from_handle) {
    CHECK_CTX(ctx);
    if (!buffer) return B200PPF_OK;
    DeviceGuard guard(ctx->device);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (opened_from_handle) PPF_CUDA(ctx, cudaIpcCloseMemHandle(buffer));
    else PPF_CUDA(ctx, cudaFree(buffer));
    return B200PPF_OK;
}

int b200ppf_vote(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t, const b200ppf_cloud *scene,
                 size_t ref_first, size_t ref_step, size_t ref_count, b200ppf_hypothesis *hyps_host) {
    CHECK_CTX(ctx);
    if (ref_count && !hyps_host) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote: null output pointer");
    PPF_CUDA(ctx, grow_buffer(&ctx->d_hyps, &ctx->hyps_cap, ref_count));
    b200ppf_hypothesis *const target = ctx->d_hyps;
    int rc = k3_vote(ctx, model, t, scene, ref_first, ref_step, ref_count, &target, 1, 0, 1);
    if (rc) return rc;
    if (ref_count)
        PPF_CUDA(ctx, cudaMemcpyAsync(hyps_host, ctx->d_hyps, ref_count * sizeof(b200ppf_hypothesis),
                                      cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_vote_stats(b200ppf_ctx *ctx, uint64_t *stats4) {
    CHECK_CTX(ctx);
    if (!stats4) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote stats: null output pointer");
    stats4[0] = stats4[1] = stats4[2] = stats4[3] = 0;
    if (!ctx->d_stats) return B200PPF_OK;
    unsigned long long h[4];
    PPF_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_stats, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 4; ++k) stats4[k] = h[k];
    return B200PPF_OK;
}

int b200ppf_vote_debug_pairs(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t s_r,
                             uint8_t *in_radius, int32_t *d4, float *alpha_s) {
    CHECK_CTX(ctx);
    if (!in_radius || !d4 || !alpha_s) return fail_msg(ctx, B200PPF_ERR_INVALID, "debug pairs: null output pointer");
    return k3_debug_pairs(ctx, t, scene, s_r, in_radius, d4, alpha_s);
}

int b200ppf_vote_debug_accumulator(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t s_r,
                                   uint32_t *acc) {
    CHECK_CTX(ctx);
    if (!acc) return fail_msg(ctx, B200PPF_ERR_INVALID, "debug accumulator: null output pointer");
    return k3_debug_accumulator(ctx, t, scene, s_r, acc);
}

int b200ppf_debug_alpha_bins(b200ppf_ctx *ctx, float angle_step, int alpha_mode, int nalpha_rule, const float *alpha_m,
                             const float *alpha_s, size_t n, uint32_t *fast, uint32_t *exact) {
    if (!(angle_step > 0.0f) || alpha_mode < 0 || alpha_mode > 1 || nalpha_rule < 0 || nalpha_rule > 2 ||
        (n && (!alpha_m || !alpha_s || !fast || !exact)))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "debug alpha bins: bad argument");
    if (n == 0) return B200PPF_OK;
    if (!ctx) return k3_debug_alpha_bins(nullptr, angle_step, alpha_mode, nalpha_rule, alpha_m, alpha_s, n, fast, exact);
    DeviceGuard guard(ctx->device);
    return k3_debug_alpha_bins(ctx, angle_step, alpha_mode, nalpha_rule, alpha_m, alpha_s, n, fast, exact);
}

/* ---- parity hooks of the sorted-key primitives (sort_scan.cu) ------------------------------- */

int b200ppf_debug_radix_sort(b200ppf_ctx *ctx, uint32_t *keys, uint32_t *keys_alt, uint32_t *v0, uint32_t *v0_alt, uint32_t *v1,
                             uint32_t *v1_alt, size_t n, uint64_t max_key, int v0_iota, int *result_in_alt) {
    if (!result_in_alt || (n && (!keys || !keys_alt)) || !v0 != !v0_alt || !v1 != !v1_alt)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "debug radix sort: bad argument");
    CHECK_CTX(ctx);
    StreamBuf<uint32_t> k(ctx), ka(ctx), a(ctx), aa(ctx), b(ctx), ba(ctx);
    StreamBuf<uint32_t> *const dev[6] = {&k, &ka, &a, &aa, &b, &ba};
    uint32_t *const host[6] = {keys, keys_alt, v0, v0_alt, v1, v1_alt};
    for (int i = 0; i < 6; ++i)
        if (int rc = to_device(ctx, *dev[i], host[i], n)) return rc;
    bool alt = false;
    if (int rc = radix_sort_u32(ctx, k, ka, a, aa, b, ba, n, max_key, v0_iota != 0, &alt)) return rc;
    for (int i = 0; i < 6; ++i)
        if (int rc = to_host(ctx, host[i], *dev[i], n)) return rc;
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *result_in_alt = alt ? 1 : 0;
    return B200PPF_OK;
}

int b200ppf_debug_lower_bounds(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, int64_t dev_len, uint32_t n_keys,
                               uint32_t shift, uint32_t *offsets, size_t offsets_cap) {
    if ((n && !sorted) || !offsets || offsets_cap < (size_t)n_keys + 1 || dev_len > (int64_t)n || shift >= 32)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "debug lower bounds: bad argument");
    CHECK_CTX(ctx);
    StreamBuf<uint32_t> s(ctx), len(ctx), off(ctx);
    const uint32_t len_host = dev_len < 0 ? 0u : (uint32_t)dev_len;
    if (int rc = to_device(ctx, s, sorted, n)) return rc;
    if (int rc = to_device(ctx, len, dev_len < 0 ? nullptr : &len_host, 1)) return rc;
    if (int rc = to_device(ctx, off, offsets, offsets_cap)) return rc;
    if (int rc = lower_bounds(ctx, s, n, len, n_keys, shift, off)) return rc;
    if (int rc = to_host(ctx, offsets, off, offsets_cap)) return rc;
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_debug_flag_scan(b200ppf_ctx *ctx, const uint32_t *flags, uint32_t n, uint32_t *rank, size_t rank_cap, int host_total,
                            uint32_t *total) {
    if ((n && !flags) || (rank_cap && !rank) || rank_cap < n || !total)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "debug flag scan: bad argument");
    CHECK_CTX(ctx);
    StreamBuf<uint32_t> f(ctx), r(ctx), t(ctx);
    if (int rc = to_device(ctx, f, flags, n)) return rc;
    if (int rc = to_device(ctx, r, rank, rank_cap)) return rc;
    if (host_total) {
        if (int rc = flag_scan_host(ctx, f, n, r, total)) return rc;
    } else {
        if (int rc = to_device(ctx, t, total, 1)) return rc;
        if (int rc = flag_scan(ctx, f, n, r, t)) return rc;
        if (int rc = to_host(ctx, total, t, 1)) return rc;
    }
    if (int rc = to_host(ctx, rank, r, rank_cap)) return rc;
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_debug_scan_rows(b200ppf_ctx *ctx, uint32_t *data, uint32_t n_rows, uint32_t row_len, size_t data_cap, uint32_t *totals,
                            size_t totals_cap) {
    if (!data || !totals || n_rows == 0 || (uint64_t)n_rows * row_len > data_cap || totals_cap < n_rows)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "debug scan rows: bad argument");
    CHECK_CTX(ctx);
    StreamBuf<uint32_t> d(ctx), t(ctx);
    if (int rc = to_device(ctx, d, data, data_cap)) return rc;
    if (int rc = to_device(ctx, t, totals, totals_cap)) return rc;
    if (int rc = scan_rows(ctx, d, n_rows, row_len, t)) return rc;
    if (int rc = to_host(ctx, data, d, data_cap)) return rc;
    if (int rc = to_host(ctx, totals, t, totals_cap)) return rc;
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_debug_run_heads(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, uint32_t *head, size_t head_cap) {
    if ((n && !sorted) || (head_cap && !head) || head_cap < n)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "debug run heads: bad argument");
    CHECK_CTX(ctx);
    StreamBuf<uint32_t> s(ctx), h(ctx);
    if (int rc = to_device(ctx, s, sorted, n)) return rc;
    if (int rc = to_device(ctx, h, head, head_cap)) return rc;
    if (int rc = run_heads(ctx, s, n, h)) return rc;
    if (int rc = to_host(ctx, head, h, head_cap)) return rc;
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int b200ppf_microbench_atoms(b200ppf_ctx *ctx, int pattern, double *atoms_per_sec) {
    CHECK_CTX(ctx);
    if (!atoms_per_sec || pattern < 0 || pattern > 15) return fail_msg(ctx, B200PPF_ERR_INVALID, "microbench: bad argument");
    return microbench_atoms(ctx, pattern, atoms_per_sec);
}

/* ---- K4 ----------------------------------------------------------------------------------- */

int b200ppf_cluster_device(b200ppf_ctx *ctx, const b200ppf_hypothesis *hyps_device, size_t n, float pos_thr,
                           float rot_thr, float *poses16, uint32_t *votes, size_t *n_out) {
    CHECK_CTX(ctx);
    if (!poses16 || !votes || !n_out || (n && !hyps_device)) return fail_msg(ctx, B200PPF_ERR_INVALID, "cluster: null argument");
    return k4_cluster(ctx, hyps_device, n, pos_thr, rot_thr, poses16, votes, n_out);
}

int b200ppf_cluster(b200ppf_ctx *ctx, const b200ppf_hypothesis *hyps_host, size_t n, float pos_thr, float rot_thr,
                    float *poses16, uint32_t *votes, size_t *n_out) {
    CHECK_CTX(ctx);
    if (!poses16 || !votes || !n_out || (n && !hyps_host)) return fail_msg(ctx, B200PPF_ERR_INVALID, "cluster: null argument");
    *n_out = 0;
    if (n == 0) return B200PPF_OK;
    StreamBuf<b200ppf_hypothesis> d(ctx);
    PPF_CUDA(ctx, d.alloc(n));
    PPF_CUDA(ctx, cudaMemcpyAsync(d, hyps_host, n * sizeof(b200ppf_hypothesis), cudaMemcpyHostToDevice, ctx->stream));
    return k4_cluster(ctx, d, n, pos_thr, rot_thr, poses16, votes, n_out);
}

int b200ppf_cluster_assignment(b200ppf_ctx *ctx, uint32_t *assignment, size_t n, size_t *n_clusters) {
    CHECK_CTX(ctx);
    if (n_clusters) *n_clusters = ctx->n_clusters;
    if (!assignment) return B200PPF_OK;
    if (n != ctx->assign_n || !ctx->d_assign)
        return fail_msg(ctx, B200PPF_ERR_STATE, "cluster assignment: size does not match the last cluster call");
    PPF_CUDA(ctx, cudaMemcpyAsync(assignment, ctx->d_assign, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

/* ---- K5 ----------------------------------------------------------------------------------- */

int b200ppf_transform(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, const float *pose16, float *out_host,
                      size_t out_stride_floats) {
    CHECK_CTX(ctx);
    if (!cloud || !pose16 || (cloud->n && !out_host)) return fail_msg(ctx, B200PPF_ERR_INVALID, "transform: null argument");
    return k5_transform(ctx, cloud, pose16, out_host, out_stride_floats);
}

/* ---- scene pre-processing (prep.cu) ------------------------------------------------------ */

int b200ppf_cloud_upload_xyz(b200ppf_ctx *ctx, const float *host, size_t n, size_t stride, b200ppf_cloud **out) {
    CHECK_CTX(ctx);
    if (!out) return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud upload: null output pointer");
    *out = nullptr;
    if (n && !host) return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud upload: null host pointer");
    if (stride < 3) return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud upload: rows must hold at least x y z");
    if (n > 0xFFFFFFF0ull) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "cloud upload: more than 2^32 points");
    return prep_upload_xyz(ctx, host, n, stride, out);
}

int b200ppf_cloud_download(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, float *host, size_t stride, size_t noff,
                           size_t coff) {
    CHECK_CTX(ctx);
    if (!cloud || (cloud->n && !host)) return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud download: null argument");
    if (stride < 3 || (noff && (noff < 3 || noff + 3 > stride)) || (coff && (coff < 3 || coff >= stride)) ||
        (noff && coff && coff >= noff && coff < noff + 3))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cloud download: stride / offsets do not describe [x y z .. nx ny nz .. curvature]");
    return prep_download(ctx, cloud, host, stride, noff, coff);
}

int b200ppf_voxel_grid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *leaf3, b200ppf_cloud **out) {
    CHECK_CTX(ctx);
    if (!in || !leaf3 || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "voxel grid: null argument");
    *out = nullptr;
    for (int k = 0; k < 3; ++k)
        if (!(leaf3[k] > 0.0f) || !std::isfinite(leaf3[k])) return fail_msg(ctx, B200PPF_ERR_INVALID, "voxel grid: leaf size must be positive");
    ctx->error.clear();
    return prep_voxel_grid(ctx, in, leaf3, out);
}

int b200ppf_knn(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, int k, uint32_t *idx_host, float *d2_host) {
    CHECK_CTX(ctx);
    if (!cloud) return fail_msg(ctx, B200PPF_ERR_INVALID, "knn: null cloud");
    if (k < 1 || k > 128 || (size_t)k > std::max<size_t>(1, cloud->n))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "knn: k must be in 1 .. min(n, 128)");
    return prep_knn(ctx, cloud, k, idx_host, d2_host);
}

int b200ppf_statistical_outlier_removal(b200ppf_ctx *ctx, const b200ppf_cloud *in, int mean_k, double stddev_mul,
                                        b200ppf_cloud **out, uint32_t *kept_host, float *distances_host, double *threshold) {
    CHECK_CTX(ctx);
    if (!in || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "statistical outlier removal: null argument");
    *out = nullptr;
    if (mean_k < 1 || mean_k > 127) return fail_msg(ctx, B200PPF_ERR_INVALID, "statistical outlier removal: mean_k must be in 1 .. 127");
    if (in->n < (size_t)mean_k + 1)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "statistical outlier removal: the cloud needs more than mean_k points");
    return prep_sor(ctx, in, mean_k, stddev_mul, out, kept_host, distances_host, threshold);
}

int b200ppf_normal_estimation(b200ppf_ctx *ctx, b200ppf_cloud *cloud, int k, const float *viewpoint3, int cov_mode) {
    CHECK_CTX(ctx);
    if (!cloud) return fail_msg(ctx, B200PPF_ERR_INVALID, "normal estimation: null cloud");
    if (k < 1 || k > 128) return fail_msg(ctx, B200PPF_ERR_INVALID, "normal estimation: k must be in 1 .. 128");
    if (cov_mode != B200PPF_COVARIANCE_SHIFTED && cov_mode != B200PPF_COVARIANCE_RAW)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "normal estimation: unknown covariance mode");
    return prep_normals(ctx, cloud, k, viewpoint3, cov_mode);
}

int b200ppf_curvature_edges(b200ppf_ctx *ctx, const b200ppf_cloud *in, float threshold, b200ppf_cloud **out) {
    CHECK_CTX(ctx);
    if (!in || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "curvature edges: null argument");
    *out = nullptr;
    return prep_curvature_edges(ctx, in, threshold, out);
}

int b200ppf_normalize_normals(b200ppf_ctx *ctx, b200ppf_cloud *cloud) {
    CHECK_CTX(ctx);
    if (!cloud) return fail_msg(ctx, B200PPF_ERR_INVALID, "normalize normals: null cloud");
    return prep_renormalize(ctx, cloud);
}

int b200ppf_frustum_corners(const float *depth, int rows, int cols, int box_x, int box_y, int box_w, int box_h, double fx,
                            double fy, double ppx, double ppy, float *corners12) {
    if (!depth || !corners12 || rows < 1 || cols < 1 || box_w < 0 || box_h < 0 || box_x >= cols || box_y >= rows ||
        box_x + box_w + 30 < 0 || box_y + box_h + 30 < 0 || !(fx != 0.0) || !(fy != 0.0))
        return fail_msg(nullptr, B200PPF_ERR_INVALID, "frustum corners: bad argument");
    prep_frustum_corners(depth, rows, cols, box_x, box_y, box_w, box_h, fx, fy, ppx, ppy, corners12);
    return B200PPF_OK;
}

int b200ppf_crop_pyramid(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, b200ppf_cloud **out,
                         uint32_t *kept_host) {
    CHECK_CTX(ctx);
    if (!in || !corners12 || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "crop: null argument");
    *out = nullptr;
    for (int k = 0; k < 12; ++k)
        if (!std::isfinite(corners12[k])) return fail_msg(ctx, B200PPF_ERR_INVALID, "crop: non-finite corner");
    return prep_crop_pyramid(ctx, in, corners12, out, kept_host);
}

int b200ppf_crop_pyramids(b200ppf_ctx *ctx, const b200ppf_cloud *in, const float *corners12, size_t n_boxes,
                          b200ppf_cloud **out) {
    CHECK_CTX(ctx);
    if (!in || !corners12 || !out) return fail_msg(ctx, B200PPF_ERR_INVALID, "crop: null argument");
    if (n_boxes < 1 || n_boxes > 64) return fail_msg(ctx, B200PPF_ERR_INVALID, "crop: n_boxes must be in 1 .. 64");
    for (size_t b = 0; b < n_boxes; ++b) out[b] = nullptr;
    if (in->ctx != ctx) return fail_msg(ctx, B200PPF_ERR_INVALID, "crop: the cloud belongs to another context");
    for (size_t k = 0; k < 12 * n_boxes; ++k)
        if (!std::isfinite(corners12[k])) {
            char msg[96];
            snprintf(msg, sizeof(msg), "crop: box %zu: non-finite corner", k / 12);
            return fail_msg(ctx, B200PPF_ERR_INVALID, msg);
        }
    return prep_crop_pyramids(ctx, in, corners12, n_boxes, out);
}

int b200ppf_debug_knn_host(const float *xyz, size_t n, size_t stride, int k, int mode, float cell_edge, const float *viewpoint3,
                           int cov_mode, uint32_t *idx, float *d2, float *mean_dist, float *normals4) {
    if ((n && !xyz) || stride < 3 || k < 1 || k > 128 || (size_t)k > std::max<size_t>(1, n) || mode < 0 || mode > 2 ||
        (mode == 0 && (!idx || !d2)) || (mode == 1 && (!mean_dist || k < 2)) || (mode == 2 && !normals4))
        return fail_msg(nullptr, B200PPF_ERR_INVALID, "debug knn: bad argument");
    return prep_debug_knn_host(xyz, n, stride, k, mode, cell_edge, viewpoint3, cov_mode, idx, d2, mean_dist, normals4);
}

/* ---- align -------------------------------------------------------------------------------- */

int b200ppf_icp_refine(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_cloud *scene,
                       const b200ppf_icp_params *params, double *poses16, size_t n_poses, double *residuals,
                       uint64_t *iterations) {
    CHECK_CTX(ctx);
    if (!model || !scene || (n_poses && !poses16)) return fail_msg(ctx, B200PPF_ERR_INVALID, "icp: null argument");
    DeviceGuard guard(ctx->device);
    const b200ppf_icp_params p = params ? *params : ICP_DEFAULT;
    return k6_icp_refine(ctx, model, scene, p.max_iterations, p.tolerance, p.rejection_scale, p.num_levels, poses16,
                         n_poses, residuals, iterations);
}

int b200ppf_icp_refine_batch(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_icp_params *params,
                             uint64_t *iterations) {
    CHECK_CTX(ctx);
    if (n_jobs && !jobs) return fail_msg(ctx, B200PPF_ERR_INVALID, "icp batch: null jobs");
    for (size_t j = 0; j < n_jobs; ++j) {
        char msg[128];
        const b200ppf_icp_job &jb = jobs[j];
        const char *why = !jb.model || !jb.scene || (jb.n_poses && !jb.poses16) ? "null argument"
                          : jb.model->ctx != ctx || jb.scene->ctx != ctx       ? "a cloud belongs to another context"
                                                                                : nullptr;
        if (why) {
            snprintf(msg, sizeof(msg), "icp batch: job %zu: %s", j, why);
            return fail_msg(ctx, B200PPF_ERR_INVALID, msg);
        }
    }
    const b200ppf_icp_params p = params ? *params : ICP_DEFAULT;
    return k6_icp_refine_batch(ctx, jobs, n_jobs, p.max_iterations, p.tolerance, p.rejection_scale, p.num_levels, iterations);
}

void b200ppf_verify_params_default(b200ppf_verify_params *p) {
    if (!p) return;
    p->inlier_dist = 0.01f;                              // the reference's leaf
    p->normal_angle = 30.0f / 180.0f * 3.14159265358979f;
}

int b200ppf_score_poses(b200ppf_ctx *ctx, const b200ppf_icp_job *jobs, size_t n_jobs, const b200ppf_verify_params *params,
                        b200ppf_pose_fit *fits) {
    CHECK_CTX(ctx);
    b200ppf_verify_params p;
    if (int rc = verify_params(ctx, params, &p)) return rc;
    if (n_jobs && !jobs) return fail_msg(ctx, B200PPF_ERR_INVALID, "score poses: null jobs");
    size_t n_poses = 0;
    for (size_t j = 0; j < n_jobs; ++j) {
        char msg[128];
        const b200ppf_icp_job &jb = jobs[j];
        const char *why = !jb.model || !jb.scene || (jb.n_poses && !jb.poses16) ? "null argument"
                          : jb.model->ctx != ctx || jb.scene->ctx != ctx       ? "a cloud belongs to another context"
                                                                                : nullptr;
        for (size_t k = 0; !why && k < 16 * jb.n_poses; ++k)
            if (!std::isfinite(jb.poses16[k])) why = "a pose is not finite";
        if (why) {
            snprintf(msg, sizeof(msg), "score poses: job %zu: %s", j, why);
            return fail_msg(ctx, B200PPF_ERR_INVALID, msg);
        }
        n_poses += jb.n_poses;
    }
    if (n_poses && !fits) return fail_msg(ctx, B200PPF_ERR_INVALID, "score poses: null fits");
    return verify_score_poses(ctx, jobs, n_jobs, p, fits);
}

int b200ppf_register(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t,
                     const b200ppf_cloud *scene, size_t ref_rate, float pos_thr, float rot_thr, float *final16,
                     float *poses16, uint32_t *votes, size_t *n_out) {
    CHECK_CTX(ctx);
    if (!scene || !poses16 || !votes || !n_out) return fail_msg(ctx, B200PPF_ERR_INVALID, "register: null argument");
    *n_out = 0;
    if (ref_rate == 0) ref_rate = 1;
    const size_t ref_count = (scene->n + ref_rate - 1) / ref_rate;
    if (ref_count == 0) return fail_msg(ctx, B200PPF_ERR_STATE, "register: empty scene");
    PPF_CUDA(ctx, grow_buffer(&ctx->d_hyps, &ctx->hyps_cap, ref_count));
    b200ppf_hypothesis *const reg_target = ctx->d_hyps;
    int rc = k3_vote(ctx, model, t, scene, 0, ref_rate, ref_count, &reg_target, 1, 0, 1);
    if (rc) return rc;
    rc = k4_cluster(ctx, ctx->d_hyps, ref_count, pos_thr, rot_thr, poses16, votes, n_out);
    if (rc) return rc;
    if (*n_out && final16) memcpy(final16, poses16, 16 * sizeof(float));
    return B200PPF_OK;
}

}  // extern "C"

namespace {

// the pre-processing after the crop: Subsampling -> OutlierProcessing -> NormalEstimation -> EdgeExtraction (with_edges) ->
// PointCloudXYZNormalToMat, stage sizes and times into res
template <class Params>
int object_prep(b200ppf_ctx *ctx, const b200ppf_cloud *cropped, const Params &p, bool with_edges, b200ppf_object_result *res,
                CloudPtr *object, CloudPtr *edges) {
    const float leaf3[3] = {p.leaf, p.leaf, p.leaf};
    b200ppf_cloud *sampled_c = nullptr, *object_c = nullptr, *edges_c = nullptr;  // each owned once its call returns
    int rc = b200ppf_voxel_grid(ctx, cropped, leaf3, &sampled_c);
    const CloudPtr sampled(sampled_c);
    if (rc) return rc;
    res->voxel_ms = ctx->timings.prep_ms;
    res->n_sampled = (uint32_t)sampled->n;
    rc = b200ppf_statistical_outlier_removal(ctx, sampled.get(), p.sor_mean_k, p.sor_stddev_mul, &object_c, nullptr, nullptr, nullptr);
    object->reset(object_c);
    if (rc) return rc;
    res->outlier_ms = ctx->timings.prep_ms;
    res->n_filtered = (uint32_t)object_c->n;
    if ((rc = b200ppf_normal_estimation(ctx, object_c, p.normal_k, nullptr, B200PPF_COVARIANCE_SHIFTED))) return rc;
    res->normals_ms = ctx->timings.prep_ms;
    if (with_edges) {
        rc = b200ppf_curvature_edges(ctx, object_c, p.edge_curvature, &edges_c);
        edges->reset(edges_c);
        if (rc) return rc;
        res->edges_ms = ctx->timings.prep_ms;
        res->n_edges = (uint32_t)edges_c->n;
    }
    if ((rc = b200ppf_normalize_normals(ctx, object_c))) return rc;
    if (edges_c && (rc = b200ppf_normalize_normals(ctx, edges_c))) return rc;
    return B200PPF_OK;
}

// a CUDA or memory failure ends a call; any other failure of a box's chain is that box's status
bool fatal(int rc) { return rc == B200PPF_ERR_CUDA || rc == B200PPF_ERR_NOMEM; }

// The chain of every match call, frame or per-object: crop all boxes in one pass, then per box the pre-processing and
// `match(b, object, edges, &poses, &votes)`, the engine's matching step (it fills the box's match_ms and n_poses and returns
// its best poses, 16 doubles each, most-voted first, and their clusters' votes), then one batched ICP of the top icp_poses
// poses of every box that reached it against models[b].  With verify (checked), the candidates of every such box (the
// refined poses, or the top pose alone without ICP) are then scored in one b200ppf_score_poses against models[b] and the
// box's object cloud, the best one becomes the box's result, and candidates (may be NULL) receives them all, max(icp_poses,
// 1) slots per box.  When box 0 succeeds, object_out / edges_out (either may be NULL) receive its clouds.
template <class Params, class Match>
int match_boxes(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                const b200ppf_cloud *const *models, const Params &p, bool with_edges, b200ppf_object_result *results, int *status,
                b200ppf_cloud **object_out, b200ppf_cloud **edges_out, const b200ppf_verify_params *verify,
                b200ppf_candidate *candidates, Match match) {
    const auto t0 = std::chrono::steady_clock::now();
    for (size_t b = 0; b < n_boxes; ++b) {
        memset(&results[b], 0, sizeof(results[b]));
        status[b] = B200PPF_OK;
    }
    std::vector<CloudPtr> crops(n_boxes), objects(n_boxes), edges(n_boxes);
    {
        std::vector<b200ppf_cloud *> out(n_boxes, nullptr);
        const int rc = b200ppf_crop_pyramids(ctx, scene, corners12, n_boxes, out.data());
        for (size_t b = 0; b < n_boxes; ++b) crops[b].reset(out[b]);
        if (rc) return rc;
    }
    const float crop_ms = ctx->timings.prep_ms;
    std::vector<std::vector<double>> refined(n_boxes), residuals(n_boxes);
    std::vector<std::vector<uint32_t>> votes(n_boxes);
    std::vector<size_t> n_cand(n_boxes, 0);
    std::vector<b200ppf_icp_job> jobs;
    for (size_t b = 0; b < n_boxes; ++b) {
        b200ppf_object_result *res = &results[b];
        res->n_cropped = (uint32_t)crops[b]->n;
        int rc = B200PPF_OK;
        if (crops[b]->n == 0) rc = fail_msg(ctx, B200PPF_ERR_STATE, "match: no scene point inside the box's frustum");
        if (!rc) rc = object_prep(ctx, crops[b].get(), p, with_edges, res, &objects[b], &edges[b]);
        crops[b].reset();  // the frame's crops go back to the pool as soon as their box is through
        if (!rc) rc = match(b, objects[b].get(), edges[b].get(), &refined[b], &votes[b]);
        if (!rc) res->votes = votes[b].empty() ? 0 : votes[b][0];
        if (!rc && res->n_poses == 0)  // the reference exits there, :502-507
            rc = fail_msg(ctx, B200PPF_ERR_STATE, "match: the matching returned no pose");
        if (fatal(rc)) return rc;
        status[b] = rc;
        if (rc) continue;
        const size_t n_icp = std::min<size_t>(res->n_poses, p.icp_poses > 0 ? (size_t)p.icp_poses : 0);
        n_cand[b] = std::max<size_t>(n_icp, 1);
        residuals[b].assign(n_cand[b], 0.0);
        if (n_icp) jobs.push_back(b200ppf_icp_job{models[b], objects[b].get(), refined[b].data(), n_icp, residuals[b].data()});
    }
    float icp_ms = 0.0f;
    if (!jobs.empty()) {
        if (int rc = b200ppf_icp_refine_batch(ctx, jobs.data(), jobs.size(), &p.icp, nullptr)) return rc;
        icp_ms = ctx->timings.icp_ms;
    }
    std::vector<std::vector<b200ppf_pose_fit>> fits(n_boxes);
    std::vector<size_t> best(n_boxes, 0);  // resultsSub[0] unless verified
    if (verify) {
        std::vector<b200ppf_icp_job> score_jobs;
        size_t n_scored = 0;
        for (size_t b = 0; b < n_boxes; ++b)
            if (!status[b]) {
                score_jobs.push_back(b200ppf_icp_job{models[b], objects[b].get(), refined[b].data(), n_cand[b], nullptr});
                n_scored += n_cand[b];
            }
        std::vector<b200ppf_pose_fit> all(n_scored);
        if (int rc = verify_score_poses(ctx, score_jobs.data(), score_jobs.size(), *verify, all.data())) return rc;
        size_t at = 0;
        for (size_t b = 0; b < n_boxes; ++b) {
            if (status[b]) continue;
            fits[b].assign(all.begin() + at, all.begin() + at + n_cand[b]);
            at += n_cand[b];
            for (size_t k = 1; k < n_cand[b]; ++k)
                if (fits[b][k].fit > fits[b][best[b]].fit) best[b] = k;
        }
    }
    const float wall = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    for (size_t b = 0; b < n_boxes; ++b) {
        b200ppf_object_result *res = &results[b];
        if (!status[b]) {
            memcpy(res->pose, refined[b].data() + 16 * best[b], 16 * sizeof(double));
            res->residual = residuals[b][best[b]];
            res->votes = votes[b][best[b]];
        }
        res->crop_ms = crop_ms;
        res->icp_ms = icp_ms;
        res->total_wall_ms = wall;
    }
    if (verify && candidates) {
        const size_t slots = p.icp_poses > 1 ? (size_t)p.icp_poses : 1;
        for (size_t b = 0; b < n_boxes; ++b) {
            b200ppf_candidate *c = candidates + b * slots;
            memset(c, 0, slots * sizeof(*c));
            for (size_t k = 0; k < slots; ++k) c[k].rank = UINT32_MAX;
            if (status[b]) continue;
            std::vector<size_t> order(n_cand[b]);
            for (size_t k = 0; k < order.size(); ++k) order[k] = k;
            std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) { return fits[b][x].fit > fits[b][y].fit; });
            for (size_t i = 0; i < order.size(); ++i) {
                const size_t k = order[i];
                memcpy(c[i].pose, refined[b].data() + 16 * k, 16 * sizeof(double));
                c[i].residual = residuals[b][k];
                c[i].votes = votes[b][k];
                c[i].rank = (uint32_t)k;
                c[i].fit = fits[b][k];
            }
        }
    }
    if (!status[0]) {
        if (object_out) *object_out = objects[0].release();
        if (edges_out) *edges_out = edges[0].release();
    }
    return B200PPF_OK;
}

// the argument checks both engines share
int frame_args(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12, const void *per_box,
               const b200ppf_cloud *const *models, const b200ppf_object_result *results, const int *status) {
    if (!scene || !corners12 || !per_box || !models || !results || !status)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "match: null argument");
    if (n_boxes < 1 || n_boxes > 64) return fail_msg(ctx, B200PPF_ERR_INVALID, "match: n_boxes must be in 1 .. 64");
    if (scene->ctx != ctx) return fail_msg(ctx, B200PPF_ERR_INVALID, "match: the scene belongs to another context");
    for (size_t b = 0; b < n_boxes; ++b)
        if (!models[b] || models[b]->ctx != ctx) {
            char msg[128];
            snprintf(msg, sizeof(msg), "match: box %zu: the model is NULL or belongs to another context", b);
            return fail_msg(ctx, B200PPF_ERR_INVALID, msg);
        }
    return B200PPF_OK;
}

// b200ppf_match_frame; b200ppf_match_object is this on one box.  The PCL matching does not read the edge cloud: it is
// extracted when the caller wants it (want_edges) and edge_curvature > 0.
int ppf_match(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12, const b200ppf_cloud *const *models,
              const b200ppf_table *const *tables, const b200ppf_object_params *params, b200ppf_object_result *results, int *status,
              bool want_edges, b200ppf_cloud **object_out, b200ppf_cloud **edges_out, const b200ppf_verify_params *verify = nullptr,
              b200ppf_candidate *candidates = nullptr) {
    CHECK_CTX(ctx);
    if (int rc = frame_args(ctx, scene, n_boxes, corners12, tables, models, results, status)) return rc;
    for (size_t b = 0; b < n_boxes; ++b)
        if (!tables[b] || tables[b]->ctx != ctx) {
            char msg[128];
            snprintf(msg, sizeof(msg), "match: box %zu: the table is NULL or belongs to another context", b);
            return fail_msg(ctx, B200PPF_ERR_INVALID, msg);
        }
    b200ppf_object_params p;
    b200ppf_object_params_default(&p);
    if (params) p = *params;
    auto match = [&](size_t b, const b200ppf_cloud *object, const b200ppf_cloud *, std::vector<double> *poses,
                     std::vector<uint32_t> *cluster_votes) {
        b200ppf_object_result *res = &results[b];
        float poses16[3 * 16];
        uint32_t votes[3] = {0, 0, 0};
        size_t n_poses = 0;
        if (int rc = b200ppf_register(ctx, models[b], tables[b], object, p.ref_rate, p.pos_thr, p.rot_thr, nullptr, poses16, votes,
                                      &n_poses))
            return rc;
        b200ppf_timings tm;
        b200ppf_get_timings(ctx, &tm);
        res->match_ms = tm.grid_ms + tm.vote_ms + tm.pose_ms + tm.cluster_ms;
        res->n_poses = (uint32_t)n_poses;
        poses->assign(poses16, poses16 + 16 * n_poses);
        cluster_votes->assign(votes, votes + n_poses);
        return B200PPF_OK;
    };
    return match_boxes(ctx, scene, n_boxes, corners12, models, p, p.edge_curvature > 0.0f && want_edges, results, status, object_out,
                       edges_out, verify, candidates, match);
}

// b200cv_match_frame; b200cv_match_object is this on one box.  The edge cloud is extracted when edge_curvature > 0 and
// Matching_S2B needs it (use_edges) or the caller wants it (want_edges).
int cv_match(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12, b200cv_detector *const *detectors,
             const b200ppf_cloud *const *models, const b200cv_object_params *params, b200ppf_object_result *results, int *status,
             bool want_edges, b200ppf_cloud **object_out, b200ppf_cloud **edges_out, const b200ppf_verify_params *verify = nullptr,
             b200ppf_candidate *candidates = nullptr) {
    CHECK_CTX(ctx);
    if (int rc = frame_args(ctx, scene, n_boxes, corners12, detectors, models, results, status)) return rc;
    for (size_t b = 0; b < n_boxes; ++b) {
        char msg[128];
        if (!detectors[b] || cv_detector_context(detectors[b]) != ctx) {
            snprintf(msg, sizeof(msg), "cv match: box %zu: the detector is NULL or belongs to another context", b);
            return fail_msg(ctx, B200PPF_ERR_INVALID, msg);
        }
        if (!cv_detector_trained(detectors[b])) {
            snprintf(msg, sizeof(msg), "cv match: box %zu: the detector is not trained", b);
            return fail_msg(ctx, B200PPF_ERR_STATE, msg);
        }
    }
    b200cv_object_params p;
    b200cv_object_params_default(&p);
    if (params) p = *params;
    if (p.use_edges && !(p.edge_curvature > 0.0f))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "cv match: Matching_S2B needs the edge cloud, edge_curvature must be positive");
    const size_t cap = p.icp_poses > 1 ? (size_t)p.icp_poses : 1;
    std::vector<b200cv_pose> poses(cap);
    cudaEvent_t ev[2] = {nullptr, nullptr};  // the context's events are taken by the stages inside the match
    PPF_CUDA(ctx, cudaEventCreate(&ev[0]));
    if (cudaEventCreate(&ev[1]) != cudaSuccess) {
        cudaEventDestroy(ev[0]);
        return fail_msg(ctx, B200PPF_ERR_CUDA, "cv match: cudaEventCreate failed");
    }
    auto match = [&](size_t b, const b200ppf_cloud *object, const b200ppf_cloud *edges, std::vector<double> *refined,
                     std::vector<uint32_t> *cluster_votes) {
        b200ppf_object_result *res = &results[b];
        if (p.use_edges && edges->n == 0)
            return fail_msg(ctx, B200PPF_ERR_STATE, "cv match: the object has no edge point for Matching_S2B to pair with");
        size_t n_clusters = 0;
        cudaEventRecord(ev[0], ctx->stream);
        int rc = b200cv_detector_match_cloud(detectors[b], object, p.use_edges ? edges : nullptr, p.relative_scene_sample_step,
                                             p.relative_scene_distance, poses.data(), cap, &n_clusters);
        cudaEventRecord(ev[1], ctx->stream);
        if (rc == B200PPF_OK && cudaEventSynchronize(ev[1]) == cudaSuccess) cudaEventElapsedTime(&res->match_ms, ev[0], ev[1]);
        if (rc) return rc;
        const size_t n_kept = std::min(n_clusters, cap);
        refined->resize(16 * n_kept);
        cluster_votes->resize(n_kept);
        for (size_t k = 0; k < n_kept; ++k) {
            memcpy(refined->data() + 16 * k, poses[k].pose, 16 * sizeof(double));
            (*cluster_votes)[k] = poses[k].num_votes;
        }
        res->n_poses = (uint32_t)n_clusters;
        return B200PPF_OK;
    };
    const int rc = match_boxes(ctx, scene, n_boxes, corners12, models, p, p.edge_curvature > 0.0f && (p.use_edges || want_edges),
                               results, status, object_out, edges_out, verify, candidates, match);
    cudaEventDestroy(ev[0]);
    cudaEventDestroy(ev[1]);
    return rc;
}

}  // namespace

extern "C" {

void b200ppf_object_params_default(b200ppf_object_params *p) {
    if (!p) return;
    p->leaf = 0.01f;
    p->sor_mean_k = 50;       // OutlierProcessing(50, thresh), src/YOLO_cropping_ppf_test.cpp:98
    p->sor_stddev_mul = 1.0;
    p->normal_k = 30;         // NormalEstimation(30), :101
    p->edge_curvature = 0.03f;  // EdgeExtraction(0.03), :103
    p->ref_rate = 20;         // relSceneSampleStep = 0.05, include/CloudProcessing.h:481
    p->pos_thr = 0.01f;       // PCL defaults of PPFRegistration
    p->rot_thr = 20.0f / 180.0f * 3.14159265358979f;
    p->icp_poses = 5;         // N = 5, include/CloudProcessing.h:508
    p->icp = ICP_DEFAULT;
}

int b200ppf_match_object(b200ppf_ctx *ctx, const b200ppf_cloud *scene, const float *corners12, const b200ppf_cloud *model,
                         const b200ppf_table *table, const b200ppf_object_params *params, b200ppf_object_result *res,
                         b200ppf_cloud **object_out, b200ppf_cloud **edges_out) {
    if (object_out) *object_out = nullptr;
    if (edges_out) *edges_out = nullptr;
    int status = B200PPF_OK;
    const int rc = ppf_match(ctx, scene, 1, corners12, &model, &table, params, res, &status, edges_out != nullptr, object_out, edges_out);
    return rc ? rc : status;
}

void b200cv_object_params_default(b200cv_object_params *p) {
    if (!p) return;
    p->leaf = 0.01f;
    p->sor_mean_k = 50;                   // OutlierProcessing(50, thresh), src/YOLO_cropping_ppf_test.cpp:98
    p->sor_stddev_mul = 1.0;
    p->normal_k = 30;                     // NormalEstimation(30), :101
    p->edge_curvature = 0.03f;            // EdgeExtraction(0.03), :103
    p->use_edges = 1;                     // Matching_S2B, :120
    p->relative_scene_sample_step = 0.05;  // match_S2B(object, edges, results, 0.05, 0.05), include/CloudProcessing.h:481-495
    p->relative_scene_distance = 0.05;
    p->icp_poses = 5;                     // N = 5, include/CloudProcessing.h:508
    p->icp = ICP_DEFAULT;
}

int b200cv_match_object(b200cv_detector *d, const b200ppf_cloud *scene, const float *corners12, const b200ppf_cloud *model,
                        const b200cv_object_params *params, b200ppf_object_result *res, b200ppf_cloud **object_out,
                        b200ppf_cloud **edges_out) {
    if (object_out) *object_out = nullptr;
    if (edges_out) *edges_out = nullptr;
    if (!d) return fail_msg(nullptr, B200PPF_ERR_INVALID, "cv match object: null detector");
    int status = B200PPF_OK;
    const int rc = cv_match(cv_detector_context(d), scene, 1, corners12, &d, &model, params, res, &status, edges_out != nullptr,
                            object_out, edges_out);
    return rc ? rc : status;
}

int b200cv_match_frame(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                       b200cv_detector *const *detectors, const b200ppf_cloud *const *models, const b200cv_object_params *params,
                       b200ppf_object_result *results, int *status) {
    return cv_match(ctx, scene, n_boxes, corners12, detectors, models, params, results, status, true, nullptr, nullptr);
}

int b200ppf_match_frame(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                        const b200ppf_cloud *const *models, const b200ppf_table *const *tables, const b200ppf_object_params *params,
                        b200ppf_object_result *results, int *status) {
    return ppf_match(ctx, scene, n_boxes, corners12, models, tables, params, results, status, true, nullptr, nullptr);
}

int b200cv_match_frame_verified(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                                b200cv_detector *const *detectors, const b200ppf_cloud *const *models,
                                const b200cv_object_params *params, const b200ppf_verify_params *verify,
                                b200ppf_object_result *results, int *status, b200ppf_candidate *candidates) {
    CHECK_CTX(ctx);
    b200ppf_verify_params v;
    if (int rc = verify_params(ctx, verify, &v)) return rc;
    return cv_match(ctx, scene, n_boxes, corners12, detectors, models, params, results, status, true, nullptr, nullptr, &v, candidates);
}

int b200ppf_match_frame_verified(b200ppf_ctx *ctx, const b200ppf_cloud *scene, size_t n_boxes, const float *corners12,
                                 const b200ppf_cloud *const *models, const b200ppf_table *const *tables,
                                 const b200ppf_object_params *params, const b200ppf_verify_params *verify,
                                 b200ppf_object_result *results, int *status, b200ppf_candidate *candidates) {
    CHECK_CTX(ctx);
    b200ppf_verify_params v;
    if (int rc = verify_params(ctx, verify, &v)) return rc;
    return ppf_match(ctx, scene, n_boxes, corners12, models, tables, params, results, status, true, nullptr, nullptr, &v, candidates);
}

}  // extern "C"
