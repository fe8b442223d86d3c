// k2_table.cu — K2: the model hash table as a radix-sorted CSR (replaces PPFHashMapSearch).
//
// [PCL] registration/src/ppf_registration.cpp PPFHashMapSearch::setInputFeatureCloud builds an
// unordered_multimap<HashKeyStruct,(i,j)> with one heap node per ordered model pair plus the
// alpha_m_[i][j] matrix (SURVEY.md A.3).  Here:
//   keys    quantise exactly as PCL: d = floor(f / step) per component, packed densely into one
//           32-bit integer (no hashing, hence no collisions), prefixed by the accumulator slice
//           of model row i so that one CSR serves every slice;
//   phase   when 2*pi/angle_step is an integer up to the guard band (PCL's 12 degrees is), the sort
//           key is extended by the phase cell of alpha_m — the position of (alpha_m + pi)/step inside
//           its bin, 16 cells — so that a bucket is ordered (cell, i, j) and the voting kernel can
//           shift whole ranges of it by one constant (ppf_math.cuh "constant-shift voting");
//   sort    stable LSD radix sort of (key.cell, pair index, alpha_m);
//   CSR     offsets[key] (buckets) and sub_offsets[key.cell] by binary search over the sorted keys;
//           per entry a 4-byte hot word (wrap field | accumulator byte offset of (row, bin of alpha_m)),
//           alpha_m in fixed point and as PCL's float; j survives only in entry_idx.  The API
//           exports restore the canonical (i, j) order inside a bucket.
// NaN signatures (diagonal / failed pairs) are dropped: no finite query can reach the key PCL
// files them under (A.3).
#include <algorithm>
#include <cmath>
#include <vector>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

constexpr uint32_t INVALID_KEY = 0xFFFFFFFFu;

__device__ __forceinline__ uint32_t slice_of(uint32_t i, uint32_t slice_rows) { return i / slice_rows; }

// sort key: (slice, packed feature key, phase cell of alpha_m)
__device__ __forceinline__ uint32_t sort_key(const KeyParams &kp, const BinParams &bp, uint32_t i, uint32_t k, float alpha) {
    uint32_t key = slice_of(i, kp.slice_rows) * kp.key_space + k;
    if (bp.cells_log2) {
        const uint32_t cell = filed_phase_cell(bp, alpha);  // fp32 estimate, exact at the circular edge (ppf_math.cuh)
        key = (key << bp.cells_log2) | cell;
        // merged votes: the bin of alpha_m (from the fixed-point phase the hot word is made of) follows the cell, so
        // that the entries of one (cell, bin, model row) — identical votes for every scene pair outside the cell —
        // end up adjacent after the stable sort
        if (kp.merge_bits) key = (key << kp.merge_bits) | (alpha == alpha ? phase_bin(bp, phase_of_fix(bp, alpha_to_fix(alpha))) : 0u);
    }
    return key;
}

// per-component min/max of the quantised features and max f4 (table built from a feature cloud)
__global__ void feature_range_kernel(const float *__restrict__ feats, size_t count, float angle_step,
                                     float dist_step, int *__restrict__ range /* lo[4], hi[4] */,
                                     int *__restrict__ max_f4_bits) {
    int lo[4] = {INT_MAX, INT_MAX, INT_MAX, INT_MAX}, hi[4] = {INT_MIN, INT_MIN, INT_MIN, INT_MIN};
    int mx = -1;
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < count; p += (size_t)gridDim.x * blockDim.x) {
        const float *s = feats + p * 5;
        float f[4] = {s[0], s[1], s[2], s[3]};
        if (f[0] != f[0] || f[1] != f[1] || f[2] != f[2] || f[3] != f[3]) continue;
        int d[4];
        d[0] = (int)floorf(f[0] / angle_step);
        d[1] = (int)floorf(f[1] / angle_step);
        d[2] = (int)floorf(f[2] / angle_step);
        d[3] = (int)floorf(f[3] / dist_step);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            lo[k] = min(lo[k], d[k]);
            hi[k] = max(hi[k], d[k]);
        }
        if (f[3] > 0.0f) mx = max(mx, __float_as_int(f[3]));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[k] = min(lo[k], __shfl_xor_sync(0xFFFFFFFFu, lo[k], o));
            hi[k] = max(hi[k], __shfl_xor_sync(0xFFFFFFFFu, hi[k], o));
        }
    }
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (lo[k] != INT_MAX) atomicMin(&range[k], lo[k]);
            if (hi[k] != INT_MIN) atomicMax(&range[4 + k], hi[k]);
        }
        if (mx >= 0) atomicMax(max_f4_bits, mx);
    }
}

// keys + alpha from a materialised feature cloud
__global__ void keys_from_features_kernel(const float *__restrict__ feats, uint32_t n, KeyParams kp, BinParams bp,
                                          uint32_t *__restrict__ keys, uint32_t *__restrict__ alpha_bits) {
    const size_t count = (size_t)n * n;
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < count; p += (size_t)gridDim.x * blockDim.x) {
        const float *s = feats + p * 5;
        float f[4] = {s[0], s[1], s[2], s[3]};
        uint32_t key = INVALID_KEY;
        if (f[0] == f[0] && f[1] == f[1] && f[2] == f[2] && f[3] == f[3]) {
            int d[4];
            quantise(kp, f, d);
            uint32_t k;
            if (pack_key(kp, d, k)) key = sort_key(kp, bp, (uint32_t)(p / n), k, s[4]);
        }
        keys[p] = key;
        alpha_bits[p] = __float_as_uint(s[4]);
    }
}

// K1+K2 fused: keys + alpha straight from the model cloud (no 20-byte signatures in HBM).
// Same tiling as K1: TI reference rows (point + frame in shared memory) x 256 j per block.
constexpr int FTI = 4;
constexpr int FTJ = 256;
struct RefStage {
    float px, py, pz, nx, ny, nz;
    Frame F;
};

__global__ void __launch_bounds__(FTJ)
keys_from_cloud_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm, uint32_t n, int feature_mode,
                       KeyParams kp, BinParams bp, uint32_t *__restrict__ keys, uint32_t *__restrict__ alpha_bits,
                       int *__restrict__ max_f4_bits, int *__restrict__ out_of_range) {
    __shared__ RefStage ref[FTI];
    const uint32_t i0 = blockIdx.y * FTI;
    const uint32_t j = blockIdx.x * FTJ + threadIdx.x;
    if (threadIdx.x < FTI && i0 + threadIdx.x < n) {
        float4 p = pos[i0 + threadIdx.x], q = nrm[i0 + threadIdx.x];
        RefStage &r = ref[threadIdx.x];
        r.px = p.x; r.py = p.y; r.pz = p.z;
        r.nx = q.x; r.ny = q.y; r.nz = q.z;
        ref_frame(make_v3(p.x, p.y, p.z), make_v3(q.x, q.y, q.z), r.F);
    }
    float4 pj = make_float4(0, 0, 0, 0), nj = make_float4(0, 0, 0, 0);
    if (j < n) {
        pj = pos[j];
        nj = nrm[j];
    }
    __syncthreads();
    int mx = -1;
#pragma unroll 1
    for (int r = 0; r < FTI; ++r) {
        const uint32_t i = i0 + r;
        if (i >= n) break;
        if (j < n) {
            uint32_t key = INVALID_KEY;
            float alpha = CUDART_NAN_F;
            if (i != j) {
                float f[4];
                V3 pi = make_v3(ref[r].px, ref[r].py, ref[r].pz), ni = make_v3(ref[r].nx, ref[r].ny, ref[r].nz);
                if (pair_features(feature_mode, pi, ni, v3_of(pj), v3_of(nj), f)) {
                    alpha = planar_alpha(ref[r].F, v3_of(pj));
                    int d[4];
                    quantise(kp, f, d);
                    uint32_t k;
                    if (pack_key(kp, d, k)) key = sort_key(kp, bp, i, k, alpha);
                    else if (f[0] == f[0] && f[1] == f[1] && f[2] == f[2]) *out_of_range = 1;
                    if (f[3] > 0.0f) mx = max(mx, __float_as_int(f[3]));
                }
            }
            keys[(size_t)i * n + j] = key;
            alpha_bits[(size_t)i * n + j] = __float_as_uint(alpha);
        }
    }
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx >= 0) atomicMax(max_f4_bits, mx);
}

// sub_offsets[k'] for k' = key << shift | cell: the search is confined to the key's own bucket; the sort keys carry
// low_bits more bits below the cell (the bin of alpha_m of tables with merged votes)
__global__ void csr_sub_offsets_kernel(const uint32_t *__restrict__ sorted_keys, const uint32_t *__restrict__ offsets,
                                       uint32_t total_sub, uint32_t shift, uint32_t low_bits,
                                       uint32_t *__restrict__ sub_offsets) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > total_sub) return;
    uint32_t lo = offsets[k >> shift];
    if (k < total_sub) {
        uint32_t hi = offsets[(k >> shift) + 1];
        const uint32_t want = k << low_bits;
        while (lo < hi) {
            uint32_t mid = lo + ((hi - lo) >> 1);
            if (sorted_keys[mid] < want) lo = mid + 1; else hi = mid;
        }
    }
    sub_offsets[k] = lo;
}

// ---- merged votes ------------------------------------------------------------------------------------------------
// After the sort the entries of one (slice, key, cell, bin of alpha_m) are adjacent and ordered by (i, j): a run of
// entries with the same model row i casts the same vote — same accumulator word, same shift — for every scene pair
// whose phase lies in another cell.  The run becomes ONE word of the merged array, (count << 24) | hot word, and the
// voting kernel adds `count` with one reduction (config 3: 1.74 entries per word).  Runs are cut every 255 entries.
__global__ void merge_heads_kernel(const uint32_t *__restrict__ sorted_keys, const uint32_t *__restrict__ sorted_idx,
                                   uint32_t n_entries, uint32_t n, uint32_t *__restrict__ head) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_entries) return;
    head[p] = (p == 0 || p % 255u == 0u || sorted_keys[p] != sorted_keys[p - 1] || sorted_idx[p] / n != sorted_idx[p - 1] / n) ? 1u : 0u;
}

__global__ void merge_words_kernel(const uint32_t *__restrict__ head, const uint32_t *__restrict__ rank,
                                   const uint32_t *__restrict__ entry_w, uint32_t n_entries,
                                   uint32_t *__restrict__ merged_w) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_entries || !head[p]) return;
    uint32_t q = p + 1;
    while (q < n_entries && !head[q]) ++q;  // <= 255 steps
    merged_w[rank[p]] = ((q - p) << 24) | (entry_w[p] & HOT_MASK);
}

__global__ void merge_identity_kernel(const uint32_t *__restrict__ entry_w, uint32_t n_entries, uint32_t *__restrict__ merged_w) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_entries) merged_w[p] = (1u << 24) | (entry_w[p] & HOT_MASK);
}

// merged position of every cell bound (cell starts are run heads)
__global__ void merge_offsets_kernel(const uint32_t *__restrict__ sub_offsets, uint32_t total_sub, const uint32_t *__restrict__ rank,
                                     uint32_t n_entries, uint32_t n_merged, uint32_t *__restrict__ msub_offsets) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > total_sub) return;
    const uint32_t o = sub_offsets[c];
    msub_offsets[c] = o < n_entries ? rank[o] : n_merged;
}

// distinct keys of the table: a key counts once however many accumulator slices hold entries of it
__global__ void count_nonempty_kernel(const uint32_t *__restrict__ offsets, uint32_t key_space, uint32_t n_slices,
                                      unsigned long long *__restrict__ count) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    bool ne = false;
    if (k < key_space)
        for (uint32_t s = 0; s < n_slices && !ne; ++s) {
            const size_t b = (size_t)s * key_space + k;
            ne = offsets[b + 1] > offsets[b];
        }
    uint32_t m = __ballot_sync(0xFFFFFFFFu, ne);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, (unsigned long long)__popc(m));
}

// per entry: the hot word (byte offset, inside the bin-major accumulator slice, of model row i's cell in the column of
// alpha_m's own bin — column 0 for tables without phase cells), alpha_m in fixed point for the per-entry paths, and
// the float alpha_m for the literal form of the guard-band votes and for the API exports.
__global__ void entries_kernel(const uint32_t *__restrict__ sorted_idx, const uint32_t *__restrict__ sorted_alpha,
                               uint32_t n_entries, uint32_t n, uint32_t slice_rows, uint32_t pitch, BinParams bp,
                               uint32_t *__restrict__ entry_w, uint32_t *__restrict__ entry_am,
                               float *__restrict__ entry_alpha, int *__restrict__ bad_alpha) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_entries) return;
    uint32_t i = sorted_idx[p] / n;
    uint32_t local = i - (i / slice_rows) * slice_rows;
    const float alpha = __uint_as_float(sorted_alpha[p]);
    // atan2f range; anything else cannot come from PPFEstimation and would not wrap like PCL's floats
    if (!(alpha >= -3.14159274f && alpha <= 3.14159274f)) *bad_alpha = 1;
    const uint32_t a_fix = alpha_to_fix(alpha);
    entry_w[p] = bp.bulk ? entry_word(bp, pitch, local, alpha) : 4u * local;
    entry_am[p] = a_fix;
    entry_alpha[p] = alpha;
}

// Bank ordering.  The accumulator is bin-major with a pitch that is a multiple of 32, so the shared-memory bank of a
// vote is (model row mod 32) for every scene pair.  A warp votes for 32 consecutive entries per instruction, and the
// instruction costs as many passes of the SM's data pipe as its fullest bank holds entries.  Inside each phase cell
// (where the order is free: exports re-sort to (i, j), vote counts do not depend on it) the entries are therefore laid
// out as
//   core   m = the rarest bank's count rounds of 32 entries, one per bank in bank order: ANY 32 consecutive
//          entries of this part hit 32 different banks, however the voting loop's batches are aligned;
//   tail   what the fuller banks have left, T entries sorted by bank and dealt round-robin into ceil(T / 32)
//          groups: a bank with e entries left puts ceil(e / groups) of them into each group,
// which meets the lower bound max(entries / 32, fullest bank) on the passes of a cell up to rounding.
// Only the merged words (the shift ranges' input) are ordered; the per-entry arrays of the scene phase's own cell
// (1/16 of the votes) stay in sorted order.  One warp per non-empty cell; ranks inside a bank follow the sorted
// order, so the result is deterministic.
constexpr int SPREAD_WARPS = 8;
__global__ void __launch_bounds__(SPREAD_WARPS * 32)
bank_order_kernel(const uint32_t *__restrict__ sub_offsets, uint32_t total_sub, const uint32_t *__restrict__ w_in,
                  uint32_t *__restrict__ w_out) {
    __shared__ uint32_t s_count[SPREAD_WARPS][32], s_run[SPREAD_WARPS][32], s_prefix[SPREAD_WARPS][32];
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint32_t *count = s_count[wib], *run = s_run[wib], *prefix = s_prefix[wib];
    const uint32_t n_warps = gridDim.x * SPREAD_WARPS;
    for (uint32_t c0 = (blockIdx.x * SPREAD_WARPS + wib) * 32; c0 < total_sub; c0 += n_warps * 32) {
        const uint32_t c = c0 + lane;
        uint32_t b = 0, e = 0;
        if (c < total_sub) {
            b = sub_offsets[c];
            e = sub_offsets[c + 1];
        }
        uint32_t nonempty = __ballot_sync(0xFFFFFFFFu, e > b);
        while (nonempty) {
            const int src = __ffs(nonempty) - 1;
            nonempty &= nonempty - 1;
            const uint32_t cb = __shfl_sync(0xFFFFFFFFu, b, src), ce = __shfl_sync(0xFFFFFFFFu, e, src);
            count[lane] = 0;
            run[lane] = 0;
            __syncwarp();
            for (uint32_t k = cb + lane; k < ce; k += 32) atomicAdd(&count[(w_in[k] >> 2) & 31u], 1u);
            __syncwarp();
            // m = the rarest bank's count; prefix = exclusive scan of what each bank has beyond m
            const uint32_t cnt = count[lane];
            uint32_t m = cnt;
            for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
            const uint32_t extra = cnt - m;
            uint32_t incl = extra;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= (uint32_t)o) incl += t;
            }
            prefix[lane] = incl - extra;
            const uint32_t tail = __shfl_sync(0xFFFFFFFFu, incl, 31);  // T
            const uint32_t groups = (tail + 31u) / 32u;                  // K
            const uint32_t gq = groups ? tail / groups : 0u, gr = groups ? tail % groups : 0u;
            __syncwarp();
            for (uint32_t k0 = cb; k0 < ce; k0 += 32) {
                const uint32_t k = k0 + lane;
                const bool valid = k < ce;
                const uint32_t w = valid ? w_in[k] : 0u;
                const uint32_t bank = valid ? ((w >> 2) & 31u) : 32u + lane;  // idle lanes match nobody
                const uint32_t same = __match_any_sync(0xFFFFFFFFu, bank);
                uint32_t r = 0;
                if (valid) r = run[bank] + __popc(same & ((1u << lane) - 1u));
                __syncwarp();
                if (valid && lane == (uint32_t)(31 - __clz(same))) run[bank] = r + 1;  // highest lane of the class
                __syncwarp();
                if (valid) {
                    uint32_t dest;
                    if (r < m) {
                        dest = r * 32u + bank;
                    } else {
                        const uint32_t t = prefix[bank] + (r - m);
                        const uint32_t j = t % groups, pos = t / groups;
                        dest = 32u * m + j * gq + min(j, gr) + pos;
                    }
                    w_out[cb + dest] = w;
                }
            }
            __syncwarp();
        }
    }
}

__global__ void alpha_scatter_kernel(const uint32_t *__restrict__ entry_idx, const float *__restrict__ entry_alpha,
                                     uint32_t n_entries, float *__restrict__ out) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_entries) return;
    out[entry_idx[p]] = entry_alpha[p];
}

__global__ void fill_nan_kernel(float *__restrict__ out, size_t count) {
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < count; p += (size_t)gridDim.x * blockDim.x)
        out[p] = CUDART_NAN_F;
}

int ceil_log2(uint64_t v) {
    int b = 0;
    while ((1ull << b) < v) ++b;
    return b;
}

}  // namespace

// accumulator geometry shared with K3 (k3_vote.cu): bytes of shared memory left for the
// accumulator once the candidate / work queues are taken out
size_t k3_accumulator_budget(const b200ppf_ctx *ctx);

int k2_build(b200ppf_ctx *ctx, const b200ppf_features *feat, const b200ppf_cloud *model, float angle_step,
             float dist_step, b200ppf_table **out) {
    if (!(angle_step > 0.0f) || !(dist_step > 0.0f))
        return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: discretisation steps must be positive");
    size_t n;
    if (feat) {
        n = (size_t)(unsigned int)std::sqrt((float)feat->count);  // PCL: n = sqrt(size)
        if (n * n != feat->count)
            return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: feature cloud size is not a square (n*n pairs expected)");
    } else {
        n = model->n;
    }
    if (n == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: empty model");
    if (n > 65535) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "table build: more than 65535 model points (pair index is 32-bit)");
    const size_t count = n * n;

    TablePtr t(new b200ppf_table());
    t->ctx = ctx;
    t->feature_mode = ctx->feature_mode;
    b200ppf_table_info &info = t->info;
    info.n_model = n;
    info.angle_step = angle_step;
    info.dist_step = dist_step;
    info.n_alpha = num_alpha_bins(angle_step, ctx->nalpha_rule);
    info.nalpha_rule = (uint32_t)ctx->nalpha_rule;
    if (info.n_alpha == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: angle step larger than 2*pi");
    // accumulator slices: rows per slice bounded by the shared-memory budget of the voting kernel.  The slice is held
    // bin-major with a pitch of 32-row multiples (k3_vote.cu), acc_cols columns (the FLOOR rules carry a spare one).
    t->bp = make_bin_params(angle_step, ctx->alpha_mode, ctx->nalpha_rule);
    {
        size_t budget = k3_accumulator_budget(ctx);
        size_t rows_max = budget / ((size_t)t->bp.acc_cols * sizeof(uint32_t)) / 32 * 32;
        if (rows_max == 0)
            return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "table build: angle step too fine for 32 accumulator rows in shared memory");
        if (const char *e = getenv("B200PPF_SLICE_ROWS")) {
            size_t v = (size_t)atoll(e);
            if (v > 0 && v < rows_max) rows_max = v;
        }
        uint32_t n_slices = (uint32_t)((n + rows_max - 1) / rows_max);
        info.n_slices = n_slices;
        info.slice_rows = (uint32_t)((n + n_slices - 1) / n_slices);
    }

    KeyParams &kp = t->kp;
    kp.angle_step = angle_step;
    kp.dist_step = dist_step;
    kp.slice_rows = info.slice_rows;
    kp.n_slices = info.n_slices;
    kp.row_pitch = (info.slice_rows + 31u) / 32u * 32u;

    StreamBuf<int> d_range(ctx);  // lo[4], hi[4], max_f4_bits, out_of_range, bad_alpha, pad
    PPF_CUDA(ctx, d_range.alloc(12));
    int h_range[12] = {INT_MAX, INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN, INT_MIN, -1, 0, 0, 0};
    PPF_CUDA(ctx, cudaMemcpyAsync(d_range, h_range, sizeof(h_range), cudaMemcpyHostToDevice, ctx->stream));

    cudaEventRecord(ctx->ev[0], ctx->stream);
    if (feat) {
        int blocks = (int)std::min<size_t>((count + 255) / 256, (size_t)ctx->sm_count * 16);
        PPF_LAUNCH(ctx, feature_range_kernel, blocks, 256, 0, reinterpret_cast<const float *>(feat->d), count,
                   angle_step, dist_step, d_range, d_range + 8);
        PPF_CUDA(ctx, cudaMemcpyAsync(h_range, d_range, sizeof(h_range), cudaMemcpyDeviceToHost, ctx->stream));
        PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int k = 0; k < 4; ++k) {
            if (h_range[k] == INT_MAX) {  // no valid pair at all
                kp.lo[k] = 0;
                kp.size[k] = 1;
            } else {
                kp.lo[k] = h_range[k];
                kp.size[k] = h_range[4 + k] - h_range[k] + 1;
            }
        }
    } else {
        // analytic bounds by feature functor; d4 bounded by the bounding-box diagonal
        auto q = [](float v, float step) { return (int)std::floor(v / step); };
        const float pi_hi = 3.2f;
        if (ctx->feature_mode == B200PPF_FEATURE_PCL_PFH) {
            kp.lo[0] = q(-pi_hi, angle_step) - 1; kp.size[0] = q(pi_hi, angle_step) + 1 - kp.lo[0] + 1;
            kp.lo[1] = q(-1.0f, angle_step) - 1;  kp.size[1] = q(1.0f, angle_step) + 1 - kp.lo[1] + 1;
            kp.lo[2] = kp.lo[1];                  kp.size[2] = kp.size[1];
        } else if (ctx->feature_mode == B200PPF_FEATURE_DROST_COS) {
            for (int k = 0; k < 3; ++k) {
                kp.lo[k] = q(-1.0f, angle_step) - 1;
                kp.size[k] = q(1.0f, angle_step) + 1 - kp.lo[k] + 1;
            }
        } else {
            for (int k = 0; k < 3; ++k) {
                kp.lo[k] = -1;
                kp.size[k] = q(pi_hi, angle_step) + 1 - kp.lo[k] + 1;
            }
        }
        double diag = 0;
        for (int k = 0; k < 3; ++k) {
            double e = (double)model->bbox_max[k] - (double)model->bbox_min[k];
            diag += e * e;
        }
        diag = std::sqrt(diag) * 1.001 + 1e-6;
        kp.lo[3] = 0;
        kp.size[3] = (int)std::floor(diag / dist_step) + 2;
    }
    {
        unsigned __int128 ks = 1;
        for (int k = 0; k < 4; ++k) ks *= (unsigned __int128)(uint32_t)kp.size[k];
        unsigned __int128 total = ks * info.n_slices + 1;
        if (total >= ((unsigned __int128)1 << 31))
            return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "table build: discretisation too fine (packed key space exceeds 2^31)");
        kp.key_space = (uint32_t)ks;
        // phase cells multiply the sort-key space: halve them until it fits 31 bits and 1 Gi offsets
        if (const char *e = getenv("B200PPF_PHASE_CELLS_LOG2")) {
            int v = atoi(e);
            if (v >= 0 && (uint32_t)v < t->bp.cells_log2) t->bp.cells_log2 = (uint32_t)v;
        }
        while (t->bp.cells_log2 > 0 && (total << t->bp.cells_log2) >= ((unsigned __int128)1 << 30)) --t->bp.cells_log2;
        if (t->bp.cells_log2 == 0) t->bp.bulk = 0;
    }
    for (int k = 0; k < 4; ++k) {
        info.lo[k] = kp.lo[k];
        info.size[k] = kp.size[k];
    }
    info.key_space = kp.key_space;
    const uint32_t total_keys = kp.key_space * info.n_slices;
    const uint32_t cells_log2 = t->bp.cells_log2;
    const uint32_t total_sub = total_keys << cells_log2;
    // merged votes: the bin of alpha_m joins the sort key when the key still fits 32 bits
    kp.merge_bits = 0;
    if (t->bp.bulk && !getenv("B200PPF_NO_MERGE")) {
        const uint32_t mb = (uint32_t)ceil_log2((uint64_t)t->bp.n_turn);
        if (ceil_log2((uint64_t)total_sub + 1) + (int)mb <= 32) kp.merge_bits = mb;
    }
    const uint32_t merge_bits = kp.merge_bits;
    info.key_bits = (uint32_t)ceil_log2((uint64_t)total_sub + 1) + merge_bits;
    info.phase_cells = 1u << cells_log2;

    // ---- keys ---------------------------------------------------------------------------------
    StreamBuf<uint32_t> keys0(ctx), keys1(ctx), idx0(ctx), idx1(ctx), alp0(ctx), alp1(ctx);
    PPF_CUDA(ctx, keys0.alloc(count));
    PPF_CUDA(ctx, idx0.alloc(count));
    PPF_CUDA(ctx, alp0.alloc(count));
    PPF_CUDA(ctx, keys1.alloc(count));
    PPF_CUDA(ctx, idx1.alloc(count));
    PPF_CUDA(ctx, alp1.alloc(count));
    uint32_t *keys[2] = {keys0, keys1}, *idx[2] = {idx0, idx1}, *alp[2] = {alp0, alp1};
    if (feat) {
        int blocks = (int)std::min<size_t>((count + 255) / 256, (size_t)ctx->sm_count * 32);
        PPF_LAUNCH(ctx, keys_from_features_kernel, blocks, 256, 0, reinterpret_cast<const float *>(feat->d), (uint32_t)n, kp,
                   t->bp, keys[0], alp[0]);
    } else {
        dim3 grid((unsigned)((n + FTJ - 1) / FTJ), (unsigned)((n + FTI - 1) / FTI));
        PPF_LAUNCH(ctx, keys_from_cloud_kernel, grid, FTJ, 0, model->pos, model->nrm, (uint32_t)n, ctx->feature_mode, kp, t->bp,
                   keys[0], alp[0], d_range + 8, d_range + 9);
    }
    cudaEventRecord(ctx->ev[1], ctx->stream);

    // ---- sort -----------------------------------------------------------------------------------
    bool in_alt = false;
    int rc = radix_sort_u32(ctx, keys[0], keys[1], idx[0], idx[1], alp[0], alp[1], count,
                            (1ull << info.key_bits) - 1, /*v0_iota=*/true, &in_alt);
    if (rc) return rc;
    const int s = in_alt ? 1 : 0;
    cudaEventRecord(ctx->ev[2], ctx->stream);

    // ---- CSR ------------------------------------------------------------------------------------
    // each array is allocated once what sizes it is known, with the length and pad table_arrays gives it
    auto alloc_arrays = [&](int first, int last) -> int {
        const std::array<TableArray, 8> arrs = table_arrays(t.get());
        for (int a = first; a <= last; ++a)
            if (arrs[a].used) PPF_CUDA(ctx, table_array_alloc(ctx->stream, arrs[a]));
        return B200PPF_OK;
    };
    if ((rc = alloc_arrays(0, 1))) return rc;  // offsets, sub_offsets
    // offsets[k] = first sorted position whose sort key is >= k << (cells_log2 + merge_bits), for k in [0, total_keys]
    if ((rc = lower_bounds(ctx, keys[s], (uint32_t)count, nullptr, total_keys, cells_log2 + merge_bits, t->offsets))) return rc;
    if (cells_log2)
        PPF_LAUNCH(ctx, csr_sub_offsets_kernel, (total_sub + 1 + 255) / 256, 256, 0, keys[s], t->offsets, total_sub, cells_log2,
                   merge_bits, t->sub_offsets);
    uint32_t n_entries = 0;
    PPF_CUDA(ctx, cudaMemcpyAsync(&n_entries, t->offsets + total_keys, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(h_range, d_range, sizeof(h_range), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!feat && h_range[9] != 0)
        return fail_msg(ctx, B200PPF_ERR_STATE, "table build: a model pair feature left the analytic key range (non-unit normals?)");
    info.n_entries = n_entries;
    {
        int bits = h_range[8];
        float mx;
        memcpy(&mx, &bits, sizeof(float));
        info.max_dist = bits < 0 ? -1.0f : mx;  // PCL: max_dist_ starts at -1
    }
    // the voting kernel reads whole batches: ENTRY_PAD readable (zero) words follow the last entry
    if ((rc = alloc_arrays(2, 5))) return rc;  // entry_w, entry_am, entry_alpha, entry_idx
    StreamBuf<unsigned long long> d_cnt(ctx);
    PPF_CUDA(ctx, d_cnt.alloc(1));
    PPF_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), ctx->stream));
    if (n_entries) {
        // per-entry arrays in sorted order: (key, cell, [bin of alpha_m,] i, j)
        PPF_LAUNCH(ctx, entries_kernel, (n_entries + 255) / 256, 256, 0, idx[s], alp[s], n_entries, (uint32_t)n, info.slice_rows,
                   kp.row_pitch, t->bp, t->entry_w, t->entry_am, t->entry_alpha, d_range + 10);
        PPF_CUDA(ctx, cudaMemcpyAsync(t->entry_idx, idx[s], (size_t)n_entries * sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                                      ctx->stream));
    }
    PPF_LAUNCH(ctx, count_nonempty_kernel, (kp.key_space + 255) / 256, 256, 0, t->offsets, kp.key_space, info.n_slices, d_cnt);
    // ---- merged votes + bank order (phase-sorted tables) ---------------------------------------------
    if (cells_log2 && n_entries) {
        // the free halves of the sort buffers hold the run heads, their ranks and the unordered merged words
        uint32_t *head = keys[1 - s], *rank = idx[1 - s], *mw_tmp = alp[1 - s];
        uint32_t n_merged = n_entries;
        if (merge_bits) {
            PPF_LAUNCH(ctx, merge_heads_kernel, (n_entries + 255) / 256, 256, 0, keys[s], idx[s], n_entries, (uint32_t)n, head);
            if ((rc = flag_scan_host(ctx, head, n_entries, rank, &n_merged))) return rc;
        }
        t->n_merged = n_merged;
        if ((rc = alloc_arrays(6, 7))) return rc;  // merged_w, msub_offsets
        if (merge_bits) {
            PPF_LAUNCH(ctx, merge_words_kernel, (n_entries + 255) / 256, 256, 0, head, rank, t->entry_w, n_entries, mw_tmp);
            PPF_LAUNCH(ctx, merge_offsets_kernel, (total_sub + 1 + 255) / 256, 256, 0, t->sub_offsets, total_sub, rank, n_entries,
                       n_merged, t->msub_offsets);
        } else {  // no room for the bin in the sort key: one word per entry, count 1
            PPF_LAUNCH(ctx, merge_identity_kernel, (n_entries + 255) / 256, 256, 0, t->entry_w, n_entries, mw_tmp);
            PPF_CUDA(ctx, cudaMemcpyAsync(t->msub_offsets, t->sub_offsets, ((size_t)total_sub + 1) * sizeof(uint32_t),
                                          cudaMemcpyDeviceToDevice, ctx->stream));
        }
        if (!getenv("B200PPF_NO_BANK_SPREAD")) {
            const unsigned blocks = (unsigned)std::min<size_t>(((size_t)total_sub + 32 * SPREAD_WARPS - 1) / (32 * SPREAD_WARPS),
                                                               (size_t)ctx->sm_count * 16);
            PPF_LAUNCH(ctx, bank_order_kernel, blocks, SPREAD_WARPS * 32, 0, t->msub_offsets, total_sub, mw_tmp, t->merged_w);
        } else {
            PPF_CUDA(ctx, cudaMemcpyAsync(t->merged_w, mw_tmp, (size_t)n_merged * sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                                          ctx->stream));
        }
    }
    info.n_merged = t->n_merged;
    unsigned long long h_cnt = 0;
    PPF_CUDA(ctx, cudaMemcpyAsync(&h_cnt, d_cnt, sizeof(h_cnt), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(h_range, d_range, sizeof(h_range), cudaMemcpyDeviceToHost, ctx->stream));
    cudaEventRecord(ctx->ev[3], ctx->stream);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (h_range[10] != 0)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "table build: an alpha_m lies outside [-pi, pi] (not produced by PPFEstimation::compute)");
    info.n_keys = h_cnt;
    cudaEventElapsedTime(&ctx->timings.keys_ms, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->timings.sort_ms, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&ctx->timings.csr_ms, ctx->ev[2], ctx->ev[3]);
    *out = t.release();
    return B200PPF_OK;
}

int k2_query_key(b200ppf_ctx *ctx, const b200ppf_table *t, const int32_t *d4, uint64_t *pairs, size_t cap,
                 size_t *n_found) {
    *n_found = 0;
    uint32_t key;
    int d[4] = {d4[0], d4[1], d4[2], d4[3]};
    if (!pack_key(t->kp, d, key)) return B200PPF_OK;
    const uint32_t n = (uint32_t)t->info.n_model;
    size_t written = 0, total = 0;
    std::vector<uint32_t> tmp;
    for (uint32_t s = 0; s < t->info.n_slices; ++s) {
        uint32_t off[2];
        PPF_CUDA(ctx, cudaMemcpyAsync(off, t->offsets + (size_t)s * t->kp.key_space + key, sizeof(off),
                                      cudaMemcpyDeviceToHost, ctx->stream));
        PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        uint32_t len = off[1] - off[0];
        total += len;
        size_t take = std::min<size_t>(len, cap - std::min(cap, written));
        if (take) {
            tmp.resize(len);  // the whole bucket: its canonical prefix is only known once it is sorted
            PPF_CUDA(ctx, cudaMemcpyAsync(tmp.data(), t->entry_idx + off[0], (size_t)len * sizeof(uint32_t),
                                          cudaMemcpyDeviceToHost, ctx->stream));
            PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            std::sort(tmp.begin(), tmp.end());  // phase-sorted buckets -> canonical (i, j) order
            for (size_t e = 0; e < take; ++e) {
                pairs[2 * (written + e)] = tmp[e] / n;
                pairs[2 * (written + e) + 1] = tmp[e] % n;
            }
            written += take;
        }
    }
    *n_found = total;
    return B200PPF_OK;
}

int k2_alpha_m(b200ppf_ctx *ctx, const b200ppf_table *t, float *host) {
    const size_t n = t->info.n_model, count = n * n;
    StreamBuf<float> d(ctx);
    PPF_CUDA(ctx, d.alloc(count));
    int blocks = (int)std::min<size_t>((count + 255) / 256, (size_t)ctx->sm_count * 16);
    PPF_LAUNCH(ctx, fill_nan_kernel, blocks, 256, 0, d, count);
    if (t->info.n_entries)
        PPF_LAUNCH(ctx, alpha_scatter_kernel, (unsigned)((t->info.n_entries + 255) / 256), 256, 0, t->entry_idx,
                   t->entry_alpha, (uint32_t)t->info.n_entries, d);
    PPF_CUDA(ctx, cudaMemcpyAsync(host, d, count * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

}  // namespace b200ppf
