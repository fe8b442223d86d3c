// sort_scan.cu — the sorted-key primitives of every stage that buckets its elements by a uint32 key (sm_100a):
//
//   radix_sort_u32   hand-written stable LSD radix sort (8-bit digits), its pass count derived from the largest key
//   lower_bounds     offsets[k] = first sorted position whose key is >= k << shift (bucket / cell starts)
//   flag_scan        exclusive scan of 0/1 flags: rank of every set flag, total on the device (flag_scan_host: on the host)
//   scan_rows        in-place exclusive scan of several rows of counts, one block per row
//   run_heads        head[i] = 1 where a run of equal sorted keys starts
//
// Users: K2 (order the N_m^2 model pairs by packed feature key -> CSR buckets, replacing the unordered_multimap of [PCL]
// registration/src/ppf_registration.cpp), the scene grid, K3's task order, K4 (order pose hypotheses by votes, replacing
// the std::sort of clusterPoses; per-cell lists and their compaction), the voxel grid, compaction and frame crop of the
// pre-processing, verification's grids, and K7's sampling and table.
//
// Radix sort: one pass = tile histogram -> column scan -> tile scatter.  A tile is WARPS x ROUNDS x 32 consecutive
// elements (4096 for large inputs, 512 for small ones so that every SM has a block to run); element
// order inside a tile is (warp, round, lane).
//   hist     per-tile digit counts with shared-memory atomics -> hist[tile][256] (coalesced 1 KB rows)
//   scan     column scan over tiles (three small kernels) -> global base of every (tile, digit)
//   scatter  the tile is sorted locally first: per-warp digit counts (match.any), a (digit, warp) scan in
//            shared memory, stable ranks by (warp, round, lane), keys and payloads staged in shared memory
//            at their tile-local sorted position; then the block copies the tile out digit run by digit
//            run — consecutive threads write consecutive addresses instead of 32 scattered 4-byte stores.
// No global atomics; stable.  HBM traffic per pass: keys read twice, payloads read once, everything
// written once, in runs of (tile / 256 ... tile) elements.
//
// Flag scan: per-block counts -> one block scans the block counts -> per-block ranks (three launches, no host wait).
#include "ppf_common.cuh"

namespace b200ppf {

namespace {

constexpr int RADIX = 256;
constexpr int WARPS = 8;            // warps per block / tile
constexpr int ROUNDS_BIG = 16;      // 4096-element tiles
constexpr int ROUNDS_SMALL = 2;     // 512-element tiles
constexpr int SCAN_CHUNK = 256;     // histogram rows per column-scan chunk

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

template <int ROUNDS>
__global__ void __launch_bounds__(WARPS * 32)
radix_hist_kernel(const uint32_t *__restrict__ keys, uint32_t n, int shift, uint32_t *__restrict__ hist) {
    constexpr uint32_t TILE = WARPS * ROUNDS * 32;
    __shared__ uint32_t cnt[RADIX];
    for (int d = threadIdx.x; d < RADIX; d += WARPS * 32) cnt[d] = 0;
    __syncthreads();
    const uint32_t begin = blockIdx.x * TILE;
    const uint32_t end = min(n, begin + TILE);  // begin < n, no overflow: n < 2^32 - TILE
#pragma unroll 4
    for (uint32_t idx = begin + threadIdx.x; idx < end; idx += WARPS * 32)
        atomicAdd(&cnt[(keys[idx] >> shift) & (RADIX - 1)], 1u);
    __syncthreads();
    uint32_t *row = hist + (size_t)blockIdx.x * RADIX;
    for (int d = threadIdx.x; d < RADIX; d += WARPS * 32) row[d] = cnt[d];
}

// column scan, step 1: per chunk of rows, per digit totals
__global__ void __launch_bounds__(RADIX)
radix_col_reduce_kernel(const uint32_t *__restrict__ hist, uint32_t nseg, uint32_t *__restrict__ chunk_tot) {
    const uint32_t d = threadIdx.x;
    const uint32_t r0 = blockIdx.x * SCAN_CHUNK, r1 = min(nseg, r0 + SCAN_CHUNK);
    uint32_t s = 0;
    for (uint32_t r = r0; r < r1; ++r) s += hist[(size_t)r * RADIX + d];
    chunk_tot[(size_t)blockIdx.x * RADIX + d] = s;
}

// step 2 (one block): exclusive scan over chunks per digit, then over digits
__global__ void __launch_bounds__(RADIX)
radix_col_scan_chunks_kernel(uint32_t *__restrict__ chunk_tot, uint32_t nchunks, uint32_t *__restrict__ digit_base) {
    __shared__ uint32_t tot[RADIX];
    const uint32_t d = threadIdx.x;
    uint32_t run = 0;
    for (uint32_t c = 0; c < nchunks; ++c) {
        uint32_t t = chunk_tot[(size_t)c * RADIX + d];
        chunk_tot[(size_t)c * RADIX + d] = run;
        run += t;
    }
    tot[d] = run;
    __syncthreads();
    // exclusive scan of 256 totals: warp 0, 8 values per lane
    if (d < 32) {
        uint32_t v[8], s = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[k] = tot[d * 8 + k];
            s += v[k];
        }
        uint32_t incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (d >= (uint32_t)o) incl += t;
        }
        uint32_t excl = incl - s;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            digit_base[d * 8 + k] = excl;
            excl += v[k];
        }
    }
}

// step 3: rewrite every histogram row as global bases
__global__ void __launch_bounds__(RADIX)
radix_col_apply_kernel(uint32_t *__restrict__ hist, uint32_t nseg, const uint32_t *__restrict__ chunk_tot,
                       const uint32_t *__restrict__ digit_base) {
    const uint32_t d = threadIdx.x;
    const uint32_t r0 = blockIdx.x * SCAN_CHUNK, r1 = min(nseg, r0 + SCAN_CHUNK);
    uint32_t run = chunk_tot[(size_t)blockIdx.x * RADIX + d] + digit_base[d];
    for (uint32_t r = r0; r < r1; ++r) {
        uint32_t t = hist[(size_t)r * RADIX + d];
        hist[(size_t)r * RADIX + d] = run;
        run += t;
    }
}

template <int ROUNDS, bool IOTA, bool HAS_V0, bool HAS_V1>
__global__ void __launch_bounds__(WARPS * 32)
radix_scatter_kernel(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ v0,
                     const uint32_t *__restrict__ v1, uint32_t n, int shift, const uint32_t *__restrict__ hist,
                     uint32_t *__restrict__ keys_out, uint32_t *__restrict__ v0_out, uint32_t *__restrict__ v1_out) {
    constexpr uint32_t TILE = WARPS * ROUNDS * 32;
    extern __shared__ uint32_t smem[];
    uint32_t *s_key = smem;                                  // [TILE] tile-local sorted order
    uint32_t *s_v0 = s_key + TILE;                           // [TILE]
    uint32_t *s_v1 = s_v0 + (HAS_V0 ? TILE : 0);             // [TILE]
    uint32_t *run = s_v1 + (HAS_V1 ? TILE : 0);              // [WARPS][RADIX] next local slot of (warp, digit)
    uint32_t *dstart = run + WARPS * RADIX;                  // [RADIX] first local slot of a digit
    uint32_t *gbase = dstart + RADIX;                        // [RADIX] global base of (this tile, digit)
    __shared__ uint32_t s_tot[8];

    const uint32_t tid = threadIdx.x, w = tid >> 5, lane = lane_id();
    const uint32_t begin = blockIdx.x * TILE;
    const uint32_t end = min(n, begin + TILE);
    const uint32_t lt = (1u << lane) - 1u;
    for (uint32_t k = tid; k < WARPS * RADIX; k += WARPS * 32) run[k] = 0;
    gbase[tid] = hist[(size_t)blockIdx.x * RADIX + tid];
    __syncthreads();

    // 1. keys into registers; per-warp digit counts
    uint32_t key[ROUNDS];
    uint32_t *mine = run + w * RADIX;
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const uint32_t idx = begin + (w * ROUNDS + r) * 32 + lane;
        const bool valid = idx < end;
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, valid);
        key[r] = 0;
        if (valid) {
            key[r] = keys[idx];
            const uint32_t digit = (key[r] >> shift) & (RADIX - 1);
            const uint32_t peers = __match_any_sync(mask, digit);
            if ((uint32_t)(__ffs(peers) - 1) == lane) mine[digit] += __popc(peers);
        }
        __syncwarp();
    }
    __syncthreads();
    // 2. (digit, warp) exclusive scan: thread d owns digit d
    {
        uint32_t c[WARPS], tot = 0;
#pragma unroll
        for (int ww = 0; ww < WARPS; ++ww) {
            c[ww] = run[ww * RADIX + tid];
            tot += c[ww];
        }
        uint32_t incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if ((int)lane >= o) incl += t;
        }
        if (lane == 31) s_tot[w] = incl;
        __syncthreads();
        uint32_t before = 0;
#pragma unroll
        for (int ww = 0; ww < WARPS; ++ww) before += (ww < (int)w) ? s_tot[ww] : 0u;
        uint32_t excl = before + incl - tot;
        dstart[tid] = excl;
#pragma unroll
        for (int ww = 0; ww < WARPS; ++ww) {
            run[ww * RADIX + tid] = excl;
            excl += c[ww];
        }
    }
    __syncthreads();
    // 3. stable tile-local positions; stage keys and payloads in sorted order
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const uint32_t idx = begin + (w * ROUNDS + r) * 32 + lane;
        const bool valid = idx < end;
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, valid);
        uint32_t digit = 0, peers = 0, pos = 0;
        if (valid) {
            digit = (key[r] >> shift) & (RADIX - 1);
            peers = __match_any_sync(mask, digit);
            pos = mine[digit] + __popc(peers & lt);
        }
        __syncwarp();
        if (valid && (uint32_t)(__ffs(peers) - 1) == lane) mine[digit] += __popc(peers);
        __syncwarp();
        if (valid) {
            s_key[pos] = key[r];
            if (HAS_V0) s_v0[pos] = IOTA ? idx : v0[idx];
            if (HAS_V1) s_v1[pos] = v1[idx];
        }
    }
    __syncthreads();
    // 4. copy out: local slot p of digit d goes to gbase[d] + (p - dstart[d]); runs are contiguous
    const uint32_t count = end - begin;
    for (uint32_t p = tid; p < count; p += WARPS * 32) {
        const uint32_t k = s_key[p];
        const uint32_t dg = (k >> shift) & (RADIX - 1);
        const uint32_t o = gbase[dg] + (p - dstart[dg]);
        keys_out[o] = k;
        if (HAS_V0) v0_out[o] = s_v0[p];
        if (HAS_V1) v1_out[o] = s_v1[p];
    }
}

// ---- bucket offsets, flag scan, run heads -------------------------------------------------------------------------
constexpr int SCAN_BLOCK = 1024;

// n_dev, when non-null, holds the length of the list instead of n.  The target is compared in 64 bits: k << shift may
// reach 2^32 (offsets[n_keys] of a full key range), which is past every key, not 0.
__global__ void lower_bounds_kernel(const uint32_t *__restrict__ sorted_keys, uint32_t n, const uint32_t *__restrict__ n_dev,
                                    uint32_t n_keys, uint32_t shift, uint32_t *__restrict__ offsets) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > n_keys) return;
    const uint64_t want = (uint64_t)k << shift;
    uint32_t lo = 0, hi = n_dev ? *n_dev : n;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if ((uint64_t)sorted_keys[mid] < want) lo = mid + 1; else hi = mid;
    }
    offsets[k] = lo;
}

__global__ void __launch_bounds__(SCAN_BLOCK)
flag_count_kernel(const uint32_t *__restrict__ flags, uint32_t n, uint32_t *__restrict__ block_sums) {
    const uint32_t k = blockIdx.x * SCAN_BLOCK + threadIdx.x;
    const int c = __syncthreads_count(k < n && flags[k] == 1u);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = (uint32_t)c;
}

// block b of the grid scans row b: data[b * row_len ...] in place (exclusive), its sum into total[b]
__global__ void __launch_bounds__(SCAN_BLOCK)
scan_rows_kernel(uint32_t *__restrict__ data, uint32_t row_len, uint32_t *__restrict__ total) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry;
    data += (size_t)blockIdx.x * row_len;
    total += blockIdx.x;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < row_len; base += SCAN_BLOCK) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < row_len ? data[i] : 0u;
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if ((threadIdx.x & 31) >= (uint32_t)o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = warp_tot[threadIdx.x], wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, o);
                if (threadIdx.x >= (uint32_t)o) wi += t;
            }
            warp_tot[threadIdx.x] = wi - w;  // exclusive
        }
        __syncthreads();
        const uint32_t excl = carry + warp_tot[threadIdx.x >> 5] + incl - v;
        if (i < row_len) data[i] = excl;
        __syncthreads();
        if (threadIdx.x == SCAN_BLOCK - 1) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// rank[k] = number of flags equal to 1 before k (written for every k)
__global__ void __launch_bounds__(SCAN_BLOCK)
flag_rank_kernel(const uint32_t *__restrict__ flags, uint32_t n, const uint32_t *__restrict__ block_sums,
                 uint32_t *__restrict__ rank) {
    __shared__ uint32_t warp_tot[32];
    const uint32_t k = blockIdx.x * SCAN_BLOCK + threadIdx.x;
    const uint32_t v = (k < n && flags[k] == 1u) ? 1u : 0u;
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, v);
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_tot[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t w = warp_tot[threadIdx.x], wi = w;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, o);
            if (threadIdx.x >= (uint32_t)o) wi += t;
        }
        warp_tot[threadIdx.x] = wi - w;
    }
    __syncthreads();
    if (k < n) rank[k] = block_sums[blockIdx.x] + warp_tot[warp] + __popc(m & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(256)
run_heads_kernel(const uint32_t *__restrict__ sorted_keys, uint32_t n, uint32_t *__restrict__ head) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) head[i] = (i == 0 || sorted_keys[i] != sorted_keys[i - 1]) ? 1u : 0u;
}

}  // namespace

// v0_iota: on entry v0 is taken to be the identity permutation 0..n-1 (its contents are not read).
namespace {

template <int ROUNDS>
int radix_sort_impl(b200ppf_ctx *ctx, uint32_t *keys, uint32_t *keys_alt, uint32_t *v0, uint32_t *v0_alt, uint32_t *v1,
                    uint32_t *v1_alt, size_t n, int bits, bool v0_iota, bool *result_in_alt) {
    constexpr uint32_t TILE = WARPS * ROUNDS * 32;
    const uint32_t ntiles = (uint32_t)((n + TILE - 1) / TILE);
    const uint32_t nchunks = (ntiles + SCAN_CHUNK - 1) / SCAN_CHUNK;
    StreamBuf<uint32_t> hist(ctx), chunk_tot(ctx), digit_base(ctx);
    PPF_CUDA(ctx, hist.alloc((size_t)ntiles * RADIX));
    PPF_CUDA(ctx, chunk_tot.alloc((size_t)nchunks * RADIX));
    PPF_CUDA(ctx, digit_base.alloc(RADIX));

    const bool has_v0 = v0 != nullptr && v0_alt != nullptr, has_v1 = v1 != nullptr && v1_alt != nullptr;
    bool iota = has_v0 && v0_iota;
    const size_t smem = ((size_t)TILE * (1 + (has_v0 ? 1 : 0) + (has_v1 ? 1 : 0)) + WARPS * RADIX + 2 * RADIX) * sizeof(uint32_t);
    uint32_t *ki = keys, *ko = keys_alt, *v0i = v0, *v0o = v0_alt, *v1i = v1, *v1o = v1_alt;
    bool in_alt = false;
    for (int shift = 0; shift < bits; shift += 8) {
        PPF_LAUNCH(ctx, radix_hist_kernel<ROUNDS>, ntiles, WARPS * 32, 0, ki, (uint32_t)n, shift, hist);
        PPF_LAUNCH(ctx, radix_col_reduce_kernel, nchunks, RADIX, 0, hist, ntiles, chunk_tot);
        PPF_LAUNCH(ctx, radix_col_scan_chunks_kernel, 1, RADIX, 0, chunk_tot, nchunks, digit_base);
        PPF_LAUNCH(ctx, radix_col_apply_kernel, nchunks, RADIX, 0, hist, ntiles, chunk_tot, digit_base);
#define SCATTER(I, A, B)                                                                                                \
    do {                                                                                                                 \
        PPF_CUDA(ctx, cudaFuncSetAttribute(radix_scatter_kernel<ROUNDS, I, A, B>,                                        \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                     \
        PPF_LAUNCH(ctx, (radix_scatter_kernel<ROUNDS, I, A, B>), ntiles, WARPS * 32, smem, ki, v0i, v1i, (uint32_t)n,    \
                   shift, hist, ko, v0o, v1o);                                                                           \
    } while (0)
        if (has_v0 && has_v1) {
            if (iota) SCATTER(true, true, true); else SCATTER(false, true, true);
        } else if (has_v0) {
            if (iota) SCATTER(true, true, false); else SCATTER(false, true, false);
        } else if (has_v1) {
            SCATTER(false, false, true);
        } else {
            SCATTER(false, false, false);
        }
#undef SCATTER
        iota = false;
        uint32_t *t;
        t = ki; ki = ko; ko = t;
        t = v0i; v0i = v0o; v0o = t;
        t = v1i; v1i = v1o; v1o = t;
        in_alt = !in_alt;
    }
    *result_in_alt = in_alt;
    return B200PPF_OK;
}

}  // namespace

int radix_sort_u32(b200ppf_ctx *ctx, uint32_t *keys, uint32_t *keys_alt, uint32_t *v0, uint32_t *v0_alt,
                   uint32_t *v1, uint32_t *v1_alt, size_t n, uint64_t max_key, bool v0_iota, bool *result_in_alt) {
    *result_in_alt = false;
    if (n == 0) return B200PPF_OK;
    if (n >= 0xFFFFFFFFull - WARPS * ROUNDS_BIG * 32)
        return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "radix sort: more than 2^32 elements");
    // the bits of max_key, at least one (a single pass also writes the iota payload), at most 32
    int bits = 1;
    while (bits < 32 && (max_key >> bits) != 0) ++bits;
    // 4096-element tiles once every SM gets a few of them, 512-element tiles for small inputs
    if (n >= (size_t)ctx->sm_count * 4 * WARPS * ROUNDS_BIG * 32)
        return radix_sort_impl<ROUNDS_BIG>(ctx, keys, keys_alt, v0, v0_alt, v1, v1_alt, n, bits, v0_iota, result_in_alt);
    return radix_sort_impl<ROUNDS_SMALL>(ctx, keys, keys_alt, v0, v0_alt, v1, v1_alt, n, bits, v0_iota, result_in_alt);
}

int lower_bounds(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, const uint32_t *n_dev, uint32_t n_keys, uint32_t shift,
                 uint32_t *offsets) {
    PPF_LAUNCH(ctx, lower_bounds_kernel, (unsigned)(((size_t)n_keys + 256) / 256), 256, 0, sorted, n, n_dev, n_keys, shift, offsets);
    return B200PPF_OK;
}

int flag_scan(b200ppf_ctx *ctx, const uint32_t *flags, uint32_t n, uint32_t *rank, uint32_t *total_dev) {
    if (n == 0) {
        PPF_CUDA(ctx, cudaMemsetAsync(total_dev, 0, sizeof(uint32_t), ctx->stream));
        return B200PPF_OK;
    }
    const uint32_t nb = (n + SCAN_BLOCK - 1) / SCAN_BLOCK;
    StreamBuf<uint32_t> block_sums(ctx);
    PPF_CUDA(ctx, block_sums.alloc(nb));
    PPF_LAUNCH(ctx, flag_count_kernel, nb, SCAN_BLOCK, 0, flags, n, block_sums);
    PPF_LAUNCH(ctx, scan_rows_kernel, 1, SCAN_BLOCK, 0, block_sums, nb, total_dev);
    PPF_LAUNCH(ctx, flag_rank_kernel, nb, SCAN_BLOCK, 0, flags, n, block_sums, rank);
    return B200PPF_OK;
}

int flag_scan_host(b200ppf_ctx *ctx, const uint32_t *flags, uint32_t n, uint32_t *rank, uint32_t *total_host) {
    *total_host = 0;
    if (n == 0) return B200PPF_OK;
    StreamBuf<uint32_t> total(ctx);
    PPF_CUDA(ctx, total.alloc(1));
    if (int rc = flag_scan(ctx, flags, n, rank, total)) return rc;
    PPF_CUDA(ctx, cudaMemcpyAsync(total_host, total, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int scan_rows(b200ppf_ctx *ctx, uint32_t *data, uint32_t n_rows, uint32_t row_len, uint32_t *totals) {
    PPF_LAUNCH(ctx, scan_rows_kernel, n_rows, SCAN_BLOCK, 0, data, row_len, totals);
    return B200PPF_OK;
}

int run_heads(b200ppf_ctx *ctx, const uint32_t *sorted, uint32_t n, uint32_t *head) {
    if (n) PPF_LAUNCH(ctx, run_heads_kernel, (n + 255) / 256, 256, 0, sorted, n, head);
    return B200PPF_OK;
}

}  // namespace b200ppf
