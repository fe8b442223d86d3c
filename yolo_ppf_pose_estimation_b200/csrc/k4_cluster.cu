// k4_cluster.cu — K4 ppf_cluster_average: greedy pose clustering and averaging on the device.
//
// Replaces PPFRegistration::clusterPoses / posesWithinErrorBounds
// ([PCL] registration/include/pcl/registration/impl/ppf_registration.hpp; SURVEY.md A.5):
//   sort hypotheses by votes (descending; ties keep reference order, A.8 rule 1);
//   each hypothesis joins the FIRST cluster (creation order) whose leader pose is within
//   (position, rotation) bounds, else it founds a new cluster; cluster votes are summed;
//   the three best clusters (votes descending, ties by creation order) are averaged
//   (mean translation, mean quaternion coefficients, normalised).
//
// PCL's loop is O(P * C) and serial.  The same assignment is computed here in parallel:
//   * "pose k founds a cluster  <=>  no EARLIER leader is within bounds of k" is the
//     lexicographically-first maximal independent set of the within-bounds graph in sorted order.
//     It is resolved in rounds: an undecided pose becomes a MEMBER as soon as an earlier within-bounds
//     pose is a LEADER, and a LEADER as soon as every earlier within-bounds pose is a MEMBER.
//     Decisions only ever use final states, so the fixpoint is PCL's result whatever the timing.
//   * within-bounds needs |dt| < pos_thr, so poses are hashed by translation cell (edge >=
//     pos_thr) and only the 27 neighbouring cells are searched: O(P) tests for realistic inputs
//     instead of P^2/2.  Hash collisions only add candidates that the exact test rejects.
//   * the poses that are not MEMBERs yet are kept as one list per translation cell, in rank order, and the
//     list is compacted after every round: a pose walks only the few earlier leaders and undecided poses of
//     its 27 cells, not the thousands of members that pile up on one object (config 3: 10 000 of them);
//   * a MEMBER's cluster is the lowest-ranked LEADER within bounds — the first hit of a walk over the
//     leaders-only lists, which are in rank order too; cluster creation indices are the exclusive prefix
//     sum of the leader flags.
#include <algorithm>
#include <cmath>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

constexpr uint32_t NONE = 0xFFFFFFFFu;
constexpr uint32_t ST_UNDECIDED = 0, ST_LEADER = 1, ST_MEMBER = 2;
static_assert(ST_LEADER == 1, "the leader numbering scans state: flag_scan counts the entries equal to 1");

struct PoseRows {  // 3x4 row-major pose as three float4 rows
    float4 r0, r1, r2;
};

__device__ __forceinline__ void rows_to_array(const PoseRows &p, float *a) {
    a[0] = p.r0.x; a[1] = p.r0.y; a[2] = p.r0.z; a[3] = p.r0.w;
    a[4] = p.r1.x; a[5] = p.r1.y; a[6] = p.r1.z; a[7] = p.r1.w;
    a[8] = p.r2.x; a[9] = p.r2.y; a[10] = p.r2.z; a[11] = p.r2.w;
}

struct HashParams {
    float inv_cell;
    uint32_t mask;  // table size - 1 (power of two)
};

__device__ __forceinline__ int cell_of(float v, float inv_cell) { return __float2int_rd(v * inv_cell); }

__device__ __forceinline__ uint32_t cell_hash(int x, int y, int z, uint32_t mask) {
    uint32_t h = ((uint32_t)x * 73856093u) ^ ((uint32_t)y * 19349663u) ^ ((uint32_t)z * 83492791u);
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 12;
    return h & mask;
}

__global__ void cluster_max_votes_kernel(const b200ppf_hypothesis *__restrict__ hyps, uint32_t n,
                                         uint32_t *__restrict__ max_votes) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t v = p < n ? hyps[p].votes : 0u;
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    if ((threadIdx.x & 31) == 0 && v) atomicMax(max_votes, v);
}

__global__ void cluster_keys_kernel(const b200ppf_hypothesis *__restrict__ hyps, uint32_t n, uint32_t max_votes,
                                    uint32_t *__restrict__ keys) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) keys[p] = max_votes - hyps[p].votes;  // ascending key == descending votes
}

__global__ void cluster_gather_kernel(const b200ppf_hypothesis *__restrict__ hyps, const uint32_t *__restrict__ order,
                                      uint32_t n, HashParams hp, PoseRows *__restrict__ poses,
                                      uint32_t *__restrict__ votes, uint32_t *__restrict__ cell_keys) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const b200ppf_hypothesis &h = hyps[order[k]];
    PoseRows p;
    p.r0 = make_float4(h.pose[0], h.pose[1], h.pose[2], h.pose[3]);
    p.r1 = make_float4(h.pose[4], h.pose[5], h.pose[6], h.pose[7]);
    p.r2 = make_float4(h.pose[8], h.pose[9], h.pose[10], h.pose[11]);
    poses[k] = p;
    votes[k] = h.votes;
    cell_keys[k] = cell_hash(cell_of(h.pose[3], hp.inv_cell), cell_of(h.pose[7], hp.inv_cell),
                             cell_of(h.pose[11], hp.inv_cell), hp.mask);
}

// Walk the earlier (rank < k) entries of the per-cell lists around pose k, in rank order inside every cell, and call
// f(rank j) for those within bounds of k; f returns true to stop.  The lists hold what is still of interest — every
// pose at first, then the non-members, finally the leaders only — and `keep(state)` skips entries untested.
template <class Keep, class F>
__device__ __forceinline__ void for_each_earlier_within(const PoseRows *__restrict__ poses,
                                                        const uint32_t *__restrict__ cell_start,
                                                        const uint32_t *__restrict__ cell_rank, HashParams hp, uint32_t k,
                                                        const float *a, float pos_thr, float rot_thr,
                                                        const volatile uint32_t *state, Keep keep, F f) {
    const int cx = cell_of(a[3], hp.inv_cell), cy = cell_of(a[7], hp.inv_cell), cz = cell_of(a[11], hp.inv_cell);
    uint32_t seen[27];
    int n_seen = 0;
    for (int dz = -1; dz <= 1; ++dz)
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                const uint32_t h = cell_hash(cx + dx, cy + dy, cz + dz, hp.mask);
                bool dup = false;  // two neighbour cells may share a bucket: visit it once
                for (int q = 0; q < n_seen; ++q) dup |= (seen[q] == h);
                if (dup) continue;
                seen[n_seen++] = h;
                const uint32_t b = cell_start[h], e = cell_start[h + 1];
                for (uint32_t s = b; s < e; ++s) {
                    const uint32_t j = cell_rank[s];
                    if (j >= k) break;  // ranks ascend inside a bucket (stable sort, order-preserving compaction)
                    const int kk = keep(state[j]);  // 0: skip untested, 1: test, 2: stop the walk
                    if (kk == 2) return;
                    if (!kk) continue;
                    const PoseRows pj = poses[j];
                    const float ddx = a[3] - pj.r0.w, ddy = a[7] - pj.r1.w, ddz = a[11] - pj.r2.w;
                    if (!(sqrtf((ddx * ddx + ddy * ddy) + ddz * ddz) < pos_thr)) continue;
                    float bb[12];
                    rows_to_array(pj, bb);
                    if (poses_within(a, bb, pos_thr, rot_thr) && f(j)) return;
                }
            }
}

// one round of the ordered independent-set resolution.  Two sets of per-cell lists, both in rank order: the leaders found
// so far (short) and the poses that are not members yet.  An earlier LEADER within bounds makes the pose a MEMBER; failing
// that, an earlier UNDECIDED pose within bounds blocks it for this round; a pose that meets neither is a LEADER.
__global__ void __launch_bounds__(128)
cluster_round_kernel(const PoseRows *__restrict__ poses, const uint32_t *__restrict__ cell_start,
                     const uint32_t *__restrict__ cell_rank, const uint32_t *__restrict__ lcell_start,
                     const uint32_t *__restrict__ lcell_rank, HashParams hp, uint32_t n, float pos_thr, float rot_thr,
                     volatile uint32_t *state, uint32_t *__restrict__ undecided) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || state[k] != ST_UNDECIDED) return;
    float a[12];
    rows_to_array(poses[k], a);
    bool blocked = false, member = false;
    // every leader the lists know of (those made in this very round are met next round: a stale view costs a round, not
    // correctness — decisions only ever use final states)
    for_each_earlier_within(
        poses, lcell_start, lcell_rank, hp, k, a, pos_thr, rot_thr, state, [&](uint32_t) -> int { return 1; },
        [&](uint32_t) {
            member = true;
            return true;
        });
    if (!member) {
        // A pose that has compared itself with UNDECIDED_TESTS earlier undecided poses without finding one within bounds
        // gives up for this round (it stays undecided: always safe) — the poses of a crowded cell that resemble nobody would
        // otherwise compare themselves with thousands of poses each.  The lowest-ranked undecided pose has no undecided pose
        // before it, so it never gives up and every round decides at least one pose.
        constexpr int UNDECIDED_TESTS = 48;
        int tested = 0;
        for_each_earlier_within(
            poses, cell_start, cell_rank, hp, k, a, pos_thr, rot_thr, state,
            [&](uint32_t sj) -> int {
                if (sj == ST_LEADER) return 1;  // possibly one made in this very round, which the leaders' lists do not hold yet
                if (sj != ST_UNDECIDED) return 0;
                if (++tested > UNDECIDED_TESTS) {
                    blocked = true;
                    return 2;
                }
                return 1;
            },
            [&](uint32_t j) {
                const uint32_t sj = state[j];
                if (sj == ST_LEADER) {
                    member = true;
                    return true;
                }
                if (sj == ST_UNDECIDED) {
                    blocked = true;
                    return true;
                }
                return false;
            });
    }
    if (member) state[k] = ST_MEMBER;
    else if (!blocked) state[k] = ST_LEADER;
    else atomicAdd(undecided, 1u);
}

// list compaction: keep[s] = the entry's pose is (still) of interest; the scan that follows preserves the order.  n bounds
// the list's length *n_list on the host: the entries between the two are not kept.
__global__ void cluster_keep_flags_kernel(const uint32_t *__restrict__ cell_rank, uint32_t n, const uint32_t *__restrict__ n_list,
                                          const uint32_t *__restrict__ state, uint32_t leaders_only,
                                          uint32_t *__restrict__ keep) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t k = 0;
    if (s < *n_list) {
        const uint32_t st = state[cell_rank[s]];
        k = leaders_only ? (st == ST_LEADER) : (st != ST_MEMBER);
    }
    keep[s] = k;
}

__global__ void cluster_compact_kernel(const uint32_t *__restrict__ cell_rank, const uint32_t *__restrict__ cell_keys,
                                       const uint32_t *__restrict__ n_list, const uint32_t *__restrict__ keep,
                                       const uint32_t *__restrict__ pos, uint32_t *__restrict__ rank_out,
                                       uint32_t *__restrict__ keys_out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_list || !keep[s]) return;
    rank_out[pos[s]] = cell_rank[s];
    keys_out[pos[s]] = cell_keys[s];
}

// every pose -> its cluster (leaders: their own; members: the lowest-ranked leader within bounds).  The lists hold
// leaders only by now; inside a cell they are in rank order, so the walk of a cell stops at its first hit.
__global__ void __launch_bounds__(128)
cluster_assign_kernel(const PoseRows *__restrict__ poses, const uint32_t *__restrict__ cell_start,
                      const uint32_t *__restrict__ cell_rank, HashParams hp, uint32_t n, float pos_thr, float rot_thr,
                      const uint32_t *__restrict__ state, const uint32_t *__restrict__ leader_id,
                      const uint32_t *__restrict__ votes, const uint32_t *__restrict__ order,
                      uint32_t *__restrict__ assign_sorted, uint32_t *__restrict__ assign_input,
                      uint32_t *__restrict__ cluster_votes, uint32_t *__restrict__ cluster_size) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint32_t c;
    if (state[k] == ST_LEADER) {
        c = leader_id[k];
    } else {
        float a[12];
        rows_to_array(poses[k], a);
        uint32_t best = NONE;
        const int cx = cell_of(a[3], hp.inv_cell), cy = cell_of(a[7], hp.inv_cell), cz = cell_of(a[11], hp.inv_cell);
        uint32_t seen[27];
        int n_seen = 0;
        for (int dz = -1; dz <= 1; ++dz)
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const uint32_t h = cell_hash(cx + dx, cy + dy, cz + dz, hp.mask);
                    bool dup = false;
                    for (int q = 0; q < n_seen; ++q) dup |= (seen[q] == h);
                    if (dup) continue;
                    seen[n_seen++] = h;
                    const uint32_t b = cell_start[h], e = cell_start[h + 1];
                    for (uint32_t s = b; s < e; ++s) {
                        const uint32_t j = cell_rank[s];
                        if (j >= k || j >= best) break;  // ranks ascend: nothing better further on in this cell
                        const PoseRows pj = poses[j];
                        const float ddx = a[3] - pj.r0.w, ddy = a[7] - pj.r1.w, ddz = a[11] - pj.r2.w;
                        if (!(sqrtf((ddx * ddx + ddy * ddy) + ddz * ddz) < pos_thr)) continue;
                        float bb[12];
                        rows_to_array(pj, bb);
                        if (poses_within(a, bb, pos_thr, rot_thr)) {
                            best = j;
                            break;
                        }
                    }
                }
        c = best != NONE ? leader_id[best] : 0u;  // a MEMBER always has an earlier leader; guard only
    }
    assign_sorted[k] = c;
    assign_input[order[k]] = c;
    atomicAdd(&cluster_votes[c], votes[k]);
    atomicAdd(&cluster_size[c], 1u);
}

// three best clusters: votes descending, creation index ascending (one CTA)
__global__ void __launch_bounds__(1024)
cluster_top3_kernel(const uint32_t *__restrict__ cluster_votes, const uint32_t *__restrict__ n_clusters_ptr,
                    uint32_t *__restrict__ top /* [3] cluster ids, NONE if absent */) {
    __shared__ unsigned long long s_best[32];
    __shared__ uint32_t chosen[3];
    const uint32_t nc = *n_clusters_ptr;
    for (int round = 0; round < 3; ++round) {
        unsigned long long best = 0;
        for (uint32_t c = threadIdx.x; c < nc; c += blockDim.x) {
            bool taken = false;
            for (int q = 0; q < round; ++q) taken |= (chosen[q] == c);
            if (taken) continue;
            // +1 so that a zero-vote cluster still beats "nothing"
            unsigned long long key = (((unsigned long long)cluster_votes[c] + 1ull) << 32) | (0xFFFFFFFFu - c);
            best = max(best, key);
        }
        for (int o = 16; o > 0; o >>= 1) best = max(best, (unsigned long long)__shfl_xor_sync(0xFFFFFFFFu, best, o));
        if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < 32; ++w) best = max(best, s_best[w]);
            chosen[round] = best ? 0xFFFFFFFFu - (uint32_t)(best & 0xFFFFFFFFu) : NONE;
            top[round] = chosen[round];
        }
        __syncthreads();
    }
}

// mean translation + mean quaternion of one top cluster per CTA (deterministic tree reduction)
__global__ void __launch_bounds__(256)
cluster_average_kernel(const PoseRows *__restrict__ poses, const uint32_t *__restrict__ assign_sorted, uint32_t n,
                       const uint32_t *__restrict__ top, const uint32_t *__restrict__ cluster_votes,
                       const uint32_t *__restrict__ cluster_size, float *__restrict__ out_poses /* [3][16] */,
                       uint32_t *__restrict__ out_votes /* [3] */) {
    __shared__ double red[256][7];
    const uint32_t c = top[blockIdx.x];
    if (c == NONE) {
        if (threadIdx.x == 0) out_votes[blockIdx.x] = 0;
        return;
    }
    double acc[7] = {0, 0, 0, 0, 0, 0, 0};
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
        if (assign_sorted[k] != c) continue;
        float a[12], q[4];
        rows_to_array(poses[k], a);
        const float R[9] = {a[0], a[1], a[2], a[4], a[5], a[6], a[8], a[9], a[10]};
        quat_from_matrix(R, q);
        acc[0] += a[3]; acc[1] += a[7]; acc[2] += a[11];
        acc[3] += q[0]; acc[4] += q[1]; acc[5] += q[2]; acc[6] += q[3];
    }
    for (int v = 0; v < 7; ++v) red[threadIdx.x][v] = acc[v];
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s)
            for (int v = 0; v < 7; ++v) red[threadIdx.x][v] += red[threadIdx.x + s][v];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float cnt = (float)cluster_size[c];
        float t[3], q[4];
        for (int v = 0; v < 3; ++v) t[v] = (float)red[0][v] / cnt;
        for (int v = 0; v < 4; ++v) q[v] = (float)red[0][3 + v] / cnt;
        const float qn = sqrtf(((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2]) + q[3] * q[3]);
        if (qn > 0.0f)
            for (int v = 0; v < 4; ++v) q[v] /= qn;
        float R[9];
        quat_to_matrix(q, R);
        float *M = out_poses + 16 * blockIdx.x;
        M[0] = R[0]; M[1] = R[1]; M[2] = R[2]; M[3] = t[0];
        M[4] = R[3]; M[5] = R[4]; M[6] = R[5]; M[7] = t[1];
        M[8] = R[6]; M[9] = R[7]; M[10] = R[8]; M[11] = t[2];
        M[12] = 0.0f; M[13] = 0.0f; M[14] = 0.0f; M[15] = 1.0f;
        out_votes[blockIdx.x] = cluster_votes[c];
    }
}

}  // namespace

int k4_cluster(b200ppf_ctx *ctx, const b200ppf_hypothesis *hyps, size_t n_, float pos_thr, float rot_thr,
               float *poses16, uint32_t *votes_out, size_t *n_out) {
    *n_out = 0;
    if (n_ == 0) return B200PPF_OK;
    if (n_ >= 0x7FFFFFFFull) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "cluster: too many hypotheses");
    const uint32_t n = (uint32_t)n_;
    cudaStream_t st = ctx->stream;
    cudaEventRecord(ctx->ev[0], st);

    // translation hash grid: cell edge >= pos_thr (margin absorbs the rounding of the cell coordinate)
    HashParams hp;
    {
        double cell = std::isinf(pos_thr) ? 1e30 : (pos_thr > 0.0f ? (double)pos_thr * 1.001 : 1e-6);
        cell = std::max(cell, 1e-6);
        hp.inv_cell = (float)(1.0 / cell);
        int bits = 8;
        while ((1u << bits) < 2u * n && bits < 22) ++bits;
        hp.mask = (1u << bits) - 1u;
    }
    const uint32_t n_cells = hp.mask + 1u;

    // one pooled allocation for all scratch
    uint32_t *keys[2], *order[2], *ckeys[2], *crank[2];
    uint32_t *votes, *state, *leader_id, *assign_sorted, *cl_votes, *cl_size, *cell_start, *small;
    PoseRows *poses;
    float *d_out;
    size_t words = 0;
    auto take = [&](size_t w) { size_t o = words; words += (w + 3) & ~size_t(3); return o; };
    const size_t o_keys0 = take(n), o_keys1 = take(n), o_ord0 = take(n), o_ord1 = take(n), o_ck0 = take(n),
                 o_ck1 = take(n), o_cr0 = take(n), o_cr1 = take(n), o_votes = take(n), o_state = take(n),
                 o_lid = take(n), o_as = take(n), o_cv = take(n), o_cs = take(n), o_cell = take((size_t)n_cells + 1),
                 o_small = take(16), o_out = take(48), o_poses = take((size_t)n * 12),
                 o_lr = take(n), o_lk = take(n), o_lcell = take((size_t)n_cells + 1);
    StreamBuf<uint32_t> pool_owner(ctx);  // returned to the pool on every path out of this function
    PPF_CUDA(ctx, pool_owner.alloc(words));
    uint32_t *pool = pool_owner.p;
    keys[0] = pool + o_keys0; keys[1] = pool + o_keys1; order[0] = pool + o_ord0; order[1] = pool + o_ord1;
    ckeys[0] = pool + o_ck0; ckeys[1] = pool + o_ck1; crank[0] = pool + o_cr0; crank[1] = pool + o_cr1;
    votes = pool + o_votes; state = pool + o_state; leader_id = pool + o_lid; assign_sorted = pool + o_as;
    cl_votes = pool + o_cv; cl_size = pool + o_cs; cell_start = pool + o_cell;
    small = pool + o_small; d_out = reinterpret_cast<float *>(pool + o_out);
    poses = reinterpret_cast<PoseRows *>(pool + o_poses);
    uint32_t *lrank = pool + o_lr, *lkeys = pool + o_lk, *lcell_start = pool + o_lcell;
    // state .. cl_size are contiguous: one memset clears state (UNDECIDED), leader ids, assignments, cluster sums
    PPF_CUDA(ctx, cudaMemsetAsync(state, 0, (o_cell - o_state) * sizeof(uint32_t), st));
    PPF_CUDA(ctx, cudaMemsetAsync(small, 0, (16 + 48) * sizeof(uint32_t), st));
    ctx->assign_n = 0;
    PPF_CUDA(ctx, grow_buffer(&ctx->d_assign, &ctx->assign_cap, n));
    ctx->assign_n = n;

    // small[0] = max votes, small[1] = undecided counter, small[2] = n_clusters, small[3..5] = top, small[6..8] = votes
    const unsigned g = (n + 255) / 256;
    uint32_t h_small[16];
    PPF_LAUNCH(ctx, cluster_max_votes_kernel, g, 256, 0, hyps, n, small);
    PPF_CUDA(ctx, cudaMemcpyAsync(h_small, small, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PPF_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t max_votes = h_small[0];
    PPF_LAUNCH(ctx, cluster_keys_kernel, g, 256, 0, hyps, n, max_votes, keys[0]);
    bool in_alt = false;
    int rc = radix_sort_u32(ctx, keys[0], keys[1], order[0], order[1], nullptr, nullptr, n, max_votes, /*v0_iota=*/true,
                            &in_alt);
    if (rc) return rc;
    const uint32_t *ord = order[in_alt ? 1 : 0];
    PPF_LAUNCH(ctx, cluster_gather_kernel, g, 256, 0, hyps, ord, n, hp, poses, votes, ckeys[0]);
    rc = radix_sort_u32(ctx, ckeys[0], ckeys[1], crank[0], crank[1], nullptr, nullptr, n, n_cells - 1, /*v0_iota=*/true,
                        &in_alt);
    if (rc) return rc;
    const uint32_t *cell_keys_sorted = ckeys[in_alt ? 1 : 0], *cell_rank = crank[in_alt ? 1 : 0];
    if ((rc = lower_bounds(ctx, cell_keys_sorted, n, nullptr, n_cells, 0, cell_start))) return rc;

    // The per-cell lists (cell_rank / cell keys, sorted by cell then rank) start with every pose and are compacted to
    // the non-members after each round, to the leaders at the end.  keep flags and positions live in the first
    // sort's buffers (free by now); small[9] = current list length.
    uint32_t *keep = keys[0], *pos = keys[1];
    int cur = in_alt ? 1 : 0;  // which crank / ckeys buffer holds the current lists
    uint32_t n_list = n;
    PPF_CUDA(ctx, cudaMemcpyAsync(small + 9, &n_list, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    // compaction of the current non-member lists: into themselves without the members (mode 0: small[9] <- new length), or
    // into the leaders-only lists (mode 1: small[11] <- their length); n_list bounds the source length on the host
    auto compact = [&](uint32_t leaders_only) -> int {
        const unsigned gl = (n_list + 255) / 256;
        uint32_t *dst_rank = leaders_only ? lrank : crank[1 - cur], *dst_keys = leaders_only ? lkeys : ckeys[1 - cur];
        uint32_t *dst_n = small + (leaders_only ? 11 : 10);
        if (n_list == 0) {
            PPF_CUDA(ctx, cudaMemsetAsync(dst_n, 0, sizeof(uint32_t), st));
        } else {
            PPF_LAUNCH(ctx, cluster_keep_flags_kernel, gl, 256, 0, crank[cur], n_list, small + 9, state, leaders_only, keep);
            if (int rc = flag_scan(ctx, keep, n_list, pos, dst_n)) return rc;
            PPF_LAUNCH(ctx, cluster_compact_kernel, gl, 256, 0, crank[cur], ckeys[cur], small + 9, keep, pos, dst_rank, dst_keys);
        }
        if (leaders_only) return lower_bounds(ctx, lkeys, 0, small + 11, n_cells, 0, lcell_start);
        PPF_CUDA(ctx, cudaMemcpyAsync(small + 9, small + 10, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        cur = 1 - cur;
        return lower_bounds(ctx, ckeys[cur], 0, small + 9, n_cells, 0, cell_start);
    };
    // no leader yet: empty leaders-only lists
    PPF_CUDA(ctx, cudaMemsetAsync(lcell_start, 0, ((size_t)n_cells + 1) * sizeof(uint32_t), st));
    // ordered independent-set rounds until nothing is undecided
    const unsigned gr = (n + 127) / 128;
    for (int iter = 0;; ++iter) {
        PPF_CUDA(ctx, cudaMemsetAsync(small + 1, 0, sizeof(uint32_t), st));
        PPF_LAUNCH(ctx, cluster_round_kernel, gr, 128, 0, poses, cell_start, crank[cur], lcell_start, lrank, hp, n, pos_thr, rot_thr,
                   state, small + 1);
        // the members leave the lists (worth it while the lists are long: a pose's walk is as long as the non-members of its
        // 27 cells), then the leaders-only lists are drawn from what is left
        if (n_list > 2048 && iter > 0 && (rc = compact(0u))) return rc;
        if ((rc = compact(1u))) return rc;
        PPF_CUDA(ctx, cudaMemcpyAsync(h_small, small, sizeof(h_small), cudaMemcpyDeviceToHost, st));
        PPF_CUDA(ctx, cudaStreamSynchronize(st));
        n_list = h_small[9];
        if (h_small[1] == 0) break;
        if (iter > (int)n) return fail_msg(ctx, B200PPF_ERR_CUDA, "cluster: leader resolution did not converge");
    }
    // lcell_start / lrank now hold every leader, in rank order inside every cell.  No pose is undecided any more, so the
    // entries of state equal to 1 are the leaders: leader_id[k] = leaders before k, the creation index of leader k (the
    // values at members are never read), small[2] = the number of clusters.
    if ((rc = flag_scan(ctx, state, n, leader_id, small + 2))) return rc;
    PPF_LAUNCH(ctx, cluster_assign_kernel, gr, 128, 0, poses, lcell_start, lrank, hp, n, pos_thr, rot_thr, state,
               leader_id, votes, ord, assign_sorted, ctx->d_assign, cl_votes, cl_size);
    PPF_LAUNCH(ctx, cluster_top3_kernel, 1, 1024, 0, cl_votes, small + 2, small + 3);
    PPF_LAUNCH(ctx, cluster_average_kernel, 3, 256, 0, poses, assign_sorted, n, small + 3, cl_votes, cl_size, d_out,
               small + 6);
    float h_out[48];
    PPF_CUDA(ctx, cudaMemcpyAsync(h_small, small, sizeof(h_small), cudaMemcpyDeviceToHost, st));
    PPF_CUDA(ctx, cudaMemcpyAsync(h_out, d_out, sizeof(h_out), cudaMemcpyDeviceToHost, st));
    cudaEventRecord(ctx->ev[1], st);
    PPF_CUDA(ctx, cudaStreamSynchronize(st));
    cudaEventElapsedTime(&ctx->timings.cluster_ms, ctx->ev[0], ctx->ev[1]);
    ctx->n_clusters = h_small[2];
    size_t k = 0;
    for (int r = 0; r < 3; ++r) {
        if (h_small[3 + r] == NONE) break;
        memcpy(poses16 + 16 * k, h_out + 16 * r, 16 * sizeof(float));
        votes_out[k] = h_small[6 + r];
        ++k;
    }
    *n_out = k;
    return B200PPF_OK;
}

}  // namespace b200ppf
