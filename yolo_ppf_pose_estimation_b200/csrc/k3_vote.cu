// k3_vote.cu — K3 ppf_vote_argmax: scene voting, peak pick and pose assembly.
//
// Replaces the voting loop of PPFRegistration::computeTransformation
// ([PCL] registration/include/pcl/registration/impl/ppf_registration.hpp; SURVEY.md A.4):
//   for every scene reference point s_r: frame T_sg; every scene point within max_dist/2 gives a
//   pair feature -> bucket -> for every (i, alpha_m) in the bucket acc[i][bin(alpha_m - alpha_s)]++;
//   first maximum of acc (lowest flat index wins ties) -> pose = T_sg^-1 * Rx(theta) * T_mg.
//
// One task per (reference point, accumulator slice): one CTA each, or persistent CTAs drawing them from a counter.  The accumulator slice — up to ~1600 model
// rows x n_alpha 32-bit counters — lives in shared memory for the CTA's whole life, votes are
// shared-memory reductions (red.shared.add), the peak is a warp-shuffle argmax, and slices merge
// through one 64-bit atomicMax per CTA on a packed (votes, ~flat index) word, which reproduces
// PCL's tie-break.  Three phases keep the lanes busy:
//   A  sweep  the 27-cell neighbourhood of the reference point in the cell-sorted scene
//             (scene_grid.cu) is 9 contiguous runs of float4 positions; the radius predicate
//             survivors are compacted into a shared candidate queue (one warp-aggregated atomic);
//   B  pair   one thread per candidate: pair feature, key, alpha_s -> up to three work items.
//             Buckets are ordered by the phase cell of alpha_m (k2_table.cu): the cells below the
//             scene pair's phase and the cells above it are two "shift" items whose every vote lands
//             at (entry's hot word - one constant); the scene phase's own cell is a "per-entry" item;
//   C  vote   warps pull work items.  Shift items: 8 x 32 hot words in flight per lane, a vote is
//             load / subtract / add-min / red.shared (ppf_math.cuh "constant-shift voting").
//             The scene phase's own cell compares phases per entry — on folding tables, whose cells the build
//             orders by sub-phase block, a group of steps whose entries all lie on one side of the scene phase
//             votes with one shift; tables whose 2*pi/step is not an integer bin every entry in fixed point
//             with guard bands, the literal double-precision form inside the bands.
//   D  fold   tables of 2 M+ entries, tasks that flush more than once or hold FOLD_MIN_PAIRS+ candidates: a pair on the
//             constant-shift path keeps only its own cell in phase C and leaves a code (key, q, cell) in its CTA's fold
//             buffer, across flushes.  At the end of the task (or of a scope of FOLD_SCOPE codes) the codes are sorted; for
//             every (bucket, shift s) they touch, a warp reads off per cell how many pairs vote on it with that shift
//             (prefix / suffix counts of the cells at q = s and q = s - 1) and walks the cell once, adding count x pairs.
//             Sums of integers in any order: the accumulators are those of one walk per pair.
// The accumulator slice is bin-major (word = bin * pitch + row, pitch a multiple of 32): the bank of a vote
// is (row mod 32) whatever the scene pair, and the table build orders every phase cell so that 32
// consecutive entries hit 32 different banks.
// Roofline (profiles/): the SM's L1 data pipe — one wavefront per 32 gathered hot words plus one per
// distinct bank conflict degree of the 32 reductions; HBM sees the table and the scene once.
#include <algorithm>
#include <cmath>
#include <type_traits>

#include "ppf_common.cuh"

namespace b200ppf {

namespace {

#ifndef B200PPF_VOTE_MINBLOCKS
#define B200PPF_VOTE_MINBLOCKS 2
#endif
// Two launch shapes: 512 threads with two CTAs per SM when the accumulator slice leaves room for both,
// 1024 threads with one CTA per SM (the same 32 warps) for the large slices of sliced tables.
constexpr int VOTE_THREADS_SMALL = 512;
constexpr int VOTE_THREADS_LARGE = 1024;
#ifndef B200PPF_OWN_UNROLL
#define B200PPF_OWN_UNROLL 4
#endif
constexpr int OWN_UNROLL = B200PPF_OWN_UNROLL;  // steps of 32 entries in flight in the scene phase's own cell
#ifndef B200PPF_OWN_SUB_MIN
#define B200PPF_OWN_SUB_MIN 96
#endif
constexpr uint32_t OWN_SUB_MIN = B200PPF_OWN_SUB_MIN;  // shorter own cells are compared in full (config 2: ~10 entries per cell)
constexpr int FULL_UNROLL = 2;  // steps in flight of the full comparison
#ifndef B200PPF_CAND_CAP
#define B200PPF_CAND_CAP 2048
#endif
constexpr int CAND_CAP = B200PPF_CAND_CAP;  // in-radius candidates buffered between flushes
#ifndef B200PPF_VOTE_UNROLL
#define B200PPF_VOTE_UNROLL 4
#endif
constexpr int VOTE_UNROLL = B200PPF_VOTE_UNROLL;
static_assert(CAND_CAP >= 2 * VOTE_THREADS_LARGE, "flush threshold must leave one sweep iteration of room");
#ifndef B200PPF_FOLD_MIN_PAIRS
#define B200PPF_FOLD_MIN_PAIRS 1024
#endif
constexpr uint32_t FOLD_MIN_PAIRS = B200PPF_FOLD_MIN_PAIRS;  // single-flush tasks with fewer candidates keep one walk per pair
constexpr size_t FOLD_MIN_ENTRIES = 1u << 21;  // tables below this walk short buckets: folding does not repay its sort

// One in-radius scene pair with a non-empty bucket.  Phase-sorted tables: the bucket's merged words are
// [off, off + len); those below k_below lie under the scene pair's phase (shift constant c_below), those from
// k_above on over it (c_below minus one bin); the scene phase's own cell — or the whole bucket when the phase sits
// on a cell edge, then k_below = k_above = len — takes the per-entry path over the unmerged entries
// [e_off, e_off + e_len).  Other tables: off = len = 0, every entry is in [e_off, e_off + e_len).
struct __align__(16) WorkItem {
    uint32_t off, len;
    uint32_t k_below, k_above;
    uint32_t e_off, e_len;      // per-entry range in the unmerged entry arrays
    uint32_t sub_range;         // own cell: sub_lo | sub_hi << 8 | 1 << 16 (ppf_math.cuh, sub_phase); 0: compare every entry in full
    uint32_t pad1;
    uint32_t c_below;           // constant subtracted from the hot words below the scene phase: 4 * pitch * (q + 1)
    uint32_t c_s;               // per-entry path: alpha_to_fix(alpha_s) - 2^31
    float alpha_s;              // per-entry path: PCL's float (literal form of the guard-band votes)
    uint32_t phi;               // the scene pair's phase inside its bin (fix_shift bits); 0xFFFFFFFF: every entry takes the literal form
};

// candidate queue + one work item per thread (phase B turns THREADS candidates into items per round)
constexpr size_t queue_bytes(int threads) { return CAND_CAP * sizeof(uint32_t) + (size_t)threads * sizeof(WorkItem); }
constexpr size_t SMALL_SHAPE_SMEM_MAX = 111 * 1024;  // two such CTAs (+ static + system reserve) share one SM
constexpr size_t STATIC_RESERVE = 2048;  // static shared + the 1 KB the system reserves per CTA
// Fold scope: a task's fold codes collect in its CTA's slot of a global buffer (L2-resident) across flushes, and phase D
// folds them once the next flush might not fit, or at the end of the task.  D sorts the codes where the idle candidate and
// item queues are, so the scope is the largest power of two of words both launch shapes' queues hold (8 192 words = the
// 512-thread shape's queues exactly).  The groups (at most two per code) then overwrite the codes in the slot, which the
// sort has taken into shared memory: a slot is 2 * FOLD_SCOPE words.
constexpr uint32_t FOLD_SCOPE = 8192;
constexpr size_t FOLD_SLOT_WORDS = 2 * (size_t)FOLD_SCOPE;
static_assert(FOLD_SCOPE * sizeof(uint32_t) <= queue_bytes(VOTE_THREADS_SMALL) && (FOLD_SCOPE & (FOLD_SCOPE - 1)) == 0,
              "the fold codes of a scope are sorted in the idle queues (bitonic)");
static_assert(FOLD_SCOPE >= CAND_CAP, "a scope must take one whole flush");

struct VoteArgs {
    const float4 *pos, *nrm;    // scene, original order (reference points are addressed by index)
    const float4 *gpos, *gnrm;  // scene, cell-sorted (gpos.w: the bits of the point's original index)
    const uint32_t *cell_start;
    GridParams gp;
    uint32_t n_s;
    uint32_t ref_first, ref_step, ref_count;
    const uint32_t *ref_order;    // task position -> reference slot, heaviest neighbourhood first (nullptr: identity)
    const uint32_t *sub_offsets;  // phase-cell bounds (bucket bounds when the table has no phase cells)
    const uint32_t *msub_offsets; // the same bounds in the merged-vote array (phase-sorted tables)
    const uint32_t *merged_w;     // (count << 24) | hot word
    const uint32_t *entry_w;
    const uint32_t *entry_am;
    const float *entry_alpha;
    KeyParams kp;
    BinParams bp;
    int feature_mode;
    float radius;
    float radius_sq_bound;  // smallest float x with sqrtf(x) >= radius:  sqrtf(d2) < radius <=> d2 < bound
    uint32_t n_model;
    unsigned long long *peaks;
    unsigned long long *stats;
    uint32_t *acc_dump;  // debug: full accumulator of reference 0 (n_model * n_alpha)
    // Persistent CTAs (as many as the device holds at once) draw (reference, slice) tasks from a counter.  One GPU, a
    // folding table: the counter is the context's, peaks are local.  Several GPUs sharing ONE work queue (b200ppf_group):
    // the counter is in rank 0's memory, drawn with system-scope atomics over NVLink — whichever GPU is free takes the next task, so the
    // ranks finish together whatever the scene's cost distribution — and each task's peak is merged into EVERY rank's peak
    // array with a system-scope 64-bit atomicMax.  When its queue is exhausted, the last CTA of a rank raises that rank's
    // flag in every rank's flag array.
    uint32_t *queue;  // nullptr: the grid is (reference, slice)
    unsigned long long *peer_peaks[MAX_PEERS];
    uint32_t *peer_flags[MAX_PEERS];
    int n_peers;  // 0: one GPU
    uint32_t signal_slot, signal_value;
    uint32_t *done_counter;
    int no_sub_phase;  // debug (B200PPF_NO_SUB_PHASE): compare every own-cell entry in full
    uint32_t fold_qbits;  // bits of q in a fold code (key, q, cell); 0: every pair walks its own bucket
    uint32_t *fold_buf;   // folding tables: FOLD_SLOT_WORDS per CTA of the launch, slot = blockIdx.x
};

__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int o) {
    return __shfl_xor_sync(0xFFFFFFFFu, v, o);
}

// keeps a loop-invariant value in a register (an opaque move the compiler cannot rematerialise)
__device__ __forceinline__ uint32_t pin_register(uint32_t v) {
    uint32_t r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
    return r;
}
// shared-memory increment without a return value (ATOMS.POPC.INC on the CTA's shared window)
__device__ __forceinline__ void red_shared_inc(uint32_t addr) {
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
}
// shared-memory add of a merged vote's count (ATOMS.ADD without a return value)
__device__ __forceinline__ void red_shared_add(uint32_t addr, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void red_shared_add_if_lt(uint32_t addr, uint32_t v, uint32_t k, uint32_t len) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %2, %3;\n\t@p red.shared.add.u32 [%0], %1;\n\t}" ::"r"(addr), "r"(v), "r"(k),
                 "r"(len)
                 : "memory");
}
// increment predicated on x >= lo && k < len (the scene phase's own cell: outside the guard band, inside the bucket)
__device__ __forceinline__ void red_shared_inc_if_ge_lt(uint32_t addr, uint32_t x, uint32_t lo, uint32_t k, uint32_t len) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ge.u32 p, %1, %2;\n\tsetp.lt.and.u32 q, %3, %4, p;\n\t@q red.shared.add.u32 [%0], 1;\n\t}" ::"r"(addr),
        "r"(x), "r"(lo), "r"(k), "r"(len)
        : "memory");
}
// the same, predicated on k < len (the partial last step of a shift item)
__device__ __forceinline__ void red_shared_inc_if_lt(uint32_t addr, uint32_t k, uint32_t len) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p red.shared.add.u32 [%0], 1;\n\t}" ::"r"(addr), "r"(k), "r"(len)
                 : "memory");
}

// count of a merged word times the scene pairs that cast it: one pair's item (the constant 1) or a folded group
__device__ __forceinline__ uint32_t times(uint32_t cnt, std::integral_constant<uint32_t, 1>) { return cnt; }
__device__ __forceinline__ uint32_t times(uint32_t cnt, uint32_t pairs) { return cnt * pairs; }

// Phase timing (instrumented builds only: -DB200PPF_PHASE_TIMING, e.g. tools/build_variant.sh).  Thread 0 reads
// %globaltimer after the barriers that end each phase and sums the CTA's wall time per phase over the launch's tasks,
// apart for single-flush and multi-flush tasks; lane 0 of every warp sums its own time in phase C's shift ranges and in
// its own cells.  The last CTA of the launch prints one line per task class and clears the sums.
#ifdef B200PPF_PHASE_TIMING
enum { PT_PROLOGUE, PT_SWEEP, PT_PAIRS, PT_VOTES, PT_FOLD, PT_PEAK, PT_C_SHIFT, PT_C_OWN, PT_TASKS, PT_N };
__device__ unsigned long long g_phase_ns[2][PT_N];
__device__ unsigned int g_phase_done;
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define PT_MARK(k)                                      \
    do {                                                \
        if (tid == 0) {                                 \
            const unsigned long long now_ = global_ns(); \
            pt[k] += now_ - pt_t;                       \
            pt_t = now_;                                \
        }                                               \
    } while (0)
#else
#define PT_MARK(k) \
    do {           \
    } while (0)
#endif

// One vote of the per-entry path of tables without phase cells (alpha mode A), in fixed point (ppf_math.cuh,
// alpha_bin_fixed):  X = A_m - C_s  (wraps like the angle),  hi = mulhi(X, T_fix) = bin.position,
// (bin, frac) = hi * 2^(32-s).  The increment is unconditional — a select is cheaper than a divergent branch —
// but when frac lies in the guard band around a bin edge (or X in the band around the +-pi seam), or the lane
// is past the end of the bucket, it is steered to a scratch word; a guard-band hit returns true and the
// caller settles that entry with the literal double-precision form.  en.x = byte offset of the row.
template <bool SEAM>
__device__ __forceinline__ bool vote_fixed(const BinParams &bp, uint32_t acc_addr, uint32_t unit, uint32_t scratch_addr,
                                           uint2 en, uint32_t c_s, bool valid) {
    const uint32_t x = en.y - c_s;
    const uint32_t hi = __umulhi(x, bp.fix_mul);
    const unsigned long long p2 = (unsigned long long)hi * bp.frac_mul;  // runtime multiplier: stays an IMAD (FMA pipe)
    const uint32_t bin = (uint32_t)(p2 >> 32), frac = (uint32_t)p2;
    bool sure = (frac - bp.fix_guard) < (0u - 2u * bp.fix_guard);
    if (SEAM) sure = sure && ((x + bp.seam_guard) >= 2u * bp.seam_guard);
    red_shared_inc((sure && valid) ? acc_addr + en.x + unit * bin : scratch_addr);
    return valid && !sure;
}

// the rare path, and every vote of alpha mode B: literal form on PCL's floats.  row_bytes = 4 * row.
template <int MODE>
__device__ __forceinline__ void vote_exact(const BinParams &bp, uint32_t acc_addr, uint32_t unit, uint32_t row_bytes,
                                           float alpha_m, float alpha_s, uint32_t &skipped) {
    const uint32_t bin = MODE == ALPHA_MODE_B
                             ? alpha_bin_fast(bp, alpha_m, alpha_s)
                             : alpha_bin_exact(ALPHA_MODE_A, bp.angle_step, bp.n_alpha, bp.overflow_bin, alpha_m, alpha_s);
    if (bin == 0xFFFFFFFFu) ++skipped;  // NaN alpha: no vote (SURVEY.md A.8)
    else red_shared_inc(acc_addr + row_bytes + unit * bin);
}

// one (reference point, accumulator slice) task; ref_i = reference slot of this launch
// FOLD: the table folds (phase D); the other tables run a kernel without it
template <int MODE, bool SEAM, bool BULK, int THREADS, bool FOLD>
__device__ __forceinline__ void vote_task(const VoteArgs &a, const uint32_t ref_i, const uint32_t slice,
                                          uint32_t *next_task) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ Frame s_sg;
    __shared__ uint32_t s_ncand, s_nitems, s_next, s_scratch, s_nfold, s_ngroups;
    __shared__ uint32_t s_cls[8];  // work items per length class of the current round
    __shared__ uint32_t s_run_start[9], s_run_end[9];
    __shared__ unsigned long long s_best[(THREADS / 32)];
    __shared__ unsigned long long s_stat[4];

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef B200PPF_PHASE_TIMING
    __shared__ unsigned long long s_warp_ns[2];
    unsigned long long pt[PT_N] = {}, pt_t = global_ns(), wt_shift = 0, wt_own = 0;
    if (tid == 0) s_warp_ns[0] = s_warp_ns[1] = 0;
#endif
    const uint32_t slice_base = slice * a.kp.slice_rows;
    const uint32_t rows = min(a.kp.slice_rows, a.n_model - slice_base);
    const uint32_t pitch = a.kp.row_pitch;               // words between two alpha columns (multiple of 32)
    const uint32_t unit = 4u * pitch;                    // bytes per alpha position
    const uint32_t wrap_bytes = unit * a.bp.n_turn;      // one turn
    const uint32_t acc_len = a.bp.acc_cols * pitch;
    // queues first; the accumulator starts on a 128-byte boundary, so a vote's bank is its row mod 32
    uint32_t *cand = reinterpret_cast<uint32_t *>(smem_raw);
    WorkItem *items = reinterpret_cast<WorkItem *>(cand + CAND_CAP);
    uint32_t *acc = reinterpret_cast<uint32_t *>(items + THREADS);
    const uint32_t acc_addr = (uint32_t)__cvta_generic_to_shared(acc);
    const uint32_t scratch_addr = (uint32_t)__cvta_generic_to_shared(&s_scratch);

    // shared queue: one thread draws the NEXT task now and parks it in shared memory once the accumulator is clear —
    // the round trip (over NVLink on the other ranks) overlaps the prologue and costs no register in the vote loops
    const bool draws = next_task != nullptr && tid == THREADS - 1;
    uint32_t drawn = 0;
    if (draws) drawn = atomicAdd_system(a.queue, 1u);
    const uint32_t s_r = a.ref_first + ref_i * a.ref_step;
    const float4 pr4 = a.pos[s_r], nr4 = a.nrm[s_r];
    const V3 p_r = v3_of(pr4), n_r = v3_of(nr4);
    if (tid == 0) {
        ref_frame(p_r, n_r, s_sg);
        s_ncand = 0;
        s_nitems = 0;
        s_next = 0;
        s_nfold = 0;
        s_ngroups = 0;
    }
    if (tid < 4) s_stat[tid] = 0;
    if (tid >= 64 && tid < 72) s_cls[tid - 64] = 0;
    if (tid >= 32 && tid < 41) {
        // the 3 x-adjacent cells of row (cy+dy, cz+dz) are one contiguous run of the sorted scene
        const int r = (int)tid - 32;
        const int cx = grid_cell_coord(a.gp, p_r.x, 0), cy = grid_cell_coord(a.gp, p_r.y, 1),
                  cz = grid_cell_coord(a.gp, p_r.z, 2);
        const int y = cy + (r % 3) - 1, z = cz + (r / 3) - 1;
        uint32_t b = 0, e = 0;
        if (y >= 0 && y < a.gp.dims[1] && z >= 0 && z < a.gp.dims[2]) {
            const int x0 = max(cx - 1, 0), x1 = min(cx + 1, a.gp.dims[0] - 1);
            b = a.cell_start[grid_cell_linear(a.gp, x0, y, z)];
            e = a.cell_start[grid_cell_linear(a.gp, x1, y, z) + 1];
        }
        s_run_start[r] = b;
        s_run_end[r] = e;
    }
    for (uint32_t k = tid; k < acc_len; k += THREADS) acc[k] = 0;
    __syncthreads();
    if (draws) *next_task = drawn;  // everyone has read the current task before the barrier above
    PT_MARK(PT_PROLOGUE);

    const uint32_t lf = a.bp.cells_log2;
    const uint32_t *slice_offsets = a.sub_offsets + (((size_t)slice * a.kp.key_space) << lf);
    const uint32_t *slice_moffsets = BULK ? a.msub_offsets + (((size_t)slice * a.kp.key_space) << lf) : nullptr;
    const uint32_t fmask = (1u << a.bp.fix_shift) - 1u;
    uint32_t st_examined = 0, st_in_radius = 0, st_nonempty = 0, st_votes = 0, st_skipped = 0;
    uint32_t neighbourhood = 0;
#pragma unroll
    for (int r = 0; r < 9; ++r) neighbourhood += s_run_end[r] - s_run_start[r];

    // shift range [kb, ke) of merged words mp[]: add count * mult at umin(hot word - c, hot word - c + one turn).  The
    // arrays carry ENTRY_PAD readable words past the end, so the partial batch loads unclamped.  mult is the constant 1
    // for one scene pair's item, the number of folded pairs for a folded group (D).
    auto shift_range = [&](const uint32_t *mp, uint32_t kb, uint32_t ke, uint32_t c0v, auto mult) {
        const uint32_t c1v = c0v - wrap_bytes;
        uint32_t k0 = kb + lane;
        auto vote = [&](uint32_t w) {
            const uint32_t off = w & 0xFFFFFFu;
            red_shared_add(acc_addr + min(off - c0v, off - c1v), times(w >> 24, mult));
        };
        // long ranges: 8 x 32 words in flight per lane (the gathers are latency-bound)
        for (; k0 - lane + 64 * VOTE_UNROLL <= ke; k0 += 64 * VOTE_UNROLL) {  // warp-uniform: a double batch
            uint32_t hw[2 * VOTE_UNROLL];
#pragma unroll
            for (int u = 0; u < 2 * VOTE_UNROLL; ++u) hw[u] = __ldg(mp + k0 + u * 32);
#pragma unroll
            for (int u = 0; u < 2 * VOTE_UNROLL; ++u) vote(hw[u]);
        }
        if (k0 - lane + 32 * VOTE_UNROLL <= ke) {  // warp-uniform: one more full batch
            uint32_t hw[VOTE_UNROLL];
#pragma unroll
            for (int u = 0; u < VOTE_UNROLL; ++u) hw[u] = __ldg(mp + k0 + u * 32);
#pragma unroll
            for (int u = 0; u < VOTE_UNROLL; ++u) vote(hw[u]);
            k0 += 32 * VOTE_UNROLL;
        }
        if (k0 - lane < ke) {  // warp-uniform: a partial batch remains; votes are predicated
            uint32_t hw[VOTE_UNROLL];
#pragma unroll
            for (int u = 0; u < VOTE_UNROLL; ++u) hw[u] = __ldg(mp + k0 + u * 32);
#pragma unroll
            for (int u = 0; u < VOTE_UNROLL; ++u) {
                const uint32_t off = hw[u] & 0xFFFFFFu;
                red_shared_add_if_lt(acc_addr + min(off - c0v, off - c1v), times(hw[u] >> 24, mult), k0 + u * 32, ke);
            }
        }
    };

    // this CTA's fold buffer: the codes of the current scope, then the groups of phase D
    uint32_t *const fold_slot = FOLD ? a.fold_buf + (size_t)blockIdx.x * FOLD_SLOT_WORDS : nullptr;

    // phases B + C (+ D) over the buffered candidates; `last`: the task's final flush (earlier ones are taken mid-sweep)
    bool flushed = false;  // an earlier flush was taken: the task flushes more than once
    auto flush = [&](const bool last) {
        PT_MARK(PT_SWEEP);
        const uint32_t ncand = s_ncand;
        // Fold the constant-shift walks of the task's pairs (D below) on tables of FOLD_MIN_ENTRIES+ entries, when the task
        // has enough pairs to share buckets: it flushes more than once (every flush folds, a short last one too) or its
        // one flush holds FOLD_MIN_PAIRS+ candidates.  Light reference points keep one walk per pair.
        const bool fold = FOLD && BULK && (!last || flushed || ncand >= FOLD_MIN_PAIRS);
        for (uint32_t c0 = 0; c0 < ncand; c0 += THREADS) {
            // ---- B: pair features -> work items -------------------------------------------------
            const uint32_t c = c0 + tid;
            // the bucket [o0, oF) of unmerged entries; phase-sorted tables: its merged words [m0, mF) split at the scene
            // phase's cell [ma, mb) into below / above, and the cell's own unmerged entries are [oa, ob)
            uint32_t o0 = 0, oa = 0, ob = 0, oF = 0, q = 0, c_s = 0, phi = 0, sub_range = 0;
            uint32_t m0 = 0, ma = 0, mb = 0, mF = 0;
            uint32_t code = 0;  // folding pair: (key, q, cell)
            bool folds = false;
            float alpha_s = 0.0f;
            if (tid < THREADS && c < ncand) {
                const uint32_t s = cand[c];
                const float4 p4 = __ldg(a.gpos + s), n4 = __ldg(a.gnrm + s);
                float f[4];
                if (pair_features(a.feature_mode, p_r, n_r, v3_of(p4), v3_of(n4), f)) {
                    ++st_in_radius;
                    int d[4];
                    quantise(a.kp, f, d);
                    uint32_t key;
                    if (pack_key(a.kp, d, key)) {
                        const uint32_t *so = slice_offsets + ((size_t)key << lf);
                        o0 = __ldg(so);
                        oF = __ldg(so + (1u << lf));
                        oa = o0;
                        ob = oF;  // the whole bucket takes the per-entry path unless it splits below
                        if (oF > o0) {
                            alpha_s = planar_alpha(s_sg, v3_of(p4));
                            c_s = alpha_to_fix(alpha_s) - 0x80000000u;
                            ++st_nonempty;
                            st_votes += oF - o0;
                            if (BULK) {
                                uint32_t cell;
                                const bool split = phase_split(a.bp, c_s, q, cell);
                                // per-entry phase comparison needs the scene pair's own position; in the sliver
                                // between N_T and T (q == N_T) every entry takes the literal form
                                phi = q < a.bp.n_turn ? (phase_of_fix(a.bp, c_s) & fmask) : 0xFFFFFFFFu;
                                if (split) {
                                    const uint32_t in = phi & ((1u << (a.bp.fix_shift - lf)) - 1u), sh = sub_phase_shift(a.bp);
                                    sub_range = ((in - a.bp.phase_guard) >> sh) | (((in + a.bp.phase_guard - 1u) >> sh) << 8) | 0x10000u;
                                    const uint32_t *mo = slice_moffsets + ((size_t)key << lf);
                                    m0 = __ldg(mo);
                                    mF = __ldg(mo + (1u << lf));
                                    ma = __ldg(mo + cell);
                                    mb = __ldg(mo + cell + 1);
                                    oa = __ldg(so + cell);
                                    ob = __ldg(so + cell + 1);
                                    if (fold) {  // the shift ranges go to a folded group; the item keeps the own cell
                                        folds = true;
                                        code = (((key << a.fold_qbits) | q) << lf) | cell;
                                        m0 = ma = mb = mF = 0;
                                    }
                                }
                            }
                        }
                    }
                }
            }
            // Items enter the queue longest class first (classes = powers of two of the bucket length): the
            // warps then finish on short items and the CTA's barrier is not held up by one long bucket.
            const bool push = oF > o0;
            const uint32_t work = (mF - m0) + (ob - oa);  // words this item walks
            const uint32_t cls = push ? (uint32_t)min(7, max(0, 23 - (int)__clz(work))) : 8u + (lane & 7u);
            uint32_t rank = 0;
            {
                const uint32_t same = __match_any_sync(0xFFFFFFFFu, cls);
                if (push) {
                    const int leader = __ffs(same) - 1;
                    if ((int)lane == leader) rank = atomicAdd(&s_cls[cls], __popc(same));
                    rank = __shfl_sync(same, rank, leader) + __popc(same & ((1u << lane) - 1u));
                }
            }
            if (fold) {  // the fold codes join the scope's codes in the CTA's fold buffer
                const uint32_t fm = __ballot_sync(0xFFFFFFFFu, folds);
                if (fm) {
                    uint32_t b = 0;
                    if (lane == (uint32_t)(__ffs(fm) - 1)) b = atomicAdd(&s_nfold, __popc(fm));
                    b = __shfl_sync(0xFFFFFFFFu, b, __ffs(fm) - 1);
                    if (folds) fold_slot[b + __popc(fm & ((1u << lane) - 1u))] = code;
                }
            }
            __syncthreads();
            if (push) {
                uint32_t slot = rank;
#pragma unroll
                for (uint32_t k = 7; k > 0; --k) slot += (k > cls) ? s_cls[k] : 0u;
                WorkItem it;
                it.off = m0;
                it.len = mF - m0;
                it.k_below = ma - m0;
                it.k_above = mb - m0;
                it.e_off = oa;
                it.e_len = ob - oa;
                it.sub_range = a.no_sub_phase ? 0u : sub_range;
                it.pad1 = 0;
                it.c_below = unit * (q + 1u);
                it.c_s = c_s;
                it.alpha_s = alpha_s;
                it.phi = phi;
                items[slot] = it;
            }
            if (tid == 0) {
                uint32_t total = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) total += s_cls[k];
                s_nitems = total;
            }
            __syncthreads();
            PT_MARK(PT_PAIRS);
            // ---- C: votes ---------------------------------------------------------------------
            const uint32_t nitems = s_nitems;
            for (;;) {
                uint32_t w = 0;
                if (lane == 0) w = atomicAdd(&s_next, 1u);
                w = __shfl_sync(0xFFFFFFFFu, w, 0);
                if (w >= nitems) break;
                const WorkItem wi = items[w];
                const uint32_t len = wi.len;
                const uint32_t *mp = a.merged_w + wi.off;
#ifdef B200PPF_PHASE_TIMING
                unsigned long long wt0 = global_ns();
#endif
                if (BULK) {
                    const std::integral_constant<uint32_t, 1> one;
                    if (wi.k_below) shift_range(mp, 0u, wi.k_below, wi.c_below, one);
                    if (wi.k_above < len) shift_range(mp, wi.k_above, len, wi.c_below - unit, one);
                }
#ifdef B200PPF_PHASE_TIMING
                {
                    const unsigned long long t = global_ns();
                    wt_shift += t - wt0;
                    wt0 = t;
                }
#endif
                if (wi.e_len) {
                    // per-entry range [0, e_end) of the unmerged entry arrays
                    const uint32_t *wp = a.entry_w + wi.e_off;
                    const uint32_t *ap = a.entry_am + wi.e_off;
                    const float *fp = a.entry_alpha + wi.e_off;
                    const uint32_t e_end = wi.e_len;
                    if (BULK && wi.phi != 0xFFFFFFFFu) {
                        // the scene phase's own cell (or the whole bucket when the phase sits on a cell edge): an entry
                        // whose phase is below the scene's shifts by q + 1, the others by q; within the guard band of
                        // the scene phase the literal form decides.  32 entries per step, two steps in flight.
                        const uint32_t guard2 = 2u * a.bp.phase_guard, phi_g = wi.phi - a.bp.phase_guard;
                        const uint32_t c_lo = wi.c_below, c_hi = wi.c_below - unit;
                        if (wi.sub_range && e_end >= OWN_SUB_MIN) {
                            // pinned in registers: left to itself the compiler re-derives the accumulator base (S2UR of
                            // the CTA id + three uniform ops) and c_hi inside every predicated increment
                            const uint32_t acc_own = pin_register(acc_addr), c_hi_own = pin_register(c_hi);
                            // the scene phase's own cell by sub-phase: rel = (entry's sub-phase) - sub_lo.  rel > span
                            // (unsigned) = outside the scene's own sub-phases, and then the sign of rel tells the side.
                            const uint32_t sub_lo = wi.sub_range & 0xFFu, sub_hi = (wi.sub_range >> 8) & 0xFFu, span = sub_hi - sub_lo;
                            // The sub-phase is the word's top byte: w < below_lim <=> below the scene's own sub-phases,
                            // w > above_lim <=> above them (never when sub_hi = 255).
                            const uint32_t below_lim = sub_lo << 24, above_lim = (sub_hi << 24) | HOT_MASK;
                            // The increment stays the +1 form (ATOMS.POPC.INC): the entries of one model row are adjacent
                            // in the cell, and lanes of one instruction that hit the same word are counted in one pass —
                            // adding the decision as a value (ATOMS.ADD) serialises them and measured 2 % slower.
                            auto own_step = [&](auto steps, const uint32_t k0, const bool tail) {
                                constexpr int U = decltype(steps)::value;
                                uint32_t w[U], v[U], settled = 0;
#pragma unroll
                                for (int u = 0; u < U; ++u) w[u] = __ldg(wp + k0 + u * 32);
                                // Every live entry of these steps below the scene's own sub-phases (or every one above
                                // them): all vote with one shift, like a shift range.  The table orders each cell by
                                // sub-phase block (k2_table.cu), so that this is the case for all steps but those that
                                // touch the scene's own block; the test reads each entry's own byte and holds in any order.
                                // Folding tables only (2 M+ entries, long own cells): on small tables the own cells that
                                // reach this loop are few and short, and the extra code measured 1 % slower on C2.
                                if constexpr (FOLD) {
                                    bool below = true, above = true;
#pragma unroll
                                    for (int u = 0; u < U; ++u) {
                                        const bool live = !tail || k0 + u * 32 < e_end;
                                        below = below && (!live || w[u] < below_lim);
                                        above = above && (!live || w[u] > above_lim);
                                    }
                                    const uint32_t side = __reduce_and_sync(0xFFFFFFFFu, (below ? 1u : 0u) | (above ? 2u : 0u));
                                    if (side) {  // warp-uniform: the vote of a shift range, with the +1 increment
                                        const uint32_t c0v = (side & 1u) ? c_lo : c_hi, c1v = c0v - wrap_bytes;
#pragma unroll
                                        for (int u = 0; u < U; ++u) {
                                            const uint32_t off = w[u] & HOT_MASK;
                                            if (!tail || k0 + u * 32 < e_end) red_shared_inc(acc_addr + min(off - c0v, off - c1v));
                                        }
                                        return;
                                    }
                                }
#pragma unroll
                                for (int u = 0; u < U; ++u) {
                                    const uint32_t rel = (w[u] >> 24) - sub_lo;
                                    const bool past = tail && k0 + u * 32 >= e_end;
                                    v[u] = (rel > span && !past) ? 1u : 0u;
                                    const uint32_t t = (w[u] & HOT_MASK) - ((int)rel > (int)span ? c_hi_own : c_lo);
                                    if (v[u]) red_shared_inc(acc_own + min(t, t + wrap_bytes));
                                    settled += past ? 1u : v[u];
                                }
                                if (__any_sync(0xFFFFFFFFu, settled != U)) {  // ~1 entry in 256: the full comparison
#pragma unroll
                                    for (int u = 0; u < U; ++u)
                                        if (!v[u] && !(tail && k0 + u * 32 >= e_end)) {
                                            const uint32_t pu = __umulhi(__ldg(ap + k0 + u * 32), a.bp.fix_mul);
                                            const uint32_t dg = (pu & fmask) - phi_g;
                                            if (dg >= guard2) {
                                                const uint32_t t = (w[u] & HOT_MASK) - ((int)dg >= 0 ? c_hi : c_lo);
                                                red_shared_inc(acc_addr + min(t, t + wrap_bytes));
                                            } else {
                                                vote_exact<MODE>(a.bp, acc_addr, unit, (w[u] & HOT_MASK) - unit * phase_bin(a.bp, pu),
                                                                 __ldg(fp + k0 + u * 32), wi.alpha_s, st_skipped);
                                            }
                                        }
                                }
                            };
                            uint32_t k0 = lane;
                            for (; k0 - lane + 32 * OWN_UNROLL <= e_end; k0 += 32 * OWN_UNROLL)  // warp-uniform
                                own_step(std::integral_constant<int, OWN_UNROLL>(), k0, false);
                            for (; k0 - lane < e_end; k0 += 32) own_step(std::integral_constant<int, 1>(), k0, true);
                        } else
                        // the scene phase sits on a cell edge and the whole bucket is compared in full:
                        // dg = (entry phase in its cell) - (scene phase) + guard.  Outside [0, 2 guard) the comparison is
                        // safe: dg negative as a signed number = the entry lies below the scene phase and shifts one more.
                        for (uint32_t k0 = lane; k0 - lane < e_end; k0 += 32 * FULL_UNROLL) {  // warp-uniform
                            uint32_t w[FULL_UNROLL], pu[FULL_UNROLL];
#pragma unroll
                            for (int u = 0; u < FULL_UNROLL; ++u) {
                                w[u] = __ldg(wp + k0 + u * 32) & HOT_MASK;
                                pu[u] = __ldg(ap + k0 + u * 32);
                            }
                            bool risky = false;
#pragma unroll
                            for (int u = 0; u < FULL_UNROLL; ++u) {
                                pu[u] = __umulhi(pu[u], a.bp.fix_mul);
                                const uint32_t dg = (pu[u] & fmask) - phi_g;
                                const uint32_t t = w[u] - ((int)dg >= 0 ? c_hi : c_lo);
                                // the guard band is circular: with the scene phase within the guard of a bin edge (the
                                // whole bucket is here then) an entry just across that edge is as close as one beside it
                                red_shared_inc_if_ge_lt(acc_addr + min(t, t + wrap_bytes), dg & fmask, guard2, k0 + u * 32, e_end);
                                risky |= (dg & fmask) < guard2 && k0 + u * 32 < e_end;
                            }
                            if (__any_sync(0xFFFFFFFFu, risky)) {  // one entry in ~10^3 sits within the guard band
#pragma unroll
                                for (int u = 0; u < FULL_UNROLL; ++u)
                                    if ((((pu[u] & fmask) - phi_g) & fmask) < guard2 && k0 + u * 32 < e_end)
                                        vote_exact<MODE>(a.bp, acc_addr, unit, w[u] - unit * phase_bin(a.bp, pu[u]),
                                                         __ldg(fp + k0 + u * 32), wi.alpha_s, st_skipped);
                            }
                        }
                    } else if (BULK) {
                        // the sliver between N_T and T: literal form for every entry (one scene pair in ~10^7)
                        for (uint32_t k = lane; k < e_end; k += 32) {
                            const uint32_t w = __ldg(wp + k) & HOT_MASK;
                            vote_exact<MODE>(a.bp, acc_addr, unit, w - unit * phase_bin(a.bp, __umulhi(__ldg(ap + k), a.bp.fix_mul)),
                                             __ldg(fp + k), wi.alpha_s, st_skipped);
                        }
                    } else if (MODE == ALPHA_MODE_A) {
                        // tables without phase cells: branch-free fixed-point votes, 32 entries per step (two steps in
                        // flight); lanes past the end read the padding and vote into the scratch word
                        for (uint32_t k0 = lane; k0 - lane < e_end; k0 += 64) {  // warp-uniform
                            uint2 en[2];
#pragma unroll
                            for (int u = 0; u < 2; ++u) en[u] = make_uint2(__ldg(wp + k0 + u * 32), __ldg(ap + k0 + u * 32));
                            bool risky[2];
#pragma unroll
                            for (int u = 0; u < 2; ++u) {
                                risky[u] = false;
                                if (k0 - lane + u * 32 < e_end)  // warp-uniform
                                    risky[u] = vote_fixed<SEAM>(a.bp, acc_addr, unit, scratch_addr, en[u], wi.c_s,
                                                                k0 + u * 32 < e_end);
                            }
#pragma unroll
                            for (int u = 0; u < 2; ++u)
                                if (risky[u])
                                    vote_exact<MODE>(a.bp, acc_addr, unit, en[u].x, __ldg(fp + k0 + u * 32),
                                                     wi.alpha_s, st_skipped);
                        }
                    } else {
                        for (uint32_t k = lane; k < e_end; k += 32)
                            vote_exact<MODE>(a.bp, acc_addr, unit, __ldg(wp + k), __ldg(fp + k), wi.alpha_s,
                                             st_skipped);
                    }
                }
#ifdef B200PPF_PHASE_TIMING
                wt_own += global_ns() - wt0;
#endif
            }
            __syncthreads();
            PT_MARK(PT_VOTES);
            if (tid == 0) {
                s_nitems = 0;
                s_next = 0;
            }
            if (tid >= 64 && tid < 72) s_cls[tid - 64] = 0;
            __syncthreads();
        }
        // the scope ends with the task, or when the next flush might not fit the fold buffer
        const uint32_t n = fold ? s_nfold : 0u;
        if (n && (last || n > FOLD_SCOPE - CAND_CAP)) {
            // ---- D: folded shift ranges ------------------------------------------------------------
            // A folding pair (q, c) votes on cell k of its bucket with shift q + 1 below c and q above it, so the pairs
            // of one bucket that vote on cell k with shift s number
            //     m_s(k) = #{q = s, c < k} + #{q = s - 1 (mod N_T), c > k},
            // and one walk of the cell adding count * m_s(k) casts all their votes.  The codes (key, q, c) are sorted
            // (bitonic, in the idle candidate and item queues), so both terms are differences of lower bounds.
            const uint32_t qb = a.fold_qbits, qmask = (1u << qb) - 1u, ncell = 1u << lf;
            uint32_t np = 32;
            while (np < n) np <<= 1;
            for (uint32_t i = tid; i < np; i += THREADS) cand[i] = i < n ? fold_slot[i] : 0xFFFFFFFFu;  // codes have at most 31 bits
            __syncthreads();
            for (uint32_t k = 2; k <= np; k <<= 1)
                for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                    for (uint32_t i = tid; i < np / 2; i += THREADS) {
                        const uint32_t lo = ((i & ~(j - 1u)) << 1) | (i & (j - 1u)), hi = lo + j;
                        const uint32_t x = cand[lo], y = cand[hi];
                        if ((x > y) == ((lo & k) == 0)) {
                            cand[lo] = y;
                            cand[hi] = x;
                        }
                    }
                    __syncthreads();
                }
            auto first_at_least = [&](uint32_t x) {
                uint32_t lo = 0, len = n;
                while (len) {
                    const uint32_t half = len >> 1;
                    if (cand[lo + half] < x) {
                        lo += half + 1;
                        len -= half + 1;
                    } else {
                        len = half;
                    }
                }
                return lo;
            };
            // one group (key, s) per s that some run (key, q) touches: s = q, and s = q + 1 when no run (key, q + 1) exists
            uint32_t *const groups = fold_slot;  // the codes are in shared memory now
            for (uint32_t i = tid; i < n; i += THREADS) {
                const uint32_t run = cand[i] >> lf;
                if (i == 0 || (cand[i - 1] >> lf) != run) {
                    const uint32_t q = run & qmask;
                    const uint32_t next = ((run - q) | (q + 1u == a.bp.n_turn ? 0u : q + 1u)) << lf;
                    const uint32_t p = first_at_least(next);
                    const bool alone = p == n || (cand[p] >> lf) != (next >> lf);
                    const uint32_t slot = atomicAdd(&s_ngroups, alone ? 2u : 1u);
                    groups[slot] = run << lf;
                    if (alone) groups[slot + 1] = next;
                }
            }
            __syncthreads();
            const uint32_t ngroups = s_ngroups;
            for (;;) {
                uint32_t w = 0;
                if (lane == 0) w = atomicAdd(&s_next, 1u);
                w = __shfl_sync(0xFFFFFFFFu, w, 0);
                if (w >= ngroups) break;
                const uint32_t g = groups[w], run = g >> lf, s = run & qmask;
                const uint32_t gp = ((run - s) | (s == 0 ? a.bp.n_turn - 1u : s - 1u)) << lf;
                // lane k < 16: first code >= (key, s, k); lane 16 + k: first code >= (key, s - 1, k + 1)
                const uint32_t kk = lane & 15u;
                const uint32_t pos = first_at_least(lane < 16 ? g + kk : gp + kk + 1u);
                const uint32_t m = (pos - __shfl_sync(0xFFFFFFFFu, pos, 0)) +
                                   (__shfl_sync(0xFFFFFFFFu, pos, 15 + ncell) - __shfl_sync(0xFFFFFFFFu, pos, 16 + kk));
                // lane k <= ncell: start of cell k of the bucket in the merged words
                const uint32_t mo = __ldg(slice_moffsets + ((size_t)(run >> qb) << lf) + min(lane, ncell));
                const uint32_t m_prev = __shfl_up_sync(0xFFFFFFFFu, m, 1), m_next = __shfl_down_sync(0xFFFFFFFFu, m, 1);
                // consecutive cells with the same multiplier are one range
                const bool live = lane < ncell && m != 0;
                uint32_t starts = __ballot_sync(0xFFFFFFFFu, live && (lane == 0 || m_prev != m));
                const uint32_t ends = __ballot_sync(0xFFFFFFFFu, live && (lane + 1 == ncell || m_next != m));
                while (starts) {
                    const uint32_t b = __ffs(starts) - 1, e = __ffs(ends & (0xFFFFFFFFu << b)) - 1;
                    shift_range(a.merged_w, __shfl_sync(0xFFFFFFFFu, mo, b), __shfl_sync(0xFFFFFFFFu, mo, e + 1), unit * s,
                                __shfl_sync(0xFFFFFFFFu, m, b));
                    starts &= starts - 1;
                }
            }
            __syncthreads();
            PT_MARK(PT_FOLD);
            if (tid == 0) {
                s_next = 0;
                s_nfold = 0;
                s_ngroups = 0;
            }
        }
        if (tid == 0) s_ncand = 0;
        if (!last) flushed = true;
        __syncthreads();
    };

    // ---- A: sweep the 27-cell neighbourhood ---------------------------------------------------------
    auto test_and_queue = [&](uint32_t s, uint32_t re) {
        bool in = false;
        if (s < re) {
            const float4 p4 = __ldg(a.gpos + s);
            const float dx = p4.x - p_r.x, dy = p4.y - p_r.y, dz = p4.z - p_r.z;
            const float d2 = (dx * dx + dy * dy) + dz * dz;
            // radius predicate on f4 itself (SURVEY.md A.8 rule 7): sqrtf(d2) < radius, evaluated
            // through the equivalent threshold on d2 (sqrtf is monotone and correctly rounded); the point's index (w) is
            // read after the test, as holding p4.w across it costs some instantiations a register
            in = d2 < a.radius_sq_bound && __float_as_uint(__ldg(&a.gpos[s].w)) != s_r;
            ++st_examined;
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, in);
        if (m) {
            uint32_t b = 0;
            if (lane == (uint32_t)(__ffs(m) - 1)) b = atomicAdd(&s_ncand, __popc(m));
            b = __shfl_sync(0xFFFFFFFFu, b, __ffs(m) - 1);
            if (in) cand[b + __popc(m & ((1u << lane) - 1u))] = s;
        }
    };
    if (neighbourhood <= CAND_CAP) {
        // the common case: every point of the 27 cells fits the queue — no barriers inside the sweep
        for (int r = 0; r < 9; ++r) {
            const uint32_t rb = s_run_start[r], re = s_run_end[r];
            for (uint32_t base = rb; base < re; base += THREADS) test_and_queue(base + tid, re);
        }
        __syncthreads();
    } else {
        for (int r = 0; r < 9; ++r) {
            const uint32_t rb = s_run_start[r], re = s_run_end[r];
            for (uint32_t base = rb; base < re; base += THREADS) {
                test_and_queue(base + tid, re);
                __syncthreads();
                const uint32_t buffered = s_ncand;
                __syncthreads();  // nobody may start the next sweep's atomics before everyone has read
                if (buffered > CAND_CAP - THREADS) flush(false);
            }
        }
    }
    flush(true);

    // ---- peak: first maximum in (i, bin) order == max of (votes, ~flat) ---------------------------
    // one thread per model row (consecutive threads read consecutive words of a column): the spare column n_alpha
    // (bins past the last column) joins column n_alpha - 1 under the FLOOR_CLAMP rule and is ignored otherwise
    // (FLOOR_DROP: the vote is lost; CEIL: there is no such column)
    const uint32_t n_alpha = a.bp.n_alpha;
    unsigned long long best = 0;
    for (uint32_t r = tid; r < rows; r += THREADS) {
        uint32_t bv = 0, bc = 0;
        for (uint32_t c = 0; c < n_alpha; ++c) {
            uint32_t v = acc[c * pitch + r];
            if (a.bp.fold && c == n_alpha - 1) v += acc[n_alpha * pitch + r];
            if (v > bv) {  // strict: the first maximum of the row
                bv = v;
                bc = c;
            }
            if (a.acc_dump) a.acc_dump[(size_t)(slice_base + r) * n_alpha + c] = v;
        }
        if (bv) {
            const unsigned long long cnd =
                ((unsigned long long)bv << 32) | (unsigned long long)(0xFFFFFFFFu - ((slice_base + r) * n_alpha + bc));
            best = max(best, cnd);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = max(best, shfl_xor_u64(best, o));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        st_examined += __shfl_xor_sync(0xFFFFFFFFu, st_examined, o);
        st_in_radius += __shfl_xor_sync(0xFFFFFFFFu, st_in_radius, o);
        st_nonempty += __shfl_xor_sync(0xFFFFFFFFu, st_nonempty, o);
        st_votes += __shfl_xor_sync(0xFFFFFFFFu, st_votes, o);
        st_skipped += __shfl_xor_sync(0xFFFFFFFFu, st_skipped, o);
    }
    if (lane == 0) {
        s_best[warp] = best;
        atomicAdd(&s_stat[0], (unsigned long long)st_examined);
        atomicAdd(&s_stat[1], (unsigned long long)st_in_radius);
        atomicAdd(&s_stat[2], (unsigned long long)st_nonempty);
        atomicAdd(&s_stat[3], (unsigned long long)st_votes);
        atomicAdd(&s_stat[3], 0ull - (unsigned long long)st_skipped);  // NaN alphas cast no vote
#ifdef B200PPF_PHASE_TIMING
        atomicAdd(&s_warp_ns[0], wt_shift);
        atomicAdd(&s_warp_ns[1], wt_own);
#endif
    }
    __syncthreads();
    PT_MARK(PT_PEAK);
#ifdef B200PPF_PHASE_TIMING
    if (tid == 0) {
        unsigned long long *g = g_phase_ns[flushed ? 1 : 0];
        for (int k = 0; k < PT_C_SHIFT; ++k) atomicAdd(g + k, pt[k]);
        atomicAdd(g + PT_C_SHIFT, s_warp_ns[0]);
        atomicAdd(g + PT_C_OWN, s_warp_ns[1]);
        atomicAdd(g + PT_TASKS, 1ull);
    }
#endif
    if (tid == 0) {
#pragma unroll
        for (int w = 1; w < (THREADS / 32); ++w) best = max(best, s_best[w]);
        if (best) {
            if (a.n_peers) {
                for (int g = 0; g < a.n_peers; ++g) atomicMax_system(a.peer_peaks[g] + ref_i, best);
            } else {
                atomicMax(a.peaks + ref_i, best);
            }
        }
        if (slice == 0) {
            atomicAdd(a.stats + 0, s_stat[0]);
            atomicAdd(a.stats + 1, s_stat[1]);
        }
        atomicAdd(a.stats + 2, s_stat[2]);
        atomicAdd(a.stats + 3, s_stat[3]);
    }
}

// Task order.  A task's cost follows the number of scene points around its reference point (C3: 81 % of the tasks take
// ~0.1 ms, 9 % take 4-9 ms, profiles/r2_queue_task_histogram.txt), and a heavy task drawn last leaves every other CTA
// idle while it runs — 13 ms per launch on C3, the same on one GPU or eight.  So each slice hands out its reference
// points heaviest neighbourhood first (the 27 grid cells the task will sweep), and the launch ends on the 0.1 ms tasks.
__global__ void ref_cost_kernel(const float4 *__restrict__ pos, const uint32_t *__restrict__ cell_start, GridParams gp,
                                uint32_t ref_first, uint32_t ref_step, uint32_t ref_count, uint32_t n_s,
                                uint32_t *__restrict__ inv_cost) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= ref_count) return;
    const float4 p = pos[ref_first + r * ref_step];
    const int cx = grid_cell_coord(gp, p.x, 0), cy = grid_cell_coord(gp, p.y, 1), cz = grid_cell_coord(gp, p.z, 2);
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, gp.dims[0] - 1);
    uint32_t n = 0;
    for (int z = max(cz - 1, 0); z <= min(cz + 1, gp.dims[2] - 1); ++z)
        for (int y = max(cy - 1, 0); y <= min(cy + 1, gp.dims[1] - 1); ++y)
            n += cell_start[grid_cell_linear(gp, x1, y, z) + 1] - cell_start[grid_cell_linear(gp, x0, y, z)];
    inv_cost[r] = n_s - n;  // ascending sort = heaviest first; equal costs keep reference order (stable sort)
}

template <int MODE, bool SEAM, bool BULK, int THREADS, bool FOLD>
__global__ void __launch_bounds__(THREADS, THREADS == 1024 ? 1 : B200PPF_VOTE_MINBLOCKS)
ppf_vote_kernel(const VoteArgs a) {
    // Either one CTA per (reference point, slice) — the grid is (positions, slices) — or persistent CTAs drawing those
    // tasks from a queue counter (folding tables: a CTA owns one slot of the fold buffer for all its tasks; several GPUs:
    // the queue shared by all ranks).  One call site serves both, so the two modes run the same machine code.  Slice-major
    // order either way: the CTAs in flight share one slice of the table in L2.
    __shared__ uint32_t s_task;
    const bool persistent = a.queue != nullptr;
    const uint32_t total = a.ref_count * a.kp.n_slices;
    if (threadIdx.x == 0) s_task = persistent ? atomicAdd_system(a.queue, 1u) : blockIdx.y * a.ref_count + blockIdx.x;
    for (;;) {
        __syncthreads();
        const uint32_t task = s_task;
        if (task >= total) break;
        const uint32_t pos = task % a.ref_count;
        vote_task<MODE, SEAM, BULK, THREADS, FOLD>(a, a.ref_order ? a.ref_order[pos] : pos, task / a.ref_count,
                                                   persistent ? &s_task : nullptr);
        if (!persistent) break;
    }
#ifdef B200PPF_PHASE_TIMING
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&g_phase_done, 1u) == gridDim.x * gridDim.y - 1) {
            __threadfence();
            for (int c = 0; c < 2; ++c) {
                unsigned long long *g = g_phase_ns[c];
                printf("k3_phase_ns flushes=%s tasks=%llu prologue=%llu sweep=%llu pairs=%llu votes=%llu fold=%llu peak=%llu "
                       "votes_shift_warp=%llu votes_own_warp=%llu\n",
                       c ? "many" : "one", g[PT_TASKS], g[PT_PROLOGUE], g[PT_SWEEP], g[PT_PAIRS], g[PT_VOTES], g[PT_FOLD],
                       g[PT_PEAK], g[PT_C_SHIFT], g[PT_C_OWN]);
                for (int k = 0; k < PT_N; ++k) g[k] = 0;
            }
            g_phase_done = 0;
        }
    }
#endif
    if (threadIdx.x == 0 && a.done_counter) {
        __threadfence_system();  // this CTA's peaks are visible everywhere before it counts as done
        if (atomicAdd(a.done_counter, 1u) == gridDim.x - 1) {
            *a.done_counter = 0;
            __threadfence_system();
            for (int g = 0; g < a.n_peers; ++g)
                *reinterpret_cast<volatile uint32_t *>(a.peer_flags[g] + a.signal_slot) = a.signal_value;
            __threadfence_system();
        }
    }
}

// Where the 64-byte records go.  Single GPU: one buffer, record r in slot r.  Several GPUs: the epilogue IS the
// all-gather — every rank writes its record r straight into slot (slot_first + r * slot_step) of every peer's
// buffer over NVLink (peer pointers from cudaIpcOpenMemHandle), so the gathered array is complete and already in
// reference order on every GPU when the kernels have finished; no staging copy, no NCCL all-gather, no reorder.
struct PeerTargets {
    b200ppf_hypothesis *base[MAX_PEERS];
    int n;
    uint32_t slot_first, slot_step;
    // optional completion signal (b200ppf_group): when the last block of the pose kernel has written its records,
    // flag word `signal_slot` of every peer's flag array is set to signal_value (system-scope, after a fence)
    uint32_t *flags[MAX_PEERS];
    uint32_t signal_slot, signal_value;
    uint32_t *done_counter;  // blocks finished so far (this device)
};

// pose of every peak: one thread per reference point
__global__ void ppf_peak_pose_kernel(const float4 *__restrict__ spos, const float4 *__restrict__ snrm,
                                     const float4 *__restrict__ mpos, const float4 *__restrict__ mnrm,
                                     uint32_t ref_first, uint32_t ref_step, uint32_t ref_count,
                                     const unsigned long long *__restrict__ peaks, BinParams bp,
                                     const PeerTargets out) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < ref_count) {
    const uint32_t s_r = ref_first + r * ref_step;
    const unsigned long long pk = peaks[r];
    const uint32_t votes = (uint32_t)(pk >> 32);
    const uint32_t flat = votes ? 0xFFFFFFFFu - (uint32_t)(pk & 0xFFFFFFFFu) : 0u;
    const uint32_t i = flat / bp.n_alpha, bin = flat - i * bp.n_alpha;
    Frame sg, mg;
    ref_frame(v3_of(spos[s_r]), v3_of(snrm[s_r]), sg);
    ref_frame(v3_of(mpos[i]), v3_of(mnrm[i]), mg);
    b200ppf_hypothesis h;
    compose_pose(sg, peak_theta(bp.mode, bp.angle_step, bin), mg, h.pose);
    h.votes = votes;
    h.model_index = i;
    h.alpha_bin = bin;
    h.scene_index = s_r;
    const size_t slot = (size_t)out.slot_first + (size_t)r * out.slot_step;
    const uint4 *src = reinterpret_cast<const uint4 *>(&h);
    for (int g = 0; g < out.n; ++g) {
        uint4 *dst = reinterpret_cast<uint4 *>(out.base[g] + slot);
#pragma unroll
        for (int q = 0; q < 4; ++q) dst[q] = src[q];  // 4 x 16 bytes: one full 64-byte record per peer
    }
    if (out.n > 1) __threadfence_system();
    }
    if (out.done_counter) {
        // the last block to finish tells every peer that this rank's records have landed
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();
            if (atomicAdd(out.done_counter, 1u) == gridDim.x - 1) {
                *out.done_counter = 0;
                __threadfence_system();
                for (int g = 0; g < out.n; ++g)
                    *reinterpret_cast<volatile uint32_t *>(out.flags[g] + out.signal_slot) = out.signal_value;
                __threadfence_system();
            }
        }
    }
}

// spin until every rank's flag has reached `value` (one thread; the flags are written by the peers' pose kernels)
__global__ void group_wait_kernel(const uint32_t *flags, int world, uint32_t value) {
    for (int g = 0; g < world; ++g) {
        const volatile uint32_t *f = flags + g;
        while ((int32_t)(*f - value) < 0) __nanosleep(200);
    }
    __threadfence_system();
}

// parity hook: per-scene-point quantities of one reference point, exactly as phases A/B see them
__global__ void ppf_debug_pairs_kernel(const float4 *__restrict__ pos, const float4 *__restrict__ nrm, uint32_t n_s,
                                       uint32_t s_r, KeyParams kp, int feature_mode, float radius,
                                       uint8_t *__restrict__ in_radius, int *__restrict__ d4,
                                       float *__restrict__ alpha_s) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_s) return;
    in_radius[s] = 0;
    d4[4 * s] = d4[4 * s + 1] = d4[4 * s + 2] = d4[4 * s + 3] = 0;
    alpha_s[s] = 0.0f;
    if (s == s_r) return;
    const V3 p_r = v3_of(pos[s_r]), n_r = v3_of(nrm[s_r]);
    const V3 p = v3_of(pos[s]), n = v3_of(nrm[s]);
    const V3 d = make_v3(p.x - p_r.x, p.y - p_r.y, p.z - p_r.z);
    if (!(norm3(d) < radius)) return;
    float f[4];
    if (!pair_features(feature_mode, p_r, n_r, p, n, f)) return;
    int q[4];
    quantise(kp, f, q);
    Frame sg;
    ref_frame(p_r, n_r, sg);
    in_radius[s] = 1;
    d4[4 * s] = q[0];
    d4[4 * s + 1] = q[1];
    d4[4 * s + 2] = q[2];
    d4[4 * s + 3] = q[3];
    alpha_s[s] = planar_alpha(sg, p);
}

__global__ void debug_alpha_bins_kernel(BinParams bp, const float *__restrict__ am, const float *__restrict__ as,
                                        uint32_t n, uint32_t *__restrict__ fast, uint32_t *__restrict__ exact) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    fast[p] = alpha_bin_phase(bp, am[p], as[p]);
    exact[p] = alpha_bin_exact(bp.mode, bp.angle_step, bp.n_alpha, bp.overflow_bin, am[p], as[p]);
}

size_t accumulator_bytes(const b200ppf_table *t) {
    return (size_t)t->kp.row_pitch * t->bp.acc_cols * sizeof(uint32_t);
}
// launch shape of a table: 512 x 2 CTAs/SM when the slice is small enough, else 1024 x 1
int vote_threads(const b200ppf_table *t) {
    return accumulator_bytes(t) + queue_bytes(VOTE_THREADS_SMALL) <= SMALL_SHAPE_SMEM_MAX ? VOTE_THREADS_SMALL
                                                                                        : VOTE_THREADS_LARGE;
}
size_t vote_smem_bytes(const b200ppf_table *t) { return accumulator_bytes(t) + queue_bytes(vote_threads(t)); }

// smallest float x with sqrtf(x) >= r (host sqrtf and device sqrtf are both correctly rounded)
float radius_sq_bound(float r) {
    if (!(r > 0.0f)) return 0.0f;
    float x = r * r;
    while (std::sqrt(x) >= r) x = std::nextafter(x, 0.0f);
    while (std::sqrt(x) < r) x = std::nextafter(x, INFINITY);
    return x;
}

int launch_vote(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t ref_first,
                size_t ref_step, size_t ref_count, uint32_t *acc_dump, const VoteQueue *queue = nullptr) {
    const float radius = t->info.max_dist * 0.5f;
    SceneGrids grid(ctx);
    if (int rc = scene_grid_build_one(ctx, scene, radius, &grid)) return rc;
    VoteArgs a;
    a.pos = scene->pos;
    a.nrm = scene->nrm;
    a.gpos = grid.pos;
    a.gnrm = grid.nrm;
    a.cell_start = grid.cell_start;
    a.gp = grid.scenes[0].gp;
    a.n_s = (uint32_t)scene->n;
    a.ref_first = (uint32_t)ref_first;
    a.ref_step = (uint32_t)ref_step;
    a.ref_count = (uint32_t)ref_count;
    a.sub_offsets = t->sub_offsets ? t->sub_offsets : t->offsets;
    a.msub_offsets = t->msub_offsets;
    a.merged_w = t->merged_w;
    a.entry_w = t->entry_w;
    a.entry_am = t->entry_am;
    a.entry_alpha = t->entry_alpha;
    a.kp = t->kp;
    a.bp = t->bp;
    a.bp.mode = ctx->alpha_mode;
    a.feature_mode = t->feature_mode;
    a.radius = radius;
    a.radius_sq_bound = radius_sq_bound(radius);
    a.n_model = (uint32_t)t->info.n_model;
    a.peaks = ctx->d_peaks;
    a.stats = ctx->d_stats;
    a.acc_dump = acc_dump;
    a.queue = nullptr;
    a.n_peers = 0;
    a.signal_slot = a.signal_value = 0;
    a.done_counter = nullptr;
    a.no_sub_phase = getenv("B200PPF_NO_SUB_PHASE") ? 1 : 0;
    a.fold_qbits = a.bp.mode == ALPHA_MODE_A ? k3_fold_qbits(t) : 0u;
    for (int g = 0; g < MAX_PEERS; ++g) {
        a.peer_peaks[g] = nullptr;
        a.peer_flags[g] = nullptr;
    }
    const size_t smem = vote_smem_bytes(t);
    const int threads = vote_threads(t);
    // persistent: as many CTAs as the device holds at once (one GPU: no more than there are tasks)
    unsigned ctas = (unsigned)(ctx->sm_count * (threads == VOTE_THREADS_SMALL ? B200PPF_VOTE_MINBLOCKS : 1));
    dim3 grid_dim(ctas);
    if (queue) {
        a.queue = queue->counter;
        a.n_peers = queue->n_peers;
        a.signal_slot = queue->slot;
        a.signal_value = queue->value;
        a.done_counter = queue->done_counter;
        for (int g = 0; g < queue->n_peers; ++g) {
            a.peer_peaks[g] = queue->peer_peaks[g];
            a.peer_flags[g] = queue->flags[g];
        }
    } else if (a.fold_qbits) {
        // a folding table on one GPU: persistent CTAs on the context's counter, so that each owns a fold-buffer slot
        ctas = (unsigned)std::min<size_t>(ctas, ref_count * t->info.n_slices);
        grid_dim = dim3(ctas);
        if (!ctx->d_vote_queue) PPF_CUDA(ctx, cudaMalloc(&ctx->d_vote_queue, sizeof(uint32_t)));
        PPF_CUDA(ctx, cudaMemsetAsync(ctx->d_vote_queue, 0, sizeof(uint32_t), ctx->stream));
        a.queue = ctx->d_vote_queue;
    } else {
        // the other tables on one GPU: one CTA per task (C1's 54 µs vote kernel measured 60-61 µs persistent, DESIGN §3)
        grid_dim = dim3((unsigned)ref_count, t->info.n_slices);
    }
    a.fold_buf = nullptr;
    if (a.fold_qbits) {
        PPF_CUDA(ctx, grow_buffer(&ctx->d_fold, &ctx->fold_cap, ctas * FOLD_SLOT_WORDS));
        a.fold_buf = ctx->d_fold;
    }
    cudaEventRecord(ctx->ev_vote[1], ctx->stream);  // grid build ends, voting starts
    // heaviest neighbourhood first once the launch is several waves deep and the buckets long enough for a task to take
    // longer than the ordering does (see ref_cost_kernel; config 2's 295 k-entry table gains nothing from it)
    StreamBuf<uint32_t> cost(ctx), cost_alt(ctx), order(ctx), order_alt(ctx);
    a.ref_order = nullptr;
    if (ref_count * t->info.n_slices >= 8 * (size_t)ctx->sm_count && t->info.n_entries >= (1u << 21) && !getenv("B200PPF_NO_TASK_ORDER")) {
        PPF_CUDA(ctx, cost.alloc(ref_count));
        PPF_CUDA(ctx, cost_alt.alloc(ref_count));
        PPF_CUDA(ctx, order.alloc(ref_count));
        PPF_CUDA(ctx, order_alt.alloc(ref_count));
        PPF_LAUNCH(ctx, ref_cost_kernel, (unsigned)((ref_count + 255) / 256), 256, 0, scene->pos, grid.cell_start.p, a.gp,
                   (uint32_t)ref_first, (uint32_t)ref_step, (uint32_t)ref_count, (uint32_t)scene->n, cost.p);
        bool in_alt = false;  // costs are counts of scene points
        if (int rc = radix_sort_u32(ctx, cost.p, cost_alt.p, order.p, order_alt.p, nullptr, nullptr, ref_count, scene->n,
                                    /*v0_iota=*/true, &in_alt))
            return rc;
        a.ref_order = in_alt ? order_alt.p : order.p;
    }
#define LAUNCH_VOTE_T(M, S, B, T, F)                                                                                  \
    do {                                                                                                            \
        PPF_CUDA(ctx, cudaFuncSetAttribute(ppf_vote_kernel<M, S, B, T, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           (int)smem));                                                             \
        PPF_LAUNCH(ctx, (ppf_vote_kernel<M, S, B, T, F>), grid_dim, T, smem, a);                                       \
    } while (0)
#define LAUNCH_VOTE(M, S, B, F)                                                          \
    do {                                                                                 \
        if (threads == VOTE_THREADS_SMALL) LAUNCH_VOTE_T(M, S, B, VOTE_THREADS_SMALL, F);  \
        else LAUNCH_VOTE_T(M, S, B, VOTE_THREADS_LARGE, F);                            \
    } while (0)
    if (ctx->alpha_mode == ALPHA_MODE_B) LAUNCH_VOTE(ALPHA_MODE_B, false, false, false);
    else if (a.bp.bulk && a.fold_qbits) LAUNCH_VOTE(ALPHA_MODE_A, false, true, true);
    else if (a.bp.bulk) LAUNCH_VOTE(ALPHA_MODE_A, false, true, false);  // an integer T has no separate seam band
    else if (a.bp.seam_guard) LAUNCH_VOTE(ALPHA_MODE_A, true, false, false);
    else LAUNCH_VOTE(ALPHA_MODE_A, false, false, false);
#undef LAUNCH_VOTE_T
#undef LAUNCH_VOTE
    cudaEventRecord(ctx->ev_vote[2], ctx->stream);
    return B200PPF_OK;
}

int ensure_vote_scratch(b200ppf_ctx *ctx, size_t ref_count) {
    if (!ctx->d_stats) PPF_CUDA(ctx, cudaMalloc(&ctx->d_stats, 4 * sizeof(unsigned long long)));
    PPF_CUDA(ctx, grow_buffer(&ctx->d_peaks, &ctx->peaks_cap, ref_count));
    PPF_CUDA(ctx, cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    PPF_CUDA(ctx, cudaMemsetAsync(ctx->d_peaks, 0, ref_count * sizeof(unsigned long long), ctx->stream));
    return B200PPF_OK;
}

int check_vote_inputs(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t ref_first,
                      size_t ref_step, size_t ref_count) {
    if (!t || !scene) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote: null table or scene");
    if (ref_step == 0) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote: reference step must be >= 1");
    if (ref_count && ref_first + (ref_count - 1) * ref_step >= scene->n)
        return fail_msg(ctx, B200PPF_ERR_INVALID, "vote: reference index range exceeds the scene");
    if (scene->n >= 0xFFFFFFFFull) return fail_msg(ctx, B200PPF_ERR_UNSUPPORTED, "vote: scene too large");
    if (vote_smem_bytes(t) + STATIC_RESERVE > ctx->smem_optin)
        return fail_msg(ctx, B200PPF_ERR_STATE, "vote: table was sliced for a larger shared-memory budget than this device has");
    return B200PPF_OK;
}

}  // namespace

// folded shift ranges: phase-sorted tables of FOLD_MIN_ENTRIES+ entries whose fold codes (key, q, cell) fit 31 bits
uint32_t k3_fold_qbits(const b200ppf_table *t) {
    if (!t->bp.bulk || t->info.n_entries < FOLD_MIN_ENTRIES) return 0;
    auto bits = [](uint32_t x) { uint32_t b = 0; while (b < 32 && (x >> b) != 0) ++b; return b; };
    const uint32_t qbits = bits(t->bp.n_turn - 1u);
    return bits(t->kp.key_space - 1u) + qbits + t->bp.cells_log2 <= 31 ? qbits : 0u;
}

uint32_t num_alpha_bins(float angle_step, int nalpha_rule) {
    const double t = 2.0 * M_PI / (double)angle_step;
    return (uint32_t)(nalpha_rule == NALPHA_CEIL ? ceil(t) : floor(t));
}

BinParams make_bin_params(float angle_step, int alpha_mode, int nalpha_rule) {
    BinParams bp;
    bp.angle_step = angle_step;
    bp.inv_step = 1.0f / angle_step;
    bp.n_alpha = num_alpha_bins(angle_step, nalpha_rule);
    bp.nalpha_rule = nalpha_rule;
    bp.overflow_bin = nalpha_rule == NALPHA_FLOOR_DROP ? bp.n_alpha : bp.n_alpha - 1;
    bp.fold = nalpha_rule == NALPHA_FLOOR_CLAMP ? 1u : 0u;
    bp.mode = alpha_mode;
    bp.mode_b_offset = (int)floor(M_PI / (double)angle_step);
    bp.guard = std::max(2e-4f, 1e-5f * bp.inv_step);
    bp.acc_cols = nalpha_rule == NALPHA_CEIL ? bp.n_alpha : bp.n_alpha + 1;
    // fixed-point hot loop: T bins per turn, multiplier with as many fractional bits as fit 32 bits
    const double T = 2.0 * M_PI / (double)angle_step;
    int kbits = 1;
    while ((double)(1ull << kbits) <= T + 1.0) ++kbits;  // integer bits of T
    bp.fix_shift = (uint32_t)std::min(31, std::max(1, 32 - kbits - 1));
    bp.fix_mul = (uint32_t)llrint(T * (double)(1ull << bp.fix_shift));
    bp.frac_mul = 1u << (32u - bp.fix_shift);
    // PCL's float rounding moves alpha by <= 3.6e-7 rad; guard = 4e-6 rad on both sides of an edge
    const double guard_rad = 4e-6;
    const double guard_bins = std::min(0.25, guard_rad / (double)angle_step);
    bp.fix_guard = (uint32_t)(guard_bins * 4294967296.0);
    // the +-pi seam sits at X = 0 (mod 2^32): below it the position inside the last bin is frac(T).
    // If frac(T) itself is inside the bin guard the seam is already covered.
    const double fracT = T - floor(T);
    const bool covered = fracT < guard_bins || fracT > 1.0 - guard_bins;
    bp.seam_guard = covered ? 0u : (uint32_t)(guard_rad / (2.0 * M_PI) * 4294967296.0);
    // phase-sorted buckets / constant-shift voting (ppf_math.cuh): T must be an integer up to the guard band
    bp.bulk = 0;
    bp.n_turn = (uint32_t)llrint(T);
    bp.cells_log2 = 0;
    bp.phase_guard = 0;
    const double off_int = fabs(T - (double)bp.n_turn);
    // the spare column must be able to hold position N_T - 1 and the column count must cover one turn
    if (alpha_mode == ALPHA_MODE_A && bp.n_turn >= 2 && bp.n_turn <= bp.acc_cols && off_int < 0.25 * guard_bins) {
        const double unit = (double)(1u << bp.fix_shift);
        bp.bulk = 1;
        bp.cells_log2 = 4;
        bp.phase_guard = (uint32_t)ceil(guard_bins * unit) + (uint32_t)ceil(off_int * unit) + 16u;
        // the guard must stay a small part of a phase cell
        while (bp.cells_log2 > 0 && (8ull * bp.phase_guard > (1ull << (bp.fix_shift - bp.cells_log2)) || bp.fix_shift < bp.cells_log2 + 8u))
            --bp.cells_log2;  // ... and hold the 8-bit sub-phase of the entry words
        if (bp.cells_log2 == 0) bp.bulk = 0;
    }
    return bp;
}

int k3_debug_alpha_bins(b200ppf_ctx *ctx, float angle_step, int alpha_mode, int nalpha_rule, const float *alpha_m,
                        const float *alpha_s, size_t n, uint32_t *fast, uint32_t *exact) {
    const BinParams bp = make_bin_params(angle_step, alpha_mode, nalpha_rule);
    if (!ctx) {  // host build of the same inline functions
        for (size_t p = 0; p < n; ++p) {
            fast[p] = alpha_bin_phase(bp, alpha_m[p], alpha_s[p]);
            exact[p] = alpha_bin_exact(bp.mode, bp.angle_step, bp.n_alpha, bp.overflow_bin, alpha_m[p], alpha_s[p]);
        }
        return B200PPF_OK;
    }
    StreamBuf<float> d_am(ctx), d_as(ctx);
    StreamBuf<uint32_t> d_f(ctx), d_e(ctx);
    PPF_CUDA(ctx, d_am.alloc(n));
    PPF_CUDA(ctx, d_as.alloc(n));
    PPF_CUDA(ctx, d_f.alloc(n));
    PPF_CUDA(ctx, d_e.alloc(n));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_am, alpha_m, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(d_as, alpha_s, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    PPF_LAUNCH(ctx, debug_alpha_bins_kernel, (unsigned)((n + 255) / 256), 256, 0, bp, d_am, d_as, (uint32_t)n, d_f, d_e);
    PPF_CUDA(ctx, cudaMemcpyAsync(fast, d_f, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(exact, d_e, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

size_t k3_accumulator_budget(const b200ppf_ctx *ctx) {
    size_t total = ctx->smem_optin ? ctx->smem_optin : kSmemPerBlockMax;
    return total - queue_bytes(VOTE_THREADS_LARGE) - STATIC_RESERVE;
}

int k3_group_wait(b200ppf_ctx *ctx, const uint32_t *flags, int world, uint32_t value) {
    PPF_LAUNCH(ctx, group_wait_kernel, 1, 1, 0, flags, world, value);
    return B200PPF_OK;
}

int k3_vote(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t, const b200ppf_cloud *scene,
            size_t ref_first, size_t ref_step, size_t ref_count, b200ppf_hypothesis *const *targets, int n_targets,
            size_t slot_first, size_t slot_step, const VoteSignal *signal) {
    if (n_targets < 1 || n_targets > MAX_PEERS) return fail_msg(ctx, B200PPF_ERR_INVALID, "vote: 1..16 output buffers");
    PeerTargets out;
    for (int g = 0; g < MAX_PEERS; ++g) {
        out.base[g] = g < n_targets ? targets[g] : nullptr;
        out.flags[g] = signal && g < n_targets ? signal->flags[g] : nullptr;
    }
    out.signal_slot = signal ? signal->slot : 0u;
    out.signal_value = signal ? signal->value : 0u;
    out.done_counter = signal ? signal->done_counter : nullptr;
    out.n = n_targets;
    out.slot_first = (uint32_t)slot_first;
    out.slot_step = (uint32_t)slot_step;
    int rc = check_vote_inputs(ctx, t, scene, ref_first, ref_step, ref_count);
    if (rc) return rc;
    if (!model || model->n != t->info.n_model)
        return fail_msg(ctx, B200PPF_ERR_STATE, "vote: model cloud does not match the table (setInputSource vs setSearchMethod)");
    if (ref_count == 0 && !signal) return B200PPF_OK;
    rc = ensure_vote_scratch(ctx, std::max<size_t>(1, ref_count));
    if (rc) return rc;
    cudaEventRecord(ctx->ev_vote[0], ctx->stream);
    if (ref_count) {
        rc = launch_vote(ctx, t, scene, ref_first, ref_step, ref_count, nullptr);  // records ev_vote[1], [2]
        if (rc) return rc;
    } else {  // a rank without reference points still signals its peers
        cudaEventRecord(ctx->ev_vote[1], ctx->stream);
        cudaEventRecord(ctx->ev_vote[2], ctx->stream);
    }
    BinParams bp = t->bp;
    bp.mode = ctx->alpha_mode;
    PPF_LAUNCH(ctx, ppf_peak_pose_kernel, (unsigned)((std::max<size_t>(1, ref_count) + 127) / 128), 128, 0, scene->pos, scene->nrm,
               model->pos, model->nrm, (uint32_t)ref_first, (uint32_t)ref_step, (uint32_t)ref_count, ctx->d_peaks, bp, out);
    cudaEventRecord(ctx->ev_vote[3], ctx->stream);
    ctx->vote_timed = true;
    return B200PPF_OK;
}

// group mode, first half: this rank's persistent CTAs on the shared queue over ALL reference points of the scene
int k3_vote_shared(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t ref_rate, size_t n_ref,
                   const VoteQueue *queue) {
    int rc = check_vote_inputs(ctx, t, scene, 0, ref_rate, n_ref);
    if (rc) return rc;
    if (!ctx->d_stats) PPF_CUDA(ctx, cudaMalloc(&ctx->d_stats, 4 * sizeof(unsigned long long)));
    PPF_CUDA(ctx, cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    cudaEventRecord(ctx->ev_vote[0], ctx->stream);
    rc = launch_vote(ctx, t, scene, 0, ref_rate, n_ref, nullptr, queue);  // records ev_vote[1], [2]
    if (rc) return rc;
    cudaEventRecord(ctx->ev_vote[3], ctx->stream);
    ctx->vote_timed = true;
    return B200PPF_OK;
}

// group mode, second half: the poses of all reference points from the complete peak array
int k3_poses(b200ppf_ctx *ctx, const b200ppf_cloud *model, const b200ppf_table *t, const b200ppf_cloud *scene, size_t ref_rate,
             size_t n_ref, const unsigned long long *peaks, b200ppf_hypothesis *out_records) {
    if (!model || model->n != t->info.n_model)
        return fail_msg(ctx, B200PPF_ERR_STATE, "vote: model cloud does not match the table (setInputSource vs setSearchMethod)");
    PeerTargets out;
    for (int g = 0; g < MAX_PEERS; ++g) {
        out.base[g] = g == 0 ? out_records : nullptr;
        out.flags[g] = nullptr;
    }
    out.n = 1;
    out.slot_first = 0;
    out.slot_step = 1;
    out.signal_slot = out.signal_value = 0;
    out.done_counter = nullptr;
    BinParams bp = t->bp;
    bp.mode = ctx->alpha_mode;
    PPF_LAUNCH(ctx, ppf_peak_pose_kernel, (unsigned)((n_ref + 127) / 128), 128, 0, scene->pos, scene->nrm, model->pos, model->nrm, 0u,
               (uint32_t)ref_rate, (uint32_t)n_ref, peaks, bp, out);
    return B200PPF_OK;
}

int k3_debug_pairs(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t s_r,
                   uint8_t *in_radius, int32_t *d4, float *alpha_s) {
    if (!t || !scene || s_r >= scene->n) return fail_msg(ctx, B200PPF_ERR_INVALID, "debug pairs: bad arguments");
    const size_t n = scene->n;
    StreamBuf<uint8_t> d_in(ctx);
    StreamBuf<int> d_d(ctx);
    StreamBuf<float> d_a(ctx);
    PPF_CUDA(ctx, d_in.alloc(n));
    PPF_CUDA(ctx, d_d.alloc(n * 4));
    PPF_CUDA(ctx, d_a.alloc(n));
    PPF_LAUNCH(ctx, ppf_debug_pairs_kernel, (unsigned)((n + 255) / 256), 256, 0, scene->pos, scene->nrm, (uint32_t)n,
               (uint32_t)s_r, t->kp, t->feature_mode, t->info.max_dist * 0.5f, d_in, d_d, d_a);
    PPF_CUDA(ctx, cudaMemcpyAsync(in_radius, d_in, n, cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(d4, d_d, n * 4 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaMemcpyAsync(alpha_s, d_a, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

int k3_debug_accumulator(b200ppf_ctx *ctx, const b200ppf_table *t, const b200ppf_cloud *scene, size_t s_r,
                         uint32_t *acc) {
    int rc = check_vote_inputs(ctx, t, scene, s_r, 1, 1);
    if (rc) return rc;
    rc = ensure_vote_scratch(ctx, 1);
    if (rc) return rc;
    const size_t len = (size_t)t->info.n_model * t->info.n_alpha;
    StreamBuf<uint32_t> d_acc(ctx);
    PPF_CUDA(ctx, d_acc.alloc(len));
    PPF_CUDA(ctx, cudaMemsetAsync(d_acc, 0, len * sizeof(uint32_t), ctx->stream));
    rc = launch_vote(ctx, t, scene, s_r, 1, 1, d_acc);
    if (rc) return rc;
    PPF_CUDA(ctx, cudaMemcpyAsync(acc, d_acc, len * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200PPF_OK;
}

}  // namespace b200ppf
