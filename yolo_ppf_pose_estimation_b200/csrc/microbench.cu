// microbench.cu — roofline denominators that MEASURED_PEAKS.json does not carry: the rate of
// shared-memory reductions (red.shared.add.u32 -> ATOMS.POPC.INC), which is what one PPF vote costs.
//   pattern 0  conflict-free: the 32 lanes of a warp hit 32 different banks
//   pattern 1  random words in a 64 KB accumulator (address from an LCG per reduction)
//   pattern 2  all lanes on one word
//   pattern 3  exactly 2 lanes per bank (different words): 2 wavefronts per instruction
//   pattern 4  exactly 4 lanes per bank: 4 wavefronts per instruction
// and the voting kernel's own shape — one coalesced 4-byte gather from an L2-resident table per reduction,
// eight gathers in flight per lane, address = loaded word - constant:
//   pattern 5  gathered, conflict-free addresses
//   pattern 6  gathered, random words (what an unordered bucket gives)
//   pattern 7  gathered, 2 lanes per bank
// Every CTA owns a 64 KB shared array; 512 threads x 2 CTAs per SM (the small voting shape) or, with
// +8 on the pattern, 1024 threads x 1 CTA per SM (the large shape).
#include "ppf_common.cuh"

namespace b200ppf {

namespace {

constexpr int MB_WORDS = 16 * 1024;
constexpr uint32_t MB_TABLE_WORDS = 16u << 20;  // 64 MB: larger than L1, resident in L2 like the model table

__device__ __forceinline__ uint32_t mb_word(int pattern, uint32_t k) {
    // k = running index of the reduction inside the table / the warp's sequence; lane = k & 31
    const uint32_t lane = k & 31u, row = k >> 5;
    switch (pattern) {
        case 0: return (row * 37u) % (MB_WORDS / 32) * 32u + lane;
        case 3: return (row * 37u) % (MB_WORDS / 64) * 64u + (lane & 15u) + (lane >> 4) * 32u;
        case 4: return (row * 37u) % (MB_WORDS / 128) * 128u + (lane & 7u) + (lane >> 3) * 32u;
        default: {
            uint32_t h = k * 2654435761u;
            h ^= h >> 15;
            h *= 0x2C1B3C6Du;
            h ^= h >> 13;
            return h % MB_WORDS;
        }
    }
}

__global__ void mb_fill_table_kernel(uint32_t *table, int pattern) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < MB_TABLE_WORDS; k += gridDim.x * blockDim.x)
        table[k] = mb_word(pattern, k) * 4u + 0x1000u;  // byte offset + the constant the kernel subtracts
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 1024 ? 1 : 2)
atoms_rate_kernel(int pattern, uint32_t iters, const uint32_t *__restrict__ table, unsigned long long *sink) {
    extern __shared__ uint32_t acc[];
    for (uint32_t k = threadIdx.x; k < MB_WORDS; k += THREADS) acc[k] = 0;
    __syncthreads();
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(acc);
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (pattern >= 5) {
        // the voting loop: 8 x 32 words in flight per lane, vote = load / subtract / reduce
        const uint32_t warps_total = gridDim.x * (THREADS / 32);
        const uint32_t span = MB_TABLE_WORDS / warps_total / 256u * 256u;
        const uint32_t *wp = table + (size_t)(blockIdx.x * (THREADS / 32) + warp) * span;
        const uint32_t c = 0x1000u - base;
        uint32_t done = 0;
        for (uint32_t it = 0; it < iters; it += 2) {  // 8 reductions per pass == 2 "iterations" of 4
            const uint32_t off = (done % span) + lane;
            uint32_t hw[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) hw[u] = __ldg(wp + off + u * 32);
#pragma unroll
            for (int u = 0; u < 8; ++u) asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(hw[u] - c) : "memory");
            done += 256u;
        }
    } else {
        uint32_t state = (blockIdx.x * THREADS + threadIdx.x) * 2654435761u + 12345u;
        for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                uint32_t word;
                if (pattern == 1) {
                    state = state * 1664525u + 1013904223u;
                    word = (state >> 10) % MB_WORDS;
                } else if (pattern == 2) {
                    word = warp;
                } else {
                    word = mb_word(pattern, ((it * 4 + u) * 64u + warp) * 32u + lane);
                }
                asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(base + word * 4) : "memory");
            }
        }
    }
    __syncthreads();
    unsigned long long s = 0;
    for (uint32_t k = threadIdx.x; k < MB_WORDS; k += THREADS) s += acc[k];
    if (s == 0xFFFFFFFFFFFFFFFFull) *sink = s;  // keep the work observable
}

template <int THREADS>
int run_rate(b200ppf_ctx *ctx, int pattern, const uint32_t *table, unsigned long long *sink, double *atoms_per_sec) {
    const size_t smem = MB_WORDS * sizeof(uint32_t);
    PPF_CUDA(ctx, cudaFuncSetAttribute(atoms_rate_kernel<THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t iters = 4096;
    const unsigned grid = (unsigned)ctx->sm_count * (1024 / THREADS) * 4;
    PPF_LAUNCH(ctx, atoms_rate_kernel<THREADS>, grid, THREADS, smem, pattern, 64u, table, sink);  // warm-up
    cudaEventRecord(ctx->ev[0], ctx->stream);
    PPF_LAUNCH(ctx, atoms_rate_kernel<THREADS>, grid, THREADS, smem, pattern, iters, table, sink);
    cudaEventRecord(ctx->ev[1], ctx->stream);
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    const double total = (double)grid * THREADS * (double)iters * 4.0;
    *atoms_per_sec = total / (ms * 1e-3);
    return B200PPF_OK;
}

}  // namespace

int microbench_atoms(b200ppf_ctx *ctx, int pattern, double *atoms_per_sec) {
    *atoms_per_sec = 0.0;
    const bool large = pattern >= 8;
    const int p = pattern & 7;
    StreamBuf<unsigned long long> sink(ctx);
    StreamBuf<uint32_t> table(ctx);
    PPF_CUDA(ctx, sink.alloc(1));
    if (p >= 5) {
        if (table.alloc(MB_TABLE_WORDS) != cudaSuccess) return fail_msg(ctx, B200PPF_ERR_NOMEM, "microbench: table allocation failed");
        mb_fill_table_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table, p == 5 ? 0 : (p == 6 ? 1 : 3));
        ctx->launches++;
    }
    return large ? run_rate<1024>(ctx, p, table, sink, atoms_per_sec) : run_rate<512>(ctx, p, table, sink, atoms_per_sec);
}

}  // namespace b200ppf
