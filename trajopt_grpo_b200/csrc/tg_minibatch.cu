// Minibatch plan of one PPO epoch (algorithms/ppo.py:147-157) over a rollout sharded by whole groups.
//
// The reference draws ONE torch.randperm over the valid steps of the whole rollout, flattened env-major, step-minor,
// and slices it into minibatches of batch_size.  A shard owns the contiguous global range [base, base + n_local) of
// that flattening (whole groups, ranks in order), so its part of minibatch b is the perm entries of
// perm[b*bs : (b+1)*bs] that fall in its range, in perm order.  Every rank holds the same perm and plans its own
// entries; summing the ranks' partial gradients gives the single-GPU minibatch gradient.
//
// Four launches, no atomics deciding positions (the plan is deterministic and stable):
//   plan_slots_kernel     one warp per env: slots[row0[n] + t] = t*N + n, the flat slot of every local valid step
//   plan_count_kernel     one CTA per chunk of PLAN_CHUNK perm entries: number of this shard's entries in the chunk
//   plan_scan_kernel      one CTA: exclusive prefix over the chunk counts (in place), total -> out_offsets[n_batches]
//   plan_scatter_kernel   one CTA per chunk again: entry i goes to out_ids[chunk prefix + rank within the chunk] as
//                         slots[perm[i] - base]; every minibatch boundary b*bs inside the chunk writes out_offsets[b]
// The slot table costs 8 bytes per local valid step written once and one random 8-byte read per entry; a binary search
// in row0 instead makes ~log2(N) random reads per entry, and at 5M entries those L2 requests bound the kernel.
#include "tg_common.cuh"

namespace {

constexpr int PLAN_NT = 256;
constexpr int PLAN_PER_THREAD = 16;
constexpr int PLAN_CHUNK = PLAN_NT * PLAN_PER_THREAD;   // perm entries per CTA
constexpr int PLAN_SCAN_NT = 1024;

// exclusive prefix of `flag` over the CTA in thread order; *total = sum over the CTA.  warp_sums: PLAN_NT / 32 ints.
__device__ __forceinline__ int cta_exclusive_scan(int flag, int *warp_sums, int *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, flag);
    const int in_warp = __popc(m & ((1u << lane) - 1u));
    if (lane == 0) warp_sums[warp] = __popc(m);
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < PLAN_NT / 32; ++w) {
        const int s = warp_sums[w];
        before += w < warp ? s : 0;
        all += s;
    }
    __syncthreads();   // warp_sums is reused by the next round
    *total = all;
    return before + in_warp;
}

__global__ void __launch_bounds__(PLAN_NT) plan_count_kernel(const int64_t *__restrict__ perm, int64_t n_total,
                                                             int64_t base, int64_t n_local,
                                                             int64_t *__restrict__ chunk_count) {
    __shared__ int warp_sums[PLAN_NT / 32];
    const int64_t c0 = (int64_t)blockIdx.x * PLAN_CHUNK;
    int cnt = 0;
#pragma unroll 4
    for (int j = 0; j < PLAN_PER_THREAD; ++j) {
        const int64_t i = c0 + j * PLAN_NT + threadIdx.x;
        if (i < n_total) {
            const uint64_t k = (uint64_t)(__ldg(perm + i) - base);   // out of range (k < base too) -> huge
            cnt += k < (uint64_t)n_local;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < PLAN_NT / 32; ++w) s += warp_sums[w];
        chunk_count[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(PLAN_SCAN_NT) plan_scan_kernel(int64_t *__restrict__ chunk, int64_t n_chunks,
                                                                 int64_t *__restrict__ total_out) {
    __shared__ int64_t warp_sums[PLAN_SCAN_NT / 32];
    __shared__ int64_t carry_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t carry = 0;
    for (int64_t c0 = 0; c0 < n_chunks; c0 += PLAN_SCAN_NT) {
        const int64_t c = c0 + threadIdx.x;
        const int64_t v = c < n_chunks ? chunk[c] : 0;
        int64_t x = v;   // inclusive warp scan
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int64_t w = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            warp_sums[lane] = w;   // inclusive over warps
            if (lane == 31) carry_s = w;
        }
        __syncthreads();
        const int64_t excl = carry + (warp > 0 ? warp_sums[warp - 1] : 0) + x - v;
        if (c < n_chunks) chunk[c] = excl;
        carry += carry_s;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_out = carry;
}

// slots[row0[n] + t] = t*N + n for every valid step of this shard: one warp per env, so the writes are contiguous
__global__ void __launch_bounds__(PLAN_NT) plan_slots_kernel(int64_t N, const int32_t *__restrict__ len,
                                                             const int64_t *__restrict__ row0, int64_t n_local,
                                                             int64_t *__restrict__ slots) {
    const int64_t n = (int64_t)blockIdx.x * (PLAN_NT / 32) + (threadIdx.x >> 5);
    if (n >= N) return;
    const int64_t r0 = row0[n];
    const int L = len[n];
    for (int t = threadIdx.x & 31; t < L && r0 + t < n_local; t += 32) slots[r0 + t] = (int64_t)t * N + n;
}

__global__ void __launch_bounds__(PLAN_NT) plan_scatter_kernel(const int64_t *__restrict__ perm, int64_t n_total,
                                                               int64_t batch_size, int64_t base, int64_t n_local,
                                                               const int64_t *__restrict__ slots,
                                                               const int64_t *__restrict__ chunk_prefix, int64_t max_ids,
                                                               int64_t *__restrict__ out_ids,
                                                               int64_t *__restrict__ out_offsets) {
    __shared__ int warp_sums[PLAN_NT / 32];
    const int64_t c0 = (int64_t)blockIdx.x * PLAN_CHUNK;
    int64_t pos0 = chunk_prefix[blockIdx.x];
    // i mod batch_size, advanced by PLAN_NT per round without a division per entry
    int64_t r = (c0 + threadIdx.x) % batch_size;
    const int64_t step = PLAN_NT % batch_size;
    for (int j = 0; j < PLAN_PER_THREAD; ++j) {
        const int64_t i = c0 + (int64_t)j * PLAN_NT + threadIdx.x;
        if (c0 + (int64_t)j * PLAN_NT >= n_total) break;   // CTA-uniform
        int64_t k = -1;
        int hit = 0;
        if (i < n_total) {
            k = __ldg(perm + i) - base;
            hit = (uint64_t)k < (uint64_t)n_local;
        }
        int round_total;
        const int rank = cta_exclusive_scan(hit, warp_sums, &round_total);
        const int64_t pos = pos0 + rank;
        if (i < n_total && r == 0) out_offsets[i / batch_size] = pos;   // boundary b*bs: entries of perm[0, b*bs)
        if (hit && pos < max_ids) out_ids[pos] = __ldg(slots + k);
        pos0 += round_total;
        r += step;
        if (r >= batch_size) r -= batch_size;
    }
}

}  // namespace

// chunk counts [n_chunks] followed by the slot table [n_total] (a shard holds at most n_total valid steps)
extern "C" int64_t tg_minibatch_plan_workspace_bytes(int64_t n_total) {
    if (n_total <= 0) return 0;
    return 8 * ((n_total + PLAN_CHUNK - 1) / PLAN_CHUNK + n_total);
}

extern "C" int tg_minibatch_plan(tg_ctx *ctx, int64_t N, const int32_t *len, const int64_t *row0, const int64_t *perm,
                                 int64_t n_total, int64_t batch_size, int64_t base, int64_t n_local, int64_t max_ids,
                                 int64_t *out_ids, int64_t *out_offsets, void *workspace, void *stream) {
    TgRange nvtx_range("tg_minibatch_plan (PPO minibatches of this shard)");
    TG_REQUIRE(ctx && len && row0 && perm && out_offsets && workspace, TG_ERR_ARG, "tg_minibatch_plan: null argument");
    TG_REQUIRE(out_ids || max_ids == 0, TG_ERR_ARG, "tg_minibatch_plan: out_ids is null");
    TG_REQUIRE(N > 0 && n_total > 0 && batch_size > 0, TG_ERR_SHAPE,
               "tg_minibatch_plan: N, n_total and batch_size must be positive");
    TG_REQUIRE(base >= 0 && n_local >= 0 && base + n_local <= n_total && max_ids >= 0, TG_ERR_SHAPE,
               "tg_minibatch_plan: shard [%lld, %lld) is not inside [0, %lld)", (long long)base,
               (long long)(base + n_local), (long long)n_total);
    const int64_t n_chunks = (n_total + PLAN_CHUNK - 1) / PLAN_CHUNK;
    TG_REQUIRE(n_chunks < ((int64_t)1 << 31), TG_ERR_SHAPE, "tg_minibatch_plan: n_total too large");
    const int64_t n_batches = (n_total + batch_size - 1) / batch_size;
    TG_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    int64_t *chunk = (int64_t *)workspace;
    int64_t *slots = chunk + n_chunks;
    if (n_local > 0) {
        plan_slots_kernel<<<(unsigned)((N + PLAN_NT / 32 - 1) / (PLAN_NT / 32)), PLAN_NT, 0, st>>>(N, len, row0, n_local,
                                                                                                  slots);
        TG_CUDA(cudaGetLastError());
    }
    plan_count_kernel<<<(unsigned)n_chunks, PLAN_NT, 0, st>>>(perm, n_total, base, n_local, chunk);
    TG_CUDA(cudaGetLastError());
    plan_scan_kernel<<<1, PLAN_SCAN_NT, 0, st>>>(chunk, n_chunks, out_offsets + n_batches);
    TG_CUDA(cudaGetLastError());
    plan_scatter_kernel<<<(unsigned)n_chunks, PLAN_NT, 0, st>>>(perm, n_total, batch_size, base, n_local, slots, chunk,
                                                                max_ids, out_ids, out_offsets);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
