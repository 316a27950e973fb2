// Length order of a rollout: the update kernels walk samples (t, env) with t < len[env] only.
// Episodes are ragged (algorithms/grpo.py:108-115 pools "all valid (episode, step) pairs"), so a
// tile of consecutive env indices at step t mixes live and finished envs and would spend tensor /
// FMA work on masked rows.  tg_len_order sorts the env indices by episode length, longest first
// (stable, so the order is a deterministic function of `len`), and counts the live envs per step:
//   perm[j]  env index at sorted position j          (int32 [N])
//   cnt[t]   number of envs with len > t             (int32 [T]) -- the live envs of step t are perm[0..cnt[t])
// The kernels then tile the sorted positions: every tile but the last of a step is fully valid.
// The sort itself is index plumbing (CUB radix sort of N small integer keys), not arithmetic of the path.
#include <cub/device/device_radix_sort.cuh>

#include "tg_common.cuh"

__global__ void order_keys_kernel(int64_t N, int T, const int32_t *__restrict__ len, uint32_t *__restrict__ key,
                                  int32_t *__restrict__ idx) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    int l = len[n];
    l = l < 0 ? 0 : (l > T ? T : l);
    key[n] = (uint32_t)(T - l);      // ascending key = descending length
    idx[n] = (int32_t)n;
}

// cnt[t] = #(len > t) = #(key < T - t) = lower bound of (T - t) in the sorted keys
__global__ void order_count_kernel(int64_t N, int T, const uint32_t *__restrict__ sorted_key, int32_t *__restrict__ cnt) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const uint32_t want = (uint32_t)(T - t);
    int64_t lo = 0, hi = N;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (sorted_key[mid] < want) lo = mid + 1;
        else hi = mid;
    }
    cnt[t] = (int32_t)lo;
}

extern "C" int tg_len_order_hold(tg_ctx *ctx, int64_t N, int T, const int32_t *len, void *stream) {
    TG_REQUIRE(ctx && len, TG_ERR_ARG, "tg_len_order_hold: null argument");
    TG_CUDA(cudaSetDevice(ctx->device));
    ctx->held_len = nullptr;
    int rc = tg_len_order(ctx, N, T, len, (cudaStream_t)stream);
    if (rc) return rc;
    ctx->held_len = len; ctx->held_N = N; ctx->held_T = T;
    return TG_OK;
}

extern "C" int tg_len_order_release(tg_ctx *ctx) {
    TG_REQUIRE(ctx != nullptr, TG_ERR_ARG, "tg_len_order_release: ctx is null");
    ctx->held_len = nullptr;
    return TG_OK;
}

int tg_len_order(tg_ctx *ctx, int64_t N, int T, const int32_t *len, cudaStream_t st) {
    TG_REQUIRE(N > 0 && N < (int64_t)1 << 31 && T > 0, TG_ERR_SHAPE, "tg_len_order: bad shape");
    if (ctx->held_len != nullptr && ctx->held_len == len && ctx->held_N == N && ctx->held_T == T) return TG_OK;
    int bits = 1;
    while ((1 << bits) <= T) ++bits;             // keys are in [0, T]
    size_t temp = 0;
    TG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp, (const uint32_t *)nullptr, (uint32_t *)nullptr,
                                            (const int32_t *)nullptr, (int32_t *)nullptr, (int)N, 0, bits, st));
    const size_t nb = ((size_t)N * 4 + 255) / 256 * 256, tb = ((size_t)T * 4 + 255) / 256 * 256;
    // [perm | cnt | key_in | key_out | idx_in | cub temp]
    int rc = tg_ctx_grow(ctx, &ctx->order_buf, &ctx->order_cap, 4 * nb + tb + temp + 256);
    if (rc) return rc;
    char *base = (char *)ctx->order_buf;
    ctx->perm = (int32_t *)base;
    ctx->cnt = (int32_t *)(base + nb);
    uint32_t *key_in = (uint32_t *)(base + nb + tb), *key_out = (uint32_t *)(base + 2 * nb + tb);
    int32_t *idx_in = (int32_t *)(base + 3 * nb + tb);
    void *tmp = base + 4 * nb + tb;
    order_keys_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(N, T, len, key_in, idx_in);
    TG_CUDA(cudaGetLastError());
    TG_CUDA(cub::DeviceRadixSort::SortPairs(tmp, temp, key_in, key_out, idx_in, ctx->perm, (int)N, 0, bits, st));
    order_count_kernel<<<(unsigned)((T + 255) / 256), 256, 0, st>>>(N, T, key_out, ctx->cnt);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
