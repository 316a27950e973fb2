// K3 on the tensor cores for WIDE policies (obs -> W -> W -> act, W = 128 or 256; BASELINE cfg 3/4/5).
//
// The three W x W GEMMs of a 128-sample tile (forward, backward-data, weight-gradient) cannot share one SM's
// memories: the weights in both operand layouts are 2 x 2W^2 x 4 bytes (512 KB..1 MB at W = 256) and the
// weight-gradient operands -- the tile's H1 and dZ2 in MN-major form, hi and lo -- another 4 x 128 x W x 4.
// So the update is two kernels per batch of tiles, both fed by streams:
//
//   kernel A  (update_tcw_fwdbwd_kernel)  forward + objective + backward-data for every tile of the batch.
//       The weights are STREAMED from L2 every tile through a 4-stage TMA ring (K-major chunks for the
//       forward, MN-major chunks for the backward), exactly like the 256-wide rollout kernel; activations go
//       registers -> tensor memory as the A operand (K halves at W = 256).  The first Linear runs on the
//       tensor core too (obs hi/lo + ones column carrying the bias).  Per tile the kernel leaves in an HBM
//       scratch, in the operand layout of kernel B:  H1, H2, dZ1 as fp32 (MN-major SW128_32B, 8-sample
//       sub-blocks) and Y = [x, 1, dmu] (fp32, K-major).  No column sums over samples are left in this kernel:
//       round 1 computed dWo = dmu^T . H2 with register butterflies here (187 us of 847 us per 2656-tile batch at
//       W = 256); dWo moved to kernel B.
//   kernel B  (update_tcw_wgrad_kernel)   split-K weight-gradient GEMMs over the batch's samples:
//       dW1 += dZ2^T . H1   and   [dW0 | db0] += dZ1^T . [x, 1]   on the tensor core (fp32 accumulators persistent in tensor
//       memory for all tiles of the launch, added to the CTA-private gradient copy at the end);
//       db1 = sum_s dZ2[s, :]   and   dWo = sum_s dmu[s] H2[s, :]   on the FP32 pipe of the converter warps (register column sums).
//       Operands are streamed from the scratch by TMA, 8 samples at a time, through two shared-memory rings (see the kernel);
//       dZ2 is not stored: the converter warps rebuild it from H2 and dmu, dZ2 = (Wo^T dmu) * act'(H2), with the operation
//       order of kernel A, while they produce the tf32 lo parts (the fp32 rows themselves serve as the hi operands: the tensor
//       core drops the low 13 bits).  W = 128: one launch.  W = 256: the [256 x 256] accumulator of dW1 fills the 512 TMEM
//       columns, so [dW0 | db0] is a second, light launch over dZ1 and Y; every scratch array is read once per update.
//       History per 2656 tiles at W = 256 (ncu, serialised): two half-output launches 2 x 241 us (8 -> 16 converter warps
//       293 -> 241) -> two rings + two converter groups 2 x 202 -> db1 / dWo as register sums 2 x 160 -> one dW1 launch +
//       one dW0 launch with warp-uniform MMA issue 201 + 80 us.
//
// Tiles are enumerated in length order (tg_order.cu): tile k of the compact list is (step t, sorted
// positions 128*blk ..), found by binary search in the per-step prefix of live tiles; k beyond the live
// total is a no-op, so the host launches ceil(upper bound / batch) batches without reading anything back.
#include <math.h>
#include <stdlib.h>

#include "tg_umma.cuh"

#define TCW_STAGES 4
#define TCW_BAR_L1 5
#define TCW_BAR_K0 6
#define TCW_BAR_K1 7

struct TcwScratch {                       // per-tile byte strides / bases inside the HBM scratch
    unsigned char *base;
    int64_t tile_bytes;                   // all arrays of one tile
    int64_t arr_bytes;                    // one of H1, dZ2, dZ1 (fp32) per tile = 16 sub-blocks * W/32 KB
    int64_t x_bytes;                      // Y per tile = 16 * XKP * 32 (fp32), XKP = roundup(O + 1 + A, 8)
};
// array order inside a tile: H1, H2, dZ1 (fp32, MN-major sub-blocks), Yh, Yl  (Y = [x, 1, dmu], K-major)

struct TcwArgs {
    TcwLayout lay;
    TcwScratch sc;
    int64_t N;
    int T;
    const float *obs, *act, *adv, *oldlp;
    const float *target;                  // value head (critic regression, ppo.py:168-169) when non-null
    const int32_t *perm, *cnt;
    const int64_t *tstart;                // [T+1] prefix of live tiles per step
    int64_t k_begin, k_count;             // this batch: compact tiles [k_begin, k_begin + k_count)
    const float *packed;
    const float *params;                  // flat torch-order parameters (kernel B reads Wo from them)
    float inv_sd[TG_MAX_ACT], inv_var[TG_MAX_ACT], log_norm;
    float eps_clip, scale, kl_scale;
    float *gpart;                         // [grid][n_params], accumulated (+=) across launches
    double *spart;                        // [grid][TG_SPART_LD], accumulated
    // forward-only mode (tg_policy_forward_traj: critic values over a rollout ppo.py:93-94, old log-probs
    // ppo.py:142-143 / grpo.py:118-119): kernel A stops after the output layer and writes these; no kernel B
    int forward_only;
    float *out_mu, *out_logp;
    // GRPO's KL term (REF instances): log-prob under a frozen reference policy and its coefficient beta * scale
    const float *reflp;
    float ref_coef;
};

bool tg_update_tcw_shape_built(const tg_mlp_cfg *mlp);

bool tg_update_tcw_eligible(const tg_mlp_cfg *mlp) {
    if (!mlp || mlp->n_layers != 3) return false;
    const int W = mlp->dims[1];
    return (W == 128 || W == 256) && mlp->dims[2] == W && mlp->dims[0] >= 1 && mlp->dims[0] <= 23 &&
           (mlp->dims[3] == 1 || mlp->dims[3] == 2 || mlp->dims[3] == 4) && mlp->activation >= 0 && mlp->activation <= 2;
}

// tstart[t] = number of live tiles of steps < t (tile = 128 sorted positions), tstart[T] = total
__global__ void tcw_tstart_kernel(int T, const int32_t *__restrict__ cnt, int64_t *__restrict__ tstart) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int64_t s = 0;
        for (int t = 0; t < T; ++t) {
            tstart[t] = s;
            s += (cnt[t] + 127) / 128;
        }
        tstart[T] = s;
    }
}

// compact tile k -> (t, blk); false when k is beyond the live tiles
TG_D bool tcw_tile_of(const int64_t *__restrict__ tstart, int T, int64_t k, int *t, int *blk) {
    if (k >= tstart[T]) return false;
    int lo = 0, hi = T - 1;             // largest t with tstart[t] <= k
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tstart[mid] <= k) lo = mid;
        else hi = mid - 1;
    }
    *t = lo;
    *blk = (int)(k - tstart[lo]);
    return true;
}

// the same for the NEXT tile of a CTA (k grows by the grid size): walk forward from the previous step instead of
// a fresh 16-load binary search -- the lookup sits on the serial per-tile chain of every warp
TG_D bool tcw_tile_next(const int64_t *__restrict__ tstart, int T, int64_t k, int *t, int *blk) {
    if (k >= tstart[T]) return false;
    int tt = *t;
    while (tt + 1 < T && tstart[tt + 1] <= k) ++tt;
    *t = tt;
    *blk = (int)(k - tstart[tt]);
    return true;
}

struct TrueTag { static constexpr bool value = true; };
struct FalseTag { static constexpr bool value = false; };

// 256-bit global accesses (sm_100): one lane moves a whole 32-byte sector, so the row-per-thread scratch traffic
// is made of full sectors instead of 16-byte halves
TG_D void stg256(void *p, const float *v) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                 "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}
TG_D void ldg256(const void *p, float *v) {
    asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p)
                 : "memory");
}

// 16-column pieces (half hh of the 32-column block): the epilogues of kernel A work at this granularity so that a
// thread holds 16 accumulator values + their hi/lo split (48 registers) instead of 32 + 32 + 32 -- at 96 registers
// per thread (18 warps) the 32-column form spilled ~0.7 KB per thread
template <int W>
TG_D void tcw_store16(unsigned char *arr, int s, int cbk, int hh, const float *v) {
    const int r = s & 7;
    unsigned char *p = arr + (size_t)(s >> 3) * (W / 32 * 1024) + (size_t)cbk * 1024 + (size_t)r * 128;
#pragma unroll
    for (int c8 = 0; c8 < 2; ++c8) stg256(p + (uint32_t)(((hh * 2 + c8) ^ (r & 3)) << 5), v + 8 * c8);
}
TG_D void tcw_tm16(const float *v, uint32_t tm_hi, uint32_t tm_lo) {
    // the raw fp32 value is the hi operand (the tensor core drops its low 13 bits), lo = x - trunc(x)
    float lo[16];
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) lo[jj] = v[jj] - tf32_trunc(v[jj]);
    tmem_st16(tm_hi, v);
    tmem_st16(tm_lo, lo);
}
// dZ2 = (Wo^T dmu) * act'(H2) for one column: the ONE definition both kernels use (kernel A for the A operand of the
// backward-data GEMM, kernel B's converter warps for the weight-gradient operand), so the two are bit-identical
template <int A>
TG_D float tcw_dz2(float h2, const float *dmu, const float *wo_col, int wo_stride, int act_kind) {
    float g = 0.0f;
#pragma unroll
    for (int o = 0; o < A; ++o) g = fmaf(dmu[o], wo_col[o * wo_stride], g);
    return g * act_bwd_from_out(h2, act_kind);
}
// the same 32 columns read back from the scratch (this thread wrote them), split, into the tensor-memory A operand.
// DZ2: the scratch holds H2; the operand is dZ2 = (Wo^T dmu) * act'(H2) (wo = this thread's first column of Wo).
template <int W, int A, bool DZ2>
TG_D void tcw_reload32(const unsigned char *arr, int s, int cbk, uint32_t tm_hi, uint32_t tm_lo, const float *dmu,
                       const float *wo, int act_kind) {
    const int r = s & 7;
    const unsigned char *p = arr + (size_t)(s >> 3) * (W / 32 * 1024) + (size_t)cbk * 1024 + (size_t)r * 128;
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        float v[16], hi[16], lo[16];
#pragma unroll
        for (int c8 = 0; c8 < 2; ++c8) ldg256(p + (uint32_t)(((hh * 2 + c8) ^ (r & 3)) << 5), v + 8 * c8);
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
            const float x = DZ2 ? tcw_dz2<A>(v[jj], dmu, wo + hh * 16 + jj, W, act_kind) : v[jj];
            hi[jj] = tf32_hi(x);
            lo[jj] = x - hi[jj];
        }
        tmem_st16(tm_hi + (uint32_t)(hh * 16), hi);
        tmem_st16(tm_lo + (uint32_t)(hh * 16), lo);
    }
}

// ============================================================================
// kernel A
// ============================================================================
// NP threads serve one sample (NP * 4 compute warps, each thread owning W / NP columns) + producer + MMA warp.
// NP = 2 keeps the CTA at 10 warps = 3 per SM sub-partition, i.e. 168 registers per thread and no spills; with
// NP = 4 (18 warps, 96 registers) the epilogues spilled ~0.8 KB per thread into an L1 that the 222 KB of shared
// memory leave almost no room for, and the serial step chain paid the L2 latency of every reload.
// REF: with GRPO's KL term to a reference policy (a.reflp).  A template flag, not a branch: at W = 256 the epilogues
// run at the 96-register cap, and a runtime branch added ~30 B of spills to the instances without the term.
template <int O, int A, bool RELU, int W, int NP, bool REF>
__global__ void __launch_bounds__(NP * 128 + 64, 1) update_tcw_fwdbwd_kernel(const __grid_constant__ TcwArgs a) {
    constexpr int HW = W / NP, NCH = HW / 32, OKP = (O + 1 + 7) / 8 * 8, KH = W / 128;
    constexpr int XKP = (O + 1 + A + 7) / 8 * 8;      // rows of Y = [x, 1, dmu, 0..] handed to kernel B
    constexpr int NCT = NP * 128;                     // compute threads
    constexpr int CNT_ALL = NCT + 32, CNT_H1 = (KH == 2 ? NCT / 2 : NCT) + 32;
    constexpr int NKC = W / 32;                       // K chunks per direction
    constexpr uint32_t CB = (uint32_t)W * 128u;       // chunk bytes
    constexpr uint32_t TM_D = 0u, TM_AHI = (uint32_t)W, TM_ALO = (uint32_t)W + 128u;
    constexpr int NS = REF ? TG_NSTAT : 4;            // statistics this instance produces
    if (a.k_begin + blockIdx.x >= a.tstart[a.T]) return;      // no live tile for this CTA in this batch (CTA-uniform)
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar, bar_d, bar_k0, full_bar[TCW_STAGES], empty_bar[TCW_STAGES];
    __shared__ uint32_t tmem_slot;
    __shared__ float muS[NP][A][128];
    __shared__ float dmuS[A][128];
    __shared__ double sred[NS][16];
    // objective / count / ratio / clip / KL statistics of sample row e, accumulated over the CTA's tiles by the part-0
    // thread of that row (shared memory instead of 10 registers per thread: the epilogues run at the 96-register cap)
    __shared__ double statS[NS][128];
    if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
    for (int i = threadIdx.x; i < NS * 128; i += blockDim.x) statS[i / 128][i % 128] = 0.0;
    unsigned char *ring = smem_raw;
    float *Rsm = reinterpret_cast<float *>(smem_raw + TCW_STAGES * CB);
    unsigned char *O_hi = reinterpret_cast<unsigned char *>(Rsm + a.lay.resident);
    unsigned char *O_lo = O_hi + 128 * OKP * 4;
    stage_weights_tma(Rsm, a.packed, a.lay.resident, &wbar);
    if (threadIdx.x == 0) {
        mbar_init(&bar_d, 1);
        mbar_init(&bar_k0, 1);
        for (int i = 0; i < TCW_STAGES; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_slot, 512);
    for (int i = threadIdx.x; i < 128 * OKP; i += blockDim.x) {
        const int r = i / OKP, c = i % OKP;
        *reinterpret_cast<float *>(O_hi + core_offset(OKP, r, c)) = c == O ? 1.0f : 0.0f;
        *reinterpret_cast<float *>(O_lo + core_offset(OKP, r, c)) = 0.0f;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t N = a.N;
    // tiles of this CTA inside the batch: slot = blockIdx.x, + gridDim.x, ...
    const int64_t k_end = a.k_begin + a.k_count;

    if (warp == NP * 4) {
        // ===== TMA producer: per tile the forward chunks (hi, lo per K chunk) then the backward chunks =====
        if (lane == 0) {
            uint32_t gi = 0;
            const float *srcf = a.packed + a.lay.chunks_f, *srcb = a.packed + a.lay.chunks_b;
            int t = 0, blk = 0;
            bool first_tile = true;
            for (int64_t k = a.k_begin + blockIdx.x; k < k_end; k += gridDim.x) {
                if (!(first_tile ? tcw_tile_of(a.tstart, a.T, k, &t, &blk) : tcw_tile_next(a.tstart, a.T, k, &t, &blk))) break;
                first_tile = false;
                for (int dir = 0; dir < (a.forward_only ? 1 : 2); ++dir) {
                    const float *src = dir ? srcb : srcf;
                    for (int i = 0; i < 2 * NKC; ++i, ++gi) {
                        const uint32_t st = gi % TCW_STAGES, ph = (gi / TCW_STAGES) & 1u;
                        mbar_wait(&empty_bar[st], ph ^ 1u);
                        mbar_expect_tx(&full_bar[st], CB);
                        tma_bulk_g2s(ring + (size_t)st * CB, src + (size_t)i * a.lay.chunk_floats, CB, &full_bar[st]);
                    }
                }
            }
        }
    } else if (warp == NP * 4 + 1) {
        // ===== MMA issuer =====
        const uint32_t idesc_f = umma_idesc_tf32(128, W, false, false);
        const uint32_t idesc_b = umma_idesc_tf32(128, W, false, true);
        const uint32_t r_u = smem_u32(Rsm), ring_u = smem_u32(ring);
        const uint32_t w0hi = r_u + (uint32_t)a.lay.w0hi * 4u, w0lo = r_u + (uint32_t)a.lay.w0lo * 4u;
        const uint32_t ohi = smem_u32(O_hi), olo = smem_u32(O_lo);
        uint32_t gi = 0;
        int t = 0, blk = 0;
        bool first_tile = true;
        for (int64_t k = a.k_begin + blockIdx.x; k < k_end; k += gridDim.x) {
            if (!(first_tile ? tcw_tile_of(a.tstart, a.T, k, &t, &blk) : tcw_tile_next(a.tstart, a.T, k, &t, &blk))) break;
            first_tile = false;
            named_sync(TCW_BAR_L1, CNT_ALL);
            tc_fence_after();
            {
                uint32_t acc = 0;
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint32_t aa = pass == 2 ? olo : ohi, bb = pass == 1 ? w0lo : w0hi;
#pragma unroll
                    for (int kk = 0; kk < OKP; kk += 8) {
                        umma_tf32_w(tmem + TM_D, umma_operand_desc(aa, OKP, false, kk), umma_operand_desc(bb, OKP, false, kk),
                                  idesc_f, acc);
                        acc = 1u;
                    }
                }
                umma_commit_w(&bar_d);
            }
            __syncwarp();
            for (int dir = 0; dir < (a.forward_only ? 1 : 2); ++dir) {   // 0: forward (K-major B), 1: backward-data (MN-major B)
                for (int half = 0; half < KH; ++half) {
                    if (half == 0) named_sync(TCW_BAR_K0, CNT_ALL);
                    else named_sync(TCW_BAR_K1, CNT_H1);
                    tc_fence_after();
                    {
                        for (int c = 0; c < 4; ++c) {
                            const uint32_t st_hi = gi % TCW_STAGES, ph_hi = (gi / TCW_STAGES) & 1u;
                            ++gi;
                            const uint32_t st_lo = gi % TCW_STAGES, ph_lo = (gi / TCW_STAGES) & 1u;
                            ++gi;
                            const uint32_t bhi = ring_u + st_hi * CB, blo = ring_u + st_lo * CB;
                            const uint32_t acol = (uint32_t)(c * 32);
                            const uint32_t idesc = dir ? idesc_b : idesc_f;
                            mbar_wait(&full_bar[st_hi], ph_hi);
                            tc_fence_after();
#pragma unroll
                            for (int ks = 0; ks < 32; ks += 8)
                                umma_tf32_ts_w(tmem + TM_D, tmem + TM_AHI + acol + (uint32_t)ks,
                                             dir ? umma_desc_mn32(bhi + (uint32_t)ks * 128u, 4096u)
                                                 : umma_operand_desc(bhi, 32, false, ks),
                                             idesc, (half | c | ks) ? 1u : 0u);
#pragma unroll
                            for (int ks = 0; ks < 32; ks += 8)
                                umma_tf32_ts_w(tmem + TM_D, tmem + TM_ALO + acol + (uint32_t)ks,
                                             dir ? umma_desc_mn32(bhi + (uint32_t)ks * 128u, 4096u)
                                                 : umma_operand_desc(bhi, 32, false, ks),
                                             idesc, 1u);
                            umma_commit_w(&empty_bar[st_hi]);
                            mbar_wait(&full_bar[st_lo], ph_lo);
                            tc_fence_after();
#pragma unroll
                            for (int ks = 0; ks < 32; ks += 8)
                                umma_tf32_ts_w(tmem + TM_D, tmem + TM_AHI + acol + (uint32_t)ks,
                                             dir ? umma_desc_mn32(blo + (uint32_t)ks * 128u, 4096u)
                                                 : umma_operand_desc(blo, 32, false, ks),
                                             idesc, 1u);
                            umma_commit_w(&empty_bar[st_lo]);
                        }
                        umma_commit_w((half == KH - 1) ? &bar_d : &bar_k0);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        // ===== compute warps =====
        const int q = warp & 3, part = warp >> 2;
        const int e = q * 32 + lane;                  // sample row of the tile = TMEM lane
        const int c0 = part * HW;
        const int my_half = c0 / 128;                 // K half this thread's columns belong to
        const uint32_t acol0 = (uint32_t)(c0 % 128);
        const uint32_t my_tm = tmem + ((uint32_t)(q * 32) << 16);
        const int act_kind = RELU ? TG_ACT_RELU : a.lay.act;
        const float *b1 = Rsm + a.lay.b1 + c0, *wo = Rsm + a.lay.wo + c0, *bo = Rsm + a.lay.bo;
        uint32_t ph_d = 0, ph_k0 = 0;
        float c_bo[A];                                 // this thread's running sum of dmu (dbo)
#pragma unroll
        for (int j = 0; j < A; ++j) c_bo[j] = 0.0f;

        // K-half protocol of the TMEM A operand (W = 256): threads whose columns belong to half 0 write it while
        // they process their chunks; threads of half 1 only write the scratch, tell the MMA warp they have read
        // D, wait until the MMAs of half 0 have consumed the operand, and then reload their chunks from the
        // scratch they just wrote (nothing is held in registers across the wait).
        constexpr bool DEFER = KH == 2;
        const bool deferred = DEFER && my_half == 1;
        float dmu_own[A];                              // d objective / d mu of this thread's sample (epilogue 2b)
#pragma unroll
        for (int j = 0; j < A; ++j) dmu_own[j] = 0.0f;
        auto finish_A = [&](const unsigned char *arr, bool dz2) {
            if (deferred) {
                tc_fence_before();
                named_arrive(TCW_BAR_K0, CNT_ALL);
                mbar_wait(&bar_k0, ph_k0);
                tc_fence_after();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    const uint32_t th = my_tm + TM_AHI + acol0 + (uint32_t)(ch * 32), tl = my_tm + TM_ALO + acol0 + (uint32_t)(ch * 32);
                    if (dz2) tcw_reload32<W, A, true>(arr, e, (c0 >> 5) + ch, th, tl, dmu_own, wo + ch * 32, act_kind);
                    else tcw_reload32<W, A, false>(arr, e, (c0 >> 5) + ch, th, tl, dmu_own, wo, act_kind);
                }
            }
            ph_k0 ^= 1u;
            tmem_st_wait();
            tc_fence_before();
            if (deferred) named_arrive(TCW_BAR_K1, CNT_H1);
            else named_arrive(TCW_BAR_K0, CNT_ALL);
        };

        int t = 0, blk = 0;
        bool first_tile = true;
        for (int64_t k = a.k_begin + blockIdx.x; k < k_end; k += gridDim.x) {
            if (!(first_tile ? tcw_tile_of(a.tstart, a.T, k, &t, &blk) : tcw_tile_next(a.tstart, a.T, k, &t, &blk))) break;
            first_tile = false;
            unsigned char *tile_sc = a.sc.base + (size_t)(k - a.k_begin) * a.sc.tile_bytes;
            unsigned char *H1s = tile_sc, *H2s = H1s + a.sc.arr_bytes, *Z1s = H2s + a.sc.arr_bytes;
            unsigned char *Xs = Z1s + a.sc.arr_bytes;      // Y = [x, 1, dmu] as fp32 (kernel B splits it)
            // ---- inputs of this thread's sample (part 0 owns the per-sample scalars)
            const int64_t j = (int64_t)blk * 128 + e;
            const bool valid = j < a.cnt[t];
            if (part == 0) {
                int64_t n = 0;
                if (valid) n = a.perm[j];
                // every global load of the tile first (they are independent gathers, mostly HBM misses), THEN the
                // stores: interleaved, the compiler must keep each load behind the previous scratch store (possible
                // aliasing) and the tile start paid O serial DRAM latencies (measured 13-25k clocks per tile)
                float x[O];
#pragma unroll
                for (int i = 0; i < O; ++i) x[i] = valid ? __ldg(a.obs + ((int64_t)t * O + i) * N + n) : 0.0f;
                // Y = [x, 1, dmu] operand of kernel B: sub-block e/8, K-major [XKP rows][8 samples]; the dmu rows are
                // filled in after the objective (epilogue 2a)
                unsigned char *xs = Xs + (size_t)(e >> 3) * (XKP * 32);
#pragma unroll
                for (int i = 0; i < O; ++i) {
                    const float xhi = tf32_hi(x[i]);
                    *reinterpret_cast<float *>(O_hi + core_offset(OKP, e, i)) = xhi;
                    *reinterpret_cast<float *>(O_lo + core_offset(OKP, e, i)) = x[i] - xhi;
                    *reinterpret_cast<float *>(xs + core_offset(8, i, e & 7)) = x[i];
                }
#pragma unroll
                for (int i = O; i < XKP; ++i)
                    *reinterpret_cast<float *>(xs + core_offset(8, i, e & 7)) = (i == O && valid) ? 1.0f : 0.0f;
            }
            if (part == 0) fence_proxy_async();       // only these threads wrote the shared-memory obs operand
            tc_fence_before();
            named_arrive(TCW_BAR_L1, CNT_ALL);
            mbar_wait(&bar_d, ph_d);
            ph_d ^= 1u;
            tc_fence_after();
            // ---- epilogue 1: H1 = act(D) (bias folded); scratch H1 hi/lo; act'(H1) mask; A operand
            // (`deferred` is warp-uniform; the two variants are separate straight-line loops -- with the branch inside
            // the unrolled body ptxas kept both paths' values alive and spilled the tile to local memory)
            uint32_t m1[NCH];
            auto epi1 = [&](auto tm_tag) {
                constexpr bool TM = decltype(tm_tag)::value;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    uint32_t m = 0;
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        float z[16];
                        tmem_ld16(my_tm + TM_D + (uint32_t)(c0 + ch * 32 + hh * 16), z);
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) {
                            z[jj] = valid ? act_fwd(z[jj], act_kind) : 0.0f;   // padding rows contribute nothing
                            m |= (z[jj] > 0.0f ? 1u : 0u) << (hh * 16 + jj);
                        }
                        tcw_store16<W>(H1s, e, (c0 >> 5) + ch, hh, z);
                        if (TM)
                            tcw_tm16(z, my_tm + TM_AHI + acol0 + (uint32_t)(ch * 32 + hh * 16),
                                     my_tm + TM_ALO + acol0 + (uint32_t)(ch * 32 + hh * 16));
                    }
                    m1[ch] = m;
                }
            };
            if (deferred) epi1(FalseTag{});
            else epi1(TrueTag{});
            finish_A(H1s, false);
            // the per-sample scalars of the objective (action, advantage / regression target, old log-prob): gathered
            // HERE, in the shadow of the forward GEMM, so that they do not occupy registers during epilogue 1
            float av[A], adv = 0.f, olp = 0.f, lr = 0.f;
            int64_t n_own = 0;
#pragma unroll
            for (int jj = 0; jj < A; ++jj) av[jj] = 0.0f;
            if (part == 0 && valid) {
                const int64_t n = a.perm[j];
                n_own = n;
                if (a.target != nullptr) {
                    adv = __ldg(a.target + (int64_t)t * N + n);       // the regression target rides in `adv`
                } else if (a.forward_only) {
                    if (a.act != nullptr) {
#pragma unroll
                        for (int jj = 0; jj < A; ++jj) av[jj] = __ldg(a.act + ((int64_t)t * A + jj) * N + n);
                    }
                } else {
#pragma unroll
                    for (int jj = 0; jj < A; ++jj) av[jj] = __ldg(a.act + ((int64_t)t * A + jj) * N + n);
                    adv = __ldg(a.adv + (int64_t)t * N + n);
                    olp = __ldg(a.oldlp + (int64_t)t * N + n);
                    if (REF) lr = __ldg(a.reflp + (int64_t)t * N + n);
                }
            }
            mbar_wait(&bar_d, ph_d);
            ph_d ^= 1u;
            tc_fence_after();
            // ---- epilogue 2a: H2 = act(D + b1), partial output-layer dot products
            {
                float pm[A];
#pragma unroll
                for (int jj = 0; jj < A; ++jj) pm[jj] = 0.0f;
#pragma unroll
                for (int c16 = 0; c16 < 2 * NCH; ++c16) {
                    float z[16];
                    tmem_ld16(my_tm + TM_D + (uint32_t)(c0 + c16 * 16), z);
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) {
                        const float h2 = act_fwd(z[jj] + b1[c16 * 16 + jj], act_kind);
#pragma unroll
                        for (int o = 0; o < A; ++o) pm[o] = fmaf(h2, wo[o * W + c16 * 16 + jj], pm[o]);
                    }
                }
#pragma unroll
                for (int jj = 0; jj < A; ++jj) muS[part][jj][e] = pm[jj];
            }
            named_sync(q + 1, NP * 32);
            if (part == 0) {
                float mu[A], dmu[A];
#pragma unroll
                for (int jj = 0; jj < A; ++jj) {
                    float m = bo[jj];
#pragma unroll
                    for (int p = 0; p < NP; ++p) m += muS[p][jj][e];
                    mu[jj] = m;
                    dmu[jj] = 0.0f;
                }
                if (a.forward_only) {
                    if (valid) {
                        if (a.out_mu) {
#pragma unroll
                            for (int jj = 0; jj < A; ++jj) a.out_mu[((int64_t)t * A + jj) * N + n_own] = mu[jj];
                        }
                        if (a.out_logp) {
                            float m2 = 0.0f;
#pragma unroll
                            for (int jj = 0; jj < A; ++jj) {
                                const float zz = (av[jj] - mu[jj]) * a.inv_sd[jj];
                                m2 += zz * zz;
                            }
                            a.out_logp[(int64_t)t * N + n_own] = -0.5f * m2 - a.log_norm;
                        }
                    }
                } else if (valid && a.target != nullptr) {
                    const float err = mu[0] - adv;                   // MSELoss(V, target), ppo.py:168-169
                    statS[0][e] += (double)err * err;
                    statS[1][e] += 1.0;
                    dmu[0] = 2.0f * a.scale * err;
                    c_bo[0] += dmu[0];
                } else if (valid) {
                    float m2 = 0.0f;
#pragma unroll
                    for (int jj = 0; jj < A; ++jj) {
                        const float zz = (av[jj] - mu[jj]) * a.inv_sd[jj];
                        m2 += zz * zz;
                    }
                    const float lp = -0.5f * m2 - a.log_norm;
                    const float ratio = expf(lp - olp);
                    const float lo = 1.0f - a.eps_clip, hi = 1.0f + a.eps_clip;
                    const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, lo), hi) * adv;
                    const bool in_range = ratio >= lo && ratio <= hi;
                    float g;
                    if (s1 < s2) g = adv;
                    else if (s1 > s2) g = in_range ? adv : 0.0f;
                    else g = 0.5f * (adv + (in_range ? adv : 0.0f));
                    float dlp = a.scale * g * ratio;
                    float eo = 0.0f;
                    if (a.kl_scale != 0.0f) {
                        eo = expf(olp);
                        dlp -= a.kl_scale * eo;
                    }
                    if (REF) {                      // k3 KL to the reference policy
                        const float u = lr - lp, em = expm1f(u);
                        const float dkl = em - u;
                        dlp += a.ref_coef * em;
                        statS[0][e] -= (double)a.ref_coef * dkl;
                        statS[NS - 1][e] += dkl;
                    }
#pragma unroll
                    for (int jj = 0; jj < A; ++jj) dmu[jj] = dlp * (av[jj] - mu[jj]) * a.inv_var[jj];
                    statS[0][e] += (double)fminf(s1, s2) * a.scale + (double)a.kl_scale * eo * (olp - lp);
                    statS[1][e] += 1.0; statS[2][e] += ratio; statS[3][e] += in_range ? 0.0 : 1.0;
#pragma unroll
                    for (int jj = 0; jj < A; ++jj) c_bo[jj] += dmu[jj];
                }
#pragma unroll
                for (int jj = 0; jj < A; ++jj) dmuS[jj][e] = dmu[jj];
                if (!a.forward_only) {
                    // dmu rows of Y (kernel B rebuilds dZ2 from them and accumulates dWo = sum dmu H2)
                    unsigned char *xs = Xs + (size_t)(e >> 3) * (XKP * 32);
#pragma unroll
                    for (int jj = 0; jj < A; ++jj)
                        *reinterpret_cast<float *>(xs + core_offset(8, O + 1 + jj, e & 7)) = dmu[jj];
                }
            }
            if (a.forward_only) {           // CTA-uniform: the next tile's L1 GEMM may overwrite D once everybody read it
                tc_fence_before();
                continue;
            }
            named_sync(q + 1, NP * 32);
            // ---- epilogue 2b: H2 -> scratch (kernel B: dWo, and dZ2 rebuilt from it); dZ2 = (Wo^T dmu) * act'(H2) -> A operand
            {
#pragma unroll
                for (int jj = 0; jj < A; ++jj) dmu_own[jj] = dmuS[jj][e];
                auto epi2b = [&](auto tm_tag) {
                    constexpr bool TM = decltype(tm_tag)::value;
#pragma unroll
                    for (int c16 = 0; c16 < 2 * NCH; ++c16) {
                        float z[16];
                        tmem_ld16(my_tm + TM_D + (uint32_t)(c0 + c16 * 16), z);
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) z[jj] = act_fwd(z[jj] + b1[c16 * 16 + jj], act_kind);
                        tcw_store16<W>(H2s, e, (c0 >> 5) + (c16 >> 1), c16 & 1, z);
                        if (TM) {
#pragma unroll
                            for (int jj = 0; jj < 16; ++jj) z[jj] = tcw_dz2<A>(z[jj], dmu_own, wo + c16 * 16 + jj, W, act_kind);
                            tcw_tm16(z, my_tm + TM_AHI + acol0 + (uint32_t)(c16 * 16), my_tm + TM_ALO + acol0 + (uint32_t)(c16 * 16));
                        }
                    }
                };
                if (deferred) epi2b(FalseTag{});
                else epi2b(TrueTag{});
            }
            finish_A(H2s, true);
            mbar_wait(&bar_d, ph_d);
            ph_d ^= 1u;
            tc_fence_after();
            // ---- epilogue 3: dZ1 = D * act'(H1) -> scratch (kernel B turns it into dW0 / db0)
#pragma unroll
            for (int c16 = 0; c16 < 2 * NCH; ++c16) {
                const int ch = c16 >> 1, hh = c16 & 1;
                float z[16];
                tmem_ld16(my_tm + TM_D + (uint32_t)(c0 + c16 * 16), z);
                if (RELU) {
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) z[jj] = ((m1[ch] >> (hh * 16 + jj)) & 1u) ? z[jj] : 0.0f;
                } else {
                    // act'(H1) from the H1 this thread stored to the scratch
                    const int r = e & 7;
                    const unsigned char *ph = H1s + (size_t)(e >> 3) * (W / 32 * 1024) + (size_t)((c0 >> 5) + ch) * 1024 + (size_t)r * 128;
#pragma unroll
                    for (int c8 = 0; c8 < 2; ++c8) {
                        float hv[8];
                        ldg256(ph + (uint32_t)(((hh * 2 + c8) ^ (r & 3)) << 5), hv);
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj) z[8 * c8 + jj] *= act_bwd_from_out(hv[jj], act_kind);
                    }
                }
                tcw_store16<W>(Z1s, e, (c0 >> 5) + ch, hh, z);
            }
            tc_fence_before();
        }
        if (!a.forward_only) {
        // ---- this CTA's butterfly partials and statistics into its private gradient copy (accumulated)
        float *gp = a.gpart + (int64_t)blockIdx.x * a.lay.n_params;
        const int64_t f2 = a.lay.flat_w[2];
        {
            double v[NS];
#pragma unroll
            for (int kq = 0; kq < NS; ++kq) v[kq] = part == 0 ? statS[kq][e] : 0.0;
#pragma unroll
            for (int kq = 0; kq < NS; ++kq) {
                for (int off = 16; off > 0; off >>= 1) v[kq] += __shfl_down_sync(0xffffffffu, v[kq], off);
                if (lane == 0) sred[kq][warp] = v[kq];
            }
            asm volatile("bar.sync 8, %0;" ::"n"(NCT) : "memory");
            if (threadIdx.x < NS && a.spart) {
                double tt = 0.0;
                for (int w = 0; w < NP * 4; ++w) tt += sred[threadIdx.x][w];
                a.spart[(int64_t)blockIdx.x * TG_SPART_LD + threadIdx.x] += tt;
            }
            asm volatile("bar.sync 8, %0;" ::"n"(NCT) : "memory");
#pragma unroll
            for (int jj = 0; jj < A; ++jj) {
                float tt = c_bo[jj];
                for (int off = 16; off > 0; off >>= 1) tt += __shfl_down_sync(0xffffffffu, tt, off);
                if (lane == 0) sred[0][warp] = (double)tt;
                asm volatile("bar.sync 8, %0;" ::"n"(NCT) : "memory");
                if (threadIdx.x == 0) {
                    float tot = 0.0f;
                    for (int w = 0; w < NP * 4; ++w) tot += (float)sred[0][w];
                    gp[f2 + (int64_t)A * W + jj] += tot;
                }
                asm volatile("bar.sync 8, %0;" ::"n"(NCT) : "memory");
            }
        }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// ============================================================================
// kernel B: split-K weight-gradient GEMMs streamed from the scratch
//   one 8-sample sub-block travels through TWO shared-memory rings:
//     raw ring     (NR slots, filled by TMA):        H2 (this half: 4 column blocks) | dZ1 (this half) | H1 (all) | Yh | Yl
//                  -- the fp32 rows of dZ1 and H1 stay there and ARE the hi operands; H2 is read by the converters only
//     derived ring (NL slots, filled by converters): Z2h, Z2l (dZ2 rebuilt from H2 and dmu) | Z1l | H1l
//   db1 = sum_s dZ2 and dWo = sum_s dmu H2 are column sums with 1 / A outputs per column: the converter thread that
//   rebuilds four dZ2 values accumulates them (and dmu x H2) in registers on the FP32 pipe -- as tcgen05 GEMMs against
//   Y they cost 5 of the 11 MMAs of a sub-block and 40 % of its operand reads for 3 % of its MACs.
//   A raw slot is busy from the TMA issue to the end of its MMAs (HBM latency + conversion + tensor time); a derived slot
//   only from the conversion on.  Two rings put NR = 8 sub-blocks of loads in flight per SM at W = 256 where one ring of
//   whole stages had room for 5 (-16 % per launch); with the register column sums below the kernel reads HBM at 76 % of
//   the measured peak, tensor pipe 41 %, issue slots 42 % (profiles/README_r2.md).
// ============================================================================
// NCV converter warps (0 .. NCV-1); warp NCV = TMA producer, warp NCV+1 = MMA issuer.
// TRUNC: the fp32 rows stay in place as the "hi" operand -- the tensor core reads only the top 19 bits of a tf32
// operand, i.e. it uses trunc(x) -- and the converter writes only lo = x - trunc(x) (one store and four cvt fewer per
// float4 than the round-to-nearest split, whose hi has to be written back).
// Geometry of the two rings for one instance.  DO_W1: dW1 (+ db1, dWo in registers); DO_W0: [dW0 | db0].  W = 128 runs both in
// one launch; at W = 256 the full dW1 accumulator [256 x 256] fills the 512 TMEM columns, so [dW0 | db0] is a second, light
// launch (it reads only dZ1 and Y) -- and H1 is read and split ONCE per sample instead of once per 128-row half (r2: the two
// half launches of the previous design read H1 twice and re-split it).
template <int O, int A, int W, bool DO_W1, bool DO_W0> struct TcwBRings {
    static constexpr int XKP = (O + 1 + A + 7) / 8 * 8;   // rows of Y = [x, 1, dmu, 0..]
    static constexpr uint32_t HB = W / 32 * 1024, XB = XKP * 32;        // bytes per piece: all W columns of 8 samples; Y
    // raw slot (TMA):            H2 | dZ1 | H1 | Y      (pieces of the instance only)
    static constexpr uint32_t R_H2 = 0, R_Z1 = DO_W1 ? HB : 0, R_H1 = R_Z1 + (DO_W0 ? HB : 0), R_X = R_H1 + (DO_W1 ? HB : 0);
    static constexpr uint32_t RAW = R_X + XB, RAW_AL = (RAW + 1023) / 1024 * 1024;
    // derived slot (converters): Z2h | Z2l | Z1l | H1l | Yl
    static constexpr uint32_t D_Z2H = 0, D_Z2L = HB, D_Z1L = DO_W1 ? 2 * HB : 0, D_H1L = D_Z1L + (DO_W0 ? HB : 0);
    static constexpr uint32_t D_XL = D_H1L + (DO_W1 ? HB : 0);
    static constexpr uint32_t DER = (D_XL + (DO_W0 ? XB : 0) + 1023) / 1024 * 1024;
    // lo part of the plain item at raw byte b (dZ1, H1, Y) sits at derived byte LO_SHIFT + b
    static constexpr uint32_t LO_SHIFT = DO_W1 ? HB : 0;
    static_assert(D_Z1L == LO_SHIFT + R_Z1 || !DO_W0, "layout");
    static_assert(D_H1L == LO_SHIFT + R_H1 || !DO_W1, "layout");
    static_assert(D_XL == LO_SHIFT + R_X, "layout");
    static constexpr int NL = 3;
    static constexpr int NR_FIT = (int)((220u * 1024u - NL * DER) / RAW_AL);
    static constexpr int NR = NR_FIT > 12 ? 12 : NR_FIT;
    static constexpr size_t BYTES = (size_t)NR * RAW_AL + (size_t)NL * DER;
};

template <int O, int A, int W, int NCV, bool TRUNC, bool DO_W1, bool DO_W0>
__global__ void __launch_bounds__((NCV + 2) * 32, 1) update_tcw_wgrad_kernel(const __grid_constant__ TcwArgs a) {
    using RG = TcwBRings<O, A, W, DO_W1, DO_W0>;
    constexpr int NGRP = 2, MB = W / 128;            // converter groups (sub-blocks g, g + 2, ...); 128-row blocks of the outputs
    static_assert(NCV % NGRP == 0, "converter groups");
    static_assert(DO_W1 || DO_W0, "nothing to do");
    constexpr int GT = NCV / NGRP * 32;              // converter threads per group
    constexpr uint32_t ZB = 4 * 1024, HB = RG::HB, XB = RG::XB, RAW_AL = RG::RAW_AL, DER = RG::DER;
    constexpr int NR = RG::NR, NL = RG::NL;
    static_assert(NR >= 4, "raw ring");
    constexpr uint32_t R_Z1 = RG::R_Z1, R_H1 = RG::R_H1, R_X = RG::R_X;
    constexpr uint32_t D_Z2H = RG::D_Z2H, D_Z2L = RG::D_Z2L, D_Z1L = RG::D_Z1L, D_H1L = RG::D_H1L, D_XL = RG::D_XL;
    constexpr uint32_t TM_DW = 0u, TM_D0 = DO_W1 ? (uint32_t)(MB * W) : 0u;        // D0 block mb at TM_D0 + 32 mb
    static_assert(TM_D0 + (DO_W0 ? 32 * MB : 0) <= 512, "tensor memory");
    constexpr int NF4 = (int)((R_X + (DO_W0 ? XB : 0)) / 16);   // float4 items per sub-block: H2 (-> dZ2, dWo, db1) | dZ1 | H1 | Y
    constexpr int NH2 = DO_W1 ? (int)(HB / 16) : 0;             // the H2 items
    constexpr int NIT = (NF4 + GT - 1) / GT, NH2_IT = DO_W1 ? (NH2 + GT - 1) / GT : 1;
    if (a.k_begin + blockIdx.x >= a.tstart[a.T]) return;      // no live tile for this CTA in this batch (CTA-uniform)
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[NR], empty_bar[NR], conv_bar[NL], der_empty_bar[NL], done_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float WoS[DO_W1 ? A : 1][DO_W1 ? W : 4];    // Wo (dZ2 = (Wo^T dmu) * act'(H2))
    if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
    if (threadIdx.x == 0) {
        for (int i = 0; i < NR; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < NL; ++i) {
            mbar_init(&conv_bar[i], GT);
            mbar_init(&der_empty_bar[i], 1);
        }
        mbar_init(&done_bar, 1);
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_slot, 512);
    if (DO_W1)
        for (int i = threadIdx.x; i < A * W; i += blockDim.x) WoS[i / W][i % W] = a.params[a.lay.flat_w[2] + i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t k_end = a.k_begin + a.k_count;
    bool any = false;
    if (warp == NCV) {
        if (lane == 0) {
            uint32_t rs = 0, rph = 0;
            int t = 0, blk = 0;
            bool first_tile = true;
            for (int64_t k = a.k_begin + blockIdx.x; k < k_end; k += gridDim.x) {
                if (!(first_tile ? tcw_tile_of(a.tstart, a.T, k, &t, &blk) : tcw_tile_next(a.tstart, a.T, k, &t, &blk))) break;
                first_tile = false;
                const unsigned char *tile_sc = a.sc.base + (size_t)(k - a.k_begin) * a.sc.tile_bytes;
                const unsigned char *arr[3];
                for (int i = 0; i < 3; ++i) arr[i] = tile_sc + (size_t)i * a.sc.arr_bytes;
                const unsigned char *Xs = tile_sc + 3 * (size_t)a.sc.arr_bytes;
                for (int sb = 0; sb < 16; ++sb) {
                    mbar_wait(&empty_bar[rs], rph ^ 1u);
                    mbar_expect_tx(&full_bar[rs], RG::RAW);
                    unsigned char *dst = smem_raw + (size_t)rs * RAW_AL;
                    const size_t sbo = (size_t)sb * HB;
                    // the fp32 rows land in the raw slot and stay there as the hi operands
                    if (DO_W1) tma_bulk_g2s(dst, arr[1] + sbo, HB, &full_bar[rs]);                    // H2
                    if (DO_W0) tma_bulk_g2s(dst + R_Z1, arr[2] + sbo, HB, &full_bar[rs]);             // dZ1
                    if (DO_W1) tma_bulk_g2s(dst + R_H1, arr[0] + sbo, HB, &full_bar[rs]);             // H1
                    tma_bulk_g2s(dst + R_X, Xs + (size_t)sb * XB, XB, &full_bar[rs]);                 // Y = [x, 1, dmu]
                    if (++rs == NR) { rs = 0; rph ^= 1u; }
                }
            }
        }
    } else if (warp == NCV + 1) {
        const uint32_t idesc_w = umma_idesc_tf32(128, W, true, true);
        const uint32_t idesc_x = umma_idesc_tf32(128, (O + 1 + 7) / 8 * 8, true, false);   // rows [x, 1] of Y only
        uint32_t rs = 0, ls = 0, lph = 0, first = 1u;
        const uint32_t tm_u = __shfl_sync(0xffffffffu, tmem, 0), smem_base = __shfl_sync(0xffffffffu, smem_u32(smem_raw), 0);
        int t = 0, blk = 0;
        bool first_tile = true;
        for (int64_t k = a.k_begin + blockIdx.x; k < k_end; k += gridDim.x) {
            if (!(first_tile ? tcw_tile_of(a.tstart, a.T, k, &t, &blk) : tcw_tile_next(a.tstart, a.T, k, &t, &blk))) break;
            first_tile = false;
            any = true;
            {
                // the whole warp runs the loop with warp-uniform operands; one elected lane issues (umma_tf32_w)
                for (int sb = 0; sb < 16; ++sb) {
                    mbar_wait(&conv_bar[ls], lph);            // landed AND split by the converter warps
                    tc_fence_after();
                    const uint32_t raw = smem_base + rs * RAW_AL;
                    const uint32_t der = smem_base + NR * RAW_AL + ls * DER;
                    const uint32_t acc0 = first ? 0u : 1u;
                    if (DO_W1) {
                        // dW1[block mb] += dZ2[:, block mb]^T . H1   (A, B MN-major: 8 reduction rows, 32-column blocks 1 KB apart)
                        const uint32_t h1h = raw + R_H1, h1l = der + D_H1L;
#pragma unroll
                        for (int mb = 0; mb < MB; ++mb) {
                            const uint32_t z2h = der + D_Z2H + (uint32_t)mb * ZB, z2l = der + D_Z2L + (uint32_t)mb * ZB;
                            const uint32_t d = tm_u + TM_DW + (uint32_t)(mb * W);
                            umma_tf32_w(d, umma_desc_mn32(z2h, 1024u), umma_desc_mn32(h1h, 1024u), idesc_w, acc0);
                            umma_tf32_w(d, umma_desc_mn32(z2h, 1024u), umma_desc_mn32(h1l, 1024u), idesc_w, 1u);
                            umma_tf32_w(d, umma_desc_mn32(z2l, 1024u), umma_desc_mn32(h1h, 1024u), idesc_w, 1u);
                        }
                    }
                    if (DO_W0) {
                        // [dW0 | db0][block mb] += dZ1[:, block mb]^T . [x, 1]   (B K-major [XKP][8]; the dmu rows of Y are not used)
                        const uint32_t xh = raw + R_X, xl = der + D_XL;
#pragma unroll
                        for (int mb = 0; mb < MB; ++mb) {
                            const uint32_t z1h = raw + R_Z1 + (uint32_t)mb * ZB, z1l = der + D_Z1L + (uint32_t)mb * ZB;
                            const uint32_t d = tm_u + TM_D0 + (uint32_t)(mb * 32);
                            umma_tf32_w(d, umma_desc_mn32(z1h, 1024u), umma_operand_desc(xh, 8, false, 0), idesc_x, acc0);
                            umma_tf32_w(d, umma_desc_mn32(z1h, 1024u), umma_operand_desc(xl, 8, false, 0), idesc_x, 1u);
                            umma_tf32_w(d, umma_desc_mn32(z1l, 1024u), umma_operand_desc(xh, 8, false, 0), idesc_x, 1u);
                        }
                    }
                    first = 0u;
                    umma_commit_w(&empty_bar[rs]);              // both slots are free once these MMAs have read them
                    umma_commit_w(&der_empty_bar[ls]);
                    if (++rs == NR) rs = 0;
                    if (++ls == NL) { ls = 0; lph ^= 1u; }
                }
            }
            __syncwarp();
        }
        if (any) umma_commit_w(&done_bar);
        __syncwarp();
    }
    if (warp < NCV) {
        // ===== converter warps: tf32 lo parts (and dZ2) of every sub-block, in shared memory =====
        const int grp = warp / (NCV / NGRP), tid_g = (int)threadIdx.x - grp * GT;
        uint32_t rs = (uint32_t)grp, rph = 0, ls = (uint32_t)grp, lph = 0;
        int t = 0, blk = 0;
        bool first_tile = true;
        const int act_kind = a.lay.act;
        // db1 and dWo on the FP32 pipe: thread <-> (sample row r, 4 columns) of its H2 items is the same in every
        // sub-block, so the column sums over samples accumulate in registers and are combined over the 8 rows at the end
        float s_db[NH2_IT][4], s_wo[NH2_IT][A][4];
#pragma unroll
        for (int i = 0; i < NH2_IT; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                s_db[i][j] = 0.0f;
#pragma unroll
                for (int o = 0; o < A; ++o) s_wo[i][o][j] = 0.0f;
            }
        for (int64_t k = a.k_begin + blockIdx.x; k < k_end; k += gridDim.x) {
            if (!(first_tile ? tcw_tile_of(a.tstart, a.T, k, &t, &blk) : tcw_tile_next(a.tstart, a.T, k, &t, &blk))) break;
            first_tile = false;
            for (int sb = grp; sb < 16; sb += NGRP) {
                mbar_wait(&full_bar[rs], rph);
                mbar_wait(&der_empty_bar[ls], lph ^ 1u);
                unsigned char *base = smem_raw + (size_t)rs * RAW_AL;
                unsigned char *der = smem_raw + (size_t)NR * RAW_AL + (size_t)ls * DER;
                // a strided walk over the items: every thread starts with its H2 item(s), the expensive ones
#pragma unroll
                for (int it = 0; it < NIT; ++it) {
                    const int f = tid_g + it * GT;
                    if (f >= NF4) break;
                    const uint32_t b = (uint32_t)f * 16u;
                    // the raw pieces are contiguous
                    const float4 v = *reinterpret_cast<const float4 *>(base + b);
                    if (DO_W1 && it < NH2_IT && b < HB) {
                        // four elements of H2: sample row r of the sub-block, columns col .. col+3 (inverse of the MN-major
                        // SW128_32B sub-block layout); dZ2 = (Wo^T dmu) * act'(H2) in kernel A's operation order
                        const int r = (int)((b & 1023u) >> 7);
                        const int col = (int)(b >> 10) * 32 + (int)((((b & 127u) >> 5) ^ (uint32_t)(r & 3)) << 3) + (int)((b & 31u) >> 2);
                        float dmu[A];
#pragma unroll
                        for (int o = 0; o < A; ++o)
                            dmu[o] = *reinterpret_cast<const float *>(base + R_X + core_offset(8, O + 1 + o, r));
                        float4 d, h4, l4;
                        d.x = tcw_dz2<A>(v.x, dmu, &WoS[0][col], W, act_kind);
                        d.y = tcw_dz2<A>(v.y, dmu, &WoS[0][col + 1], W, act_kind);
                        d.z = tcw_dz2<A>(v.z, dmu, &WoS[0][col + 2], W, act_kind);
                        d.w = tcw_dz2<A>(v.w, dmu, &WoS[0][col + 3], W, act_kind);
                        if (TRUNC) {
                            h4.x = tf32_trunc(d.x); h4.y = tf32_trunc(d.y); h4.z = tf32_trunc(d.z); h4.w = tf32_trunc(d.w);
                        } else {
                            h4.x = tf32_hi(d.x); h4.y = tf32_hi(d.y); h4.z = tf32_hi(d.z); h4.w = tf32_hi(d.w);
                        }
                        l4.x = d.x - h4.x; l4.y = d.y - h4.y; l4.z = d.z - h4.z; l4.w = d.w - h4.w;
                        *reinterpret_cast<float4 *>(der + D_Z2H + b) = TRUNC ? d : h4;
                        *reinterpret_cast<float4 *>(der + D_Z2L + b) = l4;
                        const int ii = it < NH2_IT ? it : 0;
                        s_db[ii][0] += d.x; s_db[ii][1] += d.y; s_db[ii][2] += d.z; s_db[ii][3] += d.w;
#pragma unroll
                        for (int o = 0; o < A; ++o) {
                            s_wo[ii][o][0] = fmaf(dmu[o], v.x, s_wo[ii][o][0]);
                            s_wo[ii][o][1] = fmaf(dmu[o], v.y, s_wo[ii][o][1]);
                            s_wo[ii][o][2] = fmaf(dmu[o], v.z, s_wo[ii][o][2]);
                            s_wo[ii][o][3] = fmaf(dmu[o], v.w, s_wo[ii][o][3]);
                        }
                    } else {
                        // dZ1 / H1 / Y: hi stays in place, lo = x - trunc(x) into the derived slot
                        float4 h4, l4;
                        if (TRUNC) {
                            h4.x = tf32_trunc(v.x); h4.y = tf32_trunc(v.y); h4.z = tf32_trunc(v.z); h4.w = tf32_trunc(v.w);
                        } else {
                            h4.x = tf32_hi(v.x); h4.y = tf32_hi(v.y); h4.z = tf32_hi(v.z); h4.w = tf32_hi(v.w);
                            *reinterpret_cast<float4 *>(base + b) = h4;
                        }
                        l4.x = v.x - h4.x; l4.y = v.y - h4.y; l4.z = v.z - h4.z; l4.w = v.w - h4.w;
                        *reinterpret_cast<float4 *>(der + RG::LO_SHIFT + b) = l4;
                    }
                }
                fence_proxy_async();
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&conv_bar[ls])) : "memory");
                rs += NGRP;
                if (rs >= (uint32_t)NR) { rs -= NR; rph ^= 1u; }
                ls += NGRP;
                if (ls >= (uint32_t)NL) { ls -= NL; lph ^= 1u; }
            }
        }
        if (DO_W1 && !first_tile) {
            // this thread's db1 / dWo partials -> table [group][column][sample row][1 + A] in the (now idle) rings
            mbar_wait(&done_bar, 0);                 // every MMA has read its operands
            float *tab = reinterpret_cast<float *>(smem_raw);
#pragma unroll
            for (int ii = 0; ii < NH2_IT; ++ii) {
                const int f = tid_g + ii * GT;
                if (f < NH2) {
                    const uint32_t b = (uint32_t)f * 16u;
                    const int r = (int)((b & 1023u) >> 7);
                    const int col = (int)(b >> 10) * 32 + (int)((((b & 127u) >> 5) ^ (uint32_t)(r & 3)) << 3) + (int)((b & 31u) >> 2);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float *e = tab + (size_t)(((grp * W + col + j) * 8 + r) * (A + 1));
                        e[0] = s_db[ii][j];
#pragma unroll
                        for (int o = 0; o < A; ++o) e[1 + o] = s_wo[ii][o][j];
                    }
                }
            }
        }
    }
    // did this CTA process any tile?  (uniform: its first tile index is live or not)
    {
        int t, blk;
        any = (a.k_begin + blockIdx.x < k_end) && tcw_tile_of(a.tstart, a.T, a.k_begin + blockIdx.x, &t, &blk);
    }
    __syncthreads();
    if (warp < 4 && any) {
        mbar_wait(&done_bar, 0);
        tc_fence_after();
        float *gp = a.gpart + (int64_t)blockIdx.x * a.lay.n_params;
        const int64_t f0 = a.lay.flat_w[0], f1 = a.lay.flat_w[1], f2 = a.lay.flat_w[2];
        const uint32_t my_tm = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
        for (int mb = 0; mb < MB; ++mb) {
            const int row = mb * 128 + warp * 32 + lane;     // out index (dW1) / hidden-1 index (dW0) / hidden-2 index (dWo)
            if (DO_W1) {
                for (int c = 0; c < W; c += 32) {
                    float z[32];
                    tmem_ld32(my_tm + TM_DW + (uint32_t)(mb * W + c), z);
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) gp[f1 + (int64_t)row * W + c + jj] += z[jj];
                }
                // db1 / dWo: the converter threads' partial column sums, fixed order (group, sample row)
                const float *tab = reinterpret_cast<const float *>(smem_raw);
                float acc[A + 1];
#pragma unroll
                for (int q = 0; q <= A; ++q) acc[q] = 0.0f;
                for (int g = 0; g < NGRP; ++g)
                    for (int r = 0; r < 8; ++r) {
                        const float *e = tab + (size_t)(((g * W + row) * 8 + r) * (A + 1));
#pragma unroll
                        for (int q = 0; q <= A; ++q) acc[q] += e[q];
                    }
                gp[f1 + (int64_t)W * W + row] += acc[0];
#pragma unroll
                for (int o = 0; o < A; ++o) gp[f2 + (int64_t)o * W + row] += acc[1 + o];
            }
            if (DO_W0) {
                float z[32];
                tmem_ld32(my_tm + TM_D0 + (uint32_t)(mb * 32), z);
#pragma unroll
                for (int o = 0; o < O; ++o) gp[f0 + (int64_t)row * O + o] += z[o];
                gp[f0 + (int64_t)W * O + row] += z[O];
            }
        }
        tc_fence_before();
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// ============================================================================
// host side
// ============================================================================
template <int O, int A, int W, int NP>
static int launch_tcw_np(const TcwArgs &a0, int grid, int64_t total_upper, int64_t batch_tiles, cudaStream_t st) {
    constexpr int OKP = (O + 1 + 7) / 8 * 8;
    const size_t smemA = (size_t)TCW_STAGES * W * 128 + (size_t)a0.lay.resident * 4 + 2 * (size_t)128 * OKP * 4;
    void (*kA)(const TcwArgs) = a0.reflp ? (a0.lay.act == TG_ACT_RELU ? update_tcw_fwdbwd_kernel<O, A, true, W, NP, true>
                                                                       : update_tcw_fwdbwd_kernel<O, A, false, W, NP, true>)
                                         : (a0.lay.act == TG_ACT_RELU ? update_tcw_fwdbwd_kernel<O, A, true, W, NP, false>
                                                                       : update_tcw_fwdbwd_kernel<O, A, false, W, NP, false>);
    // converter warps of kernel B: measured on B200 (profiles/README_r2.md) 8 / 12 / 16 warps = 293 / 267 / 241 us per
    // launch at W = 256 and 12 <= 16 at W = 128 (22 warps: no further gain, r2p)
    constexpr int NCV = W == 256 ? 16 : 12;
    // W = 128: one launch computes every weight gradient.  W = 256: dW1 (+ db1, dWo) fills tensor memory, [dW0 | db0] follows
    // in a light second launch that reads only dZ1 and Y.
    constexpr bool SPLIT = W == 256;
    void (*kB1)(const TcwArgs) = update_tcw_wgrad_kernel<O, A, W, NCV, true, true, !SPLIT>;
    void (*kB0)(const TcwArgs) = update_tcw_wgrad_kernel<O, A, W, NCV, true, false, true>;
    const size_t smemB1 = TcwBRings<O, A, W, true, !SPLIT>::BYTES, smemB0 = TcwBRings<O, A, W, false, true>::BYTES;
    const int threadsB = (NCV + 2) * 32;
    TG_CUDA(cudaFuncSetAttribute(kA, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemA));
    TG_CUDA(cudaFuncSetAttribute(kB1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemB1));
    if (SPLIT) TG_CUDA(cudaFuncSetAttribute(kB0, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemB0));
    for (int64_t k0 = 0; k0 < total_upper; k0 += batch_tiles) {
        TcwArgs a = a0;
        a.k_begin = k0;
        a.k_count = (total_upper - k0) < batch_tiles ? (total_upper - k0) : batch_tiles;
        kA<<<grid, NP * 128 + 64, smemA, st>>>(a);
        if (!a.forward_only) {
            kB1<<<grid, threadsB, smemB1, st>>>(a);
            if (SPLIT) kB0<<<grid, threadsB, smemB0, st>>>(a);
        }
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// threads per sample in kernel A: 2 at W = 128 (8 + 2 warps, 168 registers); 4 at W = 256 (16 + 2 warps, 96 registers:
// measured 660 us per batch against 1041 us with 2 threads per sample, profiles/README_r2.md)
template <int O, int A, int W>
static int launch_tcw(const TcwArgs &a0, int grid, int64_t total_upper, int64_t batch_tiles, cudaStream_t st) {
    return launch_tcw_np<O, A, W, (W == 256 ? 4 : 2)>(a0, grid, total_upper, batch_tiles, st);
}

// gpart [sm_count][n_params] and spart [sm_count][TG_SPART_LD] must be zeroed by the caller.
int tg_policy_grad_tcw(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                       const float *adv, const float *old_logp, const float *target, const int32_t *len, const float *params,
                       const float *inv_sd, const float *inv_var, float log_norm, float eps_clip, float scale,
                       float kl_scale, float *gpart, double *spart, int grid, cudaStream_t st, float *out_mu,
                       float *out_logp, const float *ref_logp, float ref_coef) {
    TcwArgs a;
    memset(&a, 0, sizeof(a));
    tg_build_tcw_layout(mlp, &a.lay, true);
    const int W = a.lay.W, O = a.lay.O, A = a.lay.A;
    int rc = tg_pack_weights_tcw(ctx, a.lay, params, st);
    if (rc) return rc;
    rc = tg_len_order(ctx, N, T, len, st);
    if (rc) return rc;
    // per-tile scratch; batch = as many tiles as fit the budget (a multiple of the grid)
    a.sc.arr_bytes = (int64_t)16 * (W / 32) * 1024;
    a.sc.x_bytes = (int64_t)16 * ((O + 1 + A + 7) / 8 * 8) * 32;
    a.sc.tile_bytes = 3 * a.sc.arr_bytes + a.sc.x_bytes;
    const int64_t NB = (N + 127) / 128;
    const int64_t total_upper = NB * T;                       // live tiles <= this
    // 4 GB: one batch = ~10,600 tiles at W = 256; per-batch fixed costs (3 launches, weight staging, 290 KB gradient
    // read-modify-write per CTA and launch) fall below 1 %.  TG_TCW_SCRATCH_MB overrides it (tests use a small budget
    // to cover the multi-batch path at small shapes)
    const char *budget_env = getenv("TG_TCW_SCRATCH_MB");
    const int64_t budget = budget_env ? ((int64_t)atoll(budget_env) << 20) : ((int64_t)4 << 30);
    int64_t batch_tiles = budget / a.sc.tile_bytes / grid * grid;
    if (batch_tiles < grid) batch_tiles = grid;
    if (batch_tiles > total_upper) batch_tiles = (total_upper + grid - 1) / grid * grid;
    const size_t tstart_bytes = ((size_t)(T + 1) * 8 + 255) / 256 * 256;
    rc = tg_ctx_grow(ctx, &ctx->scratch, &ctx->scratch_cap, tstart_bytes + (size_t)batch_tiles * a.sc.tile_bytes);
    if (rc) return rc;
    int64_t *tstart = reinterpret_cast<int64_t *>(ctx->scratch);
    a.sc.base = reinterpret_cast<unsigned char *>(ctx->scratch) + tstart_bytes;
    tcw_tstart_kernel<<<1, 32, 0, st>>>(T, ctx->cnt, tstart);
    TG_CUDA(cudaGetLastError());
    a.N = N; a.T = T; a.obs = obs; a.act = act; a.adv = adv; a.oldlp = old_logp; a.target = target; a.reflp = ref_logp;
    a.perm = ctx->perm; a.cnt = ctx->cnt; a.tstart = tstart;
    a.packed = ctx->packed_tc;
    a.params = params;
    for (int j = 0; j < TG_MAX_ACT; ++j) { a.inv_sd[j] = inv_sd ? inv_sd[j] : 1.0f; a.inv_var[j] = inv_var ? inv_var[j] : 1.0f; }
    a.log_norm = log_norm; a.eps_clip = eps_clip; a.scale = scale; a.kl_scale = kl_scale; a.ref_coef = ref_coef;
    a.gpart = gpart; a.spart = spart;
    a.out_mu = out_mu; a.out_logp = out_logp;
    a.forward_only = (out_mu != nullptr || out_logp != nullptr) ? 1 : 0;
#define TCW_CASE(OO, AA)                                                                                  \
    if (O == OO && A == AA)                                                                               \
        return W == 128 ? launch_tcw<OO, AA, 128>(a, grid, total_upper, batch_tiles, st)                  \
                        : launch_tcw<OO, AA, 256>(a, grid, total_upper, batch_tiles, st);
    TCW_CASE(3, 1) TCW_CASE(5, 1) TCW_CASE(10, 2) TCW_CASE(20, 4) TCW_CASE(10, 1) TCW_CASE(20, 1)
#undef TCW_CASE
    tg_set_error("no wide tensor-core update kernel instance for obs %d / act %d", O, A);
    return TG_ERR_UNSUPPORTED;
}

extern "C" int tg_policy_grad_scratch_bytes(const tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t n_tiles,
                                            int64_t *bytes_written, int64_t *bytes_read) {
    TG_REQUIRE(ctx && mlp && bytes_written && bytes_read, TG_ERR_ARG, "tg_policy_grad_scratch_bytes: null argument");
    *bytes_written = *bytes_read = 0;
    if (!tg_update_tcw_shape_built(mlp) || ctx->math_mode == TG_MATH_FP32) return TG_OK;
    TcwLayout L;
    tg_build_tcw_layout(mlp, &L, true);
    const int64_t arr = (int64_t)16 * (L.W / 32) * 1024, xb = (int64_t)16 * ((L.O + 1 + L.A + 7) / 8 * 8) * 32;
    *bytes_written = n_tiles * (3 * arr + xb);                           // kernel A: H1, H2, dZ1, [x,1,dmu], all fp32
    // kernel B: H2, H1, dZ1 once each; [x,1,dmu] once per launch (two launches at W = 256: dW1 | dW0)
    const int64_t halves = L.W / 128;
    *bytes_read = n_tiles * (3 * arr + halves * xb);
    if (halves == 2) *bytes_read += n_tiles * arr;                       // kernel A: K-half-1 threads reload H1 / dZ2 halves
    return TG_OK;
}

bool tg_update_tcw_shape_built(const tg_mlp_cfg *mlp) {
    if (!tg_update_tcw_eligible(mlp)) return false;
    const int O = mlp->dims[0], A = mlp->dims[3];
    return (O == 3 && A == 1) || (O == 5 && A == 1) || (O == 10 && A == 2) || (O == 20 && A == 4) ||
           (O == 10 && A == 1) || (O == 20 && A == 1);         // the last two: critics of the quadrotor envs
}
