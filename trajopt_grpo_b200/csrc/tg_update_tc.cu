// K3 on the tensor cores: fused clipped-surrogate objective + MLP backward for policies
// O -> 64 -> 64 -> A (two hidden layers of width TC_W; tg_policy_grad routes here under
// TG_MATH_AUTO / TG_MATH_3XTF32).  Persistent CTAs (one per SM) walk tiles of 128 samples
// (one step t x 128 consecutive envs).  8 compute warps + 1 MMA-issuer warp: sample s = TMEM lane s is served by TWO
// threads (warps q and q+4 of lane quadrant q), each owning one 32-column half of every
// 64-wide activation row -- this halves the per-thread register/ALU load of the epilogues
// and gives the scheduler 8 warps to overlap with the tensor-core round trips.
//
// Per tile i (all GEMMs are 3xTF32 tcgen05.mma, fp32 accumulation in TMEM), software-pipelined so that
// the compute warps never wait for the backward GEMM at the end of a tile:
//   P1  FP32 pipe: H1 = act(W0 x + b0); each thread writes its part of the row, hi/lo split, into
//       tensor memory (A operand buffer i%2, tcgen05.st)
//   MMA D_f[128x64] = H1 . W1^T                         (A from TMEM, B = W1 K-major in smem)
//       in its shadow: finish tile i-1 -- tcgen05.ld D_b, dZ1 = D_b * act'(H1), butterfly column sums
//       for db0 / dW0 -- then publish H1 MN-major into bufB (B operand of the weight-gradient GEMM)
//   P3  tcgen05.ld -> H2 = act(D_f + b1); output Linear (partial dot products exchanged through
//       shared memory), log-prob, ratio, clipped surrogate, d/dmu;
//       dZ2 = (Wo^T dmu) * act'(H2) -> tensor memory (A operand) and MN-major into bufC
//   MMA D_b[128x64] = dZ2 . W1                          (A from TMEM, B = W1 MN-major)
//   MMA D_w[64x64] += dZ2^T . H1                        (A = bufC, B = bufB, both MN-major, reduction
//       over the 128 samples; the accumulator stays in tensor memory for ALL tiles of the CTA and
//       is read once at the end: M = 64, row r in lane 32*(r/16) + r%16)
//       meanwhile: butterfly column sums for dWo and db1, prefetch of the next tile's inputs
// Measured and rejected (round 1): the first-layer / bias column sums as extra tcgen05 GEMMs
// (dZ1^T.[x,1], dZ2^T.1 with N = 8): correct, but bufC becomes a serial resource between three GEMMs of
// a tile and every tiny MMA still costs ~32 tensor clocks: 5.6 ms instead of 4.2 ms per update.
// Column sums over samples use a register butterfly (31 shuffles per 32-column half): lane l
// of a warp ends with the warp's sum of its column l; per-warp partials live in registers for
// the whole kernel and are combined once, in a fixed order, at the end.
// Every CTA writes its partial gradient into its private copy (gpart); grad_reduce_kernel
// (tg_update.cu) sums the copies in a fixed order -> deterministic result in flat torch layout.
#include <math.h>

#include "tg_umma.cuh"

struct UpdTcArgs {
    tg_tc_layout lay;
    int64_t N;
    int T;
    const float *obs, *act, *adv, *oldlp;
    const int32_t *len;
    const float *packed;
    float inv_sd[TG_MAX_ACT], inv_var[TG_MAX_ACT], log_norm;
    float eps_clip, scale, kl_scale;
    float *gpart;   // [grid][n_params], zero-initialised
    double *spart;  // [grid][TG_SPART_LD]
    // length order of the rollout (tg_order.cu): sorted position j of step t is env perm[j], live iff j < cnt[t]
    const int32_t *perm, *cnt;
    // GRPO's KL term (REF instances): log-prob under a frozen reference policy and its coefficient beta * scale
    const float *reflp;
    float ref_coef;
};

// butterfly column sums: v[0..32) per lane -> v[0] = sum over the warp's 32 lanes of column `lane`
template <int HALF, int OFF> TG_D void colsum_step(float *v, int lane) {
    const bool up = (lane & OFF) != 0;
#pragma unroll
    for (int j = 0; j < HALF; ++j) {
        const float send = up ? v[j] : v[j + HALF];
        const float keep = up ? v[j + HALF] : v[j];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
    }
}
TG_D float colsum32(float *v, int lane) {
    colsum_step<16, 16>(v, lane);
    colsum_step<8, 8>(v, lane);
    colsum_step<4, 4>(v, lane);
    colsum_step<2, 2>(v, lane);
    colsum_step<1, 1>(v, lane);
    return v[0];
}
// 16 columns per lane: lanes l and l^1 both end up with the sum over the warp's 32 lanes of column l >> 1
TG_D float colsum16(float *v, int lane) {
    colsum_step<8, 16>(v, lane);
    colsum_step<4, 8>(v, lane);
    colsum_step<2, 4>(v, lane);
    colsum_step<1, 2>(v, lane);
    // fixed order (even lane's partial first) so that both lanes hold the bit-identical total
    const float other = __shfl_xor_sync(0xffffffffu, v[0], 1);
    return (lane & 1) ? other + v[0] : v[0] + other;
}
// Two independent column sums interleaved level by level: a butterfly is a chain of 5 dependent shuffle rounds and
// a single one runs at ~0.15 instructions per clock; two in flight hide each other's shuffle latency.
template <int HALF, int OFF> TG_D void colsum_step2(float *v0, float *v1, int lane) {
    const bool up = (lane & OFF) != 0;
#pragma unroll
    for (int j = 0; j < HALF; ++j) {
        const float s0 = up ? v0[j] : v0[j + HALF], k0 = up ? v0[j + HALF] : v0[j];
        const float s1 = up ? v1[j] : v1[j + HALF], k1 = up ? v1[j + HALF] : v1[j];
        const float r0 = __shfl_xor_sync(0xffffffffu, s0, OFF), r1 = __shfl_xor_sync(0xffffffffu, s1, OFF);
        v0[j] = k0 + r0;
        v1[j] = k1 + r1;
    }
}
template <int NC> TG_D void colsumN2(float *v0, float *v1, int lane, float &r0, float &r1) {
    if (NC == 32) {
        colsum_step2<16, 16>(v0, v1, lane);
        colsum_step2<8, 8>(v0, v1, lane);
        colsum_step2<4, 4>(v0, v1, lane);
        colsum_step2<2, 2>(v0, v1, lane);
        colsum_step2<1, 1>(v0, v1, lane);
        r0 = v0[0];
        r1 = v1[0];
    } else {
        r0 = colsum16(v0, lane);
        r1 = colsum16(v1, lane);
    }
}
template <int NC> TG_D float colsumN(float *v, int lane) {
    if (NC == 32) return colsum32(v, lane);
    return colsum16(v, lane);
}

TG_D void split4(const float *v, float4 &hi, float4 &lo) {
    hi.x = tf32_hi(v[0]); hi.y = tf32_hi(v[1]); hi.z = tf32_hi(v[2]); hi.w = tf32_hi(v[3]);
    lo.x = v[0] - hi.x; lo.y = v[1] - hi.y; lo.z = v[2] - hi.z; lo.w = v[3] - hi.w;
}

// named barriers between the 8 compute warps (arrive, non-blocking) and the MMA issuer warp (sync)
#define BAR_FWD 5
#define BAR_BWD 6

// TMEM column map (512 columns allocated)
#define TM_DF 0u     // forward accumulator  [128 x 64]
#define TM_DB 64u    // backward-data accumulator [128 x 64]
#define TM_DW 128u   // dW1 [64 x 64], M = 64 layout, PERSISTENT across the CTA's tiles
#define TM_A0 192u   // A operand buffer 0: hi at +0, lo at +64; buffer 1 at +128

// NPART threads serve one sample: NPART*4 compute warps + the issuer warp (4 threads per sample measured no faster:
// the kernel is bound by its instruction count and phase chain, not by warp parallelism; DESIGN.md K3-TC)
constexpr int NPART = 2;
// REF: with GRPO's KL term to a reference policy (a.reflp).  A template flag, not a branch: the instances without it
// keep their register allocation and spills (the epilogues are at the 168-register cap)
template <int O, int A, bool RELU, bool REF>
__global__ void __launch_bounds__(NPART * 128 + 32, 1) update_tc_kernel(const __grid_constant__ UpdTcArgs a) {
    constexpr int W = TC_W, HW = TC_W / NPART, O4 = (O + 1 + 3) / 4 * 4;
    constexpr int NCW = NPART * 4, NT = NPART * 128 + 32;
    constexpr int NS = REF ? TG_NSTAT : 4;          // statistics this instance produces
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar, bar_a, bar_b, bar_w;
    __shared__ uint32_t tmem_slot;
    __shared__ double sred[NS][NCW];
    __shared__ float muS[NPART][A][128];
    if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
    float *Wsm = reinterpret_cast<float *>(smem_raw);
    unsigned char *bufB_hi = smem_raw + ((size_t)a.lay.total * 4 + 1023) / 1024 * 1024;   // H1, MN-major
    unsigned char *bufB_lo = bufB_hi + 128 * W * 4;
    unsigned char *bufC_hi = bufB_lo + 128 * W * 4;      // dZ2, MN-major
    unsigned char *bufC_lo = bufC_hi + 128 * W * 4;
    stage_weights_tma(Wsm, a.packed, a.lay.total, &wbar);
    if (threadIdx.x == 0) {
        mbar_init(&bar_a, 1);
        mbar_init(&bar_b, 1);
        mbar_init(&bar_w, 1);
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = warp & 3, hf = warp >> 2;        // lane quadrant, column part (0..NPART)
    const int s = q * 32 + lane;                    // sample row of this thread
    const int c0 = hf * HW;                         // first column of this thread's part
    const uint32_t my_tm = tmem + ((uint32_t)(q * 32) << 16);
    const uint32_t idesc_f = umma_idesc_tf32(128, W, false, false);
    const uint32_t idesc_b = umma_idesc_tf32(128, W, false, true);
    const uint32_t idesc_w = umma_idesc_tf32(64, W, true, true);
    const uint32_t w_u = smem_u32(Wsm);
    const uint32_t wf_hi = w_u + (uint32_t)a.lay.whi[1] * 4u, wf_lo = w_u + (uint32_t)a.lay.wlo[1] * 4u;
    const uint32_t wb_hi = w_u + (uint32_t)a.lay.wbhi[1] * 4u, wb_lo = w_u + (uint32_t)a.lay.wblo[1] * 4u;
    const uint32_t B_hi = smem_u32(bufB_hi), B_lo = smem_u32(bufB_lo), C_hi = smem_u32(bufC_hi), C_lo = smem_u32(bufC_lo);
    // this thread's part of a row in the MN-major SW128_32B layout: mn32_offset(128, s, c0 + 4*i)
    const uint32_t mn_row = (uint32_t)(c0 >> 5) * (128u * 128u) + (uint32_t)s * 128u;
    const int cb = (c0 & 31) >> 3;                  // first 32-byte chunk of this thread's columns inside the line
    const int rs = s & 3;
    const float *w1 = Wsm + a.lay.w1, *b1 = Wsm + a.lay.bias[1], *wo = Wsm + a.lay.wo, *bo = Wsm + a.lay.bo;
    const int act_kind = RELU ? TG_ACT_RELU : a.lay.act;

    // per-thread gradient partials that stay on the register butterfly (this warp's sum over its samples)
    float c_wo[A], c_b1 = 0.f, c_b0 = 0.f, c_w0[O], c_bo[A];
#pragma unroll
    for (int j = 0; j < A; ++j) c_wo[j] = c_bo[j] = 0.0f;
#pragma unroll
    for (int o = 0; o < O; ++o) c_w0[o] = 0.0f;
    double s_obj = 0.0, s_cnt = 0.0, s_ratio = 0.0, s_clip = 0.0, s_kl = 0.0;

    const int64_t N = a.N;
    const int64_t NB = (N + 127) / 128;
    const int64_t ntiles = NB * a.T;
    bool have_prev = false;      // a tile has been processed before the current one (CTA-uniform)
    if (warp == NCW) {
        // ===== MMA issuer warp.  The whole warp runs the issue loops with warp-uniform operands and ONE elected lane
        // issues each tcgen05.mma (umma_*_w): issuing from inside `if (lane == 0)` made ptxas move every descriptor
        // and TMEM address from vector to uniform registers through an ELECT / R2UR.BROADCAST waterfall, ~70 clocks
        // per MMA against the 32 clocks a [128x64x8] MMA takes (tg_tmem_probe) -- the issuing thread, not the
        // tensor pipe, bounded the kernel.  Loops are kept rolled (descriptors advance by a constant) so that the
        // uniform register file does not spill.  Tensor-pipe order per tile i:  fwd(i) | bwd(i), wgrad1(i)
        uint32_t buf = 0, first_w = 1u;
        const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
        const uint64_t d_wf_hi = umma_operand_desc(__shfl_sync(0xffffffffu, wf_hi, 0), W, false, 0);
        const uint64_t d_wf_lo = umma_operand_desc(__shfl_sync(0xffffffffu, wf_lo, 0), W, false, 0);
        const uint64_t d_wb_hi = umma_operand_desc(__shfl_sync(0xffffffffu, wb_hi, 0), W, true, 0);
        const uint64_t d_wb_lo = umma_operand_desc(__shfl_sync(0xffffffffu, wb_lo, 0), W, true, 0);
        const uint64_t d_c_hi = umma_operand_desc(__shfl_sync(0xffffffffu, C_hi, 0), 128, true, 0);
        const uint64_t d_c_lo = umma_operand_desc(__shfl_sync(0xffffffffu, C_lo, 0), 128, true, 0);
        const uint64_t d_b_hi = umma_operand_desc(__shfl_sync(0xffffffffu, B_hi, 0), 128, true, 0);
        const uint64_t d_b_lo = umma_operand_desc(__shfl_sync(0xffffffffu, B_lo, 0), 128, true, 0);
        // descriptor address field is in 16-byte units: one K step (8 elements) = 256 B K-major, 1024 B MN-major
        constexpr uint64_t STEP_K = 16, STEP_MN = 64;
        for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            if ((tile % NB) * 128 >= a.cnt[tile / NB]) continue;
            const uint32_t acol = tm + TM_A0 + buf * 128u;
            named_sync(BAR_FWD, NT);
            tc_fence_after();
            {
                uint32_t acc = 0;
#pragma unroll 1
                for (int pass = 0; pass < 3; ++pass) {
                    uint32_t ac = acol + (pass == 2 ? 64u : 0u);
                    uint64_t b = pass == 1 ? d_wf_lo : d_wf_hi;
#pragma unroll 2
                    for (int k = 0; k < W; k += 8) {
                        umma_tf32_ts_w(tm + TM_DF, ac, b, idesc_f, acc);
                        acc = 1u;
                        ac += 8u;
                        b += STEP_K;
                    }
                }
                umma_commit_w(&bar_a);
            }
            __syncwarp();
            named_sync(BAR_BWD, NT);
            tc_fence_after();
            {
                uint32_t acc = 0;
#pragma unroll 1
                for (int pass = 0; pass < 3; ++pass) {
                    uint32_t ac = acol + (pass == 2 ? 64u : 0u);
                    uint64_t b = pass == 1 ? d_wb_lo : d_wb_hi;
#pragma unroll 2
                    for (int k = 0; k < W; k += 8) {
                        umma_tf32_ts_w(tm + TM_DB, ac, b, idesc_b, acc);
                        acc = 1u;
                        ac += 8u;
                        b += STEP_MN;
                    }
                }
                umma_commit_w(&bar_b);
                // dW1 += dZ2^T . H1, accumulated in tensor memory over all of this CTA's tiles
                uint32_t accw = first_w ? 0u : 1u;
#pragma unroll 1
                for (int pass = 0; pass < 3; ++pass) {
                    uint64_t da = pass == 2 ? d_c_lo : d_c_hi;
                    uint64_t db = pass == 1 ? d_b_lo : d_b_hi;
#pragma unroll 2
                    for (int k = 0; k < 128; k += 8) {
                        umma_tf32_w(tm + TM_DW, da, db, idesc_w, accw);
                        accw = 1u;
                        da += STEP_MN;
                        db += STEP_MN;
                    }
                }
                first_w = 0u;
                umma_commit_w(&bar_w);
            }
            __syncwarp();
            have_prev = true;
            buf ^= 1u;
        }
    } else {
    // ===== compute warps =====
    // software prefetch of a tile's per-sample inputs
    float xn[O], an[A], advn = 0.f, olpn = 0.f, lrn = 0.f;
    bool vn = false;
    auto prefetch = [&](int64_t tile) {
        vn = false;
        if (tile < ntiles) {
            const int t = (int)(tile / NB);
            const int64_t j = (tile % NB) * 128 + s;
            vn = j < a.cnt[t];
            if (vn) {
                const int64_t n = a.perm[j];
#pragma unroll
                for (int o = 0; o < O; ++o) xn[o] = a.obs[((int64_t)t * O + o) * N + n];
#pragma unroll
                for (int j2 = 0; j2 < A; ++j2) an[j2] = a.act[((int64_t)t * A + j2) * N + n];
                advn = a.adv[(int64_t)t * N + n];
                olpn = a.oldlp[(int64_t)t * N + n];
                if (REF) lrn = a.reflp[(int64_t)t * N + n];
            }
        }
    };
    uint32_t ph_a = 0, ph_b = 0, ph_w = 0, buf = 0;
    float xp[O];                 // previous tile's inputs and act'(H1) mask: its dZ1 is finished one tile later
    uint32_t m1p = 0;
#pragma unroll
    for (int o = 0; o < O; ++o) xp[o] = 0.0f;
    // finish the PREVIOUS tile's backward: dZ1 = D_b * act'(H1) -> first-layer gradients (register butterflies)
    auto finish_prev = [&]() {
        mbar_wait(&bar_b, ph_b);
        ph_b ^= 1u;
        tc_fence_after();
        float d1[HW];
        tmem_ldN<HW>(my_tm + TM_DB + (uint32_t)c0, d1);
        if (RELU) {
#pragma unroll
            for (int j = 0; j < HW; ++j) d1[j] = ((m1p >> j) & 1u) ? d1[j] : 0.0f;
        } else {
#pragma unroll
            for (int i = 0; i < HW / 4; ++i) {     // bufB still holds the previous tile's H1
                const uint32_t om = mn_row + (uint32_t)((((i >> 1) + cb) ^ rs) << 5) + (uint32_t)(i & 1) * 16u;
                const float4 vh = *reinterpret_cast<const float4 *>(bufB_hi + om);
                const float4 vl = *reinterpret_cast<const float4 *>(bufB_lo + om);
                d1[4 * i] *= act_bwd_from_out(vh.x + vl.x, act_kind);
                d1[4 * i + 1] *= act_bwd_from_out(vh.y + vl.y, act_kind);
                d1[4 * i + 2] *= act_bwd_from_out(vh.z + vl.z, act_kind);
                d1[4 * i + 3] *= act_bwd_from_out(vh.w + vl.w, act_kind);
            }
        }
        // O + 1 column sums (dW0 columns and db0), two at a time
#pragma unroll
        for (int o = 0; o + 1 < O; o += 2) {
            float v0[HW], v1[HW];
#pragma unroll
            for (int e = 0; e < HW; ++e) { v0[e] = d1[e] * xp[o]; v1[e] = d1[e] * xp[o + 1]; }
            float r0, r1;
            colsumN2<HW>(v0, v1, lane, r0, r1);
            c_w0[o] += r0;
            c_w0[o + 1] += r1;
        }
        if (O % 2 == 1) {
            float v0[HW];
#pragma unroll
            for (int e = 0; e < HW; ++e) v0[e] = d1[e] * xp[O - 1];
            float r0, r1;
            colsumN2<HW>(v0, d1, lane, r0, r1);
            c_w0[O - 1] += r0;
            c_b0 += r1;
        } else {
            c_b0 += colsumN<HW>(d1, lane);
        }
        // the previous tile's weight-gradient GEMM has consumed bufB / bufC
        mbar_wait(&bar_w, ph_w);
        ph_w ^= 1u;
    };
    prefetch(blockIdx.x);
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        float x[O], av[A];
        const bool valid = vn;
        const float adv = advn, olp = olpn, lr = lrn;
#pragma unroll
        for (int o = 0; o < O; ++o) x[o] = valid ? xn[o] : 0.0f;
#pragma unroll
        for (int j = 0; j < A; ++j) av[j] = an[j];
        // whole tile is padding (fewer live envs at this step than the tile's first sorted position):
        // CTA-uniform decision from the per-step live count, no barrier needed
        if ((tile % NB) * 128 >= a.cnt[tile / NB]) { prefetch(tile + gridDim.x); continue; }
        const uint32_t my_a = my_tm + TM_A0 + buf * 128u;
        // ---- P1: first Linear on the FP32 pipe, this thread's HW neurons
        float h[HW];
#pragma unroll
        for (int i = 0; i < HW; ++i) {
            float wrow[O4];
#pragma unroll
            for (int k = 0; k < O4; k += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(w1 + (c0 + i) * O4 + k);
                wrow[k] = v.x; wrow[k + 1] = v.y; wrow[k + 2] = v.z; wrow[k + 3] = v.w;
            }
            float acc = wrow[O];
#pragma unroll
            for (int o = 0; o < O; ++o) acc = fmaf(wrow[o], x[o], acc);
            h[i] = act_fwd(acc, act_kind);
        }
        uint32_t m1 = 0;    // act'(H1) as a bit mask (ReLU); other activations re-read H1 from bufB
#pragma unroll
        for (int i = 0; i < HW; ++i) m1 |= (h[i] > 0.0f ? 1u : 0u) << i;
        {
            float hi[HW], lo[HW];
#pragma unroll
            for (int i = 0; i < HW / 4; ++i) {
                float4 h4, l4;
                split4(h + 4 * i, h4, l4);
                hi[4 * i] = h4.x; hi[4 * i + 1] = h4.y; hi[4 * i + 2] = h4.z; hi[4 * i + 3] = h4.w;
                lo[4 * i] = l4.x; lo[4 * i + 1] = l4.y; lo[4 * i + 2] = l4.z; lo[4 * i + 3] = l4.w;
            }
            tmem_stN<HW>(my_a + (uint32_t)c0, hi);
            tmem_stN<HW>(my_a + 64u + (uint32_t)c0, lo);
            tmem_st_wait();
            tc_fence_before();
            named_arrive(BAR_FWD, NT);          // -> issuer warp: forward-GEMM operands are in place
            // in the shadow of the forward GEMM: finish the previous tile's backward, then publish H1 MN-major
            if (have_prev) finish_prev();
#pragma unroll
            for (int i = 0; i < HW / 4; ++i) {
                const uint32_t om = mn_row + (uint32_t)((((i >> 1) + cb) ^ rs) << 5) + (uint32_t)(i & 1) * 16u;
                *reinterpret_cast<float4 *>(bufB_hi + om) = make_float4(hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]);
                *reinterpret_cast<float4 *>(bufB_lo + om) = make_float4(lo[4 * i], lo[4 * i + 1], lo[4 * i + 2], lo[4 * i + 3]);
            }
        }
        mbar_wait(&bar_a, ph_a);
        ph_a ^= 1u;
        tc_fence_after();
        // ---- P3: H2 (this thread's part), output Linear, objective, dZ2
        {
            float z[HW];
            tmem_ldN<HW>(my_tm + TM_DF + (uint32_t)c0, z);
#pragma unroll
            for (int j = 0; j < HW; j += 4) {
                const float4 b4 = *reinterpret_cast<const float4 *>(b1 + c0 + j);
                h[j] = act_fwd(z[j] + b4.x, act_kind);
                h[j + 1] = act_fwd(z[j + 1] + b4.y, act_kind);
                h[j + 2] = act_fwd(z[j + 2] + b4.z, act_kind);
                h[j + 3] = act_fwd(z[j + 3] + b4.w, act_kind);
            }
        }
#pragma unroll
        for (int j = 0; j < A; ++j) {
            float acc = 0.0f;
#pragma unroll
            for (int k = 0; k < HW; k += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(wo + j * W + c0 + k);
                acc = fmaf(h[k], v.x, acc); acc = fmaf(h[k + 1], v.y, acc);
                acc = fmaf(h[k + 2], v.z, acc); acc = fmaf(h[k + 3], v.w, acc);
            }
            muS[hf][j][s] = acc;
        }
        // only the warps that share this lane quadrant exchange data: named barrier
        named_sync(q + 1, NPART * 32);
        float mu[A], dmu[A];
#pragma unroll
        for (int j = 0; j < A; ++j) {
            float m = bo[j];
#pragma unroll
            for (int p = 0; p < NPART; ++p) m += muS[p][j][s];
            mu[j] = m;
            dmu[j] = 0.0f;
        }
        if (valid) {
            float m2 = 0.0f;
#pragma unroll
            for (int j = 0; j < A; ++j) {
                const float z = (av[j] - mu[j]) * a.inv_sd[j];
                m2 += z * z;
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
            float dkl = 0.0f;
            if (REF) {                          // k3 KL to the reference policy
                const float u = lr - lp, em = expm1f(u);
                dkl = em - u;
                dlp += a.ref_coef * em;
            }
#pragma unroll
            for (int j = 0; j < A; ++j) dmu[j] = dlp * (av[j] - mu[j]) * a.inv_var[j];
            if (hf == 0) {       // one of the threads of a sample keeps the statistics
                s_obj += (double)fminf(s1, s2) * a.scale + (double)a.kl_scale * eo * (olp - lp);
                if (REF) {
                    s_obj -= (double)a.ref_coef * dkl;
                    s_kl += dkl;
                }
                s_cnt += 1.0; s_ratio += ratio; s_clip += in_range ? 0.0 : 1.0;
#pragma unroll
                for (int j = 0; j < A; ++j) c_bo[j] += dmu[j];
            }
        }
        float dz[HW];
#pragma unroll
        for (int k = 0; k < HW; k += 4) {
            float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int j = 0; j < A; ++j) {
                const float4 v = *reinterpret_cast<const float4 *>(wo + j * W + c0 + k);
                s4[0] = fmaf(dmu[j], v.x, s4[0]); s4[1] = fmaf(dmu[j], v.y, s4[1]);
                s4[2] = fmaf(dmu[j], v.z, s4[2]); s4[3] = fmaf(dmu[j], v.w, s4[3]);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) dz[k + e] = s4[e] * act_bwd_from_out(h[k + e], act_kind);
        }
        {
            float hi[HW], lo[HW];
#pragma unroll
            for (int i = 0; i < HW / 4; ++i) {
                float4 h4, l4;
                split4(dz + 4 * i, h4, l4);
                hi[4 * i] = h4.x; hi[4 * i + 1] = h4.y; hi[4 * i + 2] = h4.z; hi[4 * i + 3] = h4.w;
                lo[4 * i] = l4.x; lo[4 * i + 1] = l4.y; lo[4 * i + 2] = l4.z; lo[4 * i + 3] = l4.w;
                const uint32_t om = mn_row + (uint32_t)((((i >> 1) + cb) ^ rs) << 5) + (uint32_t)(i & 1) * 16u;
                *reinterpret_cast<float4 *>(bufC_hi + om) = h4;
                *reinterpret_cast<float4 *>(bufC_lo + om) = l4;
            }
            tmem_stN<HW>(my_a + (uint32_t)c0, hi);            // the forward GEMM has consumed H1
            tmem_stN<HW>(my_a + 64u + (uint32_t)c0, lo);
            tmem_st_wait();
        }
        fence_proxy_async();
        tc_fence_before();
        named_arrive(BAR_BWD, NT);          // -> issuer warp: dZ2 (TMEM + bufC) and H1 (bufB) are in place
        // in the shadow of the GEMMs: next tile's inputs, column sums for dWo and db1
        prefetch(tile + gridDim.x);
        {
            float v0[HW];
#pragma unroll
            for (int e = 0; e < HW; ++e) v0[e] = dmu[0] * h[e];
            float r0, r1;
            colsumN2<HW>(v0, dz, lane, r0, r1);
            c_wo[0] += r0;
            c_b1 += r1;
        }
#pragma unroll
        for (int j = 1; j < A; ++j) {
            float v[HW];
#pragma unroll
            for (int e = 0; e < HW; ++e) v[e] = dmu[j] * h[e];
            c_wo[j] += colsumN<HW>(v, lane);
        }
#pragma unroll
        for (int o = 0; o < O; ++o) xp[o] = x[o];
        m1p = m1;
        have_prev = true;
        buf ^= 1u;
    }
    // ---- drain: the last tile's backward
    if (have_prev) finish_prev();
    }   // compute warps
    // ---- write this CTA's partial gradient (private copy, zero-initialised by the host)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    float *gp = a.gpart + (int64_t)blockIdx.x * a.lay.n_params;
    const int64_t f0 = a.lay.flat_w[0], f1 = a.lay.flat_w[1], f2 = a.lay.flat_w[2];
    // tensor-memory accumulators (M = 64: row r lives in lane 32*(r/16) + r%16).  have_prev is false in a CTA
    // that processed no tile: its accumulators were never written and its gradient copy stays zero.
    if (warp < NCW && have_prev) {
        const int r = q * 16 + lane;
        float z[HW];
        tmem_ldN<HW>(my_tm + TM_DW + (uint32_t)c0, z);
        if (lane < 16) {
#pragma unroll
            for (int j = 0; j < HW; ++j) gp[f1 + (int64_t)r * W + c0 + j] = z[j];       // dW1[out r][in c0+j]
        }
    }
    __syncthreads();
    // butterfly partials of the four lane quadrants, added in a fixed order
    for (int qs = 0; qs < 4; ++qs) {
        if (warp < NCW && q == qs && (HW == 32 || (lane & 1) == 0)) {
            const int col = c0 + (HW == 32 ? lane : (lane >> 1));
            gp[f1 + (int64_t)W * W + col] += c_b1;                              // b1
            gp[f0 + (int64_t)W * O + col] += c_b0;                              // b0
#pragma unroll
            for (int o = 0; o < O; ++o) gp[f0 + (int64_t)col * O + o] += c_w0[o];   // W0[col][o]
#pragma unroll
            for (int j = 0; j < A; ++j) gp[f2 + (int64_t)j * W + col] += c_wo[j];   // Wo[j][col]
        }
        __syncthreads();
    }
    // dbo and the statistics: warp shuffle, then a fixed-order sum over the warps
    {
        double v[TG_NSTAT] = {s_obj, s_cnt, s_ratio, s_clip, s_kl};
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
            if (lane == 0 && warp < NCW) sred[k][warp] = v[k];
        }
        __syncthreads();
        if (threadIdx.x < NS && a.spart) {
            double t = 0.0;
            for (int w = 0; w < NCW; ++w) t += sred[threadIdx.x][w];
            a.spart[(int64_t)blockIdx.x * TG_SPART_LD + threadIdx.x] = t;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < A; ++j) {
            float t = c_bo[j];
            for (int off = 16; off > 0; off >>= 1) t += __shfl_down_sync(0xffffffffu, t, off);
            if (lane == 0 && warp < NCW) sred[0][warp] = (double)t;
            __syncthreads();
            if (threadIdx.x == 0) {
                float tot = 0.0f;
                for (int w = 0; w < NCW; ++w) tot += (float)sred[0][w];
                gp[f2 + (int64_t)A * W + j] = tot;
            }
            __syncthreads();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

template <int O, int A, bool REF>
static int launch_update_tc_ref(const UpdTcArgs &a, int grid, size_t smem, cudaStream_t st) {
    void (*kern)(const UpdTcArgs) =
        a.lay.act == TG_ACT_RELU ? update_tc_kernel<O, A, true, REF> : update_tc_kernel<O, A, false, REF>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, NPART * 128 + 32, smem, st>>>(a);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

template <int O, int A>
static int launch_update_tc(const UpdTcArgs &a, int grid, size_t smem, cudaStream_t st) {
    return a.reflp ? launch_update_tc_ref<O, A, true>(a, grid, smem, st) : launch_update_tc_ref<O, A, false>(a, grid, smem, st);
}

bool tg_update_tc_eligible(const tg_mlp_cfg *mlp) {
    if (!tg_tc_eligible(mlp) || mlp->n_layers != 3 || mlp->dims[1] != TC_W) return false;
    const int O = mlp->dims[0], A = mlp->dims[3];
    return (O == 3 && A == 1) || (O == 5 && A == 1) || (O == 10 && A == 2) || (O == 20 && A == 4);
}

int tg_update_tc_grid(const tg_ctx *ctx) { return ctx->sm_count; }

// Launch the tensor-core update kernel.  gpart [grid][n_params] must be zeroed; spart [grid][TG_SPART_LD].
int tg_policy_grad_tc(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                      const float *adv, const float *old_logp, const float *ref_logp, const int32_t *len,
                      const float *params, const float *inv_sd, const float *inv_var, float log_norm, float eps_clip,
                      float scale, float kl_scale, float ref_coef, float *gpart, double *spart, int grid, cudaStream_t st) {
    UpdTcArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_tc_layout(mlp, &a.lay, true);
    if (rc) return rc;
    rc = tg_pack_weights_tc(ctx, a.lay, params, st);
    if (rc) return rc;
    a.N = N; a.T = T; a.obs = obs; a.act = act; a.adv = adv; a.oldlp = old_logp; a.reflp = ref_logp; a.len = len;
    a.packed = ctx->packed_tc;
    for (int j = 0; j < TG_MAX_ACT; ++j) { a.inv_sd[j] = inv_sd[j]; a.inv_var[j] = inv_var[j]; }
    a.log_norm = log_norm; a.eps_clip = eps_clip; a.scale = scale; a.kl_scale = kl_scale; a.ref_coef = ref_coef;
    a.gpart = gpart; a.spart = spart;
    rc = tg_len_order(ctx, N, T, len, st);
    if (rc) return rc;
    a.perm = ctx->perm;
    a.cnt = ctx->cnt;
    const size_t smem = ((size_t)a.lay.total * 4 + 1023) / 1024 * 1024 + 4 * (size_t)128 * TC_W * 4;
    TG_REQUIRE(smem <= (size_t)ctx->smem_optin, TG_ERR_UNSUPPORTED, "tensor-core update needs %zu B of shared memory", smem);
    const int O = a.lay.O, A = a.lay.A;
    if (O == 3 && A == 1) return launch_update_tc<3, 1>(a, grid, smem, st);
    if (O == 5 && A == 1) return launch_update_tc<5, 1>(a, grid, smem, st);
    if (O == 10 && A == 2) return launch_update_tc<10, 2>(a, grid, smem, st);
    if (O == 20 && A == 4) return launch_update_tc<20, 4>(a, grid, smem, st);
    tg_set_error("no tensor-core update instance for obs %d / act %d", O, A);
    return TG_ERR_UNSUPPORTED;
}
