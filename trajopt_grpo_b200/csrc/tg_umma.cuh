// tcgen05 (5th-gen tensor core) helpers for sm_100a: TMEM allocation, shared-memory
// matrix descriptors, kind::tf32 MMA issue, commit, TMEM loads.
//
// Operand layout used everywhere in this engine: the no-swizzle "core matrix" layout.
//   A stored matrix X[R rows][C cols] of fp32 is cut into core matrices of 8 rows x 4 cols
//   (8 x 16 bytes = 128 contiguous bytes, row r of the core at +16*r); cores are ordered
//   row-group major:  offset(r, c) = (r/8)*(C/4)*128 + (c/4)*128 + (r%8)*16 + (c%4)*4.
// The SAME buffer can be handed to the tensor core in two ways (which is why this layout is
// used instead of a swizzled one: for 32-bit operands the swizzled K-major and MN-major
// layouts differ, but the core matrix is common to both):
//   K-major view  (rows = M/N index, cols = reduction index): leading byte offset = 128
//       (next core along K), stride byte offset = (C/4)*128 (next 8-row group); one MMA of
//       kind::tf32 consumes K = 8 elements = 2 cores, i.e. +256 B per K step.
//   MN-major view (rows = reduction index, cols = M/N index): stride byte offset = 128
//       (next core along M/N), leading byte offset = (C/4)*128 (next 8-row group along the
//       reduction); one MMA consumes 8 rows = one row group, i.e. +(C/4)*128 B per K step.
// So an activation tile H[samples][features] is the K-major A operand of the next layer's
// forward GEMM AND the MN-major B operand of that layer's weight-gradient GEMM (reduction
// over samples); a weight W[out][in] is the K-major B operand of the forward GEMM AND the
// MN-major B operand of the backward-data GEMM (reduction over out).
//
// 3xTF32: the tensor core reads only the top 19 bits of each 32-bit operand.  To keep
// fp32-level accuracy every operand x is split as hi = rna_tf32(x) and lo = x - hi (exact
// in fp32, |lo| <= 2^-11 |x|), and D = A_hi*B_hi + A_hi*B_lo + A_lo*B_hi is accumulated in
// the fp32 TMEM accumulator (the dropped lo*lo term is <= 2^-22 relative).  Measured error:
// ~1e-6 of the row scale per 8 accumulation steps (the accumulator truncates), tests/test_gpu_umma.py.
#pragma once
#include "tg_mlp.cuh"

TG_D float tf32_hi(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r & 0xffffe000u);
}
// the value the tensor core uses for a raw fp32 operand of kind::tf32: the low 13 mantissa bits dropped
TG_D float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// byte offset of element (r, c) of a stored [R][C] fp32 matrix in the core-matrix layout
TG_HD uint32_t core_offset(int C, int r, int c) {
    return (uint32_t)(r >> 3) * (uint32_t)(C >> 2) * 128u + (uint32_t)(c >> 2) * 128u + (uint32_t)(r & 7) * 16u +
           (uint32_t)(c & 3) * 4u;
}
// inverse of core_offset: float index `idx` of a stored [R][C] matrix -> (row, col)
TG_HD void core_invert(int C, int64_t idx, int *r, int *c) {
    const uint32_t b = (uint32_t)idx * 4u;
    const uint32_t group = (uint32_t)(C >> 2) * 128u;
    const uint32_t rr = b % group;
    *r = (int)(b / group) * 8 + (int)((rr % 128u) >> 4);
    *c = (int)(rr / 128u) * 4 + (int)((rr & 15u) >> 2);
}

TG_D uint64_t umma_desc_raw(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) /* descriptor version (Blackwell) */;
           /* layout type bits [61,64) = 0: SWIZZLE_NONE */
}
// MN-major operands of 32-bit types have exactly one legal shared-memory layout on sm_100
// (CUTLASS sm100_common.inl: "for mn-major tf32 operands, SW128_32B is the only available smem
// layout"): a stored [R rows = reduction][C cols = M/N] matrix keeps 32 consecutive M/N elements
// of a row in one 128-byte line, lines of consecutive rows 128 B apart, the 32-byte chunk index
// inside a line XOR-ed with (row % 4) (Swizzle<2,5,2>), the next 32 M/N elements R*128 B further:
TG_HD uint32_t mn32_offset(int R, int r, int c) {
    return (uint32_t)(c >> 5) * (uint32_t)R * 128u + (uint32_t)r * 128u + (uint32_t)((((c & 31) >> 3) ^ (r & 3)) << 5) +
           (uint32_t)(c & 7) * 4u;
}
// inverse of mn32_offset: float index `idx` of a stored [R][C] matrix -> (row, col)
TG_HD void mn32_invert(int R, int64_t idx, int *r, int *c) {
    const uint32_t b = (uint32_t)idx * 4u;
    const uint32_t blk = b / ((uint32_t)R * 128u), rr = b % ((uint32_t)R * 128u);
    *r = (int)(rr / 128u);
    *c = (int)blk * 32 + (((int)((rr % 128u) >> 5) ^ (*r & 3)) << 3) + (int)((rr & 31u) >> 2);
}
// layout type 1 = SWIZZLE_128B_BASE32B; LBO = next 32-element M/N block, SBO = next 4-row group
TG_D uint64_t umma_desc_mn32(uint32_t smem_addr, uint32_t mn_block_bytes) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((mn_block_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)(512u >> 4) << 32) | (1ull << 46) | (1ull << 61);
}

// descriptor of K step `k` (k = reduction offset in elements, multiple of 8) of a stored matrix:
//   K-major : [rows = M/N][C cols = reduction] in the core-matrix layout
//   MN-major: [C rows = reduction][cols = M/N] in the SW128_32B layout (C = row count R)
TG_D uint64_t umma_operand_desc(uint32_t base, int C, bool mn_major, int k) {
    if (mn_major) return umma_desc_mn32(base + (uint32_t)k * 128u, (uint32_t)C * 128u);
    const uint32_t group = (uint32_t)(C >> 2) * 128u;     // bytes of one 8-row group
    return umma_desc_raw(base + (uint32_t)(k >> 2) * 128u, /*LBO*/ 128u, /*SBO*/ group);
}

// instruction descriptor: D fp32, A/B tf32, dense; a_mn / b_mn select MN-major operands
TG_HD uint32_t umma_idesc_tf32(int M, int N, bool a_mn = false, bool b_mn = false) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

TG_D void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {   // one full warp; ncols = power of two >= 32
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
TG_D void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// named barriers: bar.arrive does not wait, bar.sync waits until `count` threads have arrived at barrier `id`
TG_D void named_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
TG_D void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
TG_D void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
TG_D void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (UMMA operand reads)
TG_D void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], issued by ONE thread
TG_D void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Warp-uniform issue: the WHOLE warp executes the call with identical arguments and one elected lane issues the
// instruction.  With every operand warp-uniform, ptxas keeps the descriptors in uniform registers and advances
// them with the uniform datapath; issuing from inside `if (lane == 0)` instead costs R2UR moves plus 64-bit vector
// arithmetic per descriptor -- measured ~70 clocks per tcgen05.mma, more than twice the 32 clocks the MMA itself
// takes (tg_tmem_probe), so the issuing thread, not the tensor pipe, was the bottleneck.
TG_D void umma_tf32_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
TG_D void umma_tf32_ts_w(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
TG_D void umma_commit_w(uint64_t *bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
        : "memory");
}

// Same with the A operand read from tensor memory: A[M=128][K] fp32/tf32 lives in TMEM with row m in
// lane m and element k in column (a_col0 + k); one MMA consumes 8 columns.
TG_D void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 32 consecutive columns written from registers: thread i of the warp writes row (lane base + i)
TG_D void tmem_st32(uint32_t taddr, const float v[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
        "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
        "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
        "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
        "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
TG_D void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// arrive on an mbarrier when all previously issued MMAs of this thread have completed
TG_D void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives row (lane base + i)
TG_D void tmem_ld32(uint32_t taddr, float v[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 16-column variants (thread i of the warp <-> row lane base + i, 16 consecutive columns)
TG_D void tmem_st16(uint32_t taddr, const float v[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}
TG_D void tmem_ld16(uint32_t taddr, float v[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
template <int NC> TG_D void tmem_stN(uint32_t taddr, const float *v) {
    if (NC == 32) tmem_st32(taddr, v);
    else tmem_st16(taddr, v);
}
template <int NC> TG_D void tmem_ldN(uint32_t taddr, float *v) {
    if (NC == 32) tmem_ld32(taddr, v);
    else tmem_ld16(taddr, v);
}

// Issue the MMAs of one GEMM with the 3xTF32 split (ONE thread).  Each operand is a stored
// [rows][C] matrix in the core-matrix layout, read K-major or MN-major; K = reduction extent.
//   a_hi/a_lo/b_hi/b_lo: shared-memory byte addresses (u32) of the hi and lo copies.
TG_D void umma_gemm_3xtf32(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, int a_C, bool a_mn, uint32_t b_hi,
                           uint32_t b_lo, int b_C, bool b_mn, int K, uint32_t idesc, bool accumulate_first, int passes) {
    uint32_t acc = accumulate_first ? 1u : 0u;
    for (int pass = 0; pass < passes; ++pass) {
        const uint32_t a = (pass == 2) ? a_lo : a_hi;
        const uint32_t b = (pass == 1) ? b_lo : b_hi;
        for (int k = 0; k < K; k += 8) {
            umma_tf32(tmem_d, umma_operand_desc(a, a_C, a_mn, k), umma_operand_desc(b, b_C, b_mn, k), idesc, acc);
            acc = 1u;
        }
    }
}

// warp-uniform version of umma_gemm_3xtf32 (whole warp calls it, one elected lane issues)
TG_D void umma_gemm_3xtf32_w(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, int a_C, bool a_mn, uint32_t b_hi,
                             uint32_t b_lo, int b_C, bool b_mn, int K, uint32_t idesc, bool accumulate_first, int passes) {
    uint32_t acc = accumulate_first ? 1u : 0u;
    for (int pass = 0; pass < passes; ++pass) {
        const uint32_t a = (pass == 2) ? a_lo : a_hi;
        const uint32_t b = (pass == 1) ? b_lo : b_hi;
        for (int k = 0; k < K; k += 8) {
            umma_tf32_w(tmem_d, umma_operand_desc(a, a_C, a_mn, k), umma_operand_desc(b, b_C, b_mn, k), idesc, acc);
            acc = 1u;
        }
    }
}

