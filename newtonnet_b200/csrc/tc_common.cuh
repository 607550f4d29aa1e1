// Helpers shared by the tcgen05 kernels (gemm_tc.cu, gemm_ts.cu, gemm_chain.cu, gemm_tn_tc.cu, message_tc.cu): mbarriers,
// bulk async copies, UMMA descriptors, tcgen05.mma / commit / ld / st, the K-major 128B swizzle, the tf32 hi/lo split, the
// MMA issue of one TS-mode tile, PDL, and the nn_gemm128 prologues / epilogues of the SS- and TS-mode backends.
#pragma once
#include "common.cuh"

namespace tc {

constexpr int TM = 128;                       // rows per tile (UMMA M)
constexpr int KB = 32;                        // K elements per swizzle atom row (128 B)
constexpr uint32_t BLK_BYTES = TM * KB * 4;   // one [128 x 32] fp32 block = 16 KB
constexpr uint32_t STG_BYTES = 32 * 32 * 4;   // per epilogue warp: one 32 x 32 fp32 chunk, XOR-swizzled
constexpr int NKB = 4;                        // K blocks of a 128 x 128 contraction (K = 128)

// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (bits 4-5 = 1), A=B=tf32 (bits 7-9, 10-12
// = 2), both K-major (bits 15,16 = 0), N>>3 at bits 17-22, M>>4 at bits 24-28.
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor), K-major, SWIZZLE_128B:
// start>>4 | LBO(=1, unused for swizzled K-major)<<16 | SBO(1024 B between 8-row groups)>>4 <<32 |
// version=1 <<46 | layout_type=2 <<61
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
// A operand from tensor memory (TS mode): [taddr] = 128 lanes x 8 columns of tf32
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
          "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
          "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// element (row, k) of a [128 x 32] fp32 block in the K-major 128B-swizzled layout: 8-row groups of
// 1024 B, 16-byte chunk index XORed with the row index inside the group (Swizzle<3,4,3>).
__host__ __device__ __forceinline__ uint32_t swz_offset_bytes(int row, int chunk) {
    return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((chunk ^ (row & 7)) << 4));
}
// hi = x rounded to tf32 (low 13 mantissa bits zero, so the tensor core reads it exactly whatever it does
// with those bits); lo = x - hi is exact in fp32 and has at most 12 significant bits.
__device__ __forceinline__ float tf32_hi(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// MMAs of one 128 x 128 accumulator tile at d_tmem in TS mode.  K block kb of A is the hi / lo pair of 32-column groups at
// a_tmem + 64 kb in tensor memory, B the resident image at sB ([hi|lo][kb][16 KB]).  Each K block waits for its producers
// (bar_a_full[kb], parity `phase`) and is handed back to them (bar_a_empty[kb]) when its MMAs retire.
__device__ __forceinline__ void umma_tile_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t sB, uint32_t bar_a_full,
                                             uint32_t bar_a_empty, uint32_t phase) {
    for (int kb = 0; kb < NKB; ++kb) {
        mbar_wait(bar_a_full + 8 * kb, phase);
        tc_fence_after();
        const uint32_t a_hi = a_tmem + kb * 64, a_lo = a_hi + 32;
        const uint32_t b_hi = sB + kb * BLK_BYTES, b_lo = b_hi + NKB * BLK_BYTES;
#pragma unroll
        for (int ks = 0; ks < KB / 8; ++ks) {                  // UMMA_K = 8 tf32 = 8 TMEM columns / 32 bytes
            const uint64_t dbh = make_desc(b_hi + ks * 32), dbl = make_desc(b_lo + ks * 32);
            umma_tf32_ts(d_tmem, a_lo + ks * 8, dbh, (kb | ks) != 0);   // small terms first
            umma_tf32_ts(d_tmem, a_hi + ks * 8, dbl, 1);
            umma_tf32_ts(d_tmem, a_hi + ks * 8, dbh, 1);
        }
        umma_commit(bar_a_empty + 8 * kb);                     // K block's TMEM columns reusable
    }
}

// ---- nn_gemm128 prologues and epilogues (gemm_tc.cu, gemm_ts.cu) ---------------------------------------------------
// Loads are issued raw (so they stay in flight); the prologue is applied when the value is consumed.
template <int PRO>
__device__ __forceinline__ float4 load_a(const nn_gemm_args& a, int grow, int k, int M) {
    if (grow >= M) return f4_zero();
    float4 v = ld4(a.X + (size_t)grow * 128 + k);
    if (PRO == NN_PRO_ROWSCALE3) v = f4_mul(v, ld4(a.aux2 + (size_t)(grow / 3) * 128 + k));
    return v;
}
template <int PRO>
__device__ __forceinline__ float4 apply_prologue(const nn_gemm_args& a, float4 v, int grow, int k, int M) {
    if (PRO == NN_PRO_SILU) { v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w); }
    if (PRO == NN_PRO_SILU_SAVE) {
        // one sigmoid per element serves silu (this product) and silu' (kept for the reverse sweep)
        const float4 s = make_float4(sigmoid_f(v.x), sigmoid_f(v.y), sigmoid_f(v.z), sigmoid_f(v.w));
        if (grow < M)
            st4(a.aux_out + (size_t)grow * 128 + k,
                make_float4(s.x * fmaf(v.x, 1.0f - s.x, 1.0f), s.y * fmaf(v.y, 1.0f - s.y, 1.0f),
                            s.z * fmaf(v.z, 1.0f - s.z, 1.0f), s.w * fmaf(v.w, 1.0f - s.w, 1.0f)));
        v = f4_mul(v, s);
    }
    return v;
}

template <int EPI>
__device__ __forceinline__ float4 epilogue(const nn_gemm_args& a, float4 acc, int grow, int col) {
    if (EPI == NN_EPI_BIAS) {
        if (a.bias) acc = f4_add(acc, ld4(a.bias + col));
    } else if (EPI == NN_EPI_DSILU) {
        float4 p = ld4(a.aux1 + (size_t)grow * 128 + col);
        acc.x *= dsilu_f(p.x); acc.y *= dsilu_f(p.y); acc.z *= dsilu_f(p.z); acc.w *= dsilu_f(p.w);
    } else if (EPI == NN_EPI_ADD) {
        acc = f4_add(acc, ld4(a.aux1 + (size_t)grow * 128 + col));
    } else if (EPI == NN_EPI_EQUIV_BWD) {
        float4 fb = ld4(a.aux1 + (size_t)grow * 128 + col);
        float4 ab = ld4(a.aux2 + (size_t)(grow / 3) * 128 + col);
        float4 g = ld4(a.aux3 + (size_t)grow * 128 + col);
        acc = f4_add(acc, f4_fma(ab, g, fb));
    }
    return acc;
}

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------
// griddepcontrol.launch_dependents: the next kernel in the stream (if it was launched with the programmatic
// stream serialization attribute) may start once every CTA of this grid has passed this point or exited.
// griddepcontrol.wait: blocks until all prerequisite grids have COMPLETED and their memory is visible - the
// dependent kernel may only touch its own constants before it.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename Kernel, typename Args>
inline int launch_pdl(Kernel kernel, int grid, int threads, size_t smem, cudaStream_t s, const Args& args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = nn_pdl_enabled() ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args);
    if (e != cudaSuccess) { nn_set_error("kernel launch failed: %s", cudaGetErrorString(e)); return -2; }
    return 0;
}

}  // namespace tc
