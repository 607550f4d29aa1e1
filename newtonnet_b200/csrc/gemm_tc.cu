// Tensor-core backend of nn_gemm128: Y[M,128] = epi(pro(X)[M,128] @ B[128,128]) on the 5th-generation
// tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM), fp32-faithful through a 3xTF32 split:
//     X @ B  ~=  X_lo @ B_hi + X_hi @ B_lo + X_hi @ B_hi ,   hi = x rounded to tf32 (cvt.rna), lo = x - hi.
// SURVEY.md section 7 measured single-pass TF32 at 1e-3 eV/A force error (fails the 1e-4 bar) and the
// 3-pass split at the fp32 noise floor, hence three MMAs per K step.
//
// Kernel shape (persistent, one CTA per SM, 544 threads):
//   warps 0-7  producers : LDG.128 rows of X (coalesced 128 B lines) -> prologue (SiLU / row scale) ->
//                          hi/lo split -> st.shared into the UMMA K-major 128B-swizzled layout; one
//                          pipeline stage = one 32-wide K block (A_hi + A_lo = 32 KB), 2 stages; four
//                          more K blocks per thread are in flight in registers.
//   warp  16   MMA issuer: bulk-copies the prepared operand image of B (hi + lo, 128 KB) into shared
//                          memory once per CTA (cp.async.bulk + mbarrier), then issues 12 tcgen05.mma
//                          (M128 N128 K8) per stage from one elected lane; tcgen05.commit releases the
//                          stage / publishes the accumulator.
//   warps 8-15 epilogue  : tcgen05.ld the 128x128 fp32 accumulator (TMEM lane = row), apply bias /
//                          SiLU' / residual epilogues, st.global.v4.  Two accumulator buffers (2 x 128
//                          TMEM columns) let the epilogue of tile t overlap the MMAs of tile t+1.
// B stays resident in shared memory for all tiles of the CTA: per tile only X is read and Y written, so
// the kernel is bound by HBM (1 KB per row) rather than by L2 re-reads of the weights.
#include <stdlib.h>
#include "tc_common.cuh"

namespace {

using namespace tc;
constexpr int STAGES = 2;
constexpr uint32_t B_BYTES = 2 * NKB * BLK_BYTES;     // hi + lo image of B = 128 KB
constexpr uint32_t A_STAGE_BYTES = 2 * BLK_BYTES;     // A_hi + A_lo block = 32 KB
constexpr uint32_t BAR_BYTES = 256;
constexpr uint32_t SMEM_BYTES = 1024 + B_BYTES + STAGES * A_STAGE_BYTES + 8 * STG_BYTES + BAR_BYTES;
constexpr int PRODUCER_WARPS = 8, EPI_WARPS = 8;
constexpr int MMA_WARP = PRODUCER_WARPS + EPI_WARPS;
constexpr int PF = 4;                         // producer register prefetch depth in K blocks (one whole tile)
constexpr int THREADS = 32 * (PRODUCER_WARPS + EPI_WARPS + 1);
constexpr uint32_t TMEM_COLS = 256;           // two 128-column fp32 accumulators

template <int PRO, int EPI>
__global__ void __launch_bounds__(THREADS, 1) k_gemm128_tc(nn_gemm_args a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;          // swizzle atoms need 1024 B alignment
    const uint32_t sB = base;                                             // [hi|lo][kb][16 KB]
    const uint32_t sA = base + B_BYTES;                                   // [stage][hi|lo][16 KB]
    const uint32_t sStg = sA + STAGES * A_STAGE_BYTES;                    // [8 epilogue warps][4 KB]
    const uint32_t sBar = sStg + 8 * STG_BYTES;
    const uint32_t bar_b_full = sBar;                                     // 8 bytes each
    const uint32_t bar_a_full = sBar + 8;                                 // [STAGES]
    const uint32_t bar_a_empty = bar_a_full + 8 * STAGES;                 // [STAGES]
    const uint32_t bar_t_full = bar_a_empty + 8 * STAGES;                 // [2]
    const uint32_t bar_t_empty = bar_t_full + 16;                         // [2]
    const uint32_t tmem_slot = bar_t_empty + 16;                          // 4 bytes
    uint8_t* smem_gen = smem_raw + (base - smem_u32(smem_raw));           // generic pointer to `base`

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int M = a.m;
    if (a.m_dev) { long long v = (long long)a.m_dev[0] * a.m_dev_mul; M = v < a.m ? (int)v : a.m; }
    const int n_tiles = (M + TM - 1) / TM;
    const bool has_work = (int)blockIdx.x < n_tiles;

    if (warp == MMA_WARP) {
        if (lane == 0) {
            mbar_init(bar_b_full, 1);
            for (int s = 0; s < STAGES; ++s) { mbar_init(bar_a_full + 8 * s, PRODUCER_WARPS * 32); mbar_init(bar_a_empty + 8 * s, 1); }
            for (int b = 0; b < 2; ++b) { mbar_init(bar_t_full + 8 * b, 1); mbar_init(bar_t_empty + 8 * b, EPI_WARPS * 32); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));

    if (warp < PRODUCER_WARPS) {
        // ===================== producers: X rows -> hi/lo split -> swizzled smem =====================
        // Work items w = (tile, K block); each thread keeps PF items (PF x 4 LDG.128) in flight in
        // registers so ~64 KB of reads per SM are outstanding (HBM latency x bandwidth / 148 SMs).
        const int r4 = lane >> 3, chunk = lane & 7;
        const int my_tiles = has_work ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
        const int n_items = my_tiles * NKB;
        float4 v[PF][4];
        auto issue = [&](int w, float4 (&dst)[4]) {
            const int row0 = ((int)blockIdx.x + (w >> 2) * (int)gridDim.x) * TM, kb = w & 3;
#pragma unroll
            for (int it = 0; it < 4; ++it)
                dst[it] = load_a<PRO>(a, row0 + warp * 16 + it * 4 + r4, kb * KB + chunk * 4, M);
        };
#pragma unroll
        for (int u = 0; u < PF; ++u)
            if (u < n_items) issue(u, v[u]);
        uint32_t stage = 0, phase = 0;
        for (int w0 = 0; w0 < n_items; w0 += PF) {
#pragma unroll
            for (int u = 0; u < PF; ++u) {
                const int w = w0 + u;
                if (w >= n_items) break;
                const int crow0 = ((int)blockIdx.x + (w >> 2) * (int)gridDim.x) * TM, ckb = w & 3;
                mbar_wait(bar_a_empty + 8 * stage, phase ^ 1);
                uint8_t* hi = smem_gen + (sA - base) + stage * A_STAGE_BYTES;
                uint8_t* lo = hi + BLK_BYTES;
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    const int row = warp * 16 + it * 4 + r4;
                    const uint32_t off = swz_offset_bytes(row, chunk);
                    const float4 x = apply_prologue<PRO>(a, v[u][it], crow0 + row, ckb * KB + chunk * 4, M);
                    const float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
                    *reinterpret_cast<float4*>(hi + off) = h;
                    *reinterpret_cast<float4*>(lo + off) = f4_sub(x, h);
                }
                fence_proxy_async();                 // generic-proxy stores -> visible to the tensor core (async proxy)
                mbar_arrive(bar_a_full + 8 * stage);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
                if (w + PF < n_items) issue(w + PF, v[u]);
            }
        }
    } else if (warp == MMA_WARP) {
        // ===================== B load + MMA issue (one elected lane) =====================
        if (lane == 0 && has_work) {
            mbar_expect_tx(bar_b_full, B_BYTES);
            for (int c = 0; c < (int)(B_BYTES / BLK_BYTES); ++c)
                bulk_g2s(sB + c * BLK_BYTES, reinterpret_cast<const uint8_t*>(a.B_img) + (size_t)c * BLK_BYTES, BLK_BYTES, bar_b_full);
            mbar_wait(bar_b_full, 0);
            uint32_t stage = 0, phase = 0, it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(bar_t_empty + 8 * buf, acc_phase ^ 1);          // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * 128;
                for (int kb = 0; kb < NKB; ++kb) {
                    mbar_wait(bar_a_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t a_hi = sA + stage * A_STAGE_BYTES, a_lo = a_hi + BLK_BYTES;
                    const uint32_t b_hi = sB + kb * BLK_BYTES, b_lo = b_hi + NKB * BLK_BYTES;
#pragma unroll
                    for (int ks = 0; ks < KB / 8; ++ks) {                  // UMMA_K = 8 tf32 = 32 bytes
                        const uint64_t dah = make_desc(a_hi + ks * 32), dal = make_desc(a_lo + ks * 32);
                        const uint64_t dbh = make_desc(b_hi + ks * 32), dbl = make_desc(b_lo + ks * 32);
                        umma_tf32(d_tmem, dal, dbh, (kb | ks) != 0);       // small terms first
                        umma_tf32(d_tmem, dah, dbl, 1);
                        umma_tf32(d_tmem, dah, dbh, 1);
                    }
                    umma_commit(bar_a_empty + 8 * stage);                  // stage reusable once these MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(bar_t_full + 8 * buf);                         // accumulator complete
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue: TMEM -> registers -> smem transpose -> global =====================
        // 8 warps: TMEM lane quarter q = warp % 4 (hardware restriction), column half = (warp - 8) / 4.
        // tcgen05.ld hands every lane one accumulator ROW; storing that straight to global memory would
        // touch 32 cache lines per instruction.  Each 32 x 32 chunk is therefore transposed through a
        // 4 KB XOR-swizzled staging buffer (conflict-free both ways) so that 8 lanes cover one 128 B row
        // segment: 4 full lines per LDG/STG.  The residual / activation operand (aux1) is read in that
        // coalesced layout too and prefetched one chunk ahead, before the accumulator is awaited.
        const int q = warp & 3, ew = warp - PRODUCER_WARPS, half = ew >> 2;
        const int r4 = lane >> 3, c8 = lane & 7;
        constexpr bool kAux1 = (EPI == NN_EPI_DSILU || EPI == NN_EPI_ADD || EPI == NN_EPI_MUL);
        uint8_t* stg = smem_gen + (sStg - base) + ew * STG_BYTES;
        uint32_t it = 0;
        float4 ax[8];
        auto prefetch = [&](int tile, int c0) {
            if (!kAux1) return;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int grow = tile * TM + q * 32 + k * 4 + r4;
                if (grow < M) ax[k] = ld4(a.aux1 + (size_t)grow * 128 + c0 + 4 * c8);
            }
        };
        if (has_work) prefetch(blockIdx.x, half * 64);
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
            mbar_wait(bar_t_full + 8 * buf, acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * 128;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int c0 = half * 64 + c * 32;
                uint32_t v[32];
                tmem_ld32(taddr + c0, v);
                tmem_ld_wait();
                if (c == 1) {                       // accumulator fully read: hand the buffer back early
                    tc_fence_before();
                    mbar_arrive(bar_t_empty + 8 * buf);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j)         // row = lane, 16-byte chunk j -> physical chunk j ^ (lane & 7)
                    *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                        make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                    __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                __syncwarp();
                float4 cur[8];
                if (kAux1) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) cur[k] = ax[k];
                    if (c == 0) prefetch(tile, c0 + 32);
                    else if (tile + (int)gridDim.x < n_tiles) prefetch(tile + gridDim.x, half * 64);
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int row = k * 4 + r4;
                    const int grow = tile * TM + q * 32 + row;
                    float4 acc = *reinterpret_cast<const float4*>(stg + row * 128 + ((c8 ^ (row & 7)) << 4));
                    if (grow < M) {
                        const int col = c0 + 4 * c8;
                        if (EPI == NN_EPI_DSILU) {
                            const float4 p = cur[k];
                            acc.x *= dsilu_f(p.x); acc.y *= dsilu_f(p.y); acc.z *= dsilu_f(p.z); acc.w *= dsilu_f(p.w);
                        } else if (EPI == NN_EPI_ADD) {
                            acc = f4_add(acc, cur[k]);
                        } else if (EPI == NN_EPI_MUL) {
                            acc = f4_mul(acc, cur[k]);
                        } else {
                            acc = epilogue<EPI>(a, acc, grow, col);
                        }
                        st4(a.Y + (size_t)grow * 128 + col, acc);
                    }
                }
                __syncwarp();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// B [K=128][N=128] row-major  ->  image[hi|lo][kb][n][swizzled 16 B chunks] of B^T (operand rows = n)
__global__ void k_prepare_b(const float* __restrict__ B, float* __restrict__ img) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 128 * 128) return;
    int n = t >> 7, k = t & 127;
    float x = B[(size_t)k * 128 + n];
    float hi = tf32_hi(x);
    int kb = k >> 5, chunk = (k & 31) >> 2, e = k & 3;
    uint32_t off = (uint32_t)kb * BLK_BYTES + swz_offset_bytes(n, chunk) + e * 4;
    img[off / 4] = hi;
    img[(NKB * BLK_BYTES + off) / 4] = x - hi;
}

// the same for up to 64 matrices in one launch (blockIdx.y = matrix); transposed[i] != 0: the operand is src^T, i.e.
// B[k][n] = src[n][k] (a weight used in its other orientation) - no transposed copy has to be materialised
struct PrepBatch { const float* src[64]; float* img[64]; int transposed[64]; };
__global__ void k_prepare_b_batch(PrepBatch p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 128 * 128) return;
    const float* B = p.src[blockIdx.y];
    float* img = p.img[blockIdx.y];
    const int n = t >> 7, k = t & 127;
    const float x = p.transposed[blockIdx.y] ? B[(size_t)n * 128 + k] : B[(size_t)k * 128 + n];
    const float hi = tf32_hi(x);
    const int kb = k >> 5, chunk = (k & 31) >> 2, e = k & 3;
    const uint32_t off = (uint32_t)kb * BLK_BYTES + swz_offset_bytes(n, chunk) + e * 4;
    img[off / 4] = hi;
    img[(NKB * BLK_BYTES + off) / 4] = x - hi;
}

bool g_attr_set[4][5] = {};

template <int PRO, int EPI>
int launch(const nn_gemm_args& a, cudaStream_t s) {
    if (!g_attr_set[PRO][EPI]) {
        cudaError_t e = cudaFuncSetAttribute(k_gemm128_tc<PRO, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
        if (e != cudaSuccess) { nn_set_error("nn_gemm128(tc): cannot set %u B dynamic smem: %s", SMEM_BYTES, cudaGetErrorString(e)); return -2; }
        g_attr_set[PRO][EPI] = true;
    }
    const int tiles = nn_ceil_div(a.m, TM), sms = nn_num_sms();
    const int grid = tiles < sms ? tiles : sms;
    k_gemm128_tc<PRO, EPI><<<grid, THREADS, SMEM_BYTES, s>>>(a); NN_LAUNCHED(1);
    return 0;
}

}  // namespace

extern "C" int nn_gemm128_prepare_b(const float* B, float* image, void* stream) {
    NN_REQUIRE(B && image, "null pointer");
    k_prepare_b<<<128 * 128 / 256, 256, 0, (cudaStream_t)stream>>>(B, image); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("nn_gemm128_prepare_b");
    return 0;
}

extern "C" int nn_gemm128_prepare_b_batch(const float* const* src, const int32_t* transposed, float* const* image, int32_t n,
                                          void* stream) {
    NN_REQUIRE(src && transposed && image && n >= 0, "null pointer");
    for (int i0 = 0; i0 < n; i0 += 64) {
        PrepBatch p;
        const int m = n - i0 < 64 ? n - i0 : 64;
        for (int i = 0; i < m; ++i) {
            NN_REQUIRE(src[i0 + i] && image[i0 + i], "null matrix pointer");
            p.src[i] = src[i0 + i]; p.img[i] = image[i0 + i]; p.transposed[i] = transposed[i0 + i];
        }
        k_prepare_b_batch<<<dim3(128 * 128 / 256, m), 256, 0, (cudaStream_t)stream>>>(p); NN_LAUNCHED(1);
    }
    NN_CHECK_LAUNCH("nn_gemm128_prepare_b_batch");
    return 0;
}

int nn_gemm128_tc_launch(const nn_gemm_args& a, cudaStream_t s) {
    if (a.m <= 0) return 0;
    NN_REQUIRE(a.B_img != nullptr, "tensor-core backend needs B_img (nn_gemm128_prepare_b)");
    int rc = -1;
#define NN_CASE(P, E) if (a.prologue == P && a.epilogue == E) { rc = launch<P, E>(a, s); goto done; }
    NN_CASE(NN_PRO_NONE, NN_EPI_BIAS)
    NN_CASE(NN_PRO_SILU, NN_EPI_BIAS)
    NN_CASE(NN_PRO_NONE, NN_EPI_DSILU)
    NN_CASE(NN_PRO_NONE, NN_EPI_ADD)
    NN_CASE(NN_PRO_ROWSCALE3, NN_EPI_EQUIV_BWD)
    NN_CASE(NN_PRO_SILU_SAVE, NN_EPI_BIAS)
    NN_CASE(NN_PRO_NONE, NN_EPI_MUL)
#undef NN_CASE
    nn_set_error("nn_gemm128: unsupported prologue/epilogue combination %d/%d", a.prologue, a.epilogue);
    return -1;
done:
    if (rc) return rc;
    NN_CHECK_LAUNCH("nn_gemm128(tc)");
    return 0;
}
