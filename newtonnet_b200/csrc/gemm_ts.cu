// TS-mode variant of the tensor-core contraction (backend 2): the A operand lives in TENSOR MEMORY.
//
// gemm_tc.cu (SS mode) is bound by the shared-memory port of each SM: per 128-row tile the tensor core
// re-reads A_hi twice, A_lo, B_hi twice and B_lo from shared memory (384 KB), on top of 128 KB of producer
// stores and 128 KB of epilogue staging - about 5.1k of the 6.5k cycles a tile takes (throughput scales
// linearly with the number of CTAs: it is per-SM bound, not HBM bound).  Here the producers write the
// hi / lo split of X straight into TMEM (tcgen05.st, lane = row), so the MMAs read only B from shared
// memory (192 KB per tile) and the A stage ring in shared memory disappears:
//   warps 0-7  producers : coalesced LDG.128 (4 K-blocks of prefetch) -> 32x32 transpose through a 4 KB
//                          XOR-swizzled staging buffer -> row-owner layout -> prologue -> tf32 hi/lo ->
//                          tcgen05.st into the K block's TMEM columns (warp = lane quarter x K-block half)
//   warp  16   MMA issuer: tcgen05.mma kind::tf32 with A from TMEM ([taddr]) and B from the resident image
//   warps 8-15 epilogue  : unchanged (see gemm_tc.cu)
// TMEM: columns 0-255 two accumulators, 256-511 one tile of A (4 K blocks x (32 hi + 32 lo) columns).
#include <stdlib.h>
#include "tc_common.cuh"

namespace {

using namespace tc;
constexpr uint32_t B_BYTES = 2 * NKB * BLK_BYTES;     // hi + lo image of B = 128 KB
constexpr uint32_t BAR_BYTES = 256;
constexpr int PDEPTH = 2;                     // cp.async staging buffers per producer warp (items in flight)
constexpr uint32_t SMEM_BYTES = 1024 + B_BYTES + (8 * PDEPTH + 8) * STG_BYTES + BAR_BYTES;   // B image + producer / epilogue staging
constexpr int PRODUCER_WARPS = 8, EPI_WARPS = 8;
constexpr int MMA_WARP = PRODUCER_WARPS + EPI_WARPS;
// 20 warps (the MMA warp + 3 idle warps complete a warpgroup: register files are allocated per 4 warps) at 96 registers,
// rebalanced with setmaxnreg - see gemm_chain.cu.  256 R_prod + 256 R_epi + 128 R_mma <= 640 * 96.
#ifndef NN_TS_REGS_PROD
#define NN_TS_REGS_PROD 80
#define NN_TS_REGS_EPI 128
#define NN_TS_REGS_MMA 64
#endif
constexpr int THREADS = 32 * (PRODUCER_WARPS + EPI_WARPS + 4);
constexpr int REGS_PROD = NN_TS_REGS_PROD, REGS_EPI = NN_TS_REGS_EPI, REGS_MMA = NN_TS_REGS_MMA;
static_assert(256 * REGS_PROD + 256 * REGS_EPI + 128 * REGS_MMA <= 640 * 96, "register budget");
constexpr uint32_t TMEM_COLS = 512;           // 2 x 128 accumulator columns + 4 K blocks x 64 columns of A
constexpr uint32_t A_COL0 = 256;

// TILED: the EPI_MUL factor aux1 is tile-transposed (NN_TILED_INDEX), as the chained kernel writes it
template <int PRO, int EPI, bool TILED = false>
__global__ void __launch_bounds__(THREADS, 1) k_gemm128_ts(nn_gemm_args a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;          // swizzle atoms need 1024 B alignment
    const uint32_t sB = base;                                             // [hi|lo][kb][16 KB]
    const uint32_t sPst = base + B_BYTES;                                 // [8 producer warps][PDEPTH][4 KB]
    const uint32_t sStg = sPst + 8 * PDEPTH * STG_BYTES;                  // [8 epilogue warps][4 KB]
    const uint32_t sBar = sStg + 8 * STG_BYTES;
    const uint32_t bar_b_full = sBar;                                     // 8 bytes each
    const uint32_t bar_a_full = sBar + 8;                                 // [NKB] one per K block of the tile in TMEM
    const uint32_t bar_a_empty = bar_a_full + 8 * NKB;                    // [NKB]
    const uint32_t bar_t_full = bar_a_empty + 8 * NKB;                    // [2]
    const uint32_t bar_t_empty = bar_t_full + 16;                         // [2]
    const uint32_t tmem_slot = bar_t_empty + 16;                          // 4 bytes
    uint8_t* smem_gen = smem_raw + (base - smem_u32(smem_raw));           // generic pointer to `base`

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // Programmatic dependent launch: everything up to pdl_wait() touches only this kernel's constants (barriers,
    // tensor memory, the weight image), so it overlaps the tail of the preceding kernel in the stream.
    pdl_launch_dependents();
    if (warp == MMA_WARP) {
        if (lane == 0) {
            mbar_init(bar_b_full, 1);
            for (int s = 0; s < NKB; ++s) { mbar_init(bar_a_full + 8 * s, 4 * 32); mbar_init(bar_a_empty + 8 * s, 1); }
            for (int b = 0; b < 2; ++b) { mbar_init(bar_t_full + 8 * b, 1); mbar_init(bar_t_empty + 8 * b, EPI_WARPS * 32); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_expect_tx(bar_b_full, B_BYTES);
            for (int c = 0; c < (int)(B_BYTES / BLK_BYTES); ++c)
                bulk_g2s(sB + c * BLK_BYTES, reinterpret_cast<const uint8_t*>(a.B_img) + (size_t)c * BLK_BYTES, BLK_BYTES, bar_b_full);
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));
    pdl_wait();                                       // results of the preceding kernels are visible from here on
    int M = a.m;
    if (a.m_dev) { long long v = (long long)a.m_dev[0] * a.m_dev_mul; M = v < a.m ? (int)v : a.m; }
    const int n_tiles = (M + TM - 1) / TM;
    const bool has_work = (int)blockIdx.x < n_tiles;

    if (warp < PRODUCER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_PROD));
        // ===================== producers: X rows -> transpose -> hi/lo split -> TMEM =====================
        // warp = (lane quarter q, K-block half h): rows [32q, 32q+32) of K blocks 2h and 2h+1 of every tile.
        // cp.async (LDGSTS) brings each 32 x 32 block into a swizzled staging buffer in the coalesced
        // layout with no registers held (PDEPTH blocks = 8 KB per warp, 64 KB per SM in flight); the block
        // is then read back one ROW per lane, split and stored to the K block's TMEM columns.
        const int q = warp & 3, h = warp >> 2;
        const int r4 = lane >> 3, c8 = lane & 7;
        const uint32_t pst_s = sPst + warp * PDEPTH * STG_BYTES;
        uint8_t* pst_g = smem_gen + (pst_s - base);
        const int my_tiles = has_work ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
        const int n_items = my_tiles * 2;                 // item w = (tile w >> 1, K block 2h + (w & 1))
        auto issue = [&](int w) {
            const int row0 = ((int)blockIdx.x + (w >> 1) * (int)gridDim.x) * TM + q * 32, kb = 2 * h + (w & 1);
            const uint32_t dst0 = pst_s + (w % PDEPTH) * STG_BYTES;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int row = it * 4 + r4, grow = row0 + row;
                const uint32_t dst = dst0 + row * 128 + ((c8 ^ (row & 7)) << 4);
                const float* src = a.X + (size_t)(grow < M ? grow : 0) * 128 + kb * KB + c8 * 4;
                const uint32_t nbytes = grow < M ? 16u : 0u;          // rows beyond M are zero-filled
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
#pragma unroll
        for (int u = 0; u < PDEPTH; ++u) {
            if (u < n_items) issue(u);
            else asm volatile("cp.async.commit_group;" ::: "memory");    // keep the group count uniform
        }
        for (int w = 0; w < n_items; ++w) {
            const int t_local = w >> 1, kb = 2 * h + (w & 1);
            const int grow = ((int)blockIdx.x + t_local * (int)gridDim.x) * TM + q * 32 + lane;   // this lane's row
            asm volatile("cp.async.wait_group %0;" ::"n"(PDEPTH - 1) : "memory");
            __syncwarp();
            const uint8_t* blk = pst_g + (w % PDEPTH) * STG_BYTES;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + A_COL0 + kb * 64;
            bool waited = false;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {                  // 16 K values at a time: 32 live registers
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int ch = hf * 4 + j;
                    float4 x = *reinterpret_cast<const float4*>(blk + lane * 128 + ((ch ^ (lane & 7)) << 4));
                    if (PRO == NN_PRO_ROWSCALE3 && grow < M) x = f4_mul(x, ld4(a.aux2 + (size_t)(grow / 3) * 128 + kb * KB + 4 * ch));
                    x = apply_prologue<PRO>(a, x, grow, kb * KB + 4 * ch, M);
                    const float4 hh = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
                    hi[4 * j] = __float_as_uint(hh.x); hi[4 * j + 1] = __float_as_uint(hh.y);
                    hi[4 * j + 2] = __float_as_uint(hh.z); hi[4 * j + 3] = __float_as_uint(hh.w);
                    lo[4 * j] = __float_as_uint(x.x - hh.x); lo[4 * j + 1] = __float_as_uint(x.y - hh.y);
                    lo[4 * j + 2] = __float_as_uint(x.z - hh.z); lo[4 * j + 3] = __float_as_uint(x.w - hh.w);
                }
                if (!waited) {    // the MMAs of the previous tile that read this K block's columns must have retired
                    mbar_wait(bar_a_empty + 8 * kb, (t_local & 1) ^ 1);
                    tc_fence_after();
                    waited = true;
                }
                tmem_st16(taddr + hf * 16, hi);
                tmem_st16(taddr + 32 + hf * 16, lo);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(bar_a_full + 8 * kb);
            __syncwarp();                                     // every lane has read the staging block
            if (w + PDEPTH < n_items) issue(w + PDEPTH);
            else asm volatile("cp.async.commit_group;" ::: "memory");
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (warp >= MMA_WARP) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_MMA));
        // ===================== B load + MMA issue (one elected lane of warp 16; warps 17-19 idle) =====================
        if (warp == MMA_WARP && lane == 0) mbar_wait(bar_b_full, 0);           // the image copy must have landed before the CTA may exit
        if (warp == MMA_WARP && lane == 0 && has_work) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(bar_t_empty + 8 * buf, acc_phase ^ 1);          // epilogue has drained this accumulator
                tc_fence_after();
                umma_tile_ts(tmem_base + buf * 128, tmem_base + A_COL0, sB, bar_a_full, bar_a_empty, it & 1);
                umma_commit(bar_t_full + 8 * buf);                         // accumulator complete
            }
        }
        __syncwarp();
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
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
        // EPI_MUL with a tile-transposed factor (a.aux_tiled, written by the chained kernel): the factor is read and applied
        // in the row-owner layout, straight after tcgen05.ld (lane = row: 512 contiguous bytes per warp instruction)
        const int rt = q * 32 + lane;
        auto prefetch = [&](int tile, int c0) {
            if (!kAux1) return;
            if (TILED) {
#pragma unroll
                for (int j = 0; j < 8; ++j) ax[j] = ld4(a.aux1 + (((size_t)tile * 32 + (c0 >> 2) + j) * 128 + rt) * 4);
                return;
            }
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
                if (TILED) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) * ax[j].x);
                        v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) * ax[j].y);
                        v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) * ax[j].z);
                        v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) * ax[j].w);
                    }
                    if (c == 0) prefetch(tile, c0 + 32);
                    else if (tile + (int)gridDim.x < n_tiles) prefetch(tile + gridDim.x, half * 64);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j)         // row = lane, 16-byte chunk j -> physical chunk j ^ (lane & 7)
                    *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                        make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                    __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                __syncwarp();
                float4 cur[8];
                if (kAux1 && !TILED) {
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
                            if (!TILED) acc = f4_mul(acc, cur[k]);
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

bool g_attr_set[4][5][2] = {};

template <int PRO, int EPI, bool TILED = false>
int launch(const nn_gemm_args& a, cudaStream_t s) {
    if (!g_attr_set[PRO][EPI][TILED]) {
        cudaError_t e = cudaFuncSetAttribute(k_gemm128_ts<PRO, EPI, TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
        if (e != cudaSuccess) { nn_set_error("nn_gemm128(ts): cannot set %u B dynamic smem: %s", SMEM_BYTES, cudaGetErrorString(e)); return -2; }
        g_attr_set[PRO][EPI][TILED] = true;
    }
    const int tiles = nn_ceil_div(a.m, TM), sms = nn_num_sms();
    const int grid = tiles < sms ? tiles : sms;
    NN_LAUNCHED(1);
    return launch_pdl(k_gemm128_ts<PRO, EPI, TILED>, grid, THREADS, SMEM_BYTES, s, a);
}

}  // namespace

int nn_gemm128_ts_launch(const nn_gemm_args& a, cudaStream_t s) {
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
    if (a.prologue == NN_PRO_NONE && a.epilogue == NN_EPI_MUL && a.aux_tiled) { rc = launch<NN_PRO_NONE, NN_EPI_MUL, true>(a, s); goto done; }
    NN_CASE(NN_PRO_NONE, NN_EPI_MUL)
#undef NN_CASE
    nn_set_error("nn_gemm128: unsupported prologue/epilogue combination %d/%d", a.prologue, a.epilogue);
    return -1;
done:
    if (rc) return rc;
    NN_CHECK_LAUNCH("nn_gemm128(ts)");
    return 0;
}
