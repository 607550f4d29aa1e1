// Two chained 128x128 contractions in ONE kernel:  Y = epi2( mid( epi1(X · B1) ) · B2 ).
//
// Every two-layer MLP on the path (reference models/newtonnet.py:181-199: equiv_message1/2, message_nodepart,
// models/output.py:90-96: the energy head) and its reverse is a pair of 128 -> 128 products with an elementwise
// step in between.  Run as two launches of gemm_ts.cu, the intermediate [M,128] tensor costs one HBM write and one
// HBM read per row (1 KB of the 2.5 KB a forward MLP moves per row): the contractions are HBM-bound, so that
// traffic is time.  One CTA cannot hold two 3xTF32 weight images (2 x 128 KB of shared memory), so the chain runs
// on a CLUSTER OF TWO CTAs (two SMs of one TPC):
//   rank 0:  X rows -> TMEM (cp.async staging, as gemm_ts.cu) -> tcgen05.mma with B1 -> epilogue 1 in the coalesced
//            layout -> st.shared::cluster into rank 1's staging ring (the 64 KB gemm_ts.cu uses for cp.async)
//   rank 1:  ring -> hi / lo split -> TMEM -> tcgen05.mma with B2 -> epilogue 2 -> Y
// The ring holds one tile in 16 slots of 4 KB (row quarter q x K block kb); epilogue warp (q, half) of rank 0 feeds
// producer warp (q, half) of rank 1, chunk c <-> kb = 2 half + c, so flow control is one mbarrier pair per slot:
// ring_full[slot] lives in rank 1 and counts BYTES: rank 0 writes with st.async ... mbarrier::complete_tx, rank 1 arms
// 4 KB per tile (a plain remote store + release-arrive would make every chunk wait for the writer's outstanding
// global loads / stores); ring_empty[slot] lives in rank 0 (32 remote arrivals after the rows were read).  Both SMs
// do the per-tile work of one gemm_ts.cu launch; the pair moves 1.5 KB per row instead of 2.5 KB (forward).
// Measured on 1.8 M rows (B200): forward MLP 0.874 -> 0.727 ms, reverse with accumulation 1.18 -> 1.10 ms; the plain
// reverse chain is SLOWER than two launches (1.19 vs 0.86 ms: rank 0 alone has to pull X and aux1, i.e. half the SMs
// carry all the loads and there are not enough bytes in flight), and so is any chain on node-sized inputs - eval.cu
// uses the chain for the pair-level forward MLPs and the accumulating reverse ones only.  Running the activation in
// rank 1's producers instead of rank 0's epilogue was measured at 1.35 ms (worse).
//
//   MID_SILU_SAVE : q = acc + bias1;  aux_out = silu'(q)  (kept for the reverse sweep);  h = silu(q)     [forward]
//   MID_MUL       : h = acc * aux1                                                                       [reverse]
//   OUT_BIAS      : Y = acc + bias2        OUT_ADD : Y = acc + aux2
// Arithmetic is the same as the two-launch path (same formulas, same order): results are bit-identical.
#include <stdlib.h>
#include "tc_common.cuh"

namespace {

using namespace tc;
constexpr uint32_t B_BYTES = 2 * NKB * BLK_BYTES;     // hi + lo image of one weight matrix = 128 KB
constexpr uint32_t BAR_BYTES = 512;
constexpr int PDEPTH = 2;
constexpr uint32_t SMEM_BYTES = 1024 + B_BYTES + (8 * PDEPTH + 8) * STG_BYTES + BAR_BYTES;
constexpr int PRODUCER_WARPS = 8, EPI_WARPS = 8;
constexpr int MMA_WARP = PRODUCER_WARPS + EPI_WARPS;
// Register files are allocated in groups of 4 warps, so the 17th (MMA) warp is charged as a whole warpgroup: launch with
// 20 warps (3 idle ones complete that warpgroup) at 96 registers and rebalance with setmaxnreg - the MMA warpgroup and
// the producers hand registers to the epilogue warps, whose v[32] + factor prefetch + staging values spilled 120-150
// bytes per thread at 96 registers (local-memory traffic on the L1TEX pipe that already limits the kernel).  ptxas -v:
// (80, 128, 64) compiles every variant with 0-20 bytes of spill stores; the MMA-issuing code needs ~64 (descriptors).
// 256 R_prod + 256 R_epi + 128 R_mma <= 640 * 96.
#ifndef NN_CHAIN_REGS_PROD
#define NN_CHAIN_REGS_PROD 80
#define NN_CHAIN_REGS_EPI 128
#endif
constexpr int THREADS = 32 * (PRODUCER_WARPS + EPI_WARPS + 4);
constexpr int REGS_PROD = NN_CHAIN_REGS_PROD, REGS_EPI = NN_CHAIN_REGS_EPI, REGS_MMA = 64;
static_assert(256 * REGS_PROD + 256 * REGS_EPI + 128 * REGS_MMA <= 640 * 96, "register budget");
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t A_COL0 = 256;

enum { MID_SILU_SAVE = 0, MID_MUL = 1 };
enum { OUT_BIAS = 0, OUT_ADD = 1 };

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_id_x() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t n_clusters_x() { uint32_t r; asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t map_to_rank(uint32_t saddr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank)); return r;
}
__device__ __forceinline__ void st_cluster4(uint32_t raddr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(raddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// remote store that reports its 16 bytes to an mbarrier of the destination CTA when it has landed: no release fence in
// the writer (a release before a plain remote arrive would also wait for the writer's outstanding GLOBAL loads and
// stores - the aux prefetch, the silu' rows - and serialise every chunk on an HBM round trip)
__device__ __forceinline__ void st_async4(uint32_t raddr, float4 v, uint32_t rbar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(raddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(rbar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t raddr) {     // orders this thread's earlier cluster stores
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

struct ChainCtx {
    uint32_t base, sPst, sStg, tmem_base, bar_t_full, bar_t_empty, bar_ring_full, bar_ring_empty;
    uint8_t* smem_gen;
    int warp, lane, cid, ncl, M, my_tiles; bool has_work;
};

// ===================== rank-1 epilogue: output step -> Y =====================
template <int OUT>
__device__ __forceinline__ void epilogue_rank1(const nn_gemm_chain_args& a, const ChainCtx& x) {
    const uint32_t base = x.base, sStg = x.sStg, tmem_base = x.tmem_base;
    const uint32_t bar_t_full = x.bar_t_full, bar_t_empty = x.bar_t_empty;
    uint8_t* smem_gen = x.smem_gen;
    const int warp = x.warp, lane = x.lane, cid = x.cid, ncl = x.ncl, M = x.M, my_tiles = x.my_tiles;
    const int q = warp & 3, ew = warp - PRODUCER_WARPS, half = ew >> 2;
    const int r4 = lane >> 3, c8 = lane & 7;
    uint8_t* stg = smem_gen + (sStg - base) + ew * STG_BYTES;
    // Rank 1 sends nothing to its peer, so the two peer addresses (ring block, ring_full slot) are unused here.  They are
    // still computed: mapa is volatile asm, and without it ptxas schedules all four kernel variants differently.
    (void)map_to_rank(x.sPst + (half * 4 + q) * PDEPTH * STG_BYTES, 1);
    constexpr bool aux_in = OUT == OUT_ADD;
    float4 ax[8];
    auto prefetch = [&](int tile, int c0) {
        if (!aux_in) return;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int grow = tile * TM + q * 32 + k * 4 + r4;
            if (grow < M) ax[k] = ld4(a.aux2 + (size_t)grow * 128 + c0 + 4 * c8);
        }
    };
    if (x.has_work) prefetch(cid, half * 64);
    uint32_t it = 0;
    for (int t = 0; t < my_tiles; ++t, ++it) {
        const int tile = cid + t * ncl;
        const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
        mbar_wait(bar_t_full + 8 * buf, acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * 128;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int c0 = half * 64 + c * 32;
            const int kb = 2 * half + c, slot = q * 4 + kb;
            uint32_t v[32];
            tmem_ld32(taddr + c0, v);
            tmem_ld_wait();
            if (c == 1) {
                tc_fence_before();
                mbar_arrive(bar_t_empty + 8 * buf);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                    make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            __syncwarp();
            float4 cur[8];
            if (aux_in) {
#pragma unroll
                for (int k = 0; k < 8; ++k) cur[k] = ax[k];
                if (c == 0) prefetch(tile, c0 + 32);
                else if (t + 1 < my_tiles) prefetch(tile + ncl, half * 64);
            }
            const int col = c0 + 4 * c8;
            float4 bv = f4_zero();
            if (a.bias2) bv = ld4(a.bias2 + col);
            (void)map_to_rank(x.bar_ring_full + 8 * slot, 1);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int row = k * 4 + r4;
                const int grow = tile * TM + q * 32 + row;
                float4 acc = *reinterpret_cast<const float4*>(stg + row * 128 + ((c8 ^ (row & 7)) << 4));
                if (grow < M) {
                    if (OUT == OUT_ADD) acc = f4_add(acc, cur[k]);
                    else acc = f4_add(acc, bv);
                    st4(a.Y + (size_t)grow * 128 + col, acc);
                }
            }
            __syncwarp();
        }
    }
}

// ===================== rank-0 epilogue: mid step -> the peer's ring =====================
// Everything happens in the row-owner layout tcgen05.ld delivers - lane = row.  The activation-derivative tensor silu'(q) is
// held tile-transposed (NN_TILED_INDEX): it is written (MID_SILU_SAVE) or read (MID_MUL) as 512 contiguous bytes per warp
// instruction, and the tile for rank 1 is sent from the same registers, so this rank needs NO shared-memory transpose at
// all (the two-pass staging of a row-major silu' was half of the LSU shared-memory traffic of the rank that limits the
// pair, profiles/r1c_chain_summary.txt).
template <int MID>
__device__ __forceinline__ void epilogue_rank0(const nn_gemm_chain_args& a, const ChainCtx& x) {
    const uint32_t sPst = x.sPst, tmem_base = x.tmem_base;
    const uint32_t bar_t_full = x.bar_t_full, bar_t_empty = x.bar_t_empty, bar_ring_full = x.bar_ring_full,
                   bar_ring_empty = x.bar_ring_empty;
    const int warp = x.warp, lane = x.lane, cid = x.cid, ncl = x.ncl, M = x.M, my_tiles = x.my_tiles;
    const int q = warp & 3, ew = warp - PRODUCER_WARPS, half = ew >> 2;
    const int rt = q * 32 + lane;                                   // row inside the tile
    const uint32_t ring_remote = map_to_rank(sPst + (half * 4 + q) * PDEPTH * STG_BYTES, 1);
    const float* bias = a.bias1;
    auto tiled = [&](const float* base_, int tile, int chunk) { return base_ + (((size_t)tile * 32 + chunk) * 128 + rt) * 4; };
    float4 ax[8];
    auto prefetch = [&](int tile, int c0) {
        if (MID != MID_MUL) return;
#pragma unroll
        for (int j = 0; j < 8; ++j) ax[j] = ld4(tiled(a.aux1, tile, (c0 >> 2) + j));     // padded rows are allocated: always readable
    };
    if (x.has_work) prefetch(cid, half * 64);
    uint32_t it = 0;
    for (int t = 0; t < my_tiles; ++t, ++it) {
        const int tile = cid + t * ncl;
        const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
        const bool live = tile * TM + rt < M;
        mbar_wait(bar_t_full + 8 * buf, acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * 128;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int c0 = half * 64 + c * 32;
            const int kb = 2 * half + c, slot = q * 4 + kb;
            uint32_t v[32];
            tmem_ld32(taddr + c0, v);
            tmem_ld_wait();
            if (c == 1) {
                tc_fence_before();
                mbar_arrive(bar_t_empty + 8 * buf);
            }
            float4 cur[8];
            if (MID == MID_MUL) {
#pragma unroll
                for (int j = 0; j < 8; ++j) cur[j] = ax[j];
                if (c == 0) prefetch(tile, c0 + 32);
                else if (t + 1 < my_tiles) prefetch(tile + ncl, half * 64);
            }
            const uint32_t full_remote = map_to_rank(bar_ring_full + 8 * slot, 1);
            mbar_wait_cluster(bar_ring_empty + 8 * slot, (t & 1) ^ 1);       // rank 1 has read tile t-1's block
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 acc = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                               __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                float4 hmid;
                if (MID == MID_SILU_SAVE) {
                    const float4 xx = bias ? f4_add(acc, ld4(bias + c0 + 4 * j)) : acc;
                    const float4 sg = make_float4(sigmoid_f(xx.x), sigmoid_f(xx.y), sigmoid_f(xx.z), sigmoid_f(xx.w));
                    if (live)
                        st4(const_cast<float*>(tiled(a.aux_out, tile, (c0 >> 2) + j)),
                            make_float4(sg.x * fmaf(xx.x, 1.0f - sg.x, 1.0f), sg.y * fmaf(xx.y, 1.0f - sg.y, 1.0f),
                                        sg.z * fmaf(xx.z, 1.0f - sg.z, 1.0f), sg.w * fmaf(xx.w, 1.0f - sg.w, 1.0f)));
                    hmid = f4_mul(xx, sg);
                } else {
                    hmid = live ? f4_mul(acc, cur[j]) : f4_zero();
                }
                // the ring block is chunk-major ([chunk j][row]): 512 contiguous bytes per warp instruction on
                // both sides (32 separate 16-byte pieces per instruction through the cluster network were measured slower)
                st_async4(ring_remote + c * STG_BYTES + j * 512 + lane * 16, hmid, full_remote);
            }
        }
    }
}

template <int MID, int OUT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1) k_gemm128_chain(nn_gemm_chain_args a_in) {
    // dual launch (Y_b != NULL): even clusters run chain A, odd clusters chain B over the same X tiles
    nn_gemm_chain_args a = a_in;
    const bool dual = a_in.Y_b != nullptr;
    {
        uint32_t c; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(c));
        if (dual && (c & 1u)) {
            a.B1_img = a_in.B1_img_b; a.B2_img = a_in.B2_img_b; a.aux_out = a_in.aux_out_b; a.Y = a_in.Y_b;
        }
    }
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sB = base;                                             // this rank's weight image [hi|lo][kb][16 KB]
    const uint32_t sPst = base + B_BYTES;                                 // rank 0: cp.async staging; rank 1: the ring
    const uint32_t sStg = sPst + 8 * PDEPTH * STG_BYTES;                  // [8 epilogue warps][4 KB]
    const uint32_t sBar = sStg + 8 * STG_BYTES;
    const uint32_t bar_b_full = sBar;
    const uint32_t bar_a_full = sBar + 8;                                 // [NKB]
    const uint32_t bar_a_empty = bar_a_full + 8 * NKB;                    // [NKB]
    const uint32_t bar_t_full = bar_a_empty + 8 * NKB;                    // [2]
    const uint32_t bar_t_empty = bar_t_full + 16;                         // [2]
    const uint32_t bar_ring_full = bar_t_empty + 16;                      // [16] used in rank 1, slot = q * 4 + kb
    const uint32_t bar_ring_empty = bar_ring_full + 8 * 16;               // [16] used in rank 0
    const uint32_t tmem_slot = bar_ring_empty + 8 * 16;
    uint8_t* smem_gen = smem_raw + (base - smem_u32(smem_raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const int cid = dual ? (int)(cluster_id_x() >> 1) : (int)cluster_id_x();
    const int ncl = dual ? (int)(n_clusters_x() >> 1) : (int)n_clusters_x();

    pdl_launch_dependents();
    if (warp == MMA_WARP) {
        if (lane == 0) {
            mbar_init(bar_b_full, 1);
            for (int s = 0; s < NKB; ++s) { mbar_init(bar_a_full + 8 * s, 4 * 32); mbar_init(bar_a_empty + 8 * s, 1); }
            for (int b = 0; b < 2; ++b) { mbar_init(bar_t_full + 8 * b, 1); mbar_init(bar_t_empty + 8 * b, EPI_WARPS * 32); }
            for (int s = 0; s < 16; ++s) { mbar_init(bar_ring_full + 8 * s, 1); mbar_init(bar_ring_empty + 8 * s, 32); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            const uint8_t* img = reinterpret_cast<const uint8_t*>(rank == 0 ? a.B1_img : a.B2_img);
            mbar_expect_tx(bar_b_full, B_BYTES);
            for (int c = 0; c < (int)(B_BYTES / BLK_BYTES); ++c)
                bulk_g2s(sB + c * BLK_BYTES, img + (size_t)c * BLK_BYTES, BLK_BYTES, bar_b_full);
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();                               // barriers of BOTH ranks are initialised before any remote arrival
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));
    pdl_wait();
    int M = a.m;
    if (a.m_dev) { long long v = (long long)a.m_dev[0] * a.m_dev_mul; M = v < a.m ? (int)v : a.m; }
    const int n_tiles = (M + TM - 1) / TM;
    const bool has_work = cid < n_tiles;
    const int my_tiles = has_work ? (n_tiles - 1 - cid) / ncl + 1 : 0;

    ChainCtx ctx{base, sPst, sStg, tmem_base, bar_t_full, bar_t_empty, bar_ring_full, bar_ring_empty, smem_gen,
                 warp, lane, cid, ncl, M, my_tiles, has_work};
    if (warp < PRODUCER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_PROD));
        // ===================== producers: rows -> hi/lo split -> TMEM =====================
        const int q = warp & 3, h = warp >> 2;
        const int r4 = lane >> 3, c8 = lane & 7;
        const uint32_t pst_s = sPst + warp * PDEPTH * STG_BYTES;          // this warp's two 4 KB blocks: kb = 2h, 2h + 1
        uint8_t* pst_g = smem_gen + (pst_s - base);
        const int n_items = my_tiles * 2;
        auto issue = [&](int w) {                                         // rank 0 only: global -> staging
            const int row0 = (cid + (w >> 1) * ncl) * TM + q * 32, kb = 2 * h + (w & 1);
            const uint32_t dst0 = pst_s + (w % PDEPTH) * STG_BYTES;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int row = it * 4 + r4, grow = row0 + row;
                const uint32_t dst = dst0 + row * 128 + ((c8 ^ (row & 7)) << 4);
                const float* src = a.X + (size_t)(grow < M ? grow : 0) * 128 + kb * KB + c8 * 4;
                const uint32_t nbytes = grow < M ? 16u : 0u;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        if (rank == 0) {
#pragma unroll
            for (int u = 0; u < PDEPTH; ++u) {
                if (u < n_items) issue(u);
                else asm volatile("cp.async.commit_group;" ::: "memory");
            }
        } else if (lane == 0 && n_items > 0) {            // arm both slots for the first tile: 4 KB of st.async each
            mbar_expect_tx(bar_ring_full + 8 * (q * 4 + 2 * h), STG_BYTES);
            mbar_expect_tx(bar_ring_full + 8 * (q * 4 + 2 * h + 1), STG_BYTES);
        }
        for (int w = 0; w < n_items; ++w) {
            const int t_local = w >> 1, kb = 2 * h + (w & 1);
            const int slot = q * 4 + kb;
            if (rank == 0) {
                asm volatile("cp.async.wait_group %0;" ::"n"(PDEPTH - 1) : "memory");
                __syncwarp();
            } else {
                mbar_wait(bar_ring_full + 8 * slot, t_local & 1);             // all 4 KB of rank 0's st.async have landed
            }
            const uint8_t* blk = pst_g + (w % PDEPTH) * STG_BYTES;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + A_COL0 + kb * 64;
            bool waited = false;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int ch = hf * 4 + j;
                    const float4 x = rank == 1 ? *reinterpret_cast<const float4*>(blk + ch * 512 + lane * 16)
                                       : *reinterpret_cast<const float4*>(blk + lane * 128 + ((ch ^ (lane & 7)) << 4));
                    const float4 hh = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
                    hi[4 * j] = __float_as_uint(hh.x); hi[4 * j + 1] = __float_as_uint(hh.y);
                    hi[4 * j + 2] = __float_as_uint(hh.z); hi[4 * j + 3] = __float_as_uint(hh.w);
                    lo[4 * j] = __float_as_uint(x.x - hh.x); lo[4 * j + 1] = __float_as_uint(x.y - hh.y);
                    lo[4 * j + 2] = __float_as_uint(x.z - hh.z); lo[4 * j + 3] = __float_as_uint(x.w - hh.w);
                }
                if (hf == 1 && rank == 1) {                               // all rows are in registers: the slot may be refilled
                    if (lane == 0 && w + 2 < n_items) mbar_expect_tx(bar_ring_full + 8 * slot, STG_BYTES);   // re-arm first
                    mbar_arrive_remote(map_to_rank(bar_ring_empty + 8 * slot, 0));
                }
                if (!waited) {
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
            if (rank == 0) {
                __syncwarp();
                if (w + PDEPTH < n_items) issue(w + PDEPTH);
                else asm volatile("cp.async.commit_group;" ::: "memory");
            }
        }
        if (rank == 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (warp >= MMA_WARP) {                    // the MMA warp and three idle warps that complete its warpgroup
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_MMA));
        if (warp == MMA_WARP && lane == 0) mbar_wait(bar_b_full, 0);
        if (warp == MMA_WARP && lane == 0 && has_work) {
            uint32_t it = 0;
            for (int t = 0; t < my_tiles; ++t, ++it) {
                const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(bar_t_empty + 8 * buf, acc_phase ^ 1);
                tc_fence_after();
                umma_tile_ts(tmem_base + buf * 128, tmem_base + A_COL0, sB, bar_a_full, bar_a_empty, it & 1);
                umma_commit(bar_t_full + 8 * buf);
            }
        }
        __syncwarp();
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
        if (rank == 0) epilogue_rank0<MID>(a, ctx);
        else epilogue_rank1<OUT>(a, ctx);
    }
    tc_fence_before();
    cluster_sync_all();                               // no CTA leaves while its peer may still touch its shared memory
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

bool g_attr_set[2][2] = {};

template <int MID, int OUT>
int launch(const nn_gemm_chain_args& a, cudaStream_t s) {
    if (!g_attr_set[MID][OUT]) {
        cudaError_t e = cudaFuncSetAttribute(k_gemm128_chain<MID, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
        if (e != cudaSuccess) { nn_set_error("nn_gemm128_chain: cannot set %u B dynamic smem: %s", SMEM_BYTES, cudaGetErrorString(e)); return -2; }
        g_attr_set[MID][OUT] = true;
    }
    const int pairs = nn_num_sms() / 2;             // one cluster per pair of SMs
    const int tiles = nn_ceil_div(a.m, TM);
    int clusters = tiles < pairs ? tiles : pairs;
    if (a.Y_b) {                                   // dual: an even number of clusters, half per chain
        clusters = 2 * tiles < pairs ? 2 * tiles : (pairs & ~1);
        if (clusters < 2) clusters = 2;
    }
    NN_LAUNCHED(1);
    return launch_pdl(k_gemm128_chain<MID, OUT>, 2 * clusters, THREADS, SMEM_BYTES, s, a);
}

}  // namespace

extern "C" NN_API int nn_gemm128_chain(const nn_gemm_chain_args* a, void* stream) {
    NN_REQUIRE(a && a->X && a->Y && a->B1_img && a->B2_img, "null argument");
    NN_REQUIRE(a->mid == MID_SILU_SAVE || a->mid == MID_MUL, "unknown mid step");
    NN_REQUIRE(a->out == OUT_BIAS || a->out == OUT_ADD, "unknown output step");
    NN_REQUIRE(a->mid != MID_SILU_SAVE || a->aux_out, "mid = SILU_SAVE needs aux_out");
    NN_REQUIRE(a->mid != MID_MUL || a->aux1, "mid = MUL needs aux1");
    NN_REQUIRE(a->out != OUT_ADD || a->aux2, "out = ADD needs aux2");
    NN_REQUIRE(!a->Y_b || (a->B1_img_b && a->B2_img_b && (a->mid != MID_SILU_SAVE || a->aux_out_b) && a->out == OUT_BIAS && !a->bias1 && !a->bias2),
               "dual chain: needs B1_img_b, B2_img_b, aux_out_b, out = BIAS and no biases");
    if (a->m <= 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    if (a->mid == MID_SILU_SAVE) rc = a->out == OUT_BIAS ? launch<MID_SILU_SAVE, OUT_BIAS>(*a, s) : launch<MID_SILU_SAVE, OUT_ADD>(*a, s);
    else rc = a->out == OUT_BIAS ? launch<MID_MUL, OUT_BIAS>(*a, s) : launch<MID_MUL, OUT_ADD>(*a, s);
    if (rc) return rc;
    NN_CHECK_LAUNCH("nn_gemm128_chain");
    return 0;
}
