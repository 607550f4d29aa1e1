// Message kernels on the tensor cores.
//
// The edge part of the message, me_p = We rbf_p (K = 20, reference models/newtonnet.py:210), is a
// [P,20] x [20,128] contraction.  Done per lane in SIMT it costs 80 FMAs + 20 shared loads per output
// float4 and leaves the message kernels instruction-bound (24-32 % of the HBM roofline).  Here one
// tcgen05 K block (K padded 20 -> 32 = one 128-byte swizzle row) produces me for 128 pairs at a time
// (3xTF32 split, as in gemm_tc.cu), and the gather / multiply work moves into the epilogue, which runs in
// the coalesced row layout (8 lanes x 16 B per 128 B row segment):
//   forward :  m_p  = me_p * mn_i * mn_j                                     (writes 512 B / pair)
//   reverse :  mt   = mbar_p + abar_i + abar_j ;  y = mt * mn_i * mn_j
//              xbar = <y, We drbf_p>   (second accumulator, same B operand)
//              t_p  = mt * me_p        (overwrites mbar_p)
// Same persistent warp-specialised structure as gemm_tc.cu: producers (rbf rows -> hi/lo -> swizzled
// smem), one MMA-issuing lane, 8 epilogue warps with a 32x32 transposing stage, two TMEM buffers.
#include "tc_common.cuh"

namespace {

using namespace tc;
constexpr int STAGES = 2;
constexpr int PRODUCER_WARPS = 4, EPI_WARPS = 8;
constexpr int MMA_WARP = PRODUCER_WARPS + EPI_WARPS;
// register files are allocated in groups of 4 warps: 13 warps would be charged as 16, so use 16 (3 idle)
constexpr int THREADS = 32 * 16;
constexpr uint32_t B_BYTES = 2 * BLK_BYTES;            // We image: hi + lo, one K block
constexpr uint32_t BAR_BYTES = 256;
// 512 threads x 128 registers at launch; after setmaxnreg: 4 warps x 104 (producers) + 4 x 40 (MMA warpgroup) + 8 x 184
// (epilogue) = 2048 = 16 x 128
constexpr int REGS_PROD = 104, REGS_MMA = 40, REGS_EPI = 184;

// gather window of the epilogue (tools/build_variant.sh overrides these for A/B runs)
#ifndef NN_MSG_FWD_G
#define NN_MSG_FWD_G 4
#define NN_MSG_FWD_D 2
#define NN_MSG_BWD_G 2
#define NN_MSG_BWD_D 2
#endif

template <bool BWD> struct Cfg {
    static constexpr int NA = BWD ? 2 : 1;              // A operands per tile (rbf [, drbf])
    static constexpr uint32_t A_STAGE_BYTES = NA * 2 * BLK_BYTES;
    static constexpr uint32_t SMEM = 1024 + B_BYTES + STAGES * A_STAGE_BYTES + EPI_WARPS * STG_BYTES + BAR_BYTES;
    static constexpr uint32_t TMEM_COLS = BWD ? 512 : 256;
    static constexpr uint32_t ACC_COLS = BWD ? 256 : 128;   // columns per accumulator buffer
    static constexpr int PF = BWD ? 1 : 2;              // tiles of rbf rows in flight in registers per producer thread
    static constexpr int G = BWD ? NN_MSG_BWD_G : NN_MSG_FWD_G;   // rows per lane in one gather group
    static constexpr int D = BWD ? NN_MSG_BWD_D : NN_MSG_FWD_D;   // window depth: D - 1 groups in flight behind the one being consumed
};

struct MsgArgs {
    const float* rbf; const float* drbf;        // [P,20]
    const float* B_img;                          // We operand image (nn_message_prepare_b)
    const int* pair_i; const int* pair_j;
    const float* mn; const float* abar;          // [N,128]
    float* io;                                   // fwd: msg out [P,128]; bwd: mbar in / t out [P,128]
    float* x_part;                               // bwd: [2][P] partial dE/dx (column halves)
    const int* n_dev; int cap;
};

template <bool BWD>
__global__ void __launch_bounds__(THREADS, 1) k_message_tc(MsgArgs a) {
    using C = Cfg<BWD>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sB = base;
    const uint32_t sA = base + B_BYTES;
    const uint32_t sStg = sA + STAGES * C::A_STAGE_BYTES;
    const uint32_t sBar = sStg + EPI_WARPS * STG_BYTES;
    const uint32_t bar_b_full = sBar;
    const uint32_t bar_a_full = sBar + 8;
    const uint32_t bar_a_empty = bar_a_full + 8 * STAGES;
    const uint32_t bar_t_full = bar_a_empty + 8 * STAGES;
    const uint32_t bar_t_empty = bar_t_full + 16;
    const uint32_t tmem_slot = bar_t_empty + 16;
    uint8_t* smem_gen = smem_raw + (base - smem_u32(smem_raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    pdl_launch_dependents();                          // see gemm_ts.cu: the prologue overlaps the preceding kernel's tail
    if (warp == MMA_WARP) {
        if (lane == 0) {
            mbar_init(bar_b_full, 1);
            for (int s = 0; s < STAGES; ++s) { mbar_init(bar_a_full + 8 * s, PRODUCER_WARPS * 32); mbar_init(bar_a_empty + 8 * s, 1); }
            for (int b = 0; b < 2; ++b) { mbar_init(bar_t_full + 8 * b, 1); mbar_init(bar_t_empty + 8 * b, EPI_WARPS * 32); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_expect_tx(bar_b_full, B_BYTES);
            bulk_g2s(sB, a.B_img, BLK_BYTES, bar_b_full);
            bulk_g2s(sB + BLK_BYTES, reinterpret_cast<const uint8_t*>(a.B_img) + BLK_BYTES, BLK_BYTES, bar_b_full);
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(C::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));
    pdl_wait();
    int M = a.cap;
    if (a.n_dev) { int v = a.n_dev[0]; M = v < a.cap ? v : a.cap; }
    const int n_tiles = (M + TM - 1) / TM;
    const bool has_work = (int)blockIdx.x < n_tiles;

    // register files: producers and the MMA warpgroup hand registers to the two epilogue warpgroups
    if (warp < PRODUCER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_PROD));
        // ===================== producers: rbf rows (80 B) -> zero-padded 128 B swizzle rows, hi / lo =====================
        const int r4 = lane >> 3, chunk = lane & 7;
        const int my_tiles = has_work ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
        constexpr int PF = C::PF;
        float4 v[PF][C::NA][8];
        auto issue = [&](int w, float4 (&dst)[C::NA][8]) {
            const int row0 = ((int)blockIdx.x + w * (int)gridDim.x) * TM;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int p = row0 + warp * 32 + it * 4 + r4;
                const bool ok = p < M && chunk < kNB / 4;
                dst[0][it] = ok ? ld4(a.rbf + (size_t)p * kNB + chunk * 4) : f4_zero();
                if (BWD) dst[C::NA - 1][it] = ok ? ld4(a.drbf + (size_t)p * kNB + chunk * 4) : f4_zero();
            }
        };
#pragma unroll
        for (int u = 0; u < PF; ++u)
            if (u < my_tiles) issue(u, v[u]);
        uint32_t stage = 0, phase = 0;
        for (int w0 = 0; w0 < my_tiles; w0 += PF) {
#pragma unroll
            for (int u = 0; u < PF; ++u) {
                const int w = w0 + u;
                if (w >= my_tiles) break;
                mbar_wait(bar_a_empty + 8 * stage, phase ^ 1);
                uint8_t* st = smem_gen + (sA - base) + stage * C::A_STAGE_BYTES;
#pragma unroll
                for (int o = 0; o < C::NA; ++o) {
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int row = warp * 32 + it * 4 + r4;
                        const uint32_t off = swz_offset_bytes(row, chunk);
                        const float4 x = v[u][o][it];
                        const float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
                        *reinterpret_cast<float4*>(st + o * 2 * BLK_BYTES + off) = h;
                        *reinterpret_cast<float4*>(st + o * 2 * BLK_BYTES + BLK_BYTES + off) = f4_sub(x, h);
                    }
                }
                fence_proxy_async();
                mbar_arrive(bar_a_full + 8 * stage);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
                if (w + PF < my_tiles) issue(w + PF, v[u]);
            }
        }
    } else if (warp >= MMA_WARP) {                      // warpgroup 3: the MMA warp and three idle warps
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_MMA));
        if (warp == MMA_WARP && lane == 0) mbar_wait(bar_b_full, 0);
        if (warp == MMA_WARP && lane == 0 && has_work) {
            uint32_t stage = 0, phase = 0, it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(bar_t_empty + 8 * buf, acc_phase ^ 1);
                tc_fence_after();
                mbar_wait(bar_a_full + 8 * stage, phase);
                tc_fence_after();
                const uint32_t b_hi = sB, b_lo = sB + BLK_BYTES;
#pragma unroll
                for (int o = 0; o < C::NA; ++o) {
                    const uint32_t d_tmem = tmem_base + buf * C::ACC_COLS + o * 128;
                    const uint32_t a_hi = sA + stage * C::A_STAGE_BYTES + o * 2 * BLK_BYTES, a_lo = a_hi + BLK_BYTES;
#pragma unroll
                    for (int ks = 0; ks < KB / 8; ++ks) {
                        const uint64_t dah = make_desc(a_hi + ks * 32), dal = make_desc(a_lo + ks * 32);
                        const uint64_t dbh = make_desc(b_hi + ks * 32), dbl = make_desc(b_lo + ks * 32);
                        umma_tf32(d_tmem, dal, dbh, ks != 0);
                        umma_tf32(d_tmem, dah, dbl, 1);
                        umma_tf32(d_tmem, dah, dbh, 1);
                    }
                }
                umma_commit(bar_a_empty + 8 * stage);
                umma_commit(bar_t_full + 8 * buf);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue =====================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
        // The gathers (mn_i, mn_j [, abar_i, abar_j, mbar_p]) are L2 / HBM latency chains; each warp keeps a rolling
        // window of two row groups in flight (registers handed over by the producer / MMA warpgroups, setmaxnreg),
        // running across chunk and tile boundaries - the addresses depend on the pair list only, not on the MMA.
        const int q = warp & 3, ew = warp - PRODUCER_WARPS, half = ew >> 2;
        const int r4 = lane >> 3, c8 = lane & 7;
        uint8_t* stg = smem_gen + (sStg - base) + ew * STG_BYTES;
        constexpr int G = C::G, NG = 8 / G, NL = BWD ? 5 : 2, D = C::D, GT = 2 * NG;   // GT groups per tile
        static_assert(GT % D == 0, "window slots must line up across tiles");
        float4 win[D][G][NL];
        // pair endpoints of this warp's 32 rows: lane l holds row l (current tile and the next one)
        int cur_i = 0, cur_j = 0, nxt_i = 0, nxt_j = 0;
        auto load_idx = [&](int tile, int& oi, int& oj) {
            const int p = tile * TM + q * 32 + lane;
            const bool ok = tile < n_tiles && p < M;
            oi = ok ? a.pair_i[p] : 0;
            oj = ok ? a.pair_j[p] : 0;
        };
        auto issue = [&](int tile, int vi, int vj, int c, int g, float4 (&dst)[G][NL]) {
            const int col = half * 64 + c * 32 + 4 * c8;
#pragma unroll
            for (int kk = 0; kk < G; ++kk) {
                const int row = (g * G + kk) * 4 + r4;
                const int ii = __shfl_sync(0xffffffffu, vi, row), jj = __shfl_sync(0xffffffffu, vj, row);
                const int p = tile * TM + q * 32 + row;
                if (p < M) {
                    dst[kk][0] = ld4(a.mn + (size_t)ii * kF + col);
                    dst[kk][1] = ld4(a.mn + (size_t)jj * kF + col);
                    if (BWD) {
                        dst[kk][2] = ld4(a.abar + (size_t)ii * kF + col);
                        dst[kk][3] = ld4(a.abar + (size_t)jj * kF + col);
                        dst[kk][NL - 1] = ld4(a.io + (size_t)p * kF + col);
                    }
                }
            }
        };
        if (has_work) {
            load_idx(blockIdx.x, cur_i, cur_j);
#pragma unroll
            for (int m = 0; m < D - 1; ++m) issue(blockIdx.x, cur_i, cur_j, m / NG, m % NG, win[m]);
        }
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
            const int prow0 = tile * TM + q * 32;
            const int next_tile = tile + (int)gridDim.x;
            load_idx(next_tile, nxt_i, nxt_j);
            mbar_wait(bar_t_full + 8 * buf, acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * C::ACC_COLS;
            float xs[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) xs[k] = 0.f;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int c0 = half * 64 + c * 32;
                const int col = c0 + 4 * c8;
                {
                    uint32_t v[32];
                    tmem_ld32(taddr + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                            make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                        __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                }
                __syncwarp();
                float4 y[BWD ? 8 : 1];
#pragma unroll
                for (int g = 0; g < NG; ++g) {
                    const int n = c * NG + g, m = n + D - 1;            // static after unrolling; consume n, issue m
                    if (m < GT) issue(tile, cur_i, cur_j, m / NG, m % NG, win[m % D]);
                    else if (next_tile < n_tiles) issue(next_tile, nxt_i, nxt_j, (m - GT) / NG, (m - GT) % NG, win[m % D]);
                    float4 (&w)[G][NL] = win[n % D];
#pragma unroll
                    for (int kk = 0; kk < G; ++kk) {
                        const int k = g * G + kk;
                        const int row = k * 4 + r4;
                        const int p = prow0 + row;
                        const float4 me = *reinterpret_cast<const float4*>(stg + row * 128 + ((c8 ^ (row & 7)) << 4));
                        if (p < M) {
                            const float4 prod = f4_mul(w[kk][0], w[kk][1]);
                            if (!BWD) {
                                st4(a.io + (size_t)p * kF + col, f4_mul(me, prod));
                            } else {
                                const float4 mt = f4_add(w[kk][NL - 1], f4_add(w[kk][2], w[kk][3]));
                                y[BWD ? k : 0] = f4_mul(mt, prod);
                                st4(a.io + (size_t)p * kF + col, f4_mul(mt, me));
                            }
                        } else if (BWD) {
                            y[BWD ? k : 0] = f4_zero();
                        }
                    }
                }
                __syncwarp();
                if (BWD) {                              // second accumulator: dme = We drbf_p
                    uint32_t v[32];
                    tmem_ld32(taddr + 128 + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                            make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                        __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                    __syncwarp();
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const int row = k * 4 + r4;
                        const float4 dme = *reinterpret_cast<const float4*>(stg + row * 128 + ((c8 ^ (row & 7)) << 4));
                        xs[k] += f4_dot(y[BWD ? k : 0], dme);
                    }
                    __syncwarp();
                }
                if (c == 1) {                           // both accumulators fully read: hand the buffer back
                    tc_fence_before();
                    mbar_arrive(bar_t_empty + 8 * buf);
                }
            }
            if (BWD) {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    float s = xs[k];
                    s += __shfl_xor_sync(0xffffffffu, s, 1);
                    s += __shfl_xor_sync(0xffffffffu, s, 2);
                    s += __shfl_xor_sync(0xffffffffu, s, 4);
                    const int p = prow0 + k * 4 + r4;
                    if (c8 == 0 && p < M) a.x_part[(size_t)half * a.cap + p] = s;
                }
            }
            cur_i = nxt_i; cur_j = nxt_j;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS) : "memory");
    }
}

// We [128 f][20 n] (torch layout of message_edgepart.weight)  ->  image[hi|lo][f][swizzled, K padded to 32]
__global__ void k_message_prepare_b(const float* __restrict__ We, float* __restrict__ img) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 128 * 32) return;
    int n = t >> 5, k = t & 31;
    float x = k < kNB ? We[(size_t)n * kNB + k] : 0.f;
    float hi = tf32_hi(x);
    uint32_t off = swz_offset_bytes(n, k >> 2) + (k & 3) * 4;
    img[off / 4] = hi;
    img[(BLK_BYTES + off) / 4] = x - hi;
}

bool g_attr[2] = {false, false};

template <bool BWD>
int launch(const MsgArgs& a, cudaStream_t s) {
    using C = Cfg<BWD>;
    if (!g_attr[BWD]) {
        cudaError_t e = cudaFuncSetAttribute(k_message_tc<BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
        if (e != cudaSuccess) { nn_set_error("message_tc: cannot set %u B dynamic smem: %s", C::SMEM, cudaGetErrorString(e)); return -2; }
        g_attr[BWD] = true;
    }
    const int tiles = nn_ceil_div(a.cap, TM), sms = nn_num_sms();
    const int grid = tiles < sms ? tiles : sms;
    NN_LAUNCHED(1);
    return launch_pdl(k_message_tc<BWD>, grid, THREADS, C::SMEM, s, a);
}

}  // namespace

extern "C" int nn_message_prepare_b(const float* We, float* image, void* stream) {
    NN_REQUIRE(We && image, "null pointer");
    k_message_prepare_b<<<128 * 32 / 256, 256, 0, (cudaStream_t)stream>>>(We, image); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("nn_message_prepare_b");
    return 0;
}

int nn_message_fwd_tc(const nn_nbr* nl, const float* rbf, const float* mn, const float* We_img, float* msg, cudaStream_t s) {
    if (nl->cap_pairs <= 0) return 0;
    MsgArgs a{};
    a.rbf = rbf; a.B_img = We_img; a.pair_i = nl->pair_i; a.pair_j = nl->pair_j; a.mn = mn; a.io = msg;
    a.n_dev = nl->status + NN_ST_N_PAIRS; a.cap = nl->cap_pairs;
    if (int rc = launch<false>(a, s)) return rc;
    NN_CHECK_LAUNCH("message_fwd(tc)");
    return 0;
}

int nn_message_bwd_tc(const nn_nbr* nl, const float* abar, const float* mn, const float* rbf, const float* drbf,
                      const float* We_img, float* mbar_io, float* x_part, cudaStream_t s) {
    if (nl->cap_pairs <= 0) return 0;
    MsgArgs a{};
    a.rbf = rbf; a.drbf = drbf; a.B_img = We_img; a.pair_i = nl->pair_i; a.pair_j = nl->pair_j; a.mn = mn; a.abar = abar;
    a.io = mbar_io; a.x_part = x_part; a.n_dev = nl->status + NN_ST_N_PAIRS; a.cap = nl->cap_pairs;
    if (int rc = launch<true>(a, s)) return rc;
    NN_CHECK_LAUNCH("message_bwd(tc)");
    return 0;
}
