// Edge-stream kernels of the interaction layers: pair geometry, message, destination-sorted gather /
// reduce (forward and reverse sweep), energy head, force / virial reduction.
//
// All of these are HBM / L2-bandwidth-bound row streams: one warp owns one 128-float feature row
// (float4 per lane, 512 B fully coalesced), the per-atom sums run over the destination-sorted CSR in a
// fixed order (deterministic, no atomics - the reference's scatter_add_ is atomic on CUDA).
//
// Reference code replaced (paths relative to the reference repo):
//   ScaledNorm / PolynomialCutoff / RadialBesselLayer   newtonnet/layers/representations.py:118-133,155-171,223-235
//   InteractionNet.forward (message, scatter, update)   newtonnet/models/newtonnet.py:207-237
//   EnergyOutput last layer, ScaleShift, EnergyAggregator  newtonnet/models/output.py:98-100,246; layers/scalers.py:55-58
//   DerivativeProperty._save_grad (autograd replay)     newtonnet/models/output.py:66-73  -> SURVEY.md section 8a row B
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
// per-atom reductions (k_node_aggregate_*): atoms of one block are consecutive, so they share neighbours and pairs and
// L1 serves the re-reads; larger blocks = more sharing per L1 working set
#ifndef NN_AGG_THREADS
#define NN_AGG_THREADS 256      // measured on c2 / c4: 512 threads +12..20 %, 1024 threads +6..55 % kernel time
#endif
constexpr int kAggThreads = NN_AGG_THREADS;
constexpr int kAggWarps = kAggThreads / 32;

__device__ __forceinline__ int dev_count(const int* n_dev, int cap) {
    int n = n_dev ? *n_dev : cap;
    return n < cap ? n : cap;
}

// ---------------------------------------------------------------------------- geometry
// env(x) = 1 - 55x^9 + 99x^10 - 45x^11 = (1-x)^3 * sum_{k=0..8} C(k+2,2) x^k  (exact identity, see
// tests/test_oracle.py::test_cutoff_envelope_factorisation); the factored form has no cancellation
// near the cutoff.  env'(x) = -495 x^8 (1-x)^2.
__device__ __forceinline__ float envelope(float x) {
    float p = 45.f;
    p = fmaf(p, x, 36.f); p = fmaf(p, x, 28.f); p = fmaf(p, x, 21.f); p = fmaf(p, x, 15.f);
    p = fmaf(p, x, 10.f); p = fmaf(p, x, 6.f); p = fmaf(p, x, 3.f); p = fmaf(p, x, 1.f);
    float t = 1.0f - x;
    return t * t * t * p;
}
__device__ __forceinline__ float envelope_grad(float x) {
    float x2 = x * x, x4 = x2 * x2, t = 1.0f - x;
    return -495.f * x4 * x4 * t * t;
}

// Five lanes per pair, four basis functions each: every lane stores one float4 of the pair's 80-byte rbf / drbf rows,
// so a warp's stores cover consecutive 16-byte pieces (a thread-per-pair loop writes 32 different rows per instruction).
__global__ void __launch_bounds__(320)
k_edge_geom_fwd(const float* __restrict__ disp, const float* __restrict__ freq, float cutoff,
                const int* __restrict__ n_dev, int cap, float* __restrict__ rbf,
                float* __restrict__ drbf, float* __restrict__ unit, float* __restrict__ dist) {
    NN_PDL_TRIGGER();
    static_assert(kNB == 20, "five float4 per basis row");
    const int P = dev_count(n_dev, cap);
    const long long total = (long long)P * 5;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int p = (int)(t / 5), quad = (int)(t - (long long)p * 5);
        float3 d3 = make_float3(disp[3 * p], disp[3 * p + 1], disp[3 * p + 2]);
        float d = nn_norm3(d3);
        if (quad == 0) {
            unit[3 * p] = __fdiv_rn(d3.x, d); unit[3 * p + 1] = __fdiv_rn(d3.y, d); unit[3 * p + 2] = __fdiv_rn(d3.z, d);
            dist[p] = d;
        }
        float x = __fdiv_rn(d, cutoff);
        float env = envelope(x), envp = envelope_grad(x), invx = 1.0f / x;
        const float fr[4] = {freq[4 * quad], freq[4 * quad + 1], freq[4 * quad + 2], freq[4 * quad + 3]};
        float r[4], dr[4];
#pragma unroll
        for (int n = 0; n < 4; ++n) {
            float fx = fr[n] * x, sn, cs;
            sincosf(fx, &sn, &cs);
            float sb = sn * invx;
            r[n] = env * sb;
            // d/dx [env(x) sin(f x)/x] = env' sb + env (f x cos(f x) - sin(f x)) / x^2
            dr[n] = fmaf(envp, sb, env * (fx * cs - sn) * invx * invx);
        }
        st4(rbf + (size_t)p * kNB + 4 * quad, make_float4(r[0], r[1], r[2], r[3]));
        if (drbf) st4(drbf + (size_t)p * kNB + 4 * quad, make_float4(dr[0], dr[1], dr[2], dr[3]));
    }
}

// G_p = dE/d disp_p = (xbar / rc) u + (ubar - <ubar,u> u) / d, with xbar = dE/dx accumulated by the
// reverse message kernels (xbar_p = sum_layers <y_p, We drbf_p>).
__global__ void k_edge_geom_bwd(const float* __restrict__ x_bar, int n_slots, const float* __restrict__ unit_bar,
                                const float* __restrict__ unit, const float* __restrict__ dist, float cutoff,
                                const int* __restrict__ n_dev, int cap, float* __restrict__ disp_bar) {
    NN_PDL_TRIGGER();
    const int P = dev_count(n_dev, cap);
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
        float d = dist[p];
        float3 u = make_float3(unit[3 * p], unit[3 * p + 1], unit[3 * p + 2]);
        float3 ub = make_float3(unit_bar[3 * p], unit_bar[3 * p + 1], unit_bar[3 * p + 2]);
        float dot = ub.x * u.x + ub.y * u.y + ub.z * u.z;
        float xb = 0.f;
        for (int sl = 0; sl < n_slots; ++sl) xb += x_bar[(size_t)sl * cap + p];     // fixed order
        float a = xb / cutoff, invd = 1.0f / d;
        disp_bar[3 * p] = fmaf(a, u.x, (ub.x - dot * u.x) * invd);
        disp_bar[3 * p + 1] = fmaf(a, u.y, (ub.y - dot * u.y) * invd);
        disp_bar[3 * p + 2] = fmaf(a, u.z, (ub.z - dot * u.z) * invd);
    }
}

// ---------------------------------------------------------------------------- message (forward)
// me = We rbf_p (K = 20, SIMT: 0.4 % of the layer's FLOPs), m_p = me * (mn_i * mn_j).
__device__ __forceinline__ float4 edge_part(const float* __restrict__ s_wet, const float* __restrict__ rbf_row,
                                            int lane) {
    float4 me = f4_zero();
#pragma unroll 1
    for (int q = 0; q < kNB / 4; ++q) {
        float4 r = ld4(rbf_row + 4 * q);          // same address in all lanes: one broadcast transaction
        me = f4_fma(r.x, ld4(s_wet + (4 * q + 0) * kF + 4 * lane), me);
        me = f4_fma(r.y, ld4(s_wet + (4 * q + 1) * kF + 4 * lane), me);
        me = f4_fma(r.z, ld4(s_wet + (4 * q + 2) * kF + 4 * lane), me);
        me = f4_fma(r.w, ld4(s_wet + (4 * q + 3) * kF + 4 * lane), me);
    }
    return me;
}

// Pairs are stored grouped by their lower atom i (pair_ptr), so one warp walks the forward pairs of one
// atom: the i-side rows are loaded once per atom and only the j-side rows are gathered per pair.  The
// pairs of an atom are contiguous, so their rbf rows are staged into shared memory with coalesced loads
// (a chunk of pairs at a time) and the j-side gather of the next pair is issued before the current pair
// is computed (software prefetch) - the kernels are latency-bound otherwise.
constexpr int kMsgChunk = 32;
__global__ void __launch_bounds__(kThreads, 3)
k_edge_message_fwd(const int* __restrict__ pair_ptr, const int* __restrict__ pair_j, int N, int cap,
                   const float* __restrict__ rbf, const float* __restrict__ mn,
                   const float* __restrict__ Wet, float* __restrict__ msg) {
    __shared__ __align__(16) float s_wet[kNB * kF];
    __shared__ __align__(16) float s_rbf[kWarps][kMsgChunk * kNB];
    for (int k = threadIdx.x; k < kNB * kF; k += kThreads) s_wet[k] = Wet[k];
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    float* my_rbf = s_rbf[wid];
    for (int i = blockIdx.x * kWarps + wid; i < N; i += gridDim.x * kWarps) {
        const int p0 = pair_ptr[i], p1 = min(pair_ptr[i + 1], cap);
        if (p0 >= p1) continue;
        const float4 a = ld4(mn + (size_t)i * kF + 4 * lane);
        for (int c0 = p0; c0 < p1; c0 += kMsgChunk) {
            const int n = min(kMsgChunk, p1 - c0);
            const int my_j = lane < n ? pair_j[c0 + lane] : 0;
            for (int t = lane; t < n * (kNB / 4); t += 32) st4(my_rbf + 4 * t, ld4(rbf + (size_t)c0 * kNB + 4 * t));
            __syncwarp();
            float4 b_next = ld4(mn + (size_t)__shfl_sync(0xffffffffu, my_j, 0) * kF + 4 * lane);
            for (int t = 0; t < n; ++t) {
                const float4 b = b_next;
                const int jn = __shfl_sync(0xffffffffu, my_j, (t + 1) & 31);
                if (t + 1 < n) b_next = ld4(mn + (size_t)jn * kF + 4 * lane);
                float4 me = edge_part(s_wet, my_rbf + t * kNB, lane);
                st4(msg + (size_t)(c0 + t) * kF + 4 * lane, f4_mul(me, f4_mul(a, b)));
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------- gather / reduce (forward)
// a_out_i = a_i + sum_{e->i} m_p(e);  f_out_i[c] = f_i[c] + sum_{e->i} (s_e u_p[c] e1_p + e2_p * f_j[c])
template <bool FIRST>
__global__ void __launch_bounds__(kAggThreads)
k_node_aggregate_fwd(const int* __restrict__ status, const int* __restrict__ row_ptr, const int* __restrict__ col,
                     const int* __restrict__ edge_pair, int N, const float* __restrict__ msg, const float* __restrict__ e1,
                     const float* __restrict__ e2, const float* __restrict__ unit, const float* __restrict__ a_in,
                     const float* __restrict__ f_in, float* __restrict__ a_out, float* __restrict__ f_out) {
    NN_PDL_TRIGGER();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kAggWarps + (threadIdx.x >> 5);
    if (i >= N || status[NN_ST_EDGE_OVERFLOW] != 0) return;   // overflow: row_ptr is ahead of col / edge_pair
    const int r0 = row_ptr[i], r1 = row_ptr[i + 1];
    float4 am = f4_zero(), fx = f4_zero(), fy = f4_zero(), fz = f4_zero();
    for (int e0 = r0; e0 < r1; e0 += 32) {
        int my_p = 0, my_j = 0;
        float ux = 0.f, uy = 0.f, uz = 0.f;
        if (e0 + lane < r1) {
            int ep = edge_pair[e0 + lane];
            my_j = col[e0 + lane];
            my_p = ep & 0x7fffffff;
            float sgn = ep < 0 ? -1.0f : 1.0f;
            ux = sgn * unit[3 * my_p]; uy = sgn * unit[3 * my_p + 1]; uz = sgn * unit[3 * my_p + 2];
        }
        const int cnt = min(32, r1 - e0);
        for (int t = 0; t < cnt; ++t) {
            const int p = __shfl_sync(0xffffffffu, my_p, t);
            const float sx = __shfl_sync(0xffffffffu, ux, t), sy = __shfl_sync(0xffffffffu, uy, t),
                        sz = __shfl_sync(0xffffffffu, uz, t);
            const size_t po = (size_t)p * kF + 4 * lane;
            // (pair rows through L1 on purpose: the atoms of a block share pairs; L1::no_allocate loads were measured at
            //  +25 % kernel time on c2 and c4)
            am = f4_add(am, ld4(msg + po));
            float4 v1 = ld4(e1 + po);
            fx = f4_fma(sx, v1, fx); fy = f4_fma(sy, v1, fy); fz = f4_fma(sz, v1, fz);
            if (!FIRST) {
                const int j = __shfl_sync(0xffffffffu, my_j, t);
                float4 v2 = ld4(e2 + po);
                const float* fj = f_in + (size_t)j * 3 * kF + 4 * lane;
                fx = f4_fma(v2, ld4(fj), fx); fy = f4_fma(v2, ld4(fj + kF), fy); fz = f4_fma(v2, ld4(fj + 2 * kF), fz);
            }
        }
    }
    st4(a_out + (size_t)i * kF + 4 * lane, f4_add(ld4(a_in + (size_t)i * kF + 4 * lane), am));
    float* fo = f_out + (size_t)i * 3 * kF + 4 * lane;
    if (FIRST) {
        st4(fo, fx); st4(fo + kF, fy); st4(fo + 2 * kF, fz);
    } else {
        const float* fi = f_in + (size_t)i * 3 * kF + 4 * lane;
        st4(fo, f4_add(ld4(fi), fx)); st4(fo + kF, f4_add(ld4(fi + kF), fy)); st4(fo + 2 * kF, f4_add(ld4(fi + 2 * kF), fz));
    }
}

__global__ void k_equiv_update_fwd(const float* __restrict__ a_in, const float* __restrict__ f,
                                   const float* __restrict__ g, float* __restrict__ a_out, int N) {
    NN_PDL_TRIGGER();
    int t = blockIdx.x * blockDim.x + threadIdx.x;       // one float4 of one atom
    if (t >= N * (kF / 4)) return;
    int i = t / (kF / 4), q = (t % (kF / 4)) * 4;
    const float* fi = f + (size_t)i * 3 * kF + q;
    const float* gi = g + (size_t)i * 3 * kF + q;
    float4 acc = ld4(a_in + (size_t)i * kF + q);
    acc = f4_fma(ld4(fi), ld4(gi), acc);
    acc = f4_fma(ld4(fi + kF), ld4(gi + kF), acc);
    acc = f4_fma(ld4(fi + 2 * kF), ld4(gi + 2 * kF), acc);
    st4(a_out + (size_t)i * kF + q, acc);
}

__global__ void k_embed(const int64_t* __restrict__ z, const float* __restrict__ emb, float* __restrict__ a, int N,
                        int* __restrict__ status) {
    NN_PDL_TRIGGER();
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N * (kF / 4)) return;
    int i = t / (kF / 4), q = (t % (kF / 4)) * 4;
    long long zi = z[i];
    if (zi < 0 || zi > 118) { zi = 0; atomicExch(&status[NN_ST_BATCH_UNSORTED], 3); }
    st4(a + (size_t)i * kF + q, ld4(emb + (size_t)zi * kF + q));
}

// ---------------------------------------------------------------------------- layer norm (layer_norm=True)
// nn.LayerNorm(F) on atom_node at the end of a layer (models/newtonnet.py:234-235): eps 1e-5, biased variance.
__global__ void __launch_bounds__(kThreads)
k_layer_norm_fwd(float* __restrict__ a_io, const float* __restrict__ gamma, const float* __restrict__ beta,
                 float* __restrict__ xhat, float* __restrict__ rstd, int n_rows) {
    NN_PDL_TRIGGER();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    float4 x = ld4(a_io + (size_t)i * kF + 4 * lane);
    const float mean = warp_sum(x.x + x.y + x.z + x.w) * (1.0f / kF);
    const float4 d = make_float4(x.x - mean, x.y - mean, x.z - mean, x.w - mean);
    const float var = warp_sum(f4_dot(d, d)) * (1.0f / kF);
    const float r = rsqrtf(var + 1e-5f);
    const float4 h = make_float4(d.x * r, d.y * r, d.z * r, d.w * r);
    if (xhat) st4(xhat + (size_t)i * kF + 4 * lane, h);
    if (rstd && lane == 0) rstd[i] = r;
    st4(a_io + (size_t)i * kF + 4 * lane, f4_fma(h, ld4(gamma + 4 * lane), ld4(beta + 4 * lane)));
}
// abar_in = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = abar_out * gamma
__global__ void __launch_bounds__(kThreads)
k_layer_norm_bwd(float* __restrict__ abar_io, const float* __restrict__ gamma, const float* __restrict__ xhat,
                 const float* __restrict__ rstd, int n_rows) {
    NN_PDL_TRIGGER();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const float4 g = f4_mul(ld4(abar_io + (size_t)i * kF + 4 * lane), ld4(gamma + 4 * lane));
    const float4 h = ld4(xhat + (size_t)i * kF + 4 * lane);
    const float m1 = warp_sum(g.x + g.y + g.z + g.w) * (1.0f / kF);
    const float m2 = warp_sum(f4_dot(g, h)) * (1.0f / kF);
    const float r = rstd[i];
    st4(abar_io + (size_t)i * kF + 4 * lane, make_float4(r * (g.x - m1 - h.x * m2), r * (g.y - m1 - h.y * m2),
                                                          r * (g.z - m1 - h.z * m2), r * (g.w - m1 - h.w * m2)));
}

// direct_force head tail (models/output.py:129-131 + scalers.py:55-56): F_i[c] = scale[z_i] * <h_i, f_i[c]>
__global__ void __launch_bounds__(kThreads)
k_direct_force(const float* __restrict__ h, const float* __restrict__ f, const float* __restrict__ scale,
               const int64_t* __restrict__ z, int n_rows, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const float4 hv = ld4(h + (size_t)i * kF + 4 * lane);
    const float* fi = f + (size_t)i * 3 * kF + 4 * lane;
    const float sx = warp_sum(f4_dot(hv, ld4(fi))), sy = warp_sum(f4_dot(hv, ld4(fi + kF))), sz = warp_sum(f4_dot(hv, ld4(fi + 2 * kF)));
    if (lane == 0) {
        long long zi = z[i]; if (zi < 0 || zi > 118) zi = 0;
        const float sc = scale[zi];
        out[3 * i] = sc * sx; out[3 * i + 1] = sc * sy; out[3 * i + 2] = sc * sz;
    }
}

// ---------------------------------------------------------------------------- energy head
__global__ void __launch_bounds__(kThreads)
k_energy_atom(const float* __restrict__ h2pre, const float* __restrict__ w3, const float* __restrict__ b3,
              const float* __restrict__ scale, const float* __restrict__ shift, const int64_t* __restrict__ z,
              int N, float* __restrict__ e_atom) {
    NN_PDL_TRIGGER();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (i >= N) return;
    float4 h = ld4(h2pre + (size_t)i * kF + 4 * lane);
    h.x = silu_f(h.x); h.y = silu_f(h.y); h.z = silu_f(h.z); h.w = silu_f(h.w);
    float o = warp_sum(f4_dot(h, ld4(w3 + 4 * lane)));
    if (lane == 0) {
        long long zi = z[i]; if (zi < 0 || zi > 118) zi = 0;
        e_atom[i] = fmaf(o + b3[0], scale[zi], shift[zi]);
    }
}

// fixed-order fp64 sum per system (the reference sums sequentially in fp32; |shift| makes E large).  Large systems are cut
// into S slices (grid.y), one block each, and a second kernel adds the S partial sums in slice order: one block per
// system took 29 us (energy) / 215 us (virial) on the 98,304-atom box.  W values per atom.
template <int W>
__global__ void __launch_bounds__(kThreads)
k_sys_sum_partial(const float* __restrict__ val, const int* __restrict__ sys_ptr, int n_rows, int S, double* __restrict__ partial) {
    __shared__ double sm[kThreads][W];
    const int b = blockIdx.x, sl = blockIdx.y;
    const int first = sys_ptr[b], last = min(sys_ptr[b + 1], n_rows);
    const int len = max(last - first, 0);
    const int i0 = first + (int)((long long)len * sl / S), i1 = first + (int)((long long)len * (sl + 1) / S);
    double acc[W];
#pragma unroll
    for (int k = 0; k < W; ++k) acc[k] = 0.0;
    for (int i = i0 + threadIdx.x; i < i1; i += kThreads)
#pragma unroll
        for (int k = 0; k < W; ++k) acc[k] += (double)val[(size_t)i * W + k];
#pragma unroll
    for (int k = 0; k < W; ++k) sm[threadIdx.x][k] = acc[k];
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o)
#pragma unroll
            for (int k = 0; k < W; ++k) sm[threadIdx.x][k] += sm[threadIdx.x + o][k];
        __syncthreads();
    }
    if (threadIdx.x < W) partial[((size_t)b * S + sl) * W + threadIdx.x] = sm[0][threadIdx.x];
}
__global__ void k_energy_final(const double* __restrict__ partial, int S, int B, float* __restrict__ energy) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double e = 0.0;
    for (int sl = 0; sl < S; ++sl) e += partial[(size_t)b * S + sl];
    energy[b] = (float)e;
}

__global__ void k_energy_sum(const float* __restrict__ e_atom, const int* __restrict__ sys_ptr, int n_rows,
                             float* __restrict__ energy) {
    __shared__ double s[kThreads];
    int b = blockIdx.x;
    double acc = 0.0;
    const int last = min(sys_ptr[b + 1], n_rows);
    for (int i = sys_ptr[b] + threadIdx.x; i < last; i += kThreads) acc += (double)e_atom[i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) energy[b] = (float)s[0];
}

// dE/d h2pre = scale[z] * w3 * silu'(h2pre)
__global__ void k_energy_head_seed(const float* __restrict__ h2pre, const float* __restrict__ w3,
                                   const float* __restrict__ scale, const int64_t* __restrict__ z, int N,
                                   float* __restrict__ gh2) {
    NN_PDL_TRIGGER();
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N * (kF / 4)) return;
    int i = t / (kF / 4), q = (t % (kF / 4)) * 4;
    long long zi = z[i]; if (zi < 0 || zi > 118) zi = 0;
    float sc = scale[zi];
    float4 h = ld4(h2pre + (size_t)i * kF + q), w = ld4(w3 + q);
    st4(gh2 + (size_t)i * kF + q, make_float4(sc * w.x * dsilu_f(h.x), sc * w.y * dsilu_f(h.y),
                                             sc * w.z * dsilu_f(h.z), sc * w.w * dsilu_f(h.w)));
}

// ---------------------------------------------------------------------------- reverse sweep, pair side
// w[c] = dfb_i[c] - dfb_j[c];  e1bar = sum_c w[c] u[c] (overwrites e1);  ubar[c] += <w[c], e1>;
// e2bar = sum_c dfb_i[c] * f_in_j[c] + dfb_j[c] * f_in_i[c]
#ifndef NN_GATHER_BLOCKS
#define NN_GATHER_BLOCKS 2      // <= 128 registers; 3 blocks (85 registers): no change, 1 block (unbounded registers): +44 % time
#endif
template <bool FIRST>
__global__ void __launch_bounds__(kThreads, NN_GATHER_BLOCKS)
k_pair_bwd_gather(const int* __restrict__ pair_ptr, const int* __restrict__ pair_j, int N, int cap,
                  const float* __restrict__ dfb, const float* __restrict__ f_in,
                  const float* __restrict__ unit, float* __restrict__ e1_io, float* __restrict__ e2bar,
                  float* __restrict__ ubar) {
    NN_PDL_TRIGGER();
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * kWarps + (threadIdx.x >> 5); i < N; i += gridDim.x * kWarps) {
        const int p0 = pair_ptr[i], p1 = min(pair_ptr[i + 1], cap);
        if (p0 >= p1) continue;
        const float* di = dfb + (size_t)i * 3 * kF + 4 * lane;
        const float4 dix = ld4(di), diy = ld4(di + kF), diz = ld4(di + 2 * kF);
        float4 fix = f4_zero(), fiy = f4_zero(), fiz = f4_zero();
        if (!FIRST) {
            const float* fi = f_in + (size_t)i * 3 * kF + 4 * lane;
            fix = ld4(fi); fiy = ld4(fi + kF); fiz = ld4(fi + 2 * kF);
        }
        // software prefetch: the rows of pair p+1 are requested before pair p is reduced
        float4 ndx, ndy, ndz, nfx = f4_zero(), nfy = f4_zero(), nfz = f4_zero(), nv1;
        auto fetch = [&](int p) {
            const int j = pair_j[p];
            const float* dj = dfb + (size_t)j * 3 * kF + 4 * lane;
            ndx = ld4(dj); ndy = ld4(dj + kF); ndz = ld4(dj + 2 * kF);
            if (!FIRST) {
                const float* fj = f_in + (size_t)j * 3 * kF + 4 * lane;
                nfx = ld4(fj); nfy = ld4(fj + kF); nfz = ld4(fj + 2 * kF);
            }
            nv1 = ld4(e1_io + (size_t)p * kF + 4 * lane);
        };
        fetch(p0);
        for (int p = p0; p < p1; ++p) {
            const float4 djx = ndx, djy = ndy, djz = ndz, fjx = nfx, fjy = nfy, fjz = nfz, v1 = nv1;
            if (p + 1 < p1) fetch(p + 1);
            const float4 wx = f4_sub(dix, djx), wy = f4_sub(diy, djy), wz = f4_sub(diz, djz);
            const float ux = unit[3 * p], uy = unit[3 * p + 1], uz = unit[3 * p + 2];
            const size_t po = (size_t)p * kF + 4 * lane;
            float sx = warp_sum(f4_dot(wx, v1)), sy = warp_sum(f4_dot(wy, v1)), sz = warp_sum(f4_dot(wz, v1));
            if (lane == 0) { ubar[3 * p] += sx; ubar[3 * p + 1] += sy; ubar[3 * p + 2] += sz; }
            float4 e1b = f4_zero();
            e1b = f4_fma(ux, wx, e1b); e1b = f4_fma(uy, wy, e1b); e1b = f4_fma(uz, wz, e1b);
            st4(e1_io + po, e1b);
            if (!FIRST) {
                float4 acc = f4_mul(dix, fjx);
                acc = f4_fma(diy, fjy, acc); acc = f4_fma(diz, fjz, acc);
                acc = f4_fma(djx, fix, acc); acc = f4_fma(djy, fiy, acc); acc = f4_fma(djz, fiz, acc);
                st4(e2bar + po, acc);
            }
        }
    }
}

// mtot = mbar + abar_i + abar_j;  y = mtot * mn_i * mn_j;  xbar_p += <y, We drbf_p>  (one warp reduction:
// dE/dx is contracted with We here, instead of keeping a 20-wide rbf gradient per pair);
// t = mtot * (We rbf_p)  (overwrites mbar)
constexpr int kBwdChunk = 16;
__global__ void __launch_bounds__(kThreads, 3)
k_pair_bwd_message(const int* __restrict__ pair_ptr, const int* __restrict__ pair_j, int N, int cap,
                   const float* __restrict__ abar, const float* __restrict__ mn,
                   const float* __restrict__ rbf, const float* __restrict__ drbf, const float* __restrict__ Wet,
                   float* __restrict__ mbar_io, float* __restrict__ x_bar) {
    __shared__ __align__(16) float s_wet[kNB * kF];
    __shared__ __align__(16) float s_r[kWarps][kBwdChunk * kNB];
    __shared__ __align__(16) float s_d[kWarps][kBwdChunk * kNB];
    for (int k = threadIdx.x; k < kNB * kF; k += kThreads) s_wet[k] = Wet[k];
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    float* my_r = s_r[wid];
    float* my_d = s_d[wid];
    for (int i = blockIdx.x * kWarps + wid; i < N; i += gridDim.x * kWarps) {
        const int p0 = pair_ptr[i], p1 = min(pair_ptr[i + 1], cap);
        if (p0 >= p1) continue;
        const float4 ab_i = ld4(abar + (size_t)i * kF + 4 * lane);
        const float4 mn_i = ld4(mn + (size_t)i * kF + 4 * lane);
        for (int c0 = p0; c0 < p1; c0 += kBwdChunk) {
            const int n = min(kBwdChunk, p1 - c0);
            const int my_j = lane < n ? pair_j[c0 + lane] : 0;
            for (int t = lane; t < n * (kNB / 4); t += 32) {
                st4(my_r + 4 * t, ld4(rbf + (size_t)c0 * kNB + 4 * t));
                st4(my_d + 4 * t, ld4(drbf + (size_t)c0 * kNB + 4 * t));
            }
            __syncwarp();
            float4 n_m, n_ab, n_mn;
            {
                const int j0 = __shfl_sync(0xffffffffu, my_j, 0);
                n_m = ld4(mbar_io + (size_t)c0 * kF + 4 * lane);
                n_ab = ld4(abar + (size_t)j0 * kF + 4 * lane); n_mn = ld4(mn + (size_t)j0 * kF + 4 * lane);
            }
            for (int t = 0; t < n; ++t) {
                const size_t po = (size_t)(c0 + t) * kF + 4 * lane;
                const float4 mt = f4_add(n_m, f4_add(ab_i, n_ab));
                const float4 y = f4_mul(mt, f4_mul(mn_i, n_mn));
                const int jn = __shfl_sync(0xffffffffu, my_j, (t + 1) & 31);
                if (t + 1 < n) {
                    n_m = ld4(mbar_io + po + kF);
                    n_ab = ld4(abar + (size_t)jn * kF + 4 * lane); n_mn = ld4(mn + (size_t)jn * kF + 4 * lane);
                }
                // me = We rbf_p and dme = We drbf_p share the We loads
                float4 me = f4_zero(), dme = f4_zero();
                const float* r = my_r + t * kNB;
                const float* dr = my_d + t * kNB;
#pragma unroll
                for (int q = 0; q < kNB / 4; ++q) {
                    const float4 rv = ld4(r + 4 * q), dv = ld4(dr + 4 * q);
                    float4 w;
                    w = ld4(s_wet + (4 * q + 0) * kF + 4 * lane); me = f4_fma(rv.x, w, me); dme = f4_fma(dv.x, w, dme);
                    w = ld4(s_wet + (4 * q + 1) * kF + 4 * lane); me = f4_fma(rv.y, w, me); dme = f4_fma(dv.y, w, dme);
                    w = ld4(s_wet + (4 * q + 2) * kF + 4 * lane); me = f4_fma(rv.z, w, me); dme = f4_fma(dv.z, w, dme);
                    w = ld4(s_wet + (4 * q + 3) * kF + 4 * lane); me = f4_fma(rv.w, w, me); dme = f4_fma(dv.w, w, dme);
                }
                const float xs = warp_sum(f4_dot(y, dme));
                if (lane == 0) x_bar[c0 + t] = xs;                 // this layer's slot (summed in k_edge_geom_bwd)
                st4(mbar_io + po, f4_mul(mt, me));
            }
            __syncwarp();
        }
    }
}

// mnbar_k = sum_{e=(k,i)} t_p * mn_i ;  fbar_new_k[c] = dfb_k[c] + sum_{e=(k,i)} dfb_i[c] * e2_p
template <bool FIRST>
__global__ void __launch_bounds__(kAggThreads)
k_node_aggregate_bwd(const int* __restrict__ status, const int* __restrict__ row_ptr, const int* __restrict__ col,
                     const int* __restrict__ edge_pair, int N, const float* __restrict__ t, const float* __restrict__ mn, const float* __restrict__ e2,
                     const float* __restrict__ dfb, float* __restrict__ mnbar, float* __restrict__ fbar_new) {
    NN_PDL_TRIGGER();
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * kAggWarps + (threadIdx.x >> 5);
    if (k >= N || status[NN_ST_EDGE_OVERFLOW] != 0) return;
    const int r0 = row_ptr[k], r1 = row_ptr[k + 1];
    float4 am = f4_zero(), fx = f4_zero(), fy = f4_zero(), fz = f4_zero();
    for (int e0 = r0; e0 < r1; e0 += 32) {
        int my_p = 0, my_i = 0;
        if (e0 + lane < r1) { my_p = edge_pair[e0 + lane] & 0x7fffffff; my_i = col[e0 + lane]; }
        const int cnt = min(32, r1 - e0);
        for (int s = 0; s < cnt; ++s) {
            const int p = __shfl_sync(0xffffffffu, my_p, s);
            const int i = __shfl_sync(0xffffffffu, my_i, s);
            const size_t po = (size_t)p * kF + 4 * lane;
            am = f4_fma(ld4(t + po), ld4(mn + (size_t)i * kF + 4 * lane), am);
            if (!FIRST) {
                float4 v2 = ld4(e2 + po);
                const float* di = dfb + (size_t)i * 3 * kF + 4 * lane;
                fx = f4_fma(v2, ld4(di), fx); fy = f4_fma(v2, ld4(di + kF), fy); fz = f4_fma(v2, ld4(di + 2 * kF), fz);
            }
        }
    }
    st4(mnbar + (size_t)k * kF + 4 * lane, am);
    if (!FIRST) {
        const float* dk = dfb + (size_t)k * 3 * kF + 4 * lane;
        float* fo = fbar_new + (size_t)k * 3 * kF + 4 * lane;
        st4(fo, f4_add(ld4(dk), fx)); st4(fo + kF, f4_add(ld4(dk + kF), fy)); st4(fo + 2 * kF, f4_add(ld4(dk + 2 * kF), fz));
    }
}

// ---------------------------------------------------------------------------- forces and virial
// F_i = -sum_{e=(i,j)} s_e G_p(e).  Virial with the reference's strain convention
// (models/newtonnet.py:153-155: pos' = pos @ S, cell' = cell @ S, shift = cell' @ n):
//   M[a,b] = sum_p dpos_a G_b - (cell^T G)_a n_b,  dE/dD = (M + M^T)/2, virial = -dE/dD.
// With dpos = disp + cell n:  sym(M) = sym(disp (x) G) + sym(X),  X[a,b] = (cell n)_a G_b - (cell^T G)_a n_b.
// sym(X) vanishes for cubic cells, is (L_a - L_b)(n_a G_b - G_a n_b)/2 for diagonal cells, and is the
// reference's (unphysical but reproducible) extra term otherwise.  Every pair term is invariant under
// swapping the pair's orientation, so each atom takes HALF of every incident edge: under domain
// decomposition the owner of the other endpoint adds the other half.  Systems are summed in fp64 in
// fixed order.
__global__ void __launch_bounds__(128)
k_force_virial_atom(const int* __restrict__ status, const int* __restrict__ row_ptr, const int* __restrict__ col,
                    const int* __restrict__ edge_pair, int n_rows, const float* __restrict__ G,
                    const float* __restrict__ pair_disp, const float* __restrict__ pos,
                    const int64_t* __restrict__ batch, const SysMeta* __restrict__ meta,
                    float* __restrict__ forces, float* __restrict__ vir_atom) {
    NN_PDL_TRIGGER();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows || status[NN_ST_EDGE_OVERFLOW] != 0) return;
    const int r0 = row_ptr[i], r1 = row_ptr[i + 1];
    float fx = 0.f, fy = 0.f, fz = 0.f;
    float m[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const bool want_vir = vir_atom != nullptr;
    SysMeta sm;
    sm.mode = 0;
    float3 pi = make_float3(0.f, 0.f, 0.f);
    bool quirk = false;
    if (want_vir) {
        sm = meta[batch[i]];
        pi = make_float3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
        quirk = sm.mode == 2 || (sm.mode == 1 && !(sm.L[0] == sm.L[1] && sm.L[1] == sm.L[2]));
    }
    for (int e = r0; e < r1; ++e) {
        const int ep = edge_pair[e];
        const int p = ep & 0x7fffffff;
        const float sgn = ep < 0 ? -1.0f : 1.0f;
        const float gg[3] = {sgn * G[3 * p], sgn * G[3 * p + 1], sgn * G[3 * p + 2]};     // dE/d disp of THIS edge
        fx -= gg[0]; fy -= gg[1]; fz -= gg[2];
        if (!want_vir) continue;
        const float dp[3] = {sgn * pair_disp[3 * p], sgn * pair_disp[3 * p + 1], sgn * pair_disp[3 * p + 2]};
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) m[3 * a + b] += 0.25f * (dp[a] * gg[b] + dp[b] * gg[a]);
        if (quirk) {
            int j = col[e];
            float3 d = make_float3(__fsub_rn(pi.x, pos[3 * j]), __fsub_rn(pi.y, pos[3 * j + 1]), __fsub_rn(pi.z, pos[3 * j + 2]));
            float3 n3;
            nn_min_image(d, sm, &n3);
            float nn[3] = {n3.x, n3.y, n3.z};
            float X[9];
            if (sm.mode == 1) {
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) X[3 * a + b] = sm.L[a] * (nn[a] * gg[b] - gg[a] * nn[b]);
            } else {
                float hn[3], hg[3];
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    hn[a] = sm.H[3 * a] * nn[0] + sm.H[3 * a + 1] * nn[1] + sm.H[3 * a + 2] * nn[2];
                    hg[a] = sm.H[a] * gg[0] + sm.H[3 + a] * gg[1] + sm.H[6 + a] * gg[2];
                }
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) X[3 * a + b] = hn[a] * gg[b] - hg[a] * nn[b];
            }
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) m[3 * a + b] += 0.25f * (X[3 * a + b] + X[3 * b + a]);
        }
    }
    forces[3 * i] = fx; forces[3 * i + 1] = fy; forces[3 * i + 2] = fz;
    if (want_vir) {
#pragma unroll
        for (int k = 0; k < 9; ++k) vir_atom[(size_t)i * 9 + k] = m[k];
    }
}

__global__ void k_virial_sum(const float* __restrict__ vir_atom, const int* __restrict__ sys_ptr, int n_rows,
                             const float* __restrict__ cell, float* __restrict__ virial, float* __restrict__ stress) {
    __shared__ double s[kThreads][9];
    int b = blockIdx.x;
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    const int last = min(sys_ptr[b + 1], n_rows);
    for (int i = sys_ptr[b] + threadIdx.x; i < last; i += kThreads)
        for (int k = 0; k < 9; ++k) acc[k] += (double)vir_atom[(size_t)i * 9 + k];
    for (int k = 0; k < 9; ++k) s[threadIdx.x][k] = acc[k];
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o)
            for (int k = 0; k < 9; ++k) s[threadIdx.x][k] += s[threadIdx.x + o][k];
        __syncthreads();
    }
    if (threadIdx.x < 9) {
        int a = threadIdx.x / 3, c = threadIdx.x % 3;
        double gd = 0.5 * (s[0][3 * a + c] + s[0][3 * c + a]);      // dE/dD
        virial[9 * b + threadIdx.x] = (float)(-gd);
        if (stress) {
            const float* h = cell + 9 * b;
            // fp32 determinant like torch.det on the fp32 cell (models/output.py:177)
            double det = (double)h[0] * ((double)h[4] * h[8] - (double)h[5] * h[7]) -
                         (double)h[1] * ((double)h[3] * h[8] - (double)h[5] * h[6]) +
                         (double)h[2] * ((double)h[3] * h[7] - (double)h[4] * h[6]);
            stress[9 * b + threadIdx.x] = (float)(gd / det);
        }
    }
}

__global__ void k_virial_final(const double* __restrict__ partial, int S, const float* __restrict__ cell,
                               float* __restrict__ virial, float* __restrict__ stress) {
    __shared__ double m[9];
    const int b = blockIdx.x;
    if (threadIdx.x < 9) {
        double a = 0.0;
        for (int sl = 0; sl < S; ++sl) a += partial[((size_t)b * S + sl) * 9 + threadIdx.x];
        m[threadIdx.x] = a;
    }
    __syncthreads();
    if (threadIdx.x < 9) {
        int a = threadIdx.x / 3, c = threadIdx.x % 3;
        double gd = 0.5 * (m[3 * a + c] + m[3 * c + a]);      // dE/dD
        virial[9 * b + threadIdx.x] = (float)(-gd);
        if (stress) {
            const float* h = cell + 9 * b;
            double det = (double)h[0] * ((double)h[4] * h[8] - (double)h[5] * h[7]) -
                         (double)h[1] * ((double)h[3] * h[8] - (double)h[5] * h[6]) +
                         (double)h[2] * ((double)h[3] * h[7] - (double)h[4] * h[6]);
            stress[9 * b + threadIdx.x] = (float)(gd / det);
        }
    }
}

// out[k,:] = src[idx[k],:]  (rows of `width` floats, width % 4 == 0): the rows this rank sends to a peer
__global__ void k_halo_pack(const float* __restrict__ src, const int* __restrict__ idx, int n, int width4,
                            float* __restrict__ out) {
    const long long total = (long long)n * width4;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(t / width4), c = (int)(t % width4);
        st4(out + ((size_t)k * width4 + c) * 4, ld4(src + ((size_t)idx[k] * width4 + c) * 4));
    }
}

int grid_for_rows(long long rows) {
    long long g = (rows + kWarps - 1) / kWarps;
    const long long cap = (long long)nn_num_sms() * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

// ============================================================================ host launchers
extern "C" int nn_edge_geom_fwd(const float* pair_disp, const float* freq, float cutoff, const int32_t* n_pairs_dev,
                                int32_t cap_pairs, float* rbf, float* drbf, float* unit, float* dist, void* stream) {
    if (cap_pairs <= 0) return 0;
    int grid = min(nn_ceil_div((long long)cap_pairs * 5, 320), nn_num_sms() * 6);
    k_edge_geom_fwd<<<grid, 320, 0, (cudaStream_t)stream>>>(pair_disp, freq, cutoff, n_pairs_dev, cap_pairs, rbf, drbf, unit, dist); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("nn_edge_geom_fwd");
    return 0;
}

extern "C" int nn_edge_geom_bwd(const float* x_bar, int32_t n_slots, const float* unit_bar, const float* unit,
                                const float* dist, float cutoff, const int32_t* n_pairs_dev, int32_t cap_pairs,
                                float* disp_bar, void* stream) {
    if (cap_pairs <= 0) return 0;
    int grid = min(nn_ceil_div(cap_pairs, 256), nn_num_sms() * 8);
    k_edge_geom_bwd<<<grid, 256, 0, (cudaStream_t)stream>>>(x_bar, n_slots, unit_bar, unit, dist, cutoff, n_pairs_dev, cap_pairs,
                                                            disp_bar); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("nn_edge_geom_bwd");
    return 0;
}

// SIMT twin of the tensor-core message kernel; the public nn_edge_message_fwd (eval.cu) picks between them
int nn_edge_message_fwd_launch(const nn_nbr* nl, const float* rbf, const float* mn, const float* Wet, float* msg,
                               cudaStream_t s) {
    if (nl->cap_pairs <= 0) return 0;
    k_edge_message_fwd<<<grid_for_rows(nl->n_atoms), kThreads, 0, s>>>(
        nl->pair_ptr, nl->pair_j, nl->n_atoms, nl->cap_pairs, rbf, mn, Wet, msg); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("message_fwd(simt)");
    return 0;
}

int nn_node_aggregate_fwd_rows(const nn_nbr* nl, int n_rows, const float* msg, const float* e1, const float* e2,
                               const float* unit, const float* a_in, const float* f_in, float* a_out, float* f_out,
                               bool first, cudaStream_t s);
extern "C" int nn_node_aggregate_fwd(const nn_nbr* nl, const float* msg, const float* e1, const float* e2,
                                     const float* unit, const float* a_in, const float* f_in, float* a_out,
                                     float* f_out, int32_t first_layer, void* stream) {
    return nn_node_aggregate_fwd_rows(nl, nl->n_atoms, msg, e1, e2, unit, a_in, f_in, a_out, f_out, first_layer != 0,
                                      (cudaStream_t)stream);
}
int nn_node_aggregate_fwd_rows(const nn_nbr* nl, int n_rows, const float* msg, const float* e1, const float* e2,
                               const float* unit, const float* a_in, const float* f_in, float* a_out, float* f_out,
                               bool first_layer, cudaStream_t stream) {
    const int N = n_rows;
    if (N <= 0) return 0;
    int grid = nn_ceil_div(N, kAggWarps);
    if (first_layer) {
        k_node_aggregate_fwd<true><<<grid, kAggThreads, 0, (cudaStream_t)stream>>>(nl->status, nl->row_ptr, nl->col, nl->edge_pair, N, msg,
                                                                                   e1, e2, unit, a_in, f_in, a_out, f_out); NN_LAUNCHED(1);
    }
    else {
        k_node_aggregate_fwd<false><<<grid, kAggThreads, 0, (cudaStream_t)stream>>>(nl->status, nl->row_ptr, nl->col, nl->edge_pair, N, msg,
                                                                                    e1, e2, unit, a_in, f_in, a_out, f_out); NN_LAUNCHED(1);
    }
    NN_CHECK_LAUNCH("nn_node_aggregate_fwd");
    return 0;
}

extern "C" int nn_equiv_update_fwd(const float* a_in, const float* f, const float* g, float* a_out, int32_t n_atoms,
                                   void* stream) {
    if (n_atoms <= 0) return 0;
    k_equiv_update_fwd<<<nn_ceil_div((long long)n_atoms * (kF / 4), 256), 256, 0, (cudaStream_t)stream>>>(a_in, f, g, a_out, n_atoms); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("nn_equiv_update_fwd");
    return 0;
}

int nn_energy_head_fwd_rows(const float* h2pre, const float* w3, const float* b3, const float* scale, const float* shift,
                            const int64_t* z, const int32_t* sys_ptr, int n_rows, int n_systems, float* e_atom,
                            float* energy, double* partial, int slices, cudaStream_t s);
// slices per system for the two-level per-system sums: 1 (single kernel) unless systems are large
int nn_sum_slices(int n_atoms, int n_systems) {
    const long long avg = n_systems > 0 ? (long long)n_atoms / n_systems : 0;
    const long long sl = avg / 2048;
    return (int)(sl < 1 ? 1 : (sl > 64 ? 64 : sl));
}
extern "C" int nn_energy_head_fwd(const float* h2pre, const float* w3, const float* b3, const float* scale,
                                  const float* shift, const int64_t* z, const int32_t* sys_ptr, int32_t n_atoms,
                                  int32_t n_systems, float* e_atom, float* energy, void* stream) {
    return nn_energy_head_fwd_rows(h2pre, w3, b3, scale, shift, z, sys_ptr, n_atoms, n_systems, e_atom, energy, nullptr, 1,
                                   (cudaStream_t)stream);
}
int nn_energy_head_fwd_rows(const float* h2pre, const float* w3, const float* b3, const float* scale, const float* shift,
                            const int64_t* z, const int32_t* sys_ptr, int n_atoms, int n_systems, float* e_atom,
                            float* energy, double* partial, int slices, cudaStream_t s) {
    if (n_atoms > 0) {
        k_energy_atom<<<nn_ceil_div(n_atoms, kWarps), kThreads, 0, s>>>(h2pre, w3, b3, scale, shift, z, n_atoms, e_atom); NN_LAUNCHED(1);
    }
    if (partial && slices > 1) {
        k_sys_sum_partial<1><<<dim3(n_systems, slices), kThreads, 0, s>>>(e_atom, sys_ptr, n_atoms, slices, partial); NN_LAUNCHED(1);
        k_energy_final<<<nn_ceil_div(n_systems, 128), 128, 0, s>>>(partial, slices, n_systems, energy); NN_LAUNCHED(1);
    } else {
        k_energy_sum<<<n_systems, kThreads, 0, s>>>(e_atom, sys_ptr, n_atoms, energy); NN_LAUNCHED(1);
    }
    NN_CHECK_LAUNCH("nn_energy_head_fwd");
    return 0;
}

int nn_force_virial_rows(const nn_nbr* nl, int n_rows, const float* disp_bar, float* forces, float* virial, float* stress,
                         void* workspace, double* partial, int slices, cudaStream_t s) {
    float* vir_atom = virial ? (float*)workspace : nullptr;
    NN_REQUIRE(!virial || workspace, "virial needs a workspace of n_atoms*9 floats");
    if (n_rows > 0) {
        k_force_virial_atom<<<nn_ceil_div(n_rows, 128), 128, 0, s>>>(nl->status, nl->row_ptr, nl->col, nl->edge_pair, n_rows,
                                                                     disp_bar, nl->pair_disp, nl->pos, nl->batch,
                                                                     nn_nbr_sysmeta(nl), forces, vir_atom); NN_LAUNCHED(1);
    }
    if (virial && partial && slices > 1) {
        k_sys_sum_partial<9><<<dim3(nl->n_systems, slices), kThreads, 0, s>>>(vir_atom, nl->sys_ptr, n_rows, slices, partial); NN_LAUNCHED(1);
        k_virial_final<<<nl->n_systems, 32, 0, s>>>(partial, slices, nl->cell, virial, stress); NN_LAUNCHED(1);
    } else if (virial) {
        k_virial_sum<<<nl->n_systems, kThreads, 0, s>>>(vir_atom, nl->sys_ptr, n_rows, nl->cell, virial, stress); NN_LAUNCHED(1);
    }
    NN_CHECK_LAUNCH("nn_force_virial_reduce");
    return 0;
}
extern "C" int nn_force_virial_reduce(const nn_nbr* nl, const float* disp_bar, float* forces, float* virial,
                                      float* stress, void* workspace, void* stream) {
    return nn_force_virial_rows(nl, nl->n_atoms, disp_bar, forces, virial, stress, workspace, nullptr, 1, (cudaStream_t)stream);
}

extern "C" int nn_halo_pack(const float* src, const int32_t* idx, int32_t n, int32_t width, float* out, void* stream) {
    NN_REQUIRE(width > 0 && width % 4 == 0, "width must be a positive multiple of 4");
    if (n <= 0) return 0;
    long long total = (long long)n * (width / 4);
    int grid = (int)((total + 255) / 256); if (grid > nn_num_sms() * 16) grid = nn_num_sms() * 16;
    k_halo_pack<<<grid, 256, 0, (cudaStream_t)stream>>>(src, idx, n, width / 4, out); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("nn_halo_pack");
    return 0;
}

// ---- launchers used only by nn_eval (eval.cu)
int nn_layer_norm_fwd_launch(float* a_io, const float* gamma, const float* beta, float* xhat, float* rstd, int n_rows, cudaStream_t s) {
    if (n_rows <= 0) return 0;
    k_layer_norm_fwd<<<nn_ceil_div(n_rows, kWarps), kThreads, 0, s>>>(a_io, gamma, beta, xhat, rstd, n_rows); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("layer_norm_fwd");
    return 0;
}
int nn_layer_norm_bwd_launch(float* abar_io, const float* gamma, const float* xhat, const float* rstd, int n_rows, cudaStream_t s) {
    if (n_rows <= 0) return 0;
    k_layer_norm_bwd<<<nn_ceil_div(n_rows, kWarps), kThreads, 0, s>>>(abar_io, gamma, xhat, rstd, n_rows); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("layer_norm_bwd");
    return 0;
}
int nn_direct_force_launch(const float* h, const float* f, const float* scale, const int64_t* z, int n_rows, float* out, cudaStream_t s) {
    if (n_rows <= 0) return 0;
    k_direct_force<<<nn_ceil_div(n_rows, kWarps), kThreads, 0, s>>>(h, f, scale, z, n_rows, out); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("direct_force");
    return 0;
}
int nn_embed_launch(const int64_t* z, const float* emb, float* a, int N, int* status, cudaStream_t s) {
    if (N <= 0) return 0;
    k_embed<<<nn_ceil_div((long long)N * (kF / 4), 256), 256, 0, s>>>(z, emb, a, N, status); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("embed");
    return 0;
}
int nn_energy_head_seed_launch(const float* h2pre, const float* w3, const float* scale, const int64_t* z, int N,
                               float* gh2, cudaStream_t s) {
    if (N <= 0) return 0;
    k_energy_head_seed<<<nn_ceil_div((long long)N * (kF / 4), 256), 256, 0, s>>>(h2pre, w3, scale, z, N, gh2); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("energy_head_seed");
    return 0;
}
int nn_pair_bwd_gather_launch(const nn_nbr* nl, const float* dfb, const float* f_in, const float* unit, float* e1_io,
                              float* e2bar, float* ubar, bool first, cudaStream_t s) {
    if (nl->cap_pairs <= 0) return 0;
    int grid = grid_for_rows(nl->n_atoms);
    if (first) {
        k_pair_bwd_gather<true><<<grid, kThreads, 0, s>>>(nl->pair_ptr, nl->pair_j, nl->n_atoms, nl->cap_pairs,
                                                          dfb, f_in, unit, e1_io, e2bar, ubar); NN_LAUNCHED(1);
    }
    else {
        k_pair_bwd_gather<false><<<grid, kThreads, 0, s>>>(nl->pair_ptr, nl->pair_j, nl->n_atoms, nl->cap_pairs,
                                                           dfb, f_in, unit, e1_io, e2bar, ubar); NN_LAUNCHED(1);
    }
    NN_CHECK_LAUNCH("pair_bwd_gather");
    return 0;
}
int nn_pair_bwd_message_launch(const nn_nbr* nl, const float* abar, const float* mn, const float* rbf, const float* drbf,
                               const float* Wet, float* mbar_io, float* x_bar, cudaStream_t s) {
    if (nl->cap_pairs <= 0) return 0;
    k_pair_bwd_message<<<grid_for_rows(nl->n_atoms), kThreads, 0, s>>>(nl->pair_ptr, nl->pair_j, nl->n_atoms, nl->cap_pairs,
                                                                        abar, mn, rbf, drbf, Wet, mbar_io, x_bar); NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("pair_bwd_message");
    return 0;
}
int nn_node_aggregate_bwd_launch(const nn_nbr* nl, int n_rows, const float* t, const float* mn, const float* e2,
                                 const float* dfb, float* mnbar, float* fbar_new, bool first, cudaStream_t s) {
    const int N = n_rows;
    if (N <= 0) return 0;
    int grid = nn_ceil_div(N, kAggWarps);
    if (first) {
        k_node_aggregate_bwd<true><<<grid, kAggThreads, 0, s>>>(nl->status, nl->row_ptr, nl->col, nl->edge_pair, N, t, mn, e2, dfb, mnbar, fbar_new); NN_LAUNCHED(1);
    }
    else {
        k_node_aggregate_bwd<false><<<grid, kAggThreads, 0, s>>>(nl->status, nl->row_ptr, nl->col, nl->edge_pair, N, t, mn, e2, dfb, mnbar, fbar_new); NN_LAUNCHED(1);
    }
    NN_CHECK_LAUNCH("node_aggregate_bwd");
    return 0;
}
