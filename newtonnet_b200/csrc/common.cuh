// Shared device/host helpers for the newtonnet_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/newtonnet_b200.h"

#define NN_WARP 32
static constexpr int kF = NN_F;      // 128 features: one warp covers a row with one float4 per lane
static constexpr int kNB = NN_NB;    // 20 radial basis functions

void nn_set_error(const char* fmt, ...);
bool nn_pdl_enabled();     // programmatic dependent launch of the tensor-core kernels (NN_PDL=0 turns it off)
// every kernel launch of this library is counted (bench.py reports it as gpu_launches)
void nn_count_launches(int n);
// optional per-stage CUDA-event profiler (nn_profile_enable): stages are timed on the launching stream
enum { NN_STAGE_NBR = 0, NN_STAGE_GEOM, NN_STAGE_NODE_GEMM, NN_STAGE_PAIR_GEMM, NN_STAGE_MESSAGE,
       NN_STAGE_AGGREGATE, NN_STAGE_HEAD, NN_STAGE_BWD_GATHER, NN_STAGE_BWD_MESSAGE, NN_STAGE_BWD_AGGREGATE,
       NN_STAGE_FORCE, NN_STAGE_OTHER, NN_N_STAGES };
void nn_prof_begin(int stage, cudaStream_t s);
void nn_prof_end(cudaStream_t s);
struct ProfScope {
    cudaStream_t s;
    ProfScope(int stage, cudaStream_t st) : s(st) { nn_prof_begin(stage, s); }
    ~ProfScope() { nn_prof_end(s); }
};

#define NN_CHECK_LAUNCH(name)                                                       \
    do {                                                                            \
        cudaError_t err__ = cudaGetLastError();                                     \
        if (err__ != cudaSuccess) {                                                 \
            nn_set_error("%s: %s", name, cudaGetErrorString(err__));                \
            return -2;                                                              \
        }                                                                           \
    } while (0)
#define NN_LAUNCHED(n) nn_count_launches(n)
// first statement of a kernel whose successor may be a PDL kernel (tc_common.cuh): lets that kernel's prologue start
// as soon as every CTA of this grid is resident; it still waits for this grid to complete before reading its results
#define NN_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")

#define NN_REQUIRE(cond, msg)                                                       \
    do {                                                                            \
        if (!(cond)) { nn_set_error("%s: %s", __func__, msg); return -1; }          \
    } while (0)

int nn_num_sms();           // multiprocessor count of the current device (cached per device; 148 on B200)
static inline int nn_ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline size_t nn_align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct WsCarver {
    char* base; size_t off; size_t cap;
    WsCarver(void* p, size_t bytes) : base((char*)p), off(0), cap(bytes) {}
    template <typename T> T* take(size_t n) {
        size_t bytes = nn_align_up(n * sizeof(T));
        T* r = (T*)(base ? base + off : nullptr);
        off += bytes;
        return r;
    }
    bool ok() const { return off <= cap; }
};

// sigmoid via ex2.approx + rcp.approx (2 MUFU ops, ~2 ulp): the activations are evaluated 10^8 times per step
__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float silu_f(float x) { return x * sigmoid_f(x); }
// d/dx [x * sigmoid(x)] = s * (1 + x * (1 - s))
__device__ __forceinline__ float dsilu_f(float x) {
    float s = sigmoid_f(x);
    return s * fmaf(x, 1.0f - s, 1.0f);
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// streaming (read-once) 128-bit load that does not pollute L1
__device__ __forceinline__ float4 ld4_stream(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// the same without the read-only (.nc) path: for buffers the kernel also writes
__device__ __forceinline__ float4 ld4_na(const float* p) {
    float4 r;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float4 f4_mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_sub(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 f4_fma(float4 a, float4 b, float4 c) {
    return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
}
__device__ __forceinline__ float4 f4_fma(float s, float4 b, float4 c) {
    return make_float4(fmaf(s, b.x, c.x), fmaf(s, b.y, c.y), fmaf(s, b.z, c.z), fmaf(s, b.w, c.w));
}
__device__ __forceinline__ float f4_dot(float4 a, float4 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w))); }
__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Per-system description written by the neighbour-list planner and reused by the virial kernel.
struct SysMeta {
    int mode;          // 0 = not periodic, 1 = diagonal cell, 2 = general cell
    int nc[3];         // grid dimensions
    int cell_off;      // first global grid cell of this system
    int first, count;  // atom range
    int nimg;          // mode 2: lattice images n in [-nimg, nimg]^3 are enumerated; -1 = one grid cell, all pairs
    float lo[3];       // grid origin (modes 0 and 2: Cartesian grid over the bounding box of the atoms)
    float wsc[3];      // cells per unit length (modes 0, 2) / cells per unit fractional coordinate (mode 1)
    float L[3];        // diagonal cell lengths (mode 1)
    float H[9];        // cell, row-major (mode 2)
    float Hinv[9];     // (cell^T)^-1, row-major (mode 2)
};

// Minimum-image displacement with the reference's fp32 arithmetic (representations.py:85-93):
//   mode 1: per component n = rint(d / L), d' = d - L*n   (two separately rounded operations)
//   mode 2: n = rint((cell^T)^-1 d), d' = d - cell @ n    (the reference's `cell @ n`, not cell^T @ n)
// `img` receives n (needed again by the virial).
__device__ __forceinline__ float3 nn_min_image(float3 d, const SysMeta& m, float3* img) {
    float3 n = make_float3(0.f, 0.f, 0.f);
    if (m.mode == 1) {
        n.x = rintf(__fdiv_rn(d.x, m.L[0])); d.x = __fsub_rn(d.x, __fmul_rn(m.L[0], n.x));
        n.y = rintf(__fdiv_rn(d.y, m.L[1])); d.y = __fsub_rn(d.y, __fmul_rn(m.L[1], n.y));
        n.z = rintf(__fdiv_rn(d.z, m.L[2])); d.z = __fsub_rn(d.z, __fmul_rn(m.L[2], n.z));
    } else if (m.mode == 2) {
        n.x = rintf(fmaf(m.Hinv[2], d.z, fmaf(m.Hinv[1], d.y, __fmul_rn(m.Hinv[0], d.x))));
        n.y = rintf(fmaf(m.Hinv[5], d.z, fmaf(m.Hinv[4], d.y, __fmul_rn(m.Hinv[3], d.x))));
        n.z = rintf(fmaf(m.Hinv[8], d.z, fmaf(m.Hinv[7], d.y, __fmul_rn(m.Hinv[6], d.x))));
        d.x = __fsub_rn(d.x, fmaf(m.H[2], n.z, fmaf(m.H[1], n.y, __fmul_rn(m.H[0], n.x))));
        d.y = __fsub_rn(d.y, fmaf(m.H[5], n.z, fmaf(m.H[4], n.y, __fmul_rn(m.H[3], n.x))));
        d.z = __fsub_rn(d.z, fmaf(m.H[8], n.z, fmaf(m.H[7], n.y, __fmul_rn(m.H[6], n.x))));
    }
    if (img) *img = n;
    return d;
}
// torch CPU norm(dim=1) on [E,3] fp32 == sqrt(fma(z,z,fma(y,y,x*x)))  (SURVEY.md section 8a R2)
__device__ __forceinline__ float nn_norm3(float3 d) {
    return __fsqrt_rn(fmaf(d.z, d.z, fmaf(d.y, d.y, __fmul_rn(d.x, d.x))));
}

// internal launchers shared between the exported staged operators and nn_eval
int nn_gemm128_launch(const nn_gemm_args& a, cudaStream_t s);
const SysMeta* nn_nbr_sysmeta(const nn_nbr* nl);
