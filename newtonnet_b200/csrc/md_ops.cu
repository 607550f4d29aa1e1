// Device-resident molecular dynamics around the force path - SURVEY.md section 8f rank 1.
//
// The reference drives MD from ASE on the host (scripts/simulate.py:21-31: Langevin(atoms, 0.5 fs, 300 K) with
// MLAseCalculator.calculate, utils/ase_interface.py:52-81, called once per step: numpy -> torch -> H2D, forward,
// D2H -> numpy).  Here the integrator state (unwrapped positions, velocities: fp64) lives in HBM next to the
// force buffers; one step = nn_md_advance -> nn_nbr_count/fill -> nn_eval -> nn_md_finish, captured once as a
// CUDA graph and replayed without any host round trip.  The splitting is BAOAB (B half kick, A half drift,
// O exact Ornstein-Uhlenbeck, A half drift, force, B half kick); with ou_c = 1 it is velocity Verlet.
// Random numbers: Philox4x32-10 keyed by the seed, counter = (atom, step) - replaying a step reproduces it.
//
// Geometry optimisation with ASE's FIRE (ase/optimize/fire.py, FIRE.step with downhill_check=False) runs the same way,
// independently per system of a batch: nn_fire_step -> nn_nbr_count/fill -> nn_eval -> nn_fire_check, one graph.
#include "common.cuh"

namespace {

__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
}

__device__ __forceinline__ void philox4x32(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// three standard normals for (atom, step): Box-Muller on two Philox blocks' worth of uniforms
__device__ __forceinline__ void normal3(unsigned long long seed, int atom, long long step, double (&g)[3]) {
    uint32_t c[4] = {(uint32_t)atom, (uint32_t)step, (uint32_t)((unsigned long long)step >> 32), 0x4D44u};
    philox4x32(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double two32 = 1.0 / 4294967296.0;
    const double u0 = ((double)c[0] + 0.5) * two32, u1 = ((double)c[1] + 0.5) * two32;
    const double u2 = ((double)c[2] + 0.5) * two32, u3 = ((double)c[3] + 0.5) * two32;
    const double r0 = sqrt(-2.0 * log(u0)), r1 = sqrt(-2.0 * log(u2));
    double s0, c0, s1, c1;
    sincospi(2.0 * u1, &s0, &c0);
    sincospi(2.0 * u3, &s1, &c1);
    g[0] = r0 * c0; g[1] = r0 * s0; g[2] = r1 * c1;
    (void)s1;
}

// pos_model[0..2] = p wrapped into the cell Cf (rows are the lattice vectors, pos = frac @ cell); a zero (singular) cell
// leaves p as it is.  The one wrap of the device drivers: the MD step, the FIRE step and nn_wrap_positions call it.
__device__ __forceinline__ void write_wrapped(const float* __restrict__ Cf, double (&p)[3], float* __restrict__ pos_model) {
    double c[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) c[k] = (double)Cf[k];
    const double det = c[0] * (c[4] * c[8] - c[5] * c[7]) - c[1] * (c[3] * c[8] - c[5] * c[6]) + c[2] * (c[3] * c[7] - c[4] * c[6]);
    if (det != 0.0) {
        const double id = 1.0 / det;
        // inverse of cell (row-vector convention): frac = pos @ inv
        const double inv[9] = {(c[4] * c[8] - c[5] * c[7]) * id, (c[2] * c[7] - c[1] * c[8]) * id, (c[1] * c[5] - c[2] * c[4]) * id,
                               (c[5] * c[6] - c[3] * c[8]) * id, (c[0] * c[8] - c[2] * c[6]) * id, (c[2] * c[3] - c[0] * c[5]) * id,
                               (c[3] * c[7] - c[4] * c[6]) * id, (c[1] * c[6] - c[0] * c[7]) * id, (c[0] * c[4] - c[1] * c[3]) * id};
        double f[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            f[a] = p[0] * inv[a] + p[1] * inv[3 + a] + p[2] * inv[6 + a];
            f[a] -= floor(f[a]);
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) p[a] = f[0] * c[a] + f[1] * c[3 + a] + f[2] * c[6 + a];
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) pos_model[a] = (float)p[a];
}

// B A O A + wrap.  x, v: [N,3] fp64 state; force [N,3] fp32 at the current x; pos_model: wrapped fp32 copy the
// neighbour search and the network read (reference: atoms.get_positions(wrap=True), ase_interface.py:135).
__global__ void k_md_advance(int n, double* __restrict__ x, double* __restrict__ v, const float* __restrict__ force,
                             const double* __restrict__ inv_mass, const float* __restrict__ cell,
                             const long long* __restrict__ batch, float* __restrict__ pos_model, double dt, double ou_c,
                             double kT, unsigned long long seed, const long long* __restrict__ step_ctr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double im = inv_mass[i], h = 0.5 * dt;
    double p[3], u[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        u[a] = v[3 * i + a] + h * im * (double)force[3 * i + a];
        p[a] = x[3 * i + a] + h * u[a];
    }
    if (ou_c < 1.0) {
        double g[3];
        normal3(seed, i, *step_ctr, g);
        const double sigma = sqrt((1.0 - ou_c * ou_c) * kT * im);
#pragma unroll
        for (int a = 0; a < 3; ++a) u[a] = ou_c * u[a] + sigma * g[a];
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        p[a] += h * u[a];
        x[3 * i + a] = p[a];
        v[3 * i + a] = u[a];
    }
    write_wrapped(cell + 9 * batch[i], p, pos_model + 3 * i);
}

// B half kick with the new force + per-system log row {potential, kinetic} + sticky status + step counter.
// One block per system, fixed-order tree reduction (deterministic).
__global__ void __launch_bounds__(256)
k_md_finish(const int* __restrict__ sys_ptr, double* __restrict__ v, const float* __restrict__ force,
            const double* __restrict__ inv_mass, double dt, const float* __restrict__ energy, double* __restrict__ log,
            int log_cap, long long* __restrict__ step_ctr, const int* __restrict__ nbr_status, int* __restrict__ sticky,
            unsigned int* __restrict__ ticket) {
    __shared__ double red[256];
    const int b = blockIdx.x, n_sys = gridDim.x;
    const long long step = *step_ctr;
    const double h = 0.5 * dt;
    double ke = 0.0;
    for (int i = sys_ptr[b] + threadIdx.x; i < sys_ptr[b + 1]; i += blockDim.x) {
        const double im = inv_mass[i];
        double s = 0.0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const double u = v[3 * i + a] + h * im * (double)force[3 * i + a];
            v[3 * i + a] = u;
            s += u * u;
        }
        ke += im > 0.0 ? 0.5 * s / im : 0.0;
    }
    red[threadIdx.x] = ke;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double* row = log + ((size_t)(step % log_cap) * n_sys + b) * 2;
        row[0] = (double)energy[b];
        row[1] = red[0];
        if (b == 0) {
            if (nbr_status[NN_ST_EDGE_OVERFLOW]) atomicMax(&sticky[0], nbr_status[NN_ST_EDGE_OVERFLOW]);
            if (nbr_status[NN_ST_ROW_OVERFLOW]) atomicMax(&sticky[1], nbr_status[NN_ST_ROW_OVERFLOW]);
            if (nbr_status[NN_ST_SINGULAR_CELL]) sticky[2] = 1;
        }
        __threadfence();
        if (atomicAdd(ticket, 1u) == (unsigned)n_sys - 1) {     // last block: everyone has read the counter
            *ticket = 0;
            *step_ctr = step + 1;
        }
    }
}

__global__ void k_wrap(int n, const double* __restrict__ x, const float* __restrict__ cell, const long long* __restrict__ batch,
                       float* __restrict__ pos_model) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double p[3] = {x[3 * i], x[3 * i + 1], x[3 * i + 2]};
    write_wrapped(cell + 9 * batch[i], p, pos_model + 3 * i);
}

// ---- FIRE (ase.optimize.FIRE.step, downhill_check=False), one block of 256 threads per system -------------------
// Per-system state: sf [n_sys,3] fp64 {dt, a, max|f|^2}, si [n_sys,4] int32 {Nsteps, started, converged, steps}.
// Element-wise arithmetic uses the _rn intrinsics so that no multiply-add is contracted: every element follows numpy's
// operation order and rounding.  Only the three dot products and |dr|^2 are summed in another (fixed) order.
enum { FIRE_DT = 0, FIRE_A = 1, FIRE_F2 = 2 };
enum { FIRE_NSTEPS = 0, FIRE_STARTED = 1, FIRE_CONVERGED = 2, FIRE_STEPS = 3 };

__global__ void __launch_bounds__(256)
k_fire_step(const int* __restrict__ sys_ptr, double* __restrict__ x, double* __restrict__ v, const float* __restrict__ force,
            const float* __restrict__ cell, float* __restrict__ pos_model, double* __restrict__ sf, int* __restrict__ si,
            double maxstep, double dtmax, double finc, double fdec, double astart, double fa, int nmin) {
    __shared__ double red[3][256];
    __shared__ double sh[5];              // a before the update, |f|, |v|, dt after the update, |dr|
    __shared__ int mode;                  // 0 first step (v = 0), 1 downhill (mix), 2 uphill (v = 0, reset)
    const int b = blockIdx.x, t = threadIdx.x;
    if (si[4 * b + FIRE_CONVERGED]) return;                     // frozen: x and v are never written again
    const int lo = sys_ptr[b], hi = sys_ptr[b + 1];
    const bool started = si[4 * b + FIRE_STARTED] != 0;
    double fv = 0.0, ff = 0.0, vv = 0.0;
    if (started) {
        for (int i = lo + t; i < hi; i += 256) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const double f = (double)force[3 * i + c], u = v[3 * i + c];
                fv += f * u; ff += f * f; vv += u * u;
            }
        }
    }
    red[0][t] = fv; red[1][t] = ff; red[2][t] = vv;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (t < w) {
#pragma unroll
            for (int k = 0; k < 3; ++k) red[k][t] += red[k][t + w];
        }
        __syncthreads();
    }
    if (t == 0) {
        double dt = sf[3 * b + FIRE_DT], a = sf[3 * b + FIRE_A];
        int n = si[4 * b + FIRE_NSTEPS];
        sh[0] = a;
        if (!started) {                                          // ASE: self.v is None
            mode = 0;
            si[4 * b + FIRE_STARTED] = 1;
        } else if (red[0][0] > 0.0) {
            mode = 1;
            sh[1] = sqrt(red[1][0]);
            sh[2] = sqrt(red[2][0]);
            if (n > nmin) {
                dt = fmin(dt * finc, dtmax);
                a *= fa;
            }
            n += 1;
        } else {
            mode = 2;
            a = astart;
            dt *= fdec;
            n = 0;
        }
        sh[3] = dt;
        sf[3 * b + FIRE_DT] = dt; sf[3 * b + FIRE_A] = a;
        si[4 * b + FIRE_NSTEPS] = n;
    }
    __syncthreads();
    const int m = mode;
    const double a0 = sh[0], nf = sh[1], nv = sh[2], dt = sh[3], one_minus_a = 1.0 - a0;
    double dd = 0.0;
    for (int i = lo + t; i < hi; i += 256) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double f = (double)force[3 * i + c];
            double u = v[3 * i + c];
            if (m == 0) u = 0.0;
            else if (m == 1) u = __dadd_rn(__dmul_rn(one_minus_a, u), __dmul_rn(__ddiv_rn(__dmul_rn(a0, f), nf), nv));
            else u = __dmul_rn(u, 0.0);
            u = __dadd_rn(u, __dmul_rn(dt, f));
            v[3 * i + c] = u;
            const double dr = __dmul_rn(dt, u);
            dd += dr * dr;
        }
    }
    red[0][t] = dd;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (t < w) red[0][t] += red[0][t + w];
        __syncthreads();
    }
    if (t == 0) sh[4] = sqrt(red[0][0]);
    __syncthreads();
    const double normdr = sh[4];
    const bool clip = normdr > maxstep;
    for (int i = lo + t; i < hi; i += 256) {
        double p[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            double dr = __dmul_rn(dt, v[3 * i + c]);
            if (clip) dr = __ddiv_rn(__dmul_rn(maxstep, dr), normdr);
            p[c] = __dadd_rn(x[3 * i + c], dr);
            x[3 * i + c] = p[c];
        }
        write_wrapped(cell + 9 * b, p, pos_model + 3 * i);
    }
}

// ASE's Optimizer.converged on the forces at the current positions: max_i sum_c f_ic^2 < fmax^2, in fp64 and NaN-
// propagating like numpy's max.  Fixed atoms' forces are zeroed first (FixAtoms.adjust_forces).
__global__ void __launch_bounds__(256)
k_fire_check(const int* __restrict__ sys_ptr, float* __restrict__ force, const unsigned char* __restrict__ fixed,
             const double* __restrict__ fmax2, double* __restrict__ sf, int* __restrict__ si, int advance,
             long long* __restrict__ step_ctr, const int* __restrict__ nbr_status, int* __restrict__ sticky,
             unsigned int* __restrict__ ticket) {
    __shared__ double red[256];
    const int b = blockIdx.x, t = threadIdx.x, n_sys = gridDim.x;
    const long long step = advance ? *step_ctr : 0;
    double mx = 0.0;
    for (int i = sys_ptr[b] + t; i < sys_ptr[b + 1]; i += 256) {
        if (fixed && fixed[i]) {
            force[3 * i] = 0.0f; force[3 * i + 1] = 0.0f; force[3 * i + 2] = 0.0f;
            continue;
        }
        const double f0 = force[3 * i], f1 = force[3 * i + 1], f2 = force[3 * i + 2];
        const double s = __dadd_rn(__dadd_rn(__dmul_rn(f0, f0), __dmul_rn(f1, f1)), __dmul_rn(f2, f2));
        if (s > mx || s != s) mx = s;
    }
    red[t] = mx;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (t < w && (red[t + w] > red[t] || red[t + w] != red[t + w])) red[t] = red[t + w];
        __syncthreads();
    }
    if (t == 0) {
        const double m = red[0];
        sf[3 * b + FIRE_F2] = m;
        if (advance && !si[4 * b + FIRE_CONVERGED]) si[4 * b + FIRE_STEPS] += 1;
        si[4 * b + FIRE_CONVERGED] = m < *fmax2;
        if (!advance) return;
        if (b == 0) {
            if (nbr_status[NN_ST_EDGE_OVERFLOW]) atomicMax(&sticky[0], nbr_status[NN_ST_EDGE_OVERFLOW]);
            if (nbr_status[NN_ST_ROW_OVERFLOW]) atomicMax(&sticky[1], nbr_status[NN_ST_ROW_OVERFLOW]);
            if (nbr_status[NN_ST_SINGULAR_CELL]) sticky[2] = 1;
        }
        __threadfence();
        if (atomicAdd(ticket, 1u) == (unsigned)n_sys - 1) {     // last block: everyone has read the counter
            *ticket = 0;
            *step_ctr = step + 1;
        }
    }
}

}  // namespace

extern "C" {

NN_API int nn_md_advance(int32_t n_atoms, double* x, double* v, const float* force, const double* inv_mass, const float* cell,
                         const int64_t* batch, float* pos_model, double dt, double ou_c, double kT, uint64_t seed,
                         const int64_t* step_ctr, void* stream) {
    NN_REQUIRE(n_atoms >= 0 && x && v && force && inv_mass && cell && batch && pos_model && step_ctr, "null argument");
    NN_REQUIRE(ou_c >= 0.0 && ou_c <= 1.0 && kT >= 0.0, "ou_c must be in [0, 1] and kT >= 0");
    if (n_atoms == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    k_md_advance<<<(n_atoms + 127) / 128, 128, 0, s>>>(n_atoms, x, v, force, inv_mass, cell, (const long long*)batch, pos_model,
                                                       dt, ou_c, kT, (unsigned long long)seed, (const long long*)step_ctr);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_md_advance");
    return 0;
}

NN_API int nn_md_finish(int32_t n_systems, const int32_t* sys_ptr, double* v, const float* force, const double* inv_mass, double dt,
                        const float* energy, double* log, int32_t log_cap, int64_t* step_ctr, const int32_t* nbr_status,
                        int32_t* sticky, uint32_t* ticket, void* stream) {
    NN_REQUIRE(n_systems > 0 && sys_ptr && v && force && inv_mass && energy && log && log_cap > 0 && step_ctr && nbr_status &&
               sticky && ticket, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    k_md_finish<<<n_systems, 256, 0, s>>>(sys_ptr, v, force, inv_mass, dt, energy, log, log_cap, (long long*)step_ctr,
                                          nbr_status, sticky, ticket);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_md_finish");
    return 0;
}

NN_API int nn_wrap_positions(int32_t n_atoms, const double* x, const float* cell, const int64_t* batch, float* pos_model,
                             void* stream) {
    NN_REQUIRE(n_atoms >= 0 && x && cell && batch && pos_model, "null argument");
    if (n_atoms == 0) return 0;
    k_wrap<<<(n_atoms + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n_atoms, x, cell, (const long long*)batch, pos_model);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_wrap");
    return 0;
}

NN_API int nn_fire_step(int32_t n_systems, const int32_t* sys_ptr, double* x, double* v, const float* force, const float* cell,
                        float* pos_model, double* sys_f64, int32_t* sys_i32, double maxstep, double dtmax, double finc,
                        double fdec, double astart, double fa, int32_t nmin, void* stream) {
    NN_REQUIRE(n_systems > 0 && sys_ptr && x && v && force && cell && pos_model && sys_f64 && sys_i32, "null argument");
    NN_REQUIRE(maxstep > 0.0 && dtmax > 0.0 && finc > 0.0 && fdec > 0.0, "maxstep, dtmax, finc and fdec must be > 0");
    k_fire_step<<<n_systems, 256, 0, (cudaStream_t)stream>>>(sys_ptr, x, v, force, cell, pos_model, sys_f64, sys_i32, maxstep,
                                                             dtmax, finc, fdec, astart, fa, nmin);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_fire_step");
    return 0;
}

NN_API int nn_fire_check(int32_t n_systems, const int32_t* sys_ptr, float* force, const uint8_t* fixed, const double* fmax2,
                         double* sys_f64, int32_t* sys_i32, int32_t advance, int64_t* step_ctr, const int32_t* nbr_status,
                         int32_t* sticky, uint32_t* ticket, void* stream) {
    NN_REQUIRE(n_systems > 0 && sys_ptr && force && fmax2 && sys_f64 && sys_i32, "null argument");
    NN_REQUIRE(!advance || (step_ctr && nbr_status && sticky && ticket), "null argument");
    k_fire_check<<<n_systems, 256, 0, (cudaStream_t)stream>>>(sys_ptr, force, fixed, fmax2, sys_f64, sys_i32, advance,
                                                              (long long*)step_ctr, nbr_status, sticky, ticket);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_fire_check");
    return 0;
}

}  // extern "C"
