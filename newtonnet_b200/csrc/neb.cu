// Nudged elastic band force projection for device-resident climbing-image NEB (newtonnet_b200/neb.py).
//
// A band is images 0..n+1 of one structure; the end points are fixed and the n interior images are optimised together
// as one FIRE system (nn_fire_step / nn_fire_check in md_ops.cu), as ASE's FIRE(NEB(images)) does.  One step is
// nn_fire_step (band ranges) -> nn_nbr_count/fill -> nn_eval (one system per interior image) -> nn_neb_forces ->
// nn_fire_check (band ranges), one CUDA graph.
//
// The projection is ASE's NEB.get_forces with method='improvedtangent' (ase/neb.py, ASE 3.22): the improved tangent of
// Henkelman & Jonsson, J. Chem. Phys. 113, 9978 (2000), and the climbing image of Henkelman, Uberuaga & Jonsson,
// J. Chem. Phys. 113, 9901 (2000).  oracle/neb_oracle.py restates it in numpy.
#include "common.cuh"

namespace {

constexpr int kFireConverged = 2;     // column of nn_fire_step's per-system int32 state: the system is frozen

// One block of 256 threads per interior image.  Element-wise arithmetic uses the _rn intrinsics, so no multiply-add is
// contracted there and every element follows numpy's operation order.  |t+|^2, |t-|^2, |tau|^2 and <F, tau^> are
// fixed-order tree reductions over the image's atoms (their accumulations may be contracted; the order is fixed).
// A band whose model output is not finite (an interior energy, or a force of a free atom of any interior image) gets a
// zero NEB force on every image and failed[b] = 1: nn_fire_check then finds it converged and the FIRE kernels freeze it
// at its last, finite positions.  Every block of the band reads the same values, so all of them agree.
__global__ void __launch_bounds__(256)
k_neb_forces(const int* __restrict__ img_ptr, const int* __restrict__ img_band, const int* __restrict__ band_img,
             const double* __restrict__ x, const double* __restrict__ ends, const int* __restrict__ band_ends,
             const float* __restrict__ energy, const double* __restrict__ ends_energy, const float* __restrict__ force,
             const unsigned char* __restrict__ fixed, const int* __restrict__ climb, const int* __restrict__ band_si,
             double k, float* __restrict__ neb_force, int* __restrict__ imax, int* __restrict__ failed) {
    __shared__ double red[3][256];
    __shared__ double sh[4];              // |t+|, |t-|, |tau|, <F, tau^>
    const int j = blockIdx.x, t = threadIdx.x;
    const int b = img_band[j];
    if (band_si[4 * b + kFireConverged]) return;                // frozen band: its forces stay as they are
    const int j0 = band_img[b], n = band_img[b + 1] - j0, i = j - j0 + 1;
    const int lo = img_ptr[j], na = img_ptr[j + 1] - lo;
    const double* cur = x + 3 * (size_t)lo;
    const double* prev = i > 1 ? x + 3 * (size_t)img_ptr[j - 1] : ends + 3 * (size_t)band_ends[b];
    const double* next = i < n ? x + 3 * (size_t)img_ptr[j + 1] : ends + 3 * ((size_t)band_ends[b] + na);
    const double e = (double)energy[j];
    const double em = i > 1 ? (double)energy[j - 1] : ends_energy[2 * b];
    const double ep = i < n ? (double)energy[j + 1] : ends_energy[2 * b + 1];
    // climbing image: the highest interior energy, ties to the highest index
    int im = 1;
    double best = (double)energy[j0];
    bool finite = isfinite(best);
    for (int q = 1; q < n; ++q) {
        const double eq = (double)energy[j0 + q];
        finite = finite && isfinite(eq);
        if (eq >= best) { best = eq; im = q + 1; }
    }
    int bad = 0;
    for (int a = img_ptr[j0] + t; a < img_ptr[j0 + n]; a += 256) {
        if (fixed && fixed[a]) continue;
        bad |= !(isfinite(force[3 * a]) && isfinite(force[3 * a + 1]) && isfinite(force[3 * a + 2]));
    }
    if (__syncthreads_or(bad) || !finite) {
        for (int a = t; a < 3 * na; a += 256) neb_force[3 * (size_t)lo + a] = 0.0f;
        if (i == 1 && t == 0) failed[b] = 1;
        return;
    }
    const bool climbing = climb[b] != 0 && i == im;
    if (i == 1 && t == 0) imax[b] = im;
    // tangent: mode 0 tau = t+, 1 tau = t-, 2 tau = t+ wp + t- wm
    int mode = 2;
    double wp = 0.0, wm = 0.0;
    if (ep > e && e > em) {
        mode = 0;
    } else if (ep < e && e < em) {
        mode = 1;
    } else {
        const double dp = fabs(__dsub_rn(ep, e)), dm = fabs(__dsub_rn(em, e));
        const double vmax = fmax(dp, dm), vmin = fmin(dp, dm);
        wp = ep > em ? vmax : vmin;
        wm = ep > em ? vmin : vmax;
        // three equal energies (fp32 energies tie on flat paths): the weights' limit for dV_max = dV_min, tau = t+ + t-,
        // instead of ASE's zero tangent, whose normalisation gives NaN
        if (vmax == 0.0) wp = wm = 1.0;
    }
    auto tau = [&](double tp, double tm) {
        return mode == 0 ? tp : mode == 1 ? tm : __dadd_rn(__dmul_rn(tp, wp), __dmul_rn(tm, wm));
    };
    double spp = 0.0, smm = 0.0, stt = 0.0;
    for (int a = t; a < na; a += 256) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double r = cur[3 * a + c];
            const double tp = __dsub_rn(next[3 * a + c], r), tm = __dsub_rn(r, prev[3 * a + c]), u = tau(tp, tm);
            spp += tp * tp; smm += tm * tm; stt += u * u;
        }
    }
    red[0][t] = spp; red[1][t] = smm; red[2][t] = stt;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (t < w) {
#pragma unroll
            for (int q = 0; q < 3; ++q) red[q][t] += red[q][t + w];
        }
        __syncthreads();
    }
    if (t == 0) {
        sh[0] = sqrt(red[0][0]); sh[1] = sqrt(red[1][0]); sh[2] = sqrt(red[2][0]);
    }
    __syncthreads();
    const double nt = sh[2];
    double ft = 0.0;
    for (int a = t; a < na; a += 256) {
        const bool held = fixed && fixed[lo + a];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double r = cur[3 * a + c];
            const double u = __ddiv_rn(tau(__dsub_rn(next[3 * a + c], r), __dsub_rn(r, prev[3 * a + c])), nt);
            const double f = held ? 0.0 : (double)force[3 * (lo + a) + c];
            ft += f * u;
        }
    }
    __syncthreads();                                            // everyone has read sh[2] and red before red is reused
    red[0][t] = ft;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (t < w) red[0][t] += red[0][t + w];
        __syncthreads();
    }
    if (t == 0) sh[3] = red[0][0];
    __syncthreads();
    const double fpar = sh[3];
    // normal image: F - <F,tau^> tau^ + (|t+| k - |t-| k) tau^;  climbing image: F - (2 <F,tau^>) tau^
    const double spring = __dsub_rn(__dmul_rn(sh[0], k), __dmul_rn(sh[1], k)), twice = __dmul_rn(2.0, fpar);
    for (int a = t; a < na; a += 256) {
        const bool held = fixed && fixed[lo + a];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double r = cur[3 * a + c];
            const double u = __ddiv_rn(tau(__dsub_rn(next[3 * a + c], r), __dsub_rn(r, prev[3 * a + c])), nt);
            double f = held ? 0.0 : (double)force[3 * (lo + a) + c];
            if (climbing) f = __dsub_rn(f, __dmul_rn(twice, u));
            else f = __dadd_rn(__dsub_rn(f, __dmul_rn(fpar, u)), __dmul_rn(spring, u));
            neb_force[3 * (lo + a) + c] = held ? 0.0f : __double2float_rn(f);
        }
    }
}

}  // namespace

extern "C" {

NN_API int nn_neb_forces(int32_t n_images, const int32_t* img_ptr, const int32_t* img_band, const int32_t* band_img,
                         const double* x, const double* ends, const int32_t* band_ends, const float* energy,
                         const double* ends_energy, const float* force, const uint8_t* fixed, const int32_t* climb,
                         const int32_t* band_si, double k, float* neb_force, int32_t* imax, int32_t* failed, void* stream) {
    NN_REQUIRE(n_images > 0 && img_ptr && img_band && band_img && x && ends && band_ends && energy && ends_energy && force &&
               climb && band_si && neb_force && imax && failed, "null argument");
    NN_REQUIRE(k > 0.0, "the spring constant k must be > 0");
    k_neb_forces<<<n_images, 256, 0, (cudaStream_t)stream>>>(img_ptr, img_band, band_img, x, ends, band_ends, energy,
                                                             ends_energy, force, fixed, climb, band_si, k, neb_force, imax,
                                                             failed);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_neb_forces");
    return 0;
}

}  // extern "C"
