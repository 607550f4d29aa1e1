// Hessian in blocks of rows (newtonnet_b200/hessian.py).
//
// A pass evaluates k jobs at once.  A job is one row r of the Hessian of one frame: the pass puts k copies of frames into
// one batch (copy c = system c, atoms [c n, (c+1) n)), takes pos_grad of that batch with create_graph and differentiates
// <seed, pos_grad> with respect to the replicated positions, where the seed holds a one-hot for row r_c in copy c's block.
// Copies are independent systems, so copy c's block of that gradient is row r_c of its frame's Hessian.
//
// Plan: int32 [n_pass, k, 3] = {frame, local row (-1 = padding job), output row}.  The pass index lives in device memory
// (`pass_ctr`): expand reads it, the last block of scatter advances it, so a captured pass replays without host traffic.
#include "common.cuh"

namespace {

// one thread per replicated atom: copy the job's frame into its slot, write the one-hot seed
__global__ void k_hessian_expand(const int32_t* __restrict__ plan, const int32_t* __restrict__ pass_ctr, int k, int n_slot,
                                 const int64_t* __restrict__ z, const float* __restrict__ pos, const float* __restrict__ cell,
                                 const int32_t* __restrict__ frame_ptr, int64_t* __restrict__ z_rep, float* __restrict__ pos_rep,
                                 float* __restrict__ cell_rep, int64_t* __restrict__ batch_rep, float* __restrict__ seed) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k * n_slot) return;
    const int c = i / n_slot, a = i - c * n_slot;
    const int32_t* job = plan + ((size_t)(*pass_ctr) * k + c) * 3;
    const int f = job[0], row = job[1];
    const int src = frame_ptr[f] + a;
    z_rep[i] = z[src];
    batch_rep[i] = c;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        pos_rep[3 * i + d] = pos[3 * src + d];
        seed[3 * i + d] = (row == 3 * a + d) ? 1.0f : 0.0f;      // padding jobs (row = -1) get a zero seed
    }
    if (a == 0)
        for (int q = 0; q < 9; ++q) cell_rep[9 * c + q] = cell[9 * f + q];
}

// one block per job: the job's whole output row, columns of its own frame from its copy's gradient, every other column 0
__global__ void __launch_bounds__(256)
k_hessian_scatter(const int32_t* __restrict__ plan, int32_t* __restrict__ pass_ctr, int n_slot, const int32_t* __restrict__ frame_ptr,
                  const float* __restrict__ grad_rep, float* __restrict__ H, long long n_cols, unsigned int* __restrict__ ticket) {
    const int c = blockIdx.x, k = gridDim.x;
    const int32_t* job = plan + ((size_t)(*pass_ctr) * k + c) * 3;
    const int f = job[0], row = job[1], out = job[2];
    if (row >= 0) {
        const long long lo = 3LL * frame_ptr[f], hi = 3LL * frame_ptr[f + 1];
        const float* g = grad_rep + 3LL * c * n_slot - lo;
        float* h = H + (long long)out * n_cols;
        for (long long j = threadIdx.x; j < n_cols; j += blockDim.x) h[j] = (j >= lo && j < hi) ? g[j] : 0.0f;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(ticket, 1u) == (unsigned)k - 1) {        // last block: every block has read the pass index
            *ticket = 0;
            *pass_ctr += 1;
        }
    }
}

}  // namespace

extern "C" {

NN_API int nn_hessian_expand(const int32_t* plan, const int32_t* pass_ctr, int32_t k, int32_t n_slot, const int64_t* z,
                             const float* pos, const float* cell, const int32_t* frame_ptr, int64_t* z_rep, float* pos_rep,
                             float* cell_rep, int64_t* batch_rep, float* seed, void* stream) {
    NN_REQUIRE(plan && pass_ctr && z && pos && cell && frame_ptr && z_rep && pos_rep && cell_rep && batch_rep && seed, "null argument");
    NN_REQUIRE(k > 0 && n_slot > 0, "k and n_slot must be positive");
    const long long n = (long long)k * n_slot;
    NN_REQUIRE(n < (1LL << 31), "k * n_slot must fit in int32");
    k_hessian_expand<<<nn_ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(plan, pass_ctr, k, n_slot, z, pos, cell, frame_ptr,
                                                                           z_rep, pos_rep, cell_rep, batch_rep, seed);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_hessian_expand");
    return 0;
}

NN_API int nn_hessian_scatter(const int32_t* plan, int32_t* pass_ctr, int32_t k, int32_t n_slot, const int32_t* frame_ptr,
                              const float* grad_rep, float* H, int64_t n_cols, uint32_t* ticket, void* stream) {
    NN_REQUIRE(plan && pass_ctr && frame_ptr && grad_rep && H && ticket, "null argument");
    NN_REQUIRE(k > 0 && n_slot > 0 && n_cols > 0, "k, n_slot and n_cols must be positive");
    k_hessian_scatter<<<k, 256, 0, (cudaStream_t)stream>>>(plan, pass_ctr, n_slot, frame_ptr, grad_rep, H, (long long)n_cols, ticket);
    NN_LAUNCHED(1);
    NN_CHECK_LAUNCH("k_hessian_scatter");
    return 0;
}

}  // extern "C"
