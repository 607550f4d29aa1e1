/*
 * newtonnet_b200 - C ABI of the B200 (sm_100a) energy / force / stress path of NewtonNet.
 *
 * The reference (THGLab/NewtonNet v2.1.0) is pure Python/PyTorch and has no FFI of its own; the
 * entry points below are the "thin custom-op layer" that its hot path
 *     NewtonNet.forward(z, pos, cell, batch)            newtonnet/models/newtonnet.py:74-104
 *     MLAseCalculator.calculate                         newtonnet/utils/ase_interface.py:52-81
 * binds to (ctypes stub in INTEGRATION.md).  Each function cites the reference code it replaces;
 * citations are relative to the reference repository root.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns all memory (inputs, outputs, workspaces); nothing is allocated or freed here,
 *     except a few KB of lazily created read-only tables;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); no host sync inside;
 *   - return value 0 = launched, negative = error (see nn_last_error(), thread local);
 *   - device-side conditions (capacity overflow, unsorted batch, singular cell) are reported in a
 *     caller-provided int32 status word array `status[NN_STATUS_WORDS]`, read back by the caller
 *     together with the results;
 *   - fp32 arithmetic, int32 indices; F = 128 features, nb = 20 radial basis functions, SiLU.
 *   - atoms of one system are contiguous and `batch` is non-decreasing (PyG convention used by the
 *     reference, newtonnet/utils/ase_interface.py:141).
 *
 * Edge convention (SURVEY.md section 8): directed edge e = (i, j), i = destination = edge_index[0],
 * j = source = edge_index[1], disp_e = pos_i - pos_j (minimum image).  The neighbour list is a
 * destination-sorted CSR (row_ptr, col) with rows sorted by j (== the reference's edge order) plus the
 * list of undirected pairs p = (i < j): message, e1 and e2 are symmetric in (i, j) and are evaluated
 * once per pair; `edge_pair[e]` = pair id of directed edge e, bit 31 set when the edge is the
 * reversed orientation (j < i).
 */
#ifndef NEWTONNET_B200_H
#define NEWTONNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define NN_API __attribute__((visibility("default")))
#else
#define NN_API
#endif

#define NN_F 128            /* n_features (scripts/config.yml:32) */
#define NN_NB 20            /* n_basis    (scripts/config.yml:31) */
#define NN_MAX_LAYERS 8
#define NN_STATUS_WORDS 8
/* status word indices */
#define NN_ST_EDGE_OVERFLOW 0   /* directed edges found > capacity (value = edges needed)            */
#define NN_ST_ROW_OVERFLOW 1    /* an atom has more than NN_MAX_DEGREE neighbours                    */
#define NN_ST_BATCH_UNSORTED 2  /* batch is not non-decreasing / out of range                        */
#define NN_ST_SINGULAR_CELL 3   /* periodic batch with a singular cell (reference: _LinAlgError)     */
#define NN_ST_N_EDGES 4         /* number of directed edges E                                        */
#define NN_ST_N_PAIRS 5         /* number of undirected pairs P = E / 2                              */
#define NN_ST_N_CELLS 6         /* number of grid cells used by the neighbour search                 */
#define NN_MAX_DEGREE 512

NN_API const char* nn_last_error(void);
NN_API int nn_version(void);
/* number of CUDA kernels this library has launched since the last reset (host-side counter). */
NN_API long long nn_launch_count(int reset);
/* optional stage profiler: CUDA events recorded on the launching stream around each stage of
 * nn_nbr_count / nn_nbr_fill / nn_eval; nn_profile_collect (after a stream synchronise) returns summed
 * milliseconds and sample counts per stage and clears the samples.  Stage ids: 0 neighbour list,
 * 1 edge geometry, 2 node GEMMs, 3 pair GEMMs, 4 message, 5 aggregate, 6 energy head, 7 reverse pair
 * gather, 8 reverse message, 9 reverse aggregate, 10 force/virial, 11 other. */
#define NN_N_STAGES_API 12
NN_API int nn_profile_enable(int on);
NN_API int nn_profile_collect(float* ms_per_stage, int* n_per_stage, int n_stages);

/* ------------------------------------------------------------------ weights
 * fp32 device copies of the reference parameters (names: SURVEY.md section 8b).  A 128x128 matrix is
 * passed as `w` (torch layout [out, in]) and `wt` (its transpose [in, out]): forward products
 * x @ W^T use B = wt, reverse-sweep products g @ W use B = w (B is always row-major [K, N]).
 * `w_img` / `wt_img` are the tensor-core operand images of w / wt written by nn_gemm128_prepare_b
 * (NULL = tensor-core backend unavailable for this matrix).
 */
typedef struct {
    const float *w, *wt, *w_img, *wt_img;
} nn_mat;

typedef struct {
    nn_mat W1; const float* b1;     /* interaction_layers.l.message_nodepart.0 */
    nn_mat W2; const float* b2;     /* interaction_layers.l.message_nodepart.2 */
    const float *We, *Wet;          /* message_edgepart.weight [F, nb] and its transpose [nb, F] */
    const float *We_img;            /* tensor-core operand image of We (nn_message_prepare_b), or NULL */
    nn_mat U1, U2;                  /* equiv_message1.{0,2}.weight */
    nn_mat V1, V2;                  /* equiv_message2.{0,2}.weight */
    nn_mat Wu;                      /* equiv_update.weight */
    const float *ln_gamma, *ln_beta; /* layer_norm.{weight,bias} [F] (layer_norm=True, models/newtonnet.py:202-205) or NULL */
} nn_layer_weights;

typedef struct {
    int32_t n_layers;
    float cutoff;
    const float* embedding;         /* embedding_layers.node_embedding.weight [119, F] */
    const float* frequencies;       /* embedding_layers.edge_embedding.embedding.frequencies [nb] */
    nn_layer_weights layer[NN_MAX_LAYERS];
    nn_mat H1; const float* hb1;    /* output_layers.k.layers.0 */
    nn_mat H2; const float* hb2;    /* output_layers.k.layers.2 */
    const float *w3, *hb3;          /* output_layers.k.layers.4  ([1,F], [1]) */
    const float *scale, *shift;     /* scalers.k.{scale,shift}.weight [119] */
    /* optional direct_force head (models/output.py:115-132): layers.{0,2,4} 128->128 and its per-element scale */
    nn_mat D1; const float* db1;
    nn_mat D2; const float* db2;
    nn_mat D3; const float* db3;
    const float* dscale;            /* scalers.k.scale.weight [119] of the direct_force head, or NULL = head absent */
} nn_weights;

/* ------------------------------------------------------------------ neighbour list
 * Replaces RadiusGraph.forward, newtonnet/layers/representations.py:57-100 (dense O(N^2) mesh) with a
 * per-system cell list; each candidate pair is tested with the reference's fp32 arithmetic so the edge
 * set is bit-identical (diagonal or zero cells; other cells use the same formula with an fp32 inverse).
 */
typedef struct {
    int32_t n_atoms, n_systems;
    int32_t cap_edges;              /* capacity of col / edge_pair */
    int32_t cap_pairs;              /* capacity of pair_* (>= cap_edges / 2) */
    int32_t cap_cells;              /* capacity of the cell arrays (>= 2 * n_atoms + n_systems) */
    int32_t n_owned;                /* > 0: pairs between two atoms with index >= n_owned (ghost-ghost) are
                                       dropped (domain decomposition); 0 = keep all */
    const float* pos;               /* [N,3] */
    const float* cell;              /* [B,3,3] rows = lattice vectors; all zero = not periodic */
    const int64_t* batch;           /* [N] system id of each atom, non-decreasing */
    /* outputs */
    int32_t* sys_ptr;               /* [B+1] first atom of each system */
    int32_t* row_ptr;               /* [N+1] */
    int32_t* col;                   /* [cap_edges] source atom j, ascending within a row */
    int32_t* edge_pair;             /* [cap_edges] pair id | (reversed << 31) */
    int32_t* pair_ptr;              /* [N+1] first pair whose lower atom is i */
    int32_t* pair_i;                /* [cap_pairs] */
    int32_t* pair_j;                /* [cap_pairs] */
    float* pair_disp;               /* [cap_pairs,3] pos_i - pos_j, minimum image (reference arithmetic) */
    int32_t* status;                /* [NN_STATUS_WORDS] */
    void* workspace;                /* nn_nbr_workspace_bytes() */
    size_t workspace_bytes;
} nn_nbr;

NN_API size_t nn_nbr_workspace_bytes(int32_t n_atoms, int32_t n_systems);
/* pass 1: bins the atoms, counts neighbours, writes sys_ptr, row_ptr and status[NN_ST_N_EDGES]. */
NN_API int nn_nbr_count(const nn_nbr* nl, float cutoff, void* stream);
/* pass 2: fills col / edge_pair / pair_*; entries beyond the capacities are dropped and flagged. */
NN_API int nn_nbr_fill(const nn_nbr* nl, float cutoff, void* stream);
/* rev[e] = position of the reversed edge (j, i) of directed edge e = (i, j), rev [cap_edges]: read in row order it lists
 * the edges grouped by SOURCE atom (the transposed adjacency of the symmetric edge set), which is what the scatter to the
 * source atoms of the training path needs (models/newtonnet.py:211 mn[edge_index[1]] under autograd). */
NN_API int nn_nbr_edge_reverse(const nn_nbr* nl, int32_t* rev, void* stream);
/* edge_index [2,E] int64 in the reference's order (representations.py:74-82,97). */
NN_API int nn_nbr_edge_index(const nn_nbr* nl, int64_t* edge_index, int64_t n_edges, void* stream);

/* ------------------------------------------------------------------ dense contraction (F = 128)
 * Y[M,128] = epilogue( prologue(X)[M,128] @ B[128,128] ), B row-major [K,N].  Replaces the addmm / mm
 * calls of models/newtonnet.py:209,218,222,230 and models/output.py:98-100 and their autograd
 * transposes.  `m_dev` (optional) holds the row count on the device; then `m` is the launch capacity.
 */
/* prologues: NONE; SILU: silu(X); ROWSCALE3: X[r] * aux2[r/3]; SILU_SAVE: silu(X) and additionally
 * aux_out = silu'(X) (aux_out may alias X: the reverse sweep then needs no transcendental).
 * epilogues: BIAS: + bias (may be NULL); DSILU: * silu'(aux1); ADD: + aux1; EQUIV_BWD: + aux1 + aux2[r/3]*aux3;
 * MUL: * aux1. */
enum { NN_PRO_NONE = 0, NN_PRO_SILU = 1, NN_PRO_ROWSCALE3 = 2, NN_PRO_SILU_SAVE = 3 };
enum { NN_EPI_BIAS = 0, NN_EPI_DSILU = 1, NN_EPI_ADD = 2, NN_EPI_EQUIV_BWD = 3, NN_EPI_MUL = 4 };
#define NN_B_IMAGE_FLOATS (2 * 128 * 128)
typedef struct {
    const float* X; const float* B; float* Y;
    const float* B_img;             /* operand image of B from nn_gemm128_prepare_b (tensor-core backend) */
    const float* bias;              /* NN_EPI_BIAS: [128] or NULL */
    const float* aux1;              /* DSILU: pre-activation; ADD: addend; MUL: factor; EQUIV_BWD: fbar  (all [M,128]) */
    const float* aux2;              /* ROWSCALE3 / EQUIV_BWD: abar [M/3,128] */
    const float* aux3;              /* EQUIV_BWD: g [M,128] */
    float* aux_out;                 /* SILU_SAVE: receives silu'(X) [M,128] */
    const int32_t* m_dev; int32_t m_dev_mul;   /* rows = m_dev[0] * m_dev_mul when m_dev != NULL */
    int32_t m;
    int32_t prologue, epilogue;
    int32_t aux_tiled;              /* NN_EPI_MUL only: aux1 is stored tile-transposed (NN_TILED_INDEX), as the chained kernel writes it */
} nn_gemm_args;
/* Tile-transposed ("row-owner") layout of an [M,128] fp32 tensor: tiles of 128 rows, inside a tile the 16-byte chunk c
 * (0..31) of row r (0..127) lives at float offset ((tile * 32 + c) * 128 + r) * 4.  tcgen05.ld / st hand every lane one ROW
 * of the accumulator, so in this layout the 32 lanes of a warp touch 512 contiguous bytes per instruction and the
 * activation-derivative tensors silu'(q) that travel between the forward and the reverse MLP kernels need no
 * shared-memory transpose on either side.  Buffers in this layout hold ceil(M / 128) * 128 rows. */
#define NN_TILED_INDEX(row, col) ((((size_t)((row) >> 7) * 32 + ((col) >> 2)) * 128 + ((row) & 127)) * 4 + ((col) & 3))
NN_API int nn_gemm128(const nn_gemm_args* a, void* stream);
/* Two chained contractions in one kernel (a cluster of two CTAs, the intermediate tile travels through distributed
 * shared memory instead of HBM):  Y = out( mid(X . B1) . B2 ).  Every two-layer 128->128 MLP of the path and its
 * reverse: models/newtonnet.py:181-199 (message_nodepart, equiv_message1/2), models/output.py:90-96 (energy head).
 *   mid = NN_MID_SILU_SAVE: q = acc + bias1; aux_out = silu'(q); h = silu(q)      (forward)
 *   mid = NN_MID_MUL      : h = acc * aux1                                         (reverse)
 *   out = NN_OUT_BIAS     : Y = acc + bias2 (bias2 may be NULL)     out = NN_OUT_ADD: Y = acc + aux2
 * aux_out (mid = SILU_SAVE) and aux1 (mid = MUL) are in the tile-transposed layout (NN_TILED_INDEX) and hold whole tiles
 * of 128 rows; X, Y and aux2 are row-major.  Bit-identical to two nn_gemm128 calls (the second of a reverse pair reading
 * aux1 with aux_tiled = 1).  B1_img / B2_img: nn_gemm128_prepare_b images.  tcgen05 only. */
#define NN_MID_SILU_SAVE 0
#define NN_MID_MUL 1
#define NN_OUT_BIAS 0
#define NN_OUT_ADD 1
typedef struct {
    const float* X; const float* B1_img; const float* B2_img;
    const float* bias1; const float* bias2;
    const float* aux1; const float* aux2; float* aux_out;
    float* Y;
    const int32_t* m_dev; int32_t m_dev_mul;   /* rows = m_dev[0] * m_dev_mul when m_dev != NULL */
    int32_t m;
    int32_t mid, out;
    /* optional SECOND chain over the same X (NULL = none): Y_b = out( mid(X . B1_img_b) . B2_img_b ), aux_out_b its mid
     * output; same mid / out steps, no biases.  The two chains run in one launch, odd / even clusters walking the tiles
     * in lockstep, so X is fetched from HBM once (the second read is an L2 hit): equiv_message1 and equiv_message2 of one
     * layer share their input (models/newtonnet.py:218,222). */
    const float* B1_img_b; const float* B2_img_b; float* aux_out_b; float* Y_b;
    int32_t pad_;
} nn_gemm_chain_args;
NN_API int nn_gemm128_chain(const nn_gemm_chain_args* a, void* stream);
/* Writes the tensor-core operand image of B ([128,128] row-major K x N): B^T split into tf32 hi / lo
 * parts, laid out as UMMA K-major 128B-swizzled blocks; `image` holds NN_B_IMAGE_FLOATS floats. */
NN_API int nn_gemm128_prepare_b(const float* B, float* image, void* stream);
/* the same for n matrices in one launch; src / image are HOST arrays of device pointers, transposed[i] != 0 takes src[i]^T
 * as the operand (a weight in its other orientation: forward x W^T and reverse g W need both images of W). */
NN_API int nn_gemm128_prepare_b_batch(const float* const* src, const int32_t* transposed, float* const* image, int32_t n,
                                      void* stream);
/* backend for nn_gemm128 and nn_eval: 0 = fp32 SIMT, 1 = tcgen05 3xTF32 with A and B in shared memory,
 * 2 = tcgen05 3xTF32 with the A operand in tensor memory (TS mode). */
NN_API int nn_set_gemm_backend(int backend);
NN_API int nn_get_gemm_backend(void);

/* ------------------------------------------------------------------ whole evaluation
 * energy[B], forces[N,3], virial[B,3,3] (= -dE/dD, models/output.py:161-165), stress = -virial/det(cell)
 * (models/output.py:174-180) for NewtonNet.forward with heads energy / gradient_force / stress / virial.
 * Replaces EmbeddingNet.forward (models/newtonnet.py:139-161), EdgeEmbedding (layers/
 * representations.py:20-43), InteractionNet.forward x L (models/newtonnet.py:207-237), EnergyOutput +
 * ScaleShift + EnergyAggregator (models/output.py:98-100,246; layers/scalers.py:55-58) and the
 * autograd replay of DerivativeProperty._save_grad (models/output.py:66-73) by the hand-derived
 * reverse sweep of SURVEY.md section 8a row B.
 */
typedef struct {
    const nn_nbr* nbr;
    const nn_weights* w;
    const int64_t* z;               /* [N] atomic numbers */
    int32_t want_forces;            /* 0: energy only (no reverse sweep) */
    int32_t want_virial;
    int32_t n_owned;                /* domain decomposition: atoms [0, n_owned) are owned, [n_owned, N) are
                                       ghosts whose feature rows the caller refreshes between phases;
                                       0 = all atoms owned (single GPU) */
    int32_t pad_;
    /* outputs */
    float* energy;                  /* [B] */
    float* forces;                  /* [N,3] */
    float* virial;                  /* [B,9] */
    float* stress;                  /* [B,9] or NULL */
    float* atom_node;               /* [N,F]   final invariant features (CustomOutputSet.atom_node) */
    float* force_node;              /* [N,3,F] final equivariant features */
    float* direct_force;            /* [N,3] direct_force head output, or NULL */
    void* workspace; size_t workspace_bytes;   /* nn_eval_workspace_bytes() */
} nn_eval_args;
NN_API size_t nn_eval_workspace_bytes(int32_t n_atoms, int32_t n_systems, int32_t cap_pairs, int32_t n_layers,
                               int32_t want_forces);
NN_API int nn_eval(const nn_eval_args* a, void* stream);
/* The same evaluation split into phases, for spatial domain decomposition: node-level work covers the
 * owned atoms, pair-level work every local pair (owned-owned and owned-ghost); after the phases marked
 * [x] the caller copies the named buffers' ghost rows from their owner ranks (halo exchange).
 *   BEGIN, then per layer l: FWD_NODE(l) [mn(l), and f_out(l-1) if l>0], FWD_PAIR(l); HEAD;
 *   BWD_SEED, then per layer l = L-1..0: BWD_NODE(l) [dfb, abar], BWD_PAIR(l); FINISH.
 * energy / virial / stress then hold this rank's partial sums, forces the owned rows. */
enum { NN_PH_BEGIN = 0, NN_PH_FWD_NODE = 1, NN_PH_FWD_PAIR = 2, NN_PH_HEAD = 3, NN_PH_BWD_SEED = 4,
       NN_PH_BWD_NODE = 5, NN_PH_BWD_PAIR = 6, NN_PH_FINISH = 7,
       /* finer split, so that exchanges off the critical path can run on a second stream:
        * FWD_PAIR = FWD_PAIR_A (message, edge MLPs, aggregation: needs ghost mn(l), f_out(l-1); produces f_out(l)) +
        *            FWD_PAIR_B (equivariant update, layer norm: owned rows only);
        * BWD_NODE = BWD_NORM (layer-norm reverse: abar(l) final) + BWD_NODE_B (dfb);
        * BWD_PAIR = BWD_PAIR_A (pair gather + reverse edge MLPs: needs ghost dfb, f_out(l-1)) +
        *            BWD_PAIR_B (reverse message, aggregation, node MLP: needs ghost abar, mn(l)) */
       NN_PH_FWD_PAIR_A = 8, NN_PH_FWD_PAIR_B = 9, NN_PH_BWD_NORM = 10, NN_PH_BWD_NODE_B = 11,
       NN_PH_BWD_PAIR_A = 12, NN_PH_BWD_PAIR_B = 13 };
enum { NN_BUF_MN = 0, NN_BUF_F_OUT = 1, NN_BUF_DFB = 2, NN_BUF_ABAR = 3 };
NN_API int nn_eval_phase(const nn_eval_args* a, int32_t phase, int32_t layer, void* stream);
/* device pointer of an exchanged buffer inside the workspace: MN [N,F], F_OUT [N,3,F] (per layer),
 * DFB [N,3,F], ABAR [N,F]. */
NN_API float* nn_eval_buffer(const nn_eval_args* a, int32_t which, int32_t layer);
/* out[k, :] = src[idx[k], :] for k < n (width floats per row): packs the rows a rank sends to a peer. */
NN_API int nn_halo_pack(const float* src, const int32_t* idx, int32_t n, int32_t width, float* out, void* stream);

/* ------------------------------------------------------------------ staged operators (also used by
 * nn_eval; exported for per-kernel parity tests and for the differentiable training path) */
/* ScaledNorm + PolynomialCutoff * RadialBessel, representations.py:129-131,166-169,233,41:
 * per pair d, u = disp/d, x = d/rc, rbf[nb] = env(x) * sin(f_n x) / x and (optional, for the reverse
 * sweep) drbf[nb] = d rbf / dx. */
NN_API int nn_edge_geom_fwd(const float* pair_disp, const float* freq, float cutoff, const int32_t* n_pairs_dev,
                            int32_t cap_pairs, float* rbf, float* drbf, float* unit, float* dist, void* stream);
/* reverse of the above: G_p = dE/d disp_p from dE/dx and unit_bar [P,3]; dE/dx is given as `n_slots`
 * partial arrays x_bar[slot * cap_pairs + p] (one or two per layer) that are summed in slot order. */
NN_API int nn_edge_geom_bwd(const float* x_bar, int32_t n_slots, const float* unit_bar, const float* unit,
                            const float* dist, float cutoff, const int32_t* n_pairs_dev, int32_t cap_pairs,
                            float* disp_bar, void* stream);
/* image of message_edgepart.weight [128, 20] for the tensor-core message kernels (2 * 4096 floats). */
#define NN_WE_IMAGE_FLOATS (2 * 128 * 32)
NN_API int nn_message_prepare_b(const float* We, float* image, void* stream);
/* m_p = (We rbf_p) * mn_i * mn_j, models/newtonnet.py:210-211, for the pairs p < status[NN_ST_N_PAIRS] (rows past the
 * count are not written).  Tensor-core backend (nn_get_gemm_backend() >= 1) with We_img != NULL: the persistent tcgen05
 * kernel (3xTF32, We_img from nn_message_prepare_b) that nn_eval runs; otherwise the fp32 SIMT kernel, which needs Wet. */
NN_API int nn_edge_message_fwd(const nn_nbr* nl, const float* rbf, const float* mn, const float* Wet,
                               const float* We_img, float* msg, void* stream);
/* a_out = a + sum_e m ; f_out = f + sum_e (e1 u + e2 * f_j), models/newtonnet.py:213-227. */
NN_API int nn_node_aggregate_fwd(const nn_nbr* nl, const float* msg, const float* e1, const float* e2,
                          const float* unit, const float* a_in, const float* f_in, float* a_out,
                          float* f_out, int32_t first_layer, void* stream);
/* a_out = a + sum_c f[c] * g[c], models/newtonnet.py:230-231 (g = f @ Wu^T from nn_gemm128). */
NN_API int nn_equiv_update_fwd(const float* a_in, const float* f, const float* g, float* a_out, int32_t n_atoms,
                        void* stream);
/* atomic energy + scale/shift + per-system sum: models/output.py:100,246, layers/scalers.py:55-58. */
NN_API int nn_energy_head_fwd(const float* h2pre, const float* w3, const float* b3, const float* scale,
                       const float* shift, const int64_t* z, const int32_t* sys_ptr, int32_t n_atoms,
                       int32_t n_systems, float* e_atom, float* energy, void* stream);
/* F_i = -sum_e sign_e G_p(e); virial with the reference's strain convention (see DESIGN.md). */
NN_API int nn_force_virial_reduce(const nn_nbr* nl, const float* disp_bar, float* forces, float* virial,
                           float* stress, void* workspace, void* stream);

/* ------------------------------------------------------------------ domain decomposition over NVLink peer memory
 * SURVEY.md section 8e (the reference itself is single-process: layers/representations.py:72-93 is one dense mesh).
 * Every rank owns one arena from nn_p2p_alloc (plain cudaMalloc, zero-filled, so that CUDA IPC handles - 64 bytes,
 * exchanged by the caller - can map it into the other processes): landing buffers for ghost feature rows, flag words,
 * the complete force array [n_atoms_total,3] and a table of per-rank partial sums.  The step counter the flag epochs
 * derive from lives in device memory, so one decomposed evaluation (nn_dd_begin, nn_nbr_*, nn_eval_phase interleaved
 * with nn_dd_halo_push / nn_dd_halo_wait, nn_dd_finish) is capturable as ONE CUDA graph; there is no NCCL call on the
 * data path.  Channels: independent (landing buffers, flags, epoch sequence) triples so that a second stream can
 * exchange rows off the critical path; every rank must issue the same sequence seq = 0 .. stride[channel]-1 of
 * exchanges per channel and step (nn_dd_finish is the last exchange of channel 0). */
#define NN_DD_MAX_RANKS 16
#define NN_DD_CHANNELS 2
#define NN_DD_MAX_WIDTH 384         /* floats per exchanged row: F or 3F */
#define NN_DD_PARTIAL 32            /* floats per rank in the partial table */
#define NN_DD_STATUS_WORDS 8
enum { NN_DD_ST_STALE = 0,          /* an owned atom moved more than skin/2 since the plan was made: replan */
       NN_DD_ST_TIMEOUT = 1,        /* a peer did not publish its flag within ~2 s */
       NN_DD_ST_OVERFLOW = 2,       /* some rank's neighbour list outgrew its capacity */
       NN_DD_ST_BAD_INPUT = 3,      /* row overflow / unsorted batch / singular cell on some rank */
       NN_DD_ST_STEP = 4,           /* device step counter */
       NN_DD_ST_EDGES = 5 };        /* directed edges summed over ranks / 1024 */
typedef struct {
    int32_t world, rank, n_atoms_total, n_owned, n_ghost, pad_;
    int32_t stride[NN_DD_CHANNELS];                     /* exchanges per step on each channel */
    /* this rank's arena */
    float* landing[NN_DD_CHANNELS][2];                  /* [n_ghost, NN_DD_MAX_WIDTH] each, alternating by epoch parity */
    int32_t* flags[NN_DD_CHANNELS];                     /* [world]: last epoch each source rank has published here */
    float* forces_full;                                 /* [n_atoms_total, 3] */
    float* partials;                                    /* [world, NN_DD_PARTIAL] */
    /* the same regions of the other ranks, mapped into this process (index = rank; own entries unused) */
    float* peer_landing[NN_DD_CHANNELS][2][NN_DD_MAX_RANKS];
    int32_t* peer_flags[NN_DD_CHANNELS][NN_DD_MAX_RANKS];
    float* peer_forces_full[NN_DD_MAX_RANKS];
    float* peer_partials[NN_DD_MAX_RANKS];
    /* send plan: local rows send_idx[send_begin[s] .. send_end[s]) go to rank s and land at row row_offset[s] of its
     * ghost order; ranges are contiguous in rank order (own range empty) */
    const int32_t* send_idx;
    int32_t send_begin[NN_DD_MAX_RANKS], send_end[NN_DD_MAX_RANKS], row_offset[NN_DD_MAX_RANKS];
    int32_t* step;                                      /* device, 1 int: step counter */
    uint32_t* done;                                     /* device, NN_DD_CHANNELS zeroed counters */
    int32_t* status;                                    /* device, NN_DD_STATUS_WORDS (local flags) */
} nn_dd_comm;
NN_API int nn_p2p_alloc(size_t bytes, void** ptr);
NN_API int nn_p2p_free(void* ptr);
NN_API int nn_p2p_get_handle(void* ptr, void* handle64);
NN_API int nn_p2p_open_handle(const void* handle64, void** ptr);
NN_API int nn_p2p_close_handle(void* ptr);
/* starts a step: pos_local[i] = pos[l2g[i]], z_local[i] = z[l2g[i]] for the n_local = n_owned + n_ghost local atoms;
 * raises the sticky STALE flag when an owned atom is further than skin/2 from pos_ref or the cell differs from
 * cell_ref (the state the brick / ghost plan was made for); advances the step counter. */
NN_API int nn_dd_begin(const nn_dd_comm* c, const float* pos, const float* pos_ref, const float* cell, const float* cell_ref,
                       const int64_t* z, const int32_t* l2g, int32_t n_local, float skin, float* pos_local,
                       int64_t* z_local, void* stream);
/* owner -> ghost copy of rows [*, width] (width = F or 3F): push stores this rank's rows into the peers' landing
 * buffers and raises the flags; wait spins (bounded) on the local flags and copies the landing buffer into
 * ghost_rows = first ghost row of the same array. */
NN_API int nn_dd_halo_push(const nn_dd_comm* c, int32_t channel, int32_t seq, const float* rows, int32_t width, void* stream);
NN_API int nn_dd_halo_wait(const nn_dd_comm* c, int32_t channel, int32_t seq, float* ghost_rows, int32_t width, void* stream);
/* completes the step: owned forces are written into every rank's complete force array (owner-only writes), the
 * partial energy [1] / virial [9] / stress [9] and status words into every rank's table; after the flags,
 * forces_out [n_atoms_total,3], out_small = {energy, virial[9], stress[9]} (fp64 sums in rank order: the same
 * bits on every rank) and out_status [NN_DD_STATUS_WORDS] (OR over ranks) are written.  virial / stress may be NULL. */
NN_API int nn_dd_finish(const nn_dd_comm* c, int32_t seq, const float* forces_owned, const int32_t* l2g, const float* energy,
                        const float* virial, const float* stress, const int32_t* nbr_status, float* forces_out,
                        float* out_small, int32_t* out_status, void* stream);

/* ------------------------------------------------------------------ training-path primitives (row T)
 * Closed under differentiation together with nn_gemm128 and nn_halo_pack (= gather rows), so autograd can
 * compose the double backward of reference train/trainer.py:303-313. */
/* out[i,:] = sum over k in [row_ptr[i], row_ptr[i+1]) of src[perm ? perm[k] : k, :]  (fixed order) - the
 * deterministic form of torch_geometric.utils.scatter(reduce='sum') (models/newtonnet.py:214,226). */
NN_API int nn_segment_sum(const float* src, const int32_t* perm, const int32_t* row_ptr, int32_t n_rows,
                          int32_t width, float* out, void* stream);
/* out[128,128] = X[m,128]^T @ Y[m,128]  (weight gradients of the 128x128 linears). */
NN_API size_t nn_gemm128_tn_workspace_bytes(int32_t m);
NN_API int nn_gemm128_tn(const float* X, const float* Y, int32_t m, float* out, void* workspace, void* stream);
/* out = (accumulate ? out : 0) + X^T Y: a parameter's gradient summed over its uses (what autograd's AccumulateGrad does,
 * reference train/trainer.py:309 loss.backward()) without a separate add kernel; fixed summation order. */
NN_API int nn_gemm128_tn_acc(const float* X, const float* Y, int32_t m, float* out, void* workspace, int32_t accumulate,
                             void* stream);

/* Fused row products of the training path: the element-wise glue of InteractionNet.forward (models/newtonnet.py:211,
 * 219-226,231) as kernels that are closed under differentiation (each gradient is a combination of the others), so
 * autograd composes forward / backward / double backward from them.  Rows of F = 128 floats.
 *   nn_ew_mul3: out = a * b * c (n_floats elements).
 *   nn_ew_rows(mode): p [n,F], q3 [n,3,F], u [n,3]:
 *     0 outer      out[n,3,F] = p[e,:] * u[e,c]            1 contract_c  out[n,F] = sum_c q3[e,c,:] * u[e,c]
 *     2 row_dot    out[n,3]   = <q3[e,c,:], p[e,:]>        3 mul_b       out[n,3,F] = p[e,:] * q3[e,c,:]
 *     4 sum_mul_c  out[n,F]   = sum_c q3[e,c,:] * p3[e,c,:]   (the second [n,3,F] operand is passed as p) */
NN_API int nn_ew_mul3(const float* a, const float* b, const float* c, float* out, int64_t n_floats, void* stream);
NN_API int nn_ew_rows(int32_t mode, const float* p, const float* q3, const float* u, float* out, int32_t n_rows, void* stream);
/* The message product with GATHERED operands (no [E,F] copy of the node rows is materialised):
 *   nn_ew_gmul:        out[e,:] = a[e,:] * (b ? b[e,:] : 1) * r1[i1[e],:] * (r2 ? r2[i2[e],:] : 1)   (models/newtonnet.py:211)
 * Closed under differentiation together with nn_ew_mul3 / nn_segment_sum. */
NN_API int nn_ew_gmul(const float* a, const float* b, const float* r1, const int32_t* i1, const float* r2, const int32_t* i2,
                      float* out, int32_t n_rows, void* stream);
/* Equivariant aggregation (models/newtonnet.py:219-226) without [E,3,F] intermediates; segments are CSR rows (row_ptr, optional
 * perm = edge ids in row order), rows3 an [N,3,F] node table read through an edge index:
 *   nn_seg_prod(u):       out[k,c,:] = sum_{e in seg(k)} x[e,:] * u[e,c]
 *   nn_seg_prod(rows3):   out[k,c,:] = sum_{e in seg(k)} x[e,:] * rows3[idx[e],c,:]
 *   nn_ew_g3(0, p = u):   out[e,:] = sum_c u[e,c] * rows3[idx[e],c,:]
 *   nn_ew_g3(1, p = x):   out[e,c] = < rows3[idx[e],c,:], x[e,:] >
 *   nn_ew_g3(2):          out[e,:] = sum_c rows3[idx[e],c,:] * rowsb[idxb[e],c,:]
 * Closed under differentiation (each gradient is another member), fixed summation order. */
NN_API int nn_seg_prod(const float* x, const float* u, const float* rows3, const int32_t* idx, const int32_t* perm,
                       const int32_t* row_ptr, int32_t n_rows, float* out, void* stream);
NN_API int nn_ew_g3(int32_t mode, const float* rows3, const int32_t* idx, const float* p, const float* rowsb, const int32_t* idxb,
                    float* out, int32_t n_rows, void* stream);
/* SiLU with its first two derivatives (layers/activations.py:13 nn.SiLU under autograd twice): mode 0 out = silu(x);
 * mode 1 out = a * silu'(x); mode 2 out = a * b * silu''(x). */
/* Radial basis R_n(x) = env(x) sin(f_n x) / x (representations.py:166-169,233) with its x-derivatives of order k = 0..2:
 * op 0 (scale): out[e,n] = (a ? a[e] : 1) * R^k_n(x[e])  ([n_rows, 20]);  op 1 (dot): out[e] = sum_n a[e,n] R^k_n(x[e]). */
NN_API int nn_ew_rbf(int32_t op, int32_t k, const float* a, const float* x, const float* freq, float* out, int32_t n_rows, void* stream);
NN_API int nn_ew_silu(int32_t mode, const float* x, const float* a, const float* b, float* out, int64_t n_floats, void* stream);

/* ---- reverse-sweep operators (SURVEY.md section 8a row B) as standalone entry points; nn_eval composes exactly these.
 * They replace the autograd replay of DerivativeProperty._save_grad (models/output.py:66-73) piece by piece. */
/* Y = silu(X M1^T + b1) M2^T + b2; `mid` receives the pre-activation, or silu'(pre-activation) when save_dact != 0 (what
 * nn_mlp_bwd consumes).  m_dev != NULL: pair-level call, rows = m_dev[0] <= m.  One chained launch where it pays; then `mid`
 * is written in the tile-transposed layout (NN_TILED_INDEX) and must hold ceil(m / 128) * 128 rows - nn_mlp_mid_tiled tells
 * which, for the same (m, m_dev != NULL) that nn_mlp_fwd / nn_mlp_bwd are called with. */
NN_API int nn_mlp_mid_tiled(int32_t m, int32_t has_m_dev);
NN_API int nn_mlp_fwd(const float* X, const nn_mat* M1, const float* b1, float* mid, const nn_mat* M2, const float* b2, float* Y,
                      int32_t m, const int32_t* m_dev, int32_t save_dact, void* stream);
/* Y (+)= ((G M2) * dact) M1: the transpose of nn_mlp_fwd with respect to X.  `tmp` [m,128] may alias G. */
NN_API int nn_mlp_bwd(const float* G, const nn_mat* M2, const float* dact, float* tmp, const nn_mat* M1, float* Y, int32_t m,
                      const int32_t* m_dev, int32_t accumulate, void* stream);
/* gh2[i,:] = scale[z_i] * w3 * silu'(h2pre[i,:]): d(sum of atomic energies)/d(second hidden layer), models/output.py:98-100 */
NN_API int nn_energy_head_bwd(const float* h2pre, const float* w3, const float* scale, const int64_t* z, int32_t n_atoms,
                              float* gh2, void* stream);
/* per pair p = (i<j), with w[c] = dfb_i[c] - dfb_j[c]:  ubar_p[c] += <w[c], e1_p>;  e1_io_p <- sum_c w[c] u_p[c]  (in place);
 * e2bar_p = sum_c dfb_i[c] * f_in_j[c] + dfb_j[c] * f_in_i[c]  (skipped when f_in == NULL: first layer).  dfb, f_in [N,3,128]. */
NN_API int nn_pair_gather_bwd(const nn_nbr* nl, const float* dfb, const float* f_in, const float* unit, float* e1_io,
                              float* e2bar, float* ubar, void* stream);
/* mt = mbar_p + abar_i + abar_j;  y = mt * mn_i * mn_j;  x_part <- <y, We drbf_p> (tensor-core backend: two partial sums
 * x_part[0][p] + x_part[1][p] over the column halves; SIMT: x_part[0][p], row 1 untouched);  mbar_io_p <- mt * (We rbf_p). */
NN_API int nn_edge_message_bwd(const nn_nbr* nl, const float* abar, const float* mn, const float* rbf, const float* drbf,
                               const float* Wet, const float* We_img, float* mbar_io, float* x_part, void* stream);
/* mnbar_k = sum_{e=(k,i)} t_p(e) * mn_i;  fbar_new_k[c] = dfb_k[c] + sum_{e=(k,i)} dfb_i[c] * e2_p(e)  (skipped when e2 == NULL) */
NN_API int nn_node_aggregate_bwd(const nn_nbr* nl, const float* t, const float* mn, const float* e2, const float* dfb,
                                 float* mnbar, float* fbar_new, void* stream);

/* ---- device-resident molecular dynamics (caller side of the path; SURVEY.md 8f rank 1) --------------------
 * Replaces the per-step host loop of the reference's MD driver: scripts/simulate.py:21-31 (ASE Langevin) calling
 * MLAseCalculator.calculate, utils/ase_interface.py:52-81, i.e. numpy -> H2D -> forward -> D2H every step.
 * One step = nn_md_advance -> nn_nbr_count -> nn_nbr_fill -> nn_eval -> nn_md_finish on one stream (CUDA graph
 * capturable: every step-dependent quantity, including the step counter, lives in device memory).
 * BAOAB splitting; ou_c = exp(-friction * dt) (1.0 = velocity Verlet, no noise), kT in the energy unit.
 * x, v: [n_atoms,3] fp64 state (x unwrapped); pos_model: [n_atoms,3] fp32 wrapped positions bound to nn_nbr.pos. */
NN_API int nn_md_advance(int32_t n_atoms, double* x, double* v, const float* force, const double* inv_mass, const float* cell,
                         const int64_t* batch, float* pos_model, double dt, double ou_c, double kT, uint64_t seed,
                         const int64_t* step_ctr, void* stream);
/* second half kick with the new forces; writes log[(step % log_cap), system, {potential, kinetic}] (fp64), ORs the
 * neighbour-list status words into sticky[0..2] = {edges needed, max degree, singular cell} and increments *step_ctr. */
NN_API int nn_md_finish(int32_t n_systems, const int32_t* sys_ptr, double* v, const float* force, const double* inv_mass,
                        double dt, const float* energy, double* log, int32_t log_cap, int64_t* step_ctr,
                        const int32_t* nbr_status, int32_t* sticky, uint32_t* ticket, void* stream);
/* pos_model = x wrapped into each atom's cell, in fp32 (the wrap nn_md_advance and nn_fire_step apply after a step). */
NN_API int nn_wrap_positions(int32_t n_atoms, const double* x, const float* cell, const int64_t* batch, float* pos_model,
                             void* stream);

/* ---- device-resident geometry optimisation: FIRE per system of a batch (newtonnet_b200/optimize.py) ---------------
 * Replaces the host loop of an ASE optimiser around MLAseCalculator.calculate (utils/ase_interface.py:52-81): one step =
 * nn_fire_step -> nn_nbr_count -> nn_nbr_fill -> nn_eval -> nn_fire_check, capturable as one CUDA graph (all per-system
 * state, fmax and the step counter live in device memory).  The step is ase.optimize.FIRE.step (ASE 3.22 / 3.23,
 * downhill_check=False, no masses, ASE time units) run independently for every system b = [sys_ptr[b], sys_ptr[b+1]).
 * x, v: [n_atoms,3] fp64 (x unwrapped); force: [n_atoms,3] fp32 at x; pos_model: [n_atoms,3] fp32 wrapped, bound to
 * nn_nbr.pos; cell: [n_systems,3,3] (all zero = not periodic).
 * sys_f64: [n_systems,3] {dt, a, max_i |f_i|^2}; sys_i32: [n_systems,4] {Nsteps, started, converged, steps taken}.
 * Every sum is a fixed-order reduction over the system's own atoms, so a system's trajectory does not depend on which
 * other systems share the batch.  A converged system is not touched (its x, v and state are frozen). */
NN_API int nn_fire_step(int32_t n_systems, const int32_t* sys_ptr, double* x, double* v, const float* force, const float* cell,
                        float* pos_model, double* sys_f64, int32_t* sys_i32, double maxstep, double dtmax, double finc,
                        double fdec, double astart, double fa, int32_t nmin, void* stream);
/* After nn_eval: zeroes the forces of fixed atoms (fixed: [n_atoms] 0/1 bytes, or NULL), stores max_i |f_i|^2 over the
 * system in fp64 and sets converged = (max_i |f_i|^2 < *fmax2) (ASE's Optimizer.converged).  advance != 0 (the captured
 * step): also counts one step for every system that was not converged before the call, ORs the neighbour-list status words
 * into sticky[0..2] = {edges needed, max degree, singular cell} and increments *step_ctr (ticket: one zero-initialised
 * uint32, returned to 0).  advance = 0 only measures: step_ctr, nbr_status, sticky and ticket may be NULL. */
NN_API int nn_fire_check(int32_t n_systems, const int32_t* sys_ptr, float* force, const uint8_t* fixed, const double* fmax2,
                         double* sys_f64, int32_t* sys_i32, int32_t advance, int64_t* step_ctr, const int32_t* nbr_status,
                         int32_t* sticky, uint32_t* ticket, void* stream);

/* ---- device-resident climbing-image NEB: one FIRE system per band (newtonnet_b200/neb.py) ------------------------------
 * One step = nn_fire_step (band ranges) -> nn_nbr_count -> nn_nbr_fill -> nn_eval (one system per interior image) ->
 * nn_neb_forces -> nn_fire_check (band ranges, on neb_force), capturable as one CUDA graph.
 * NEB force of every interior image: ASE's NEB.get_forces with method='improvedtangent' and a scalar spring constant k
 * (ASE 3.22; where an image and both neighbours have equal energies the tangent is t+ + t-, not ASE's zero vector).
 * One block per interior image j of n_images; bands are stored band-major and images image-major:
 * img_ptr [n_images+1] first atom of each interior image; img_band [n_images] its band; band_img [n_bands+1] first
 * interior image of each band.  x [*,3] fp64 positions of the interior images; ends [*,3] fp64 end-point positions:
 * band b's image 0 at rows band_ends[b].., its last image right after; energy [n_images] fp32 (nn_eval's output);
 * ends_energy [n_bands,2] fp64; force [*,3] fp32 model forces (fixed: 0/1 bytes or NULL, fixed atoms' forces count as 0).
 * climb [n_bands] 0/1: the highest interior image (ties to the highest index) climbs; imax [n_bands] receives its index in
 * 1..n.  band_si: nn_fire_step's per-band int32 state: the blocks of a converged band write nothing.
 * neb_force [*,3] fp32 receives the NEB force (0 for fixed atoms).  A band whose model output is not finite (an interior
 * energy, or a force of a free atom) gets a zero NEB force on every image and failed[b] = 1 (failed: [n_bands] int32, only
 * ever set), so nn_fire_check finds it converged and the FIRE kernels leave it at its last, finite positions.  Spring vectors are never wrapped: periodic images
 * must be aligned (minimum-image displacements between consecutive images) before they are passed in. */
NN_API int nn_neb_forces(int32_t n_images, const int32_t* img_ptr, const int32_t* img_band, const int32_t* band_img,
                         const double* x, const double* ends, const int32_t* band_ends, const float* energy,
                         const double* ends_energy, const float* force, const uint8_t* fixed, const int32_t* climb,
                         const int32_t* band_si, double k, float* neb_force, int32_t* imax, int32_t* failed, void* stream);

/* ---- Hessian in blocks of rows (newtonnet_b200/hessian.py; reference models/output.py:141-152 batches rows with vmap) ----
 * A pass puts k copies of frames of n_slot atoms into one batch (copy c = system c) and differentiates <seed, pos_grad>
 * once: copy c's block of that gradient is row plan[pass][c].row of its frame's Hessian.
 * plan: [n_pass, k, 3] int32 {frame, local row in [0, 3 n_slot) or -1 for a padding job, output row};
 * frame_ptr: [n_frames + 1] first atom of each frame of the input batch; every planned frame has n_slot atoms.
 * *pass_ctr: index of the pass both calls work on (device memory: a captured pass replays without host traffic).
 * expand: z_rep [k n_slot], pos_rep [k n_slot, 3], cell_rep [k,3,3], batch_rep [k n_slot] (= copy index), seed [k n_slot, 3]
 *         (one-hot at the job's row in its copy's block; all zero for a padding job). */
NN_API int nn_hessian_expand(const int32_t* plan, const int32_t* pass_ctr, int32_t k, int32_t n_slot, const int64_t* z,
                             const float* pos, const float* cell, const int32_t* frame_ptr, int64_t* z_rep, float* pos_rep,
                             float* cell_rep, int64_t* batch_rep, float* seed, void* stream);
/* H[out, :] for each real job of the pass: columns 3 frame_ptr[f] .. 3 frame_ptr[f+1] from copy c of grad_rep [k n_slot, 3],
 * all other n_cols columns 0 (each element written once, no atomics); padding jobs write nothing.  Then advances
 * *pass_ctr by one (ticket: one zero-initialised uint32, returned to 0 by the call). */
NN_API int nn_hessian_scatter(const int32_t* plan, int32_t* pass_ctr, int32_t k, int32_t n_slot, const int32_t* frame_ptr,
                              const float* grad_rep, float* H, int64_t n_cols, uint32_t* ticket, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEWTONNET_B200_H */
