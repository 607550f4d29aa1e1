#include <cstdlib>
// nn_eval: one call = one NewtonNet energy (+ forces, virial, stress) evaluation on a prebuilt
// neighbour list.  Launches the staged kernels on one stream, no host synchronisation, all buffers
// carved from the caller's workspace; capturable in a CUDA graph.
//
// Forward follows NewtonNet.forward (reference newtonnet/models/newtonnet.py:74-104); the reverse
// sweep is the hand-derived backward of SURVEY.md section 8a row B in pair-symmetric form (checked in
// fp64 against the reference's autograd by oracle/newtonnet_oracle.py::forward_analytic).
#include <stdarg.h>
#include "common.cuh"

int nn_gemm128_simt_launch(const nn_gemm_args& a, cudaStream_t s);
int nn_sum_slices(int n_atoms, int n_systems);
int nn_gemm128_tc_launch(const nn_gemm_args& a, cudaStream_t s);
int nn_gemm128_ts_launch(const nn_gemm_args& a, cudaStream_t s);
int nn_embed_launch(const int64_t* z, const float* emb, float* a, int N, int* status, cudaStream_t s);
int nn_energy_head_seed_launch(const float* h2pre, const float* w3, const float* scale, const int64_t* z, int N,
                               float* gh2, cudaStream_t s);
int nn_pair_bwd_gather_launch(const nn_nbr* nl, const float* dfb, const float* f_in, const float* unit, float* e1_io,
                              float* e2bar, float* ubar, bool first, cudaStream_t s);
int nn_pair_bwd_message_launch(const nn_nbr* nl, const float* abar, const float* mn, const float* rbf, const float* drbf,
                               const float* Wet, float* mbar_io, float* x_bar, cudaStream_t s);
int nn_layer_norm_fwd_launch(float* a_io, const float* gamma, const float* beta, float* xhat, float* rstd, int n_rows, cudaStream_t s);
int nn_layer_norm_bwd_launch(float* abar_io, const float* gamma, const float* xhat, const float* rstd, int n_rows, cudaStream_t s);
int nn_direct_force_launch(const float* h, const float* f, const float* scale, const int64_t* z, int n_rows, float* out, cudaStream_t s);
int nn_message_fwd_tc(const nn_nbr* nl, const float* rbf, const float* mn, const float* We_img, float* msg, cudaStream_t s);
int nn_edge_message_fwd_launch(const nn_nbr* nl, const float* rbf, const float* mn, const float* Wet, float* msg,
                               cudaStream_t s);
int nn_message_bwd_tc(const nn_nbr* nl, const float* abar, const float* mn, const float* rbf, const float* drbf,
                      const float* We_img, float* mbar_io, float* x_part, cudaStream_t s);
int nn_node_aggregate_bwd_launch(const nn_nbr* nl, int n_rows, const float* t, const float* mn, const float* e2,
                                 const float* dfb, float* mnbar, float* fbar_new, bool first, cudaStream_t s);

// ---------------------------------------------------------------------------- error / backend state
static thread_local char g_err[512] = "";
void nn_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char* nn_last_error(void) { return g_err; }
extern "C" int nn_version(void) { return 100; }

// ---------------------------------------------------------------------------- launch counter / stage profiler
#include <atomic>
#include <vector>
static std::atomic<long long> g_launches{0};
void nn_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
static bool chain_enabled() {          // two-CTA chained GEMM pairs (gemm_chain.cu); NN_CHAIN=0 falls back to two launches
    static int v = -1;
    if (v < 0) { const char* e = getenv("NN_CHAIN"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

// node-level MLPs (no device row count) take the chained kernel when they are small enough to be launch-latency-bound:
// one launch instead of two (measured: see DESIGN.md).  Large node-level inputs stay on two launches.
constexpr int kChainSmallM = 20000;

bool nn_pdl_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("NN_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

int nn_num_sms() {
    static int sms[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (sms[dev] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        sms[dev] = v > 0 ? v : 148;
    }
    return sms[dev];
}

extern "C" long long nn_launch_count(int reset) {
    long long v = g_launches.load();
    if (reset) g_launches.store(0);
    return v;
}

namespace {
struct ProfSample { cudaEvent_t e0, e1; int stage; };
struct Profiler {
    bool on = false;
    std::vector<ProfSample> samples;   // recorded since the last collect
    std::vector<cudaEvent_t> pool;     // reusable events
    cudaEvent_t cur0 = nullptr; int cur_stage = -1; int depth = 0;
    cudaEvent_t get() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
} g_prof;
}  // namespace

void nn_prof_begin(int stage, cudaStream_t s) {
    if (!g_prof.on) return;
    if (g_prof.depth++ > 0) return;          // nested scopes belong to the outer stage
    g_prof.cur0 = g_prof.get(); g_prof.cur_stage = stage;
    cudaEventRecord(g_prof.cur0, s);
}
void nn_prof_end(cudaStream_t s) {
    if (!g_prof.on) return;
    if (--g_prof.depth > 0) return;
    cudaEvent_t e1 = g_prof.get();
    cudaEventRecord(e1, s);
    g_prof.samples.push_back({g_prof.cur0, e1, g_prof.cur_stage});
}
extern "C" int nn_profile_enable(int on) { g_prof.on = on != 0; g_prof.depth = 0; return 0; }
// Sums the recorded stage times (ms) and sample counts; the caller must have synchronised the stream.
extern "C" int nn_profile_collect(float* ms_per_stage, int* n_per_stage, int n_stages) {
    for (int k = 0; k < n_stages; ++k) { ms_per_stage[k] = 0.f; n_per_stage[k] = 0; }
    for (auto& sm : g_prof.samples) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, sm.e0, sm.e1) == cudaSuccess && sm.stage < n_stages) {
            ms_per_stage[sm.stage] += ms; n_per_stage[sm.stage] += 1;
        }
        g_prof.pool.push_back(sm.e0); g_prof.pool.push_back(sm.e1);
    }
    g_prof.samples.clear();
    return NN_N_STAGES;
}

static int g_backend = 0;
extern "C" int nn_set_gemm_backend(int backend) {
    if (backend < 0 || backend > 2) { nn_set_error("unknown gemm backend %d", backend); return -1; }
    g_backend = backend;
    return 0;
}
extern "C" int nn_get_gemm_backend(void) { return g_backend; }

// The chained kernel keeps the activation-derivative tensor silu'(q) in the tile-transposed layout (NN_TILED_INDEX), and
// the reverse MLP (chained or two launches) reads it there.  Writer and reader take the decision from the same predicate:
// the chained kernel ran in the forward MLP <=> pair-level call (device row count) or a small node-level call.
static bool chain_runs_fwd(const int* m_dev, int m) { return g_backend == 2 && chain_enabled() && (m_dev || m <= kChainSmallM); }
extern "C" int nn_mlp_mid_tiled(int32_t m, int32_t has_m_dev) {
    static const int one = 1;
    return chain_runs_fwd(has_m_dev ? &one : nullptr, m) ? 1 : 0;
}


int nn_gemm128_launch(const nn_gemm_args& a, cudaStream_t s) {
    if (g_backend == 2) return nn_gemm128_ts_launch(a, s);
    return g_backend == 1 ? nn_gemm128_tc_launch(a, s) : nn_gemm128_simt_launch(a, s);
}
extern "C" int nn_gemm128(const nn_gemm_args* a, void* stream) {
    NN_REQUIRE(a && a->X && a->B && a->Y, "null pointer");
    return nn_gemm128_launch(*a, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------- workspace layout
namespace {

struct LayerBuf {
    float *pre, *mn, *f_out, *g;          // node level: [N,F], [N,F], [N,3,F], [N,3,F]
    float *msg, *q1, *e1, *q2, *e2;       // pair level: [P,F] each (q2/e2 unused in layer 0)
    float *ln_xhat, *ln_rstd;             // layer norm: normalised rows [N,F] and 1/sigma [N]
};

struct EvalWs {
    LayerBuf layer[NN_MAX_LAYERS];
    float *a0, *a1;                       // [N,F] ping-pong invariant features
    float *rbf, *drbf, *unit, *dist;      // [P,nb], [P,nb] (d rbf / dx), [P,3], [P]
    float *h1pre, *h2pre, *e_atom;        // head
    float *d1, *d2;                       // direct_force head temporaries [N,F]
    // reverse sweep
    float *abar, *mnbar, *tmpN;           // [N,F]
    float *fbar, *dfb;                    // [N,3,F]
    float *e2bar, *mbar;                  // [P,F]
    float *x_bar, *ubar, *G;              // [2L][P] (dE/dx partial slots), [P,3], [P,3]
    float *vir_atom;                      // [N,9]
    double *sum_part; int slices;         // [B, slices, 9] partial per-system sums (two-level energy / virial sums)
    size_t total;
};

EvalWs carve_eval(void* base, size_t cap, int N, int B, int P, int L, bool bwd) {
    WsCarver c(base, cap);
    EvalWs w{};
    const size_t NF = (size_t)N * kF, PF = (size_t)P * kF;
    // activation-derivative buffers may be held tile-transposed (NN_TILED_INDEX): whole tiles of 128 rows
    const size_t NFt = (size_t)((N + 127) / 128 * 128) * kF, PFt = (size_t)((P + 127) / 128 * 128) * kF;
    for (int l = 0; l < L; ++l) {
        LayerBuf& b = w.layer[l];
        b.pre = c.take<float>(NFt); b.mn = c.take<float>(NF);
        b.f_out = c.take<float>(3 * NF); b.g = c.take<float>(3 * NF);
        b.msg = c.take<float>(PF); b.q1 = c.take<float>(PFt); b.e1 = c.take<float>(PF);
        if (l > 0) { b.q2 = c.take<float>(PFt); b.e2 = c.take<float>(PF); }
        b.ln_xhat = c.take<float>(NF); b.ln_rstd = c.take<float>(N);
    }
    w.a0 = c.take<float>(NF); w.a1 = c.take<float>(NF);
    w.rbf = c.take<float>((size_t)P * kNB); w.unit = c.take<float>((size_t)P * 3); w.dist = c.take<float>(P);
    w.drbf = bwd ? c.take<float>((size_t)P * kNB) : nullptr;
    w.h1pre = c.take<float>(NFt); w.h2pre = c.take<float>(NF); w.e_atom = c.take<float>(N);
    w.d1 = c.take<float>(NF); w.d2 = c.take<float>(NF);
    w.slices = nn_sum_slices(N, B);
    w.sum_part = c.take<double>((size_t)(B > 0 ? B : 1) * w.slices * 9);
    if (bwd) {
        w.abar = c.take<float>(NF); w.mnbar = c.take<float>(NF); w.tmpN = c.take<float>(NF);
        w.fbar = c.take<float>(3 * NF); w.dfb = c.take<float>(3 * NF);
        w.e2bar = c.take<float>(PF); w.mbar = c.take<float>(PF);
        w.x_bar = c.take<float>((size_t)2 * L * P); w.ubar = c.take<float>((size_t)P * 3); w.G = c.take<float>((size_t)P * 3);
        w.vir_atom = c.take<float>((size_t)N * 9);
    }
    w.total = c.off;
    return w;
}

struct Gemm {
    cudaStream_t s; int rc = 0;
    bool aux_tiled_next = false;          // the next EPI_MUL launch reads its factor in the tile-transposed layout
    // fwd(M): x @ M^T -> B = M.wt ; bwd(M): g @ M -> B = M.w
    void fwd(const float* X, const nn_mat& M, float* Y, int m, int pro, int epi, const float* bias = nullptr,
             const float* aux1 = nullptr, const float* aux2 = nullptr, const float* aux3 = nullptr,
             const int* m_dev = nullptr) { run(X, M.wt, M.wt_img, Y, m, pro, epi, bias, aux1, aux2, aux3, m_dev); }
    void bwd(const float* X, const nn_mat& M, float* Y, int m, int pro, int epi, const float* bias = nullptr,
             const float* aux1 = nullptr, const float* aux2 = nullptr, const float* aux3 = nullptr,
             const int* m_dev = nullptr) { run(X, M.w, M.w_img, Y, m, pro, epi, bias, aux1, aux2, aux3, m_dev); }
    // Y = (silu(X @ M1^T + b1)) @ M2^T + b2, silu'(.) left in `mid` (forward MLP); one chained launch when available
    void mlp_fwd(const float* X, const nn_mat& M1, const float* b1, float* mid, const nn_mat& M2, const float* b2, float* Y,
                 int m, int pro_act, const int* m_dev = nullptr) {
        if (rc) return;
        if (chain_runs_fwd(m_dev, m)) {     // gemm_chain.cu
            if (!(M1.wt_img && M2.wt_img)) { nn_set_error("mlp_fwd: the chained kernel needs the operand images of both matrices"); rc = -1; return; }
            ProfScope ps(m_dev ? NN_STAGE_PAIR_GEMM : NN_STAGE_NODE_GEMM, s);
            nn_gemm_chain_args a{};
            a.X = X; a.B1_img = M1.wt_img; a.B2_img = M2.wt_img; a.bias1 = b1; a.bias2 = b2; a.aux_out = mid; a.Y = Y;
            a.m_dev = m_dev; a.m_dev_mul = 1; a.m = m; a.mid = NN_MID_SILU_SAVE; a.out = NN_OUT_BIAS;
            rc = nn_gemm128_chain(&a, s);
            return;
        }
        fwd(X, M1, mid, m, NN_PRO_NONE, NN_EPI_BIAS, b1, nullptr, nullptr, nullptr, m_dev);
        fwd(mid, M2, Y, m, pro_act, NN_EPI_BIAS, b2, nullptr, nullptr, nullptr, m_dev);
    }
    // two forward MLPs over the same input in one dual launch (equiv_message1 / equiv_message2: X is read from HBM once)
    bool mlp_fwd_dual(const float* X, const nn_mat& A1, float* midA, const nn_mat& A2, float* YA, const nn_mat& B1, float* midB,
                      const nn_mat& B2, float* YB, int m, const int* m_dev) {
        if (rc) return true;
        if (!(g_backend == 2 && chain_enabled() && m_dev && A1.wt_img && A2.wt_img && B1.wt_img && B2.wt_img)) return false;
        ProfScope ps(NN_STAGE_PAIR_GEMM, s);
        nn_gemm_chain_args a{};
        a.X = X; a.B1_img = A1.wt_img; a.B2_img = A2.wt_img; a.aux_out = midA; a.Y = YA;
        a.B1_img_b = B1.wt_img; a.B2_img_b = B2.wt_img; a.aux_out_b = midB; a.Y_b = YB;
        a.m_dev = m_dev; a.m_dev_mul = 1; a.m = m; a.mid = NN_MID_SILU_SAVE; a.out = NN_OUT_BIAS;
        rc = nn_gemm128_chain(&a, s);
        return true;
    }
    // Y (+)= ((G @ M2) * dact) @ M1 (reverse MLP); `tmp` receives the intermediate on the two-launch path only
    void mlp_bwd(const float* G, const nn_mat& M2, const float* dact, float* tmp, const nn_mat& M1, float* Y, int m,
                 bool accumulate, const int* m_dev = nullptr) {
        if (rc) return;
        if (g_backend == 2 && chain_enabled() && ((m_dev && accumulate) || (!m_dev && m <= kChainSmallM)) && M1.w_img && M2.w_img) {
            ProfScope ps(m_dev ? NN_STAGE_PAIR_GEMM : NN_STAGE_NODE_GEMM, s);
            nn_gemm_chain_args a{};
            a.X = G; a.B1_img = M2.w_img; a.B2_img = M1.w_img; a.aux1 = dact; a.aux2 = accumulate ? Y : nullptr; a.Y = Y;
            a.m_dev = m_dev; a.m_dev_mul = 1; a.m = m; a.mid = NN_MID_MUL; a.out = accumulate ? NN_OUT_ADD : NN_OUT_BIAS;
            rc = nn_gemm128_chain(&a, s);
            return;
        }
        aux_tiled_next = chain_runs_fwd(m_dev, m);     // the forward MLP ran chained and left silu' tile-transposed
        bwd(G, M2, tmp, m, NN_PRO_NONE, NN_EPI_MUL, nullptr, dact, nullptr, nullptr, m_dev);
        aux_tiled_next = false;
        bwd(tmp, M1, Y, m, NN_PRO_NONE, accumulate ? NN_EPI_ADD : NN_EPI_BIAS, nullptr, accumulate ? Y : nullptr, nullptr, nullptr, m_dev);
    }
    void run(const float* X, const float* B, const float* B_img, float* Y, int m, int pro, int epi,
             const float* bias = nullptr, const float* aux1 = nullptr, const float* aux2 = nullptr,
             const float* aux3 = nullptr, const int* m_dev = nullptr, int mul = 1) {
        if (rc) return;
        ProfScope ps(m_dev ? NN_STAGE_PAIR_GEMM : NN_STAGE_NODE_GEMM, s);
        nn_gemm_args a{};
        // SILU_SAVE overwrites the pre-activation X with silu'(X) in place (X is not needed afterwards)
        if (pro == NN_PRO_SILU_SAVE) a.aux_out = const_cast<float*>(X);
        a.X = X; a.B = B; a.B_img = B_img; a.Y = Y; a.bias = bias; a.aux1 = aux1; a.aux2 = aux2; a.aux3 = aux3;
        a.m_dev = m_dev; a.m_dev_mul = mul; a.m = m; a.prologue = pro; a.epilogue = epi;
        a.aux_tiled = (epi == NN_EPI_MUL && aux_tiled_next) ? 1 : 0;
        rc = nn_gemm128_launch(a, s);
    }
};

}  // namespace

extern "C" size_t nn_eval_workspace_bytes(int32_t n_atoms, int32_t n_systems, int32_t cap_pairs, int32_t n_layers,
                                          int32_t want_forces) {
    if (n_layers < 1 || n_layers > NN_MAX_LAYERS) return 0;
    return carve_eval(nullptr, 0, n_atoms, n_systems, cap_pairs, n_layers, want_forces != 0).total;
}

#define NN_TRY(expr) do { int rc__ = (expr); if (rc__) return rc__; } while (0)

int nn_node_aggregate_fwd_rows(const nn_nbr* nl, int n_rows, const float* msg, const float* e1, const float* e2,
                               const float* unit, const float* a_in, const float* f_in, float* a_out, float* f_out,
                               bool first, cudaStream_t s);
int nn_energy_head_fwd_rows(const float* h2pre, const float* w3, const float* b3, const float* scale, const float* shift,
                            const int64_t* z, const int32_t* sys_ptr, int n_rows, int n_systems, float* e_atom,
                            float* energy, double* partial, int slices, cudaStream_t s);
int nn_force_virial_rows(const nn_nbr* nl, int n_rows, const float* disp_bar, float* forces, float* virial, float* stress,
                         void* workspace, double* partial, int slices, cudaStream_t s);
int nn_sum_slices(int n_atoms, int n_systems);

namespace {

struct EvalCtx {
    const nn_eval_args* a; const nn_nbr* nl; const nn_weights* W;
    int N, No, B, P, L; bool bwd; cudaStream_t s; EvalWs w; const int* np_dev; int PRO_ACT;
};

int make_ctx(const nn_eval_args* a, void* stream, EvalCtx& c) {
    NN_REQUIRE(a && a->nbr && a->w && a->z && a->energy, "null pointer");
    c.a = a; c.nl = a->nbr; c.W = a->w;
    c.N = c.nl->n_atoms; c.B = c.nl->n_systems; c.P = c.nl->cap_pairs; c.L = c.W->n_layers;
    c.No = a->n_owned > 0 ? a->n_owned : c.N;
    NN_REQUIRE(c.No <= c.N, "n_owned > n_atoms");
    NN_REQUIRE(c.L >= 1 && c.L <= NN_MAX_LAYERS, "n_layers out of range");
    c.bwd = a->want_forces != 0 || a->want_virial != 0;
    NN_REQUIRE(!c.bwd || a->forces, "forces buffer required");
    NN_REQUIRE(!a->want_virial || a->virial, "virial buffer required");
    NN_REQUIRE(a->workspace_bytes >= nn_eval_workspace_bytes(c.N, c.B, c.P, c.L, c.bwd), "workspace too small");
    c.s = (cudaStream_t)stream;
    c.w = carve_eval(a->workspace, a->workspace_bytes, c.N, c.B, c.P, c.L, c.bwd);
    c.np_dev = c.nl->status + NN_ST_N_PAIRS;
    // with a reverse sweep the activation GEMMs leave silu'(pre) behind in place of pre
    c.PRO_ACT = c.bwd ? NN_PRO_SILU_SAVE : NN_PRO_SILU;
    return 0;
}

// One phase of the evaluation.  Node-level work (GEMMs, aggregations, head) runs on the first `No` (owned)
// atoms, pair-level work on every local pair; between phases a domain-decomposed caller refreshes the
// ghost rows [No, N) of the buffer named in the comment (single-GPU: No == N, nothing to exchange).
int run_phase(EvalCtx& c, int phase, int l);
int run_phase(EvalCtx& c, int phase, int l) {
    const nn_weights& W = *c.W; EvalWs& w = c.w; const nn_nbr* nl = c.nl; cudaStream_t s = c.s;
    const int N = c.N, No = c.No, P = c.P, L = c.L; const int* np_dev = c.np_dev;
    Gemm g{s};
    float* a_cur = w.a0; float* a_nxt = w.a1;
    switch (phase) {
    case NN_PH_BEGIN: {      // edge features (R3-R6) and embedding (R1)
        { ProfScope ps(NN_STAGE_GEOM, s); NN_TRY(nn_edge_geom_fwd(nl->pair_disp, W.frequencies, W.cutoff, np_dev, P, w.rbf, w.drbf, w.unit, w.dist, s)); }
        { ProfScope ps(NN_STAGE_OTHER, s); NN_TRY(nn_embed_launch(c.a->z, W.embedding, a_cur, No, nl->status, s)); }
        return 0;
    }
    case NN_PH_FWD_NODE: {   // -> mn(l) of owned atoms            [then ghosts of: mn(l), f_out(l-1)]
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        g.mlp_fwd(a_cur, lw.W1, lw.b1, b.pre, lw.W2, lw.b2, b.mn, No, c.PRO_ACT);
        return g.rc;
    }
    case NN_PH_FWD_PAIR: {   // message, edge MLPs, aggregation, equivariant update (R7)
        NN_TRY(run_phase(c, NN_PH_FWD_PAIR_A, l));
        return run_phase(c, NN_PH_FWD_PAIR_B, l);
    }
    case NN_PH_FWD_PAIR_A: {
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        const bool first = l == 0;
        const float* f_in = first ? nullptr : w.layer[l - 1].f_out;
        {
            ProfScope ps(NN_STAGE_MESSAGE, s);
            NN_TRY(nn_edge_message_fwd(nl, w.rbf, b.mn, lw.Wet, lw.We_img, b.msg, s));
        }
        // layer 0: force_node == 0, so equiv_message2 contributes exactly nothing; other layers: both MLPs in one dual launch
        if (first || !g.mlp_fwd_dual(b.msg, lw.U1, b.q1, lw.U2, b.e1, lw.V1, b.q2, lw.V2, b.e2, P, np_dev)) {
            g.mlp_fwd(b.msg, lw.U1, nullptr, b.q1, lw.U2, nullptr, b.e1, P, c.PRO_ACT, np_dev);
            if (!first) g.mlp_fwd(b.msg, lw.V1, nullptr, b.q2, lw.V2, nullptr, b.e2, P, c.PRO_ACT, np_dev);
        }
        NN_TRY(g.rc);
        { ProfScope ps(NN_STAGE_AGGREGATE, s); NN_TRY(nn_node_aggregate_fwd_rows(nl, No, b.msg, b.e1, b.e2, w.unit, a_cur, f_in, a_nxt, b.f_out, first, s)); }
        return 0;
    }
    case NN_PH_FWD_PAIR_B: {
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        g.fwd(b.f_out, lw.Wu, b.g, 3 * No, NN_PRO_NONE, NN_EPI_BIAS);
        NN_TRY(g.rc);
        { ProfScope ps(NN_STAGE_OTHER, s); NN_TRY(nn_equiv_update_fwd(a_nxt, b.f_out, b.g, a_cur, No, s)); }
        if (lw.ln_gamma) {   // layer_norm=True (models/newtonnet.py:234-235)
            ProfScope ps(NN_STAGE_OTHER, s);
            NN_TRY(nn_layer_norm_fwd_launch(a_cur, lw.ln_gamma, lw.ln_beta, b.ln_xhat, b.ln_rstd, No, s));
        }
        return 0;
    }
    case NN_PH_HEAD: {       // energy head (R8, R9): partial energies over owned atoms
        g.mlp_fwd(a_cur, W.H1, W.hb1, w.h1pre, W.H2, W.hb2, w.h2pre, No, c.PRO_ACT);
        NN_TRY(g.rc);
        { ProfScope ps(NN_STAGE_HEAD, s); NN_TRY(nn_energy_head_fwd_rows(w.h2pre, W.w3, W.hb3, W.scale, W.shift, c.a->z, nl->sys_ptr, No, c.B, w.e_atom, c.a->energy, w.sum_part, w.slices, s)); }
        if (c.a->direct_force) {   // direct_force head (models/output.py:115-132): no reverse sweep involved
            NN_REQUIRE(W.dscale != nullptr, "direct_force requested but the weights carry no direct_force head");
            g.fwd(a_cur, W.D1, w.d1, No, NN_PRO_NONE, NN_EPI_BIAS, W.db1);
            g.fwd(w.d1, W.D2, w.d2, No, NN_PRO_SILU, NN_EPI_BIAS, W.db2);
            g.fwd(w.d2, W.D3, w.d1, No, NN_PRO_SILU, NN_EPI_BIAS, W.db3);
            NN_TRY(g.rc);
            ProfScope ps(NN_STAGE_HEAD, s);
            NN_TRY(nn_direct_force_launch(w.d1, w.layer[L - 1].f_out, W.dscale, c.a->z, No, c.a->direct_force, s));
        }
        if (c.a->atom_node) cudaMemcpyAsync(c.a->atom_node, a_cur, (size_t)No * kF * sizeof(float), cudaMemcpyDeviceToDevice, s);
        if (c.a->force_node) cudaMemcpyAsync(c.a->force_node, w.layer[L - 1].f_out, (size_t)No * 3 * kF * sizeof(float),
                                             cudaMemcpyDeviceToDevice, s);
        return 0;
    }
    case NN_PH_BWD_SEED: {   // reverse sweep (R10 / row B): dE/da of owned atoms
        { ProfScope ps(NN_STAGE_HEAD, s); NN_TRY(nn_energy_head_seed_launch(w.h2pre, W.w3, W.scale, c.a->z, No, w.tmpN, s)); }
        g.mlp_bwd(w.tmpN, W.H2, w.h1pre, w.mnbar, W.H1, w.abar, No, false);
        NN_TRY(g.rc);
        cudaMemsetAsync(w.fbar, 0, (size_t)N * 3 * kF * sizeof(float), s);
        cudaMemsetAsync(w.x_bar, 0, (size_t)2 * L * P * sizeof(float), s);
        cudaMemsetAsync(w.ubar, 0, (size_t)P * 3 * sizeof(float), s);
        return 0;
    }
    case NN_PH_BWD_NODE: {   // dfb = fbar + abar*g + (abar*f_out) @ Wu  (owned)   [then ghosts of: dfb, abar]
        NN_TRY(run_phase(c, NN_PH_BWD_NORM, l));
        return run_phase(c, NN_PH_BWD_NODE_B, l);
    }
    case NN_PH_BWD_NORM: {
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        if (lw.ln_gamma) NN_TRY(nn_layer_norm_bwd_launch(w.abar, lw.ln_gamma, b.ln_xhat, b.ln_rstd, No, s));
        return 0;
    }
    case NN_PH_BWD_NODE_B: {
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        g.bwd(b.f_out, lw.Wu, w.dfb, 3 * No, NN_PRO_ROWSCALE3, NN_EPI_EQUIV_BWD, nullptr, w.fbar, w.abar, b.g);
        return g.rc;
    }
    case NN_PH_BWD_PAIR: {
        NN_TRY(run_phase(c, NN_PH_BWD_PAIR_A, l));
        return run_phase(c, NN_PH_BWD_PAIR_B, l);
    }
    case NN_PH_BWD_PAIR_A: {
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        const bool first = l == 0;
        const float* f_in = first ? nullptr : w.layer[l - 1].f_out;
        { ProfScope ps(NN_STAGE_BWD_GATHER, s); NN_TRY(nn_pair_bwd_gather_launch(nl, w.dfb, f_in, w.unit, b.e1, w.e2bar, w.ubar, first, s)); }
        // mbar = ((e1bar @ U2) * silu'(q1)) @ U1 + ((e2bar @ V2) * silu'(q2)) @ V1
        g.mlp_bwd(b.e1, lw.U2, b.q1, b.e1, lw.U1, w.mbar, P, false, np_dev);
        if (!first) {
            g.mlp_bwd(w.e2bar, lw.V2, b.q2, w.e2bar, lw.V1, w.mbar, P, true, np_dev);
        }
        return g.rc;
    }
    case NN_PH_BWD_PAIR_B: {
        const nn_layer_weights& lw = W.layer[l]; LayerBuf& b = w.layer[l];
        const bool first = l == 0;
        {
            ProfScope ps(NN_STAGE_BWD_MESSAGE, s);
            float* slot = w.x_bar + (size_t)2 * l * P;      // two partial arrays per layer, summed in k_edge_geom_bwd
            if (g_backend >= 1 && lw.We_img) NN_TRY(nn_message_bwd_tc(nl, w.abar, b.mn, w.rbf, w.drbf, lw.We_img, w.mbar, slot, s));
            else NN_TRY(nn_pair_bwd_message_launch(nl, w.abar, b.mn, w.rbf, w.drbf, lw.Wet, w.mbar, slot, s));
        }
        { ProfScope ps(NN_STAGE_BWD_AGGREGATE, s); NN_TRY(nn_node_aggregate_bwd_launch(nl, No, w.mbar, b.mn, b.e2, w.dfb, w.mnbar, w.fbar, first, s)); }
        // abar += ((mnbar @ W2) * silu'(pre)) @ W1
        g.mlp_bwd(w.mnbar, lw.W2, b.pre, w.tmpN, lw.W1, w.abar, No, true);
        return g.rc;
    }
    case NN_PH_FINISH: {     // dE/d disp per pair, forces of owned atoms, partial virial
        { ProfScope ps(NN_STAGE_GEOM, s); NN_TRY(nn_edge_geom_bwd(w.x_bar, 2 * L, w.ubar, w.unit, w.dist, W.cutoff, np_dev, P, w.G, s)); }
        ProfScope ps(NN_STAGE_FORCE, s);
        NN_TRY(nn_force_virial_rows(nl, No, w.G, c.a->forces, c.a->want_virial ? c.a->virial : nullptr,
                                    c.a->want_virial ? c.a->stress : nullptr, w.vir_atom, w.sum_part, w.slices, s));
        return 0;
    }
    }
    nn_set_error("nn_eval_phase: unknown phase %d", phase);
    return -1;
}

}  // namespace

// ---------------------------------------------------------------- reverse-sweep operators as standalone entry points
// (SURVEY.md section 8b lists forward / backward pairs; nn_eval composes exactly these launchers)
extern "C" NN_API int nn_mlp_fwd(const float* X, const nn_mat* M1, const float* b1, float* mid, const nn_mat* M2, const float* b2,
                                 float* Y, int32_t m, const int32_t* m_dev, int32_t save_dact, void* stream) {
    NN_REQUIRE(X && M1 && M2 && mid && Y, "null pointer");
    Gemm g{(cudaStream_t)stream};
    g.mlp_fwd(X, *M1, b1, mid, *M2, b2, Y, m, save_dact ? NN_PRO_SILU_SAVE : NN_PRO_SILU, m_dev);
    if (g.rc) return g.rc;
    NN_CHECK_LAUNCH("nn_mlp_fwd");
    return 0;
}

extern "C" NN_API int nn_mlp_bwd(const float* G, const nn_mat* M2, const float* dact, float* tmp, const nn_mat* M1, float* Y,
                                 int32_t m, const int32_t* m_dev, int32_t accumulate, void* stream) {
    NN_REQUIRE(G && M1 && M2 && dact && tmp && Y, "null pointer");
    Gemm g{(cudaStream_t)stream};
    g.mlp_bwd(G, *M2, dact, tmp, *M1, Y, m, accumulate != 0, m_dev);
    if (g.rc) return g.rc;
    NN_CHECK_LAUNCH("nn_mlp_bwd");
    return 0;
}

extern "C" NN_API int nn_energy_head_bwd(const float* h2pre, const float* w3, const float* scale, const int64_t* z, int32_t n_atoms,
                                         float* gh2, void* stream) {
    NN_REQUIRE(h2pre && w3 && scale && z && gh2, "null pointer");
    return nn_energy_head_seed_launch(h2pre, w3, scale, z, n_atoms, gh2, (cudaStream_t)stream);
}

extern "C" NN_API int nn_pair_gather_bwd(const nn_nbr* nl, const float* dfb, const float* f_in, const float* unit, float* e1_io,
                                         float* e2bar, float* ubar, void* stream) {
    NN_REQUIRE(nl && dfb && unit && e1_io && ubar && (f_in == nullptr || e2bar != nullptr), "null pointer");
    return nn_pair_bwd_gather_launch(nl, dfb, f_in, unit, e1_io, e2bar, ubar, f_in == nullptr, (cudaStream_t)stream);
}

extern "C" NN_API int nn_edge_message_fwd(const nn_nbr* nl, const float* rbf, const float* mn, const float* Wet, const float* We_img,
                                          float* msg, void* stream) {
    NN_REQUIRE(nl && rbf && mn && msg && (Wet || We_img), "null pointer");
    if (g_backend >= 1 && We_img) return nn_message_fwd_tc(nl, rbf, mn, We_img, msg, (cudaStream_t)stream);
    NN_REQUIRE(Wet != nullptr, "the SIMT backend needs Wet");
    return nn_edge_message_fwd_launch(nl, rbf, mn, Wet, msg, (cudaStream_t)stream);
}

extern "C" NN_API int nn_edge_message_bwd(const nn_nbr* nl, const float* abar, const float* mn, const float* rbf, const float* drbf,
                                          const float* Wet, const float* We_img, float* mbar_io, float* x_part, void* stream) {
    NN_REQUIRE(nl && abar && mn && rbf && drbf && mbar_io && x_part && (Wet || We_img), "null pointer");
    if (g_backend >= 1 && We_img) return nn_message_bwd_tc(nl, abar, mn, rbf, drbf, We_img, mbar_io, x_part, (cudaStream_t)stream);
    NN_REQUIRE(Wet != nullptr, "the SIMT backend needs Wet");
    return nn_pair_bwd_message_launch(nl, abar, mn, rbf, drbf, Wet, mbar_io, x_part, (cudaStream_t)stream);
}

extern "C" NN_API int nn_node_aggregate_bwd(const nn_nbr* nl, const float* t, const float* mn, const float* e2, const float* dfb,
                                            float* mnbar, float* fbar_new, void* stream) {
    NN_REQUIRE(nl && t && mn && mnbar && (e2 == nullptr || (dfb && fbar_new)), "null pointer");
    const int rows = nl->n_owned > 0 ? nl->n_owned : nl->n_atoms;
    return nn_node_aggregate_bwd_launch(nl, rows, t, mn, e2, dfb, mnbar, fbar_new, e2 == nullptr, (cudaStream_t)stream);
}

extern "C" int nn_eval_phase(const nn_eval_args* a, int32_t phase, int32_t layer, void* stream) {
    EvalCtx c;
    NN_TRY(make_ctx(a, stream, c));
    NN_REQUIRE(layer >= 0 && layer < c.L, "layer out of range");
    NN_REQUIRE(c.bwd || phase < NN_PH_BWD_SEED || phase == NN_PH_FWD_PAIR_A || phase == NN_PH_FWD_PAIR_B, "reverse-sweep phase without want_forces");
    NN_TRY(run_phase(c, phase, layer));
    NN_CHECK_LAUNCH("nn_eval_phase");
    return 0;
}

extern "C" float* nn_eval_buffer(const nn_eval_args* a, int32_t which, int32_t layer) {
    EvalCtx c;
    if (make_ctx(a, nullptr, c) || layer < 0 || layer >= c.L) return nullptr;
    switch (which) {
    case NN_BUF_MN: return c.w.layer[layer].mn;
    case NN_BUF_F_OUT: return c.w.layer[layer].f_out;
    case NN_BUF_DFB: return c.w.dfb;
    case NN_BUF_ABAR: return c.w.abar;
    }
    return nullptr;
}

extern "C" int nn_eval(const nn_eval_args* a, void* stream) {
    EvalCtx c;
    NN_TRY(make_ctx(a, stream, c));
    NN_TRY(run_phase(c, NN_PH_BEGIN, 0));
    for (int l = 0; l < c.L; ++l) {
        NN_TRY(run_phase(c, NN_PH_FWD_NODE, l));
        NN_TRY(run_phase(c, NN_PH_FWD_PAIR, l));
    }
    NN_TRY(run_phase(c, NN_PH_HEAD, 0));
    if (c.bwd) {
        NN_TRY(run_phase(c, NN_PH_BWD_SEED, 0));
        for (int l = c.L - 1; l >= 0; --l) {
            NN_TRY(run_phase(c, NN_PH_BWD_NODE, l));
            NN_TRY(run_phase(c, NN_PH_BWD_PAIR, l));
        }
        NN_TRY(run_phase(c, NN_PH_FINISH, 0));
    }
    NN_CHECK_LAUNCH("nn_eval");
    return 0;
}
