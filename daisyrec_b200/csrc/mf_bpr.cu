// mf_bpr.cu -- the BPR-MF training step as ONE persistent cooperative sm_100a kernel.
//
// Stands behind GeneralRecommender.fit's step loop (daisy/model/AbstractRecommender.py:112-128)
// with MF.calc_loss (daisy/model/MFRecommender.py:70-97), BPRLoss (daisy/utils/loss.py:11),
// autograd's embedding backward (:125) and optim.SGD/Adam.step (:126, :53-56).
//
// Synchronous-step semantics (every gradient of a step is taken at the PRE-step weights, the
// Frobenius norms couple the whole batch) are kept exactly, without ever materialising the
// reference's table-sized dense gradient:
//
//   phase 1 (read-only on P,Q)   per triple (u,i,j): index tile staged by TMA (cp.async.bulk) into
//       shared memory; a group of W lanes gathers the three factor rows with 128-bit L2 loads,
//       reduces the two dot products with xor-shuffles (canonical order), evaluates
//       s = sigmoid(x), loss = -log(1e-10+s), c = -s(1-s)/(1e-10+s) and issues vector
//       RED.ADD.F32x4 reductions of the BPR part of the gradient into the L2-resident
//       accumulators gP/gQ:  gP[u] += c(q_i-q_j), gQ[i] += c p_u, gQ[j] -= c p_u; it also counts how
//       often each row occurs (cntU, cntI = pos | neg<<32) and accumulates the six batch norms.
//   -- grid barrier --           (norms and loss are now final; nobody reads P,Q any more)
//   phase 2                      every touched row is applied exactly once:
//       g = gP[r] + cnt * (reg_1 sgn(theta) + reg_2 theta / ||.||_F);  theta -= lr g  (or Adam);
//       the accumulator row and its counter are reset for the next step.  Rows are found either
//       by a dense sweep (large batches: every row is touched) or by claiming the counter with
//       atomicExch from the triple that touched it (small batches).
//   -- grid barrier --           next step.
//
// A NaN loss (ValueError in the reference, :122-123) stops the loop before the update of that step.
//
// Variants of the same kernel: GEN = false is the BPR-only hot instantiation, GEN = true selects HingeLoss / TOP1Loss
// (daisy/utils/loss.py:16-33) or the point-wise CL / SL branch (MFRecommender.py:75-81: the third plane holds the label,
// only P_u and Q_i take part) at run time; `phases` splits it into phase-1 / phase-2 launches (multi-GPU exchange,
// LightGCN, NeuMF); `neg_row_ptr` switches on the fused sampler (a fresh negative per triple drawn inside phase 1).
#include <math.h>
#include <stdlib.h>

#include <map>
#include <mutex>
#include <vector>

#include "step_kernel.cuh"

namespace drb {

// b?[k] = triples[perm[k], ?]
__global__ void gather_triples_kernel(const int32_t *__restrict__ triples, const int64_t *__restrict__ perm, long long n,
                                      int32_t *__restrict__ bu, int32_t *__restrict__ bi, int32_t *__restrict__ bj)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        long long src = perm ? perm[k] : k;
        const int32_t *t = triples + 3 * src;
        bu[k] = __ldg(t);
        bi[k] = __ldg(t + 1);
        bj[k] = __ldg(t + 2);
    }
}

// ------------------------------------------------------------------ host dispatch
typedef void (*StepKernel)(StepParams);

template <int VEC, bool GEN>
static StepKernel pick_kernel_v(int W, int NCH)
{
#define DRB_CASE(w, n) \
    if (W == w && NCH == n) return mf_bpr_steps_kernel<VEC, w, n, GEN>;
    DRB_CASE(1, 1) DRB_CASE(2, 1) DRB_CASE(4, 1) DRB_CASE(8, 1) DRB_CASE(16, 1) DRB_CASE(32, 1)
    DRB_CASE(32, 2) DRB_CASE(32, 4) DRB_CASE(32, 8)
#undef DRB_CASE
    return nullptr;
}

// The lean MF instantiation.  Its lane geometry is its own: the index loads, address arithmetic, loss chain and counter updates
// of a triple are replayed by every lane of the row's group, the row arithmetic is not -- so fewer lanes per row (more chunks of
// 4 floats per lane) means fewer issue slots per triple and more rows in flight per warp.  Candidates for a factor count are
// every (W lanes, NCH in {4, 2, 1} chunks per lane) with W a power of two; the preferred one keeps 8 lanes per row, so that one
// 128-bit access of a group still covers exactly one 128-byte line (F = 64: 8 lanes x 2 chunks, F = 128: 8 x 4).  Which
// candidate runs is decided on the device (lean_autotune).  Only the fp32 summation order of the two dot products differs from
// the canonical geometry (row_geom) that rank / predict / the oracle share.
static int lean_nch_only()
{
    static const int v = [] {
        const char *e = getenv("DRB_LEAN_NCH");   // developer switch: restrict the candidates to 1 | 2 | 4 chunks per lane
        int n = e ? atoi(e) : 0;
        return (n == 1 || n == 2 || n == 4) ? n : 0;
    }();
    return v;
}
// candidates in order of preference; returns their number (at most 3)
static int lean_candidates(int F, int (&cw)[3], int (&cn)[3])
{
    int count = 0;
    if (F <= 0 || F % 4 != 0) return 0;
    const int chunks = F / 4;
    auto valid = [&](int n) {
        if (chunks % n != 0) return false;
        const int w = chunks / n;
        return w <= 32 && (w & (w - 1)) == 0;
    };
    auto push = [&](int n) {
        for (int k = 0; k < count; ++k) if (cn[k] == n) return;
        if (lean_nch_only() != 0 && n != lean_nch_only()) return;
        cw[count] = chunks / n;
        cn[count] = n;
        ++count;
    };
    for (int n = 4; n >= 1; n >>= 1)                       // preferred: the most chunks per lane that keep whole lines (W >= 8)
        if (valid(n) && (chunks / n >= 8 || n == 1)) { push(n); break; }
    for (int n = 4; n >= 1; n >>= 1)
        if (valid(n)) push(n);
    if (count == 0 && lean_nch_only() == 0) {              // e.g. F = 100: 25 chunks on 32 lanes
        RowGeom g = row_geom(F);
        if (g.vec == 4 && g.nch == 1) { cw[0] = g.width; cn[0] = 1; count = 1; }
    }
    return count;
}
void lean_default_geom(int F, int &W, int &NCH)            // host-only: the preferred candidate
{
    int cw[3], cn[3];
    W = NCH = 0;
    if (lean_candidates(F, cw, cn) > 0) { W = cw[0]; NCH = cn[0]; }
}
static StepKernel pick_lean_wn(int W, int NCH)
{
#define DRB_LEAN(w, n) \
    if (W == w && NCH == n) return mf_bpr_steps_lean_kernel<4, w, n>;
    DRB_LEAN(1, 1) DRB_LEAN(2, 1) DRB_LEAN(4, 1) DRB_LEAN(8, 1) DRB_LEAN(16, 1) DRB_LEAN(32, 1)
    DRB_LEAN(1, 2) DRB_LEAN(2, 2) DRB_LEAN(4, 2) DRB_LEAN(8, 2) DRB_LEAN(16, 2) DRB_LEAN(32, 2)
    DRB_LEAN(1, 4) DRB_LEAN(2, 4) DRB_LEAN(4, 4) DRB_LEAN(8, 4) DRB_LEAN(16, 4) DRB_LEAN(32, 4)
#undef DRB_LEAN
    return nullptr;
}

// GEN = false: BPR only (the hot instantiation, no loss-kind branches); GEN = true: HL / TL selected at run time
static StepKernel pick_kernel(int F, bool gen)
{
    if (F <= 0) return nullptr;
    RowGeom g = row_geom(F);
    if (gen) {
        if (g.vec == 4) return pick_kernel_v<4, true>(g.width, g.nch);
        if (g.vec == 2) return pick_kernel_v<2, true>(g.width, g.nch);
        return pick_kernel_v<1, true>(g.width, g.nch);
    }
    if (g.vec == 4) return pick_kernel_v<4, false>(g.width, g.nch);
    if (g.vec == 2) return pick_kernel_v<2, false>(g.width, g.nch);
    return pick_kernel_v<1, false>(g.width, g.nch);
}

// grid / tile choice and the cooperative launch of one chosen instantiation
static int launch_kernel(StepKernel k, StepParams &p, cudaStream_t st, bool keep_status, int tile_cap = kTileDefault)
{
    // occupancy of the chosen instantiation, cached (the query costs microseconds and this runs once per step in the
    // split multi-GPU / LightGCN / NeuMF paths)
    static thread_local StepKernel cached_k = nullptr;
    static thread_local int cached_per_sm = 0;
    if (cached_k != k) {
        int q = 0;
        DRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, k, kThreads, 0));
        cached_k = k;
        cached_per_sm = q;
    }
    const int per_sm = cached_per_sm;
    DRB_REQUIRE(per_sm > 0, "step kernel does not fit on an SM");
    const int max_grid = per_sm * sm_count();
    // tile: equal tiles of at most kTileMax triples, every CTA the same number of them
    const int tile = pick_tile((p.batch + max_grid - 1) / max_grid, tile_cap);
    p.tile = tile;
    long long tiles = (p.batch + tile - 1) / tile;
    long long rows_work = ((long long)p.U + p.I + 63) / 64;
    bool dense = p.dense_hint >= 0 ? (p.dense_hint != 0)
                                   : ((p.opt != DRB_OPT_SGD) || (3 * p.batch >= ((long long)p.U + p.I) / 4));
    long long want_grid = (dense && p.apply) ? (tiles > rows_work ? tiles : rows_work) : tiles;
    int grid = (int)(want_grid < 1 ? 1 : (want_grid > max_grid ? max_grid : want_grid));
    if (p.phases & 1)
        DRB_CUDA(cudaMemsetAsync(p.ws.hdr, 0, (p.phases == 3 && !keep_status) ? sizeof(WsHeader) : kHdrResetBytes, st));
    void *args[] = {&p};
    DRB_CUDA(cudaLaunchCooperativeKernel((void *)k, dim3(grid), dim3(kThreads), args, 0, st));
    return DRB_OK;
}

// ---- on-device selection of the step instantiation (lean_autotune below): seeded problems built on the host
struct CheckProblem {
    int U, I, F, B, K;
    std::vector<float> hP, hQ;
    std::vector<int32_t> hu, hi, hj;
};
static void make_check_problem(CheckProblem &c, int U, int I, int F, int B, int K, bool hot_users)
{
    c.U = U; c.I = I; c.F = F; c.B = B; c.K = K;
    c.hP.resize((size_t)U * F);
    c.hQ.resize((size_t)I * F);
    const long long n = (long long)B * K;
    c.hu.resize(n); c.hi.resize(n); c.hj.resize(n);
    unsigned long long x = 0x9E3779B97F4A7C15ull;
    auto rnd = [&]() { x = x * 6364136223846793005ull + 1442695040888963407ull; return (uint32_t)(x >> 33); };
    for (auto &v : c.hP) v = ((float)(rnd() % 20001) - 10000.f) * 2e-5f;
    for (auto &v : c.hQ) v = ((float)(rnd() % 20001) - 10000.f) * 2e-5f;
    for (long long t = 0; t < n; ++t) {
        c.hu[t] = (int32_t)(rnd() % (uint32_t)(hot_users ? U / 4 : U));
        const unsigned long long a = rnd() % (uint32_t)I;
        c.hi[t] = (int32_t)(hot_users ? a : a * a / (unsigned)I);      // timing problem: popular items, like the bench's planes
        c.hj[t] = (int32_t)(rnd() % (uint32_t)I);
    }
}
// one launch of K steps of instantiation k on a fresh copy of the problem; optional outputs: tables, losses, milliseconds of a
// second (warm) launch
static bool run_check_variant(const CheckProblem &c, StepKernel k, int opt, float lr, std::vector<float> *outP,
                              std::vector<float> *outQ, double *loss, float *ms, int tile_cap = kTileDefault)
{
    const long long n = (long long)c.B * c.K;
    const size_t wsb = carve(nullptr, c.U, c.I, c.F, opt, nullptr);
    float *dP = nullptr, *dQ = nullptr;
    void *dws = nullptr;
    int32_t *du = nullptr, *di = nullptr, *dj = nullptr;
    double *dl = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool good = cudaMalloc(&dP, c.hP.size() * 4) == cudaSuccess && cudaMalloc(&dQ, c.hQ.size() * 4) == cudaSuccess &&
                cudaMalloc(&dws, wsb) == cudaSuccess && cudaMalloc(&du, n * 4) == cudaSuccess &&
                cudaMalloc(&di, n * 4) == cudaSuccess && cudaMalloc(&dj, n * 4) == cudaSuccess &&
                cudaMalloc(&dl, c.K * 8) == cudaSuccess && cudaEventCreate(&e0) == cudaSuccess &&
                cudaEventCreate(&e1) == cudaSuccess;
    if (good) {
        cudaMemcpy(dP, c.hP.data(), c.hP.size() * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(dQ, c.hQ.data(), c.hQ.size() * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(du, c.hu.data(), n * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(di, c.hi.data(), n * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(dj, c.hj.data(), n * 4, cudaMemcpyHostToDevice);
        cudaMemset(dws, 0, wsb);
        drb_hyper h = {lr, 0.001f, 0.001f, opt, 0.9f, 0.999f, 1e-8f, DRB_LOSS_BPR};
        StepParams p;
        good = fill_params(p, dP, dQ, dws, c.U, c.I, c.F, du, di, dj, n, c.B, 0, c.K, &h, 0, dl, 1) == DRB_OK &&
               launch_kernel(k, p, (cudaStream_t)0, false, tile_cap) == DRB_OK &&
               cudaStreamSynchronize((cudaStream_t)0) == cudaSuccess;
        if (good && ms != nullptr) {
            *ms = 0.f;
            for (int rep = 0; rep < 2 && good; ++rep) {            // best of two warm launches
                float t = 0.f;
                cudaEventRecord(e0, (cudaStream_t)0);
                good = launch_kernel(k, p, (cudaStream_t)0, false, tile_cap) == DRB_OK;
                cudaEventRecord(e1, (cudaStream_t)0);
                good = good && cudaEventSynchronize(e1) == cudaSuccess && cudaEventElapsedTime(&t, e0, e1) == cudaSuccess;
                if (good && (rep == 0 || t < *ms)) *ms = t;
            }
        }
    }
    if (good && outP != nullptr) {
        outP->resize(c.hP.size());
        outQ->resize(c.hQ.size());
        good = cudaMemcpy(outP->data(), dP, c.hP.size() * 4, cudaMemcpyDeviceToHost) == cudaSuccess &&
               cudaMemcpy(outQ->data(), dQ, c.hQ.size() * 4, cudaMemcpyDeviceToHost) == cudaSuccess &&
               cudaMemcpy(loss, dl, c.K * 8, cudaMemcpyDeviceToHost) == cudaSuccess;
    }
    cudaFree(dP); cudaFree(dQ); cudaFree(dws); cudaFree(du); cudaFree(di); cudaFree(dj); cudaFree(dl);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    return good;
}

// what the BPR + SGD / Adam steps of one factor count run with
struct LeanChoice {
    int W = 0, NCH = 0;               // lanes per row, chunks per lane of the lean instantiation; W == 0: the general one
    int tile_cap = kTileDefault;
    float ms_general = 0.f, ms_lean = 0.f;   // timed launch of the autotune (best lean candidate)
};

// same losses (1e-5 rel) and tables (1e-5 abs) as the reference outputs of the general instantiation
static bool same_results(const CheckProblem &c, int opt, const std::vector<float> &P0, const std::vector<float> &Q0,
                         const double *l0, const std::vector<float> &P1, const std::vector<float> &Q1, const double *l1)
{
    bool ok = true;
    for (int k = 0; k < c.K; ++k) ok = ok && fabs(l0[k] - l1[k]) <= 1e-5 * fabs(l0[k]) && l0[k] > 0.0;
    // Adam turns a gradient that is pure rounding noise into a +-lr step of either sign: a few such elements may differ by up to
    // 2 lr between ANY two runs (also of the same kernel); everything else agrees to 1e-5
    int bad = 0;
    float worst = 0.f;
    double moved = 0.0;
    for (size_t e = 0; e < P0.size(); ++e) {
        const float dlt = fabsf(P0[e] - P1[e]);
        if (!(dlt <= 1e-5f)) { ++bad; worst = fmaxf(worst, dlt); }
        moved = fmax(moved, fabs((double)P0[e] - c.hP[e]));
    }
    for (size_t e = 0; e < Q0.size(); ++e) {
        const float dlt = fabsf(Q0[e] - Q1[e]);
        if (!(dlt <= 1e-5f)) { ++bad; worst = fmaxf(worst, dlt); }
    }
    ok = ok && (bad == 0 || (opt == DRB_OPT_ADAM && bad <= 4 && worst <= 0.11f));
    return ok && moved > 1e-4;                                   // and the steps did move the tables
}

// The lean instantiations were written after the last GPU slot of their round, so nothing about them is assumed: once per
// process and factor count every candidate geometry (1) must reproduce the general instantiation on a small seeded problem
// (two SGD and two Adam steps), and (2) is timed against it on an L2-regime problem with the bench's index statistics
// (3 steps x 524 288 triples, best of two warm launches).  The fastest correct candidate is used if it beats the general
// instantiation, and a larger index tile if that helps it further; otherwise the general kernel stays.  Never a wrong table,
// never a slower step.
static LeanChoice lean_autotune(int F, bool hbm)
{
    LeanChoice best;
    StepKernel gen = pick_kernel(F, false);
    int cw[3], cn[3];
    const int ncand = lean_candidates(F, cw, cn);
    if (gen == nullptr || ncand == 0) return best;
    CheckProblem small, big;
    make_check_problem(small, 96, 80, F, 384, 2, true);
    // timing problem: tables + accumulators inside L2 (like BASELINE config 2) or, for the HBM regime, 2 x 134 MB of user rows
    const int rows = hbm ? 33554432 / F : (F <= 64 ? 131072 : 65536);
    make_check_problem(big, rows, hbm ? 16384 : rows / 4, F, 1 << 19, 3, false);
    std::vector<float> refP[2], refQ[2];
    double refl[2][2];
    bool ok = true;
    for (int opt = DRB_OPT_SGD; opt <= DRB_OPT_ADAM && ok; ++opt)
        ok = run_check_variant(small, gen, opt, 0.05f, &refP[opt], &refQ[opt], refl[opt], nullptr);
    ok = ok && run_check_variant(big, gen, DRB_OPT_SGD, 0.01f, nullptr, nullptr, nullptr, &best.ms_general);
    float best_ms = 0.f;
    for (int k = 0; k < ncand && ok; ++k) {
        StepKernel lean = pick_lean_wn(cw[k], cn[k]);
        if (lean == nullptr) continue;
        bool same = true;
        for (int opt = DRB_OPT_SGD; opt <= DRB_OPT_ADAM && same; ++opt) {
            std::vector<float> P1, Q1;
            double l1[2];
            same = run_check_variant(small, lean, opt, 0.05f, &P1, &Q1, l1, nullptr) &&
                   same_results(small, opt, refP[opt], refQ[opt], refl[opt], P1, Q1, l1);
        }
        cudaGetLastError();
        if (!same) {
            fprintf(stderr, "[daisyrec_b200] lean step kernel %d lanes x %d chunks (factors=%d) did not reproduce the general "
                            "instantiation: not used\n", cw[k], cn[k], F);
            continue;
        }
        float ms = 0.f;
        if (!run_check_variant(big, lean, DRB_OPT_SGD, 0.01f, nullptr, nullptr, nullptr, &ms) || !(ms > 0.f)) continue;
        if (best_ms == 0.f || ms < best_ms) { best_ms = ms; best.W = cw[k]; best.NCH = cn[k]; }
    }
    cudaGetLastError();
    best.ms_lean = best_ms;
    if (!ok || best.W == 0 || !(best_ms < 0.98f * best.ms_general)) {
        if (ok && best.W != 0)
            fprintf(stderr, "[daisyrec_b200] lean step kernel (factors=%d): %.3f ms against %.3f ms of the general instantiation on "
                            "the timing problem: keeping the general one\n", F, best_ms, best.ms_general);
        best.W = best.NCH = 0;
        return best;
    }
    float ms_big_tile = 0.f;                                      // a larger index tile for the chosen candidate?
    if (run_check_variant(big, pick_lean_wn(best.W, best.NCH), DRB_OPT_SGD, 0.01f, nullptr, nullptr, nullptr, &ms_big_tile,
                          kTileMax) && ms_big_tile > 0.f && ms_big_tile < 0.98f * best_ms) {
        best.tile_cap = kTileMax;
        best.ms_lean = ms_big_tile;
    }
    cudaGetLastError();
    return best;
}

// regime of a problem: do the two tables and their accumulators fit the L2 cache?
static bool hbm_regime(long long table_rows, int F)
{
    static const long long l2 = [] {
        int dev = 0, bytes = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&bytes, cudaDevAttrL2CacheSize, dev) != cudaSuccess) {
            cudaGetLastError();
            bytes = 0;
        }
        return (long long)(bytes > 0 ? bytes : 64 << 20);
    }();
    return table_rows * (long long)F * 8 > l2;
}

static const LeanChoice &lean_choice(int F, long long table_rows)
{
    static const bool no_lean = getenv("DRB_NO_LEAN") != nullptr;   // developer switch: A/B the instantiations
    static std::mutex mu;
    static std::map<int, LeanChoice> state;
    const bool hbm = hbm_regime(table_rows, F);
    const int key = F * 2 + (hbm ? 1 : 0);
    std::lock_guard<std::mutex> lock(mu);
    auto it = state.find(key);
    if (it == state.end()) it = state.emplace(key, no_lean ? LeanChoice() : lean_autotune(F, hbm)).first;
    return it->second;
}

// exported to p2p.cu: the lean geometry and index-tile cap chosen for this factor count and table size (W == 0: general)
bool lean_enabled(int F, long long table_rows) { return lean_choice(F, table_rows).W > 0; }
void lean_geom(int F, long long table_rows, int &W, int &NCH)
{
    const LeanChoice &c = lean_choice(F, table_rows);
    W = c.W;
    NCH = c.NCH;
}
int lean_tile_cap(int F, long long table_rows) { return lean_choice(F, table_rows).tile_cap; }

int launch_steps(StepParams &p, cudaStream_t st, bool keep_status)
{
    // lean: the MF hot path; GEN: any loss but BPR, Adagrad / RMSprop sweeps, FM biases, deterministic accumulation
    StepKernel k = nullptr;
    int tile_cap = kTileDefault;
    if (step_params_lean(p)) {
        const LeanChoice &c = lean_choice(p.F, (long long)p.U + p.I);
        if (c.W > 0) {
            k = pick_lean_wn(c.W, c.NCH);
            tile_cap = c.tile_cap;
        }
    }
    if (k == nullptr) {
        k = pick_kernel(p.F, p.loss != DRB_LOSS_BPR || p.opt > DRB_OPT_ADAM || p.bias != nullptr || p.det != 0);
        tile_cap = kTileDefault;
    }
    DRB_REQUIRE(!p.det || (p.phases == 3 && p.ws.gP64 != nullptr), "deterministic accumulation: single-GPU fused steps with a "
                "workspace from drb_mf_workspace_bytes_det");
    DRB_REQUIRE(k != nullptr, "unsupported factors=%d (row too long for 32 lanes x 8 chunks)", p.F);
    return launch_kernel(k, p, st, keep_status, tile_cap);
}

int check_nan(void *d_ws, cudaStream_t st, int64_t *nan_step)
{
    WsHeader h;
    DRB_CUDA(cudaMemcpyAsync(&h, d_ws, sizeof(WsHeader), cudaMemcpyDeviceToHost, st));
    DRB_CUDA(cudaStreamSynchronize(st));
    if (h.status == DRB_ERR_NAN_LOSS) {
        if (nan_step) *nan_step = h.nan_step;
        set_error("Loss=Nan or Infinity at step %lld: current settings does not fit the recommender", h.nan_step);
        return DRB_ERR_NAN_LOSS;
    }
    if (nan_step) *nan_step = -1;
    return DRB_OK;
}

}  // namespace drb

using namespace drb;

extern "C" size_t drb_mf_workspace_bytes(int32_t U, int32_t I, int32_t F, int32_t opt)
{
    return carve(nullptr, U, I, F, opt, nullptr);
}

// 1: BPR + SGD/Adam steps at this factor count run the lean instantiation (after its self-check), 0: the general one.
// lanes / chunks (optional) receive the lane geometry of that instantiation.
extern "C" int drb_mf_step_variant(int32_t F, int64_t table_rows, int32_t *lanes, int32_t *chunks)
{
    int W = 0, NCH = 0;
    drb::lean_geom(F, table_rows, W, NCH);
    const bool lean = W > 0;
    if (!lean && F > 0) {
        drb::RowGeom g = drb::row_geom(F);
        W = g.width;
        NCH = g.nch;
    }
    if (lanes) *lanes = W;
    if (chunks) *chunks = NCH;
    return lean ? 1 : 0;
}

// the timing half of the on-device selection for `factors`: milliseconds of the timed launch (3 steps of 524 288 triples) of the
// general instantiation and of the best lean candidate, and the index-tile cap in use (runs the selection if it has not run)
extern "C" int drb_mf_step_selfcheck_ms(int32_t F, int64_t table_rows, float *ms_general, float *ms_lean, int32_t *tile_cap)
{
    const drb::LeanChoice &c = drb::lean_choice(F, table_rows);
    if (ms_general) *ms_general = c.ms_general;
    if (ms_lean) *ms_lean = c.ms_lean;
    if (tile_cap) *tile_cap = c.tile_cap;
    return DRB_OK;
}

// host-only: the lane geometry of the lean (lean != 0) or the canonical instantiation for `factors`, and the tile size the
// launcher picks for `per_cta` triples per CTA and step (no device needed)
extern "C" int drb_mf_step_geometry(int32_t F, int32_t lean, int32_t *lanes, int32_t *chunks, int64_t per_cta, int32_t *tile)
{
    int W = 0, NCH = 0;
    if (lean) {
        drb::lean_default_geom(F, W, NCH);
    } else if (F > 0) {
        drb::RowGeom g = drb::row_geom(F);
        W = g.width;
        NCH = g.nch;
    }
    if (lanes) *lanes = W;
    if (chunks) *chunks = NCH;
    if (tile) *tile = drb::pick_tile(per_cta);
    return W > 0 ? DRB_OK : DRB_ERR_INVALID;
}

extern "C" int drb_mf_workspace_init(void *d_ws, int32_t U, int32_t I, int32_t F, int32_t opt, void *stream)
{
    DRB_REQUIRE(d_ws != nullptr && U > 0 && I > 0 && F > 0, "workspace_init: bad arguments");
    size_t bytes = carve(nullptr, U, I, F, opt, nullptr);
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, bytes, (cudaStream_t)stream));
    return DRB_OK;
}

namespace drb {
int fill_params(StepParams &p, float *P, float *Q, void *d_ws, int U, int I, int F, const int32_t *bu, const int32_t *bi,
                const int32_t *bj, long long n, long long batch, long long first, long long nsteps, const drb_hyper *h,
                long long adam_step0, double *d_step_loss, int apply, float *d_bias, int det, int shared)
{
    DRB_REQUIRE(P && Q && d_ws && bu && bi && bj && h && d_step_loss, "null pointer argument");
    DRB_REQUIRE((shared ? U == 0 && P == Q && h->loss == DRB_LOSS_CL && !d_bias && !det : U > 0) && I > 0 && F > 0 && batch > 0 && n >= 0 && first >= 0 && nsteps >= 0, "bad sizes");
    DRB_REQUIRE(h->opt >= DRB_OPT_SGD && h->opt <= DRB_OPT_RMSPROP, "unknown optimizer id %d", h->opt);
    DRB_REQUIRE(h->loss >= DRB_LOSS_BPR && h->loss <= DRB_LOSS_SL, "unknown loss id %d", h->loss);
    DRB_REQUIRE((first + nsteps - 1) * batch < n || nsteps == 0 || n == 0, "steps [%lld,%lld) exceed %lld triples", first,
                first + nsteps, n);
    p.P = P; p.Q = Q;
    carve(d_ws, U, I, F, h->opt, &p.ws, d_bias != nullptr, det);
    p.det = det;
    p.bu = bu; p.bi = bi; p.bj = bj;
    p.n = n; p.batch = batch; p.first_step = first; p.n_steps = nsteps;
    p.U = U; p.I = I; p.F = F;
    copy_hyper(p, h);
    p.loss = h->loss;
    p.adam_step0 = adam_step0;
    p.step_loss = d_step_loss;
    p.apply = apply;
    p.bias = d_bias;
    if (shared) {   // both gradient contributions of a triple accumulate into the one table's accumulator
        p.shared = 1;
        p.ws.gP = p.ws.gQ;
    }
    return DRB_OK;
}
}  // namespace drb

extern "C" int drb_mf_bpr_train_steps(float *d_P, float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F,
                                      const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n,
                                      int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *hyper,
                                      int64_t adam_step0, double *d_step_loss, int32_t sync_and_check,
                                      int64_t *nan_step, void *stream)
{
    StepParams p;
    int rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, d_bu, d_bi, d_bj, n, batch, first_step, n_steps, hyper, adam_step0,
                         d_step_loss, 1);
    if (rc != DRB_OK) return rc;
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_steps(p, st);
    if (rc != DRB_OK) return rc;
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

// Deterministic accumulation (opt-in): the same steps with every cross-thread sum taken in fixed point, so that two runs --
// and any two orders of the atomics -- give bitwise identical tables and losses.  Workspace: drb_mf_workspace_bytes_det.
extern "C" size_t drb_mf_workspace_bytes_det(int32_t U, int32_t I, int32_t F, int32_t opt)
{
    return carve(nullptr, U, I, F, opt, nullptr, 0, 1);
}

extern "C" int drb_mf_bpr_train_steps_det(float *d_P, float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F,
                                          const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n,
                                          int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *hyper,
                                          int64_t adam_step0, double *d_step_loss, int32_t sync_and_check, int64_t *nan_step,
                                          void *stream)
{
    StepParams p;
    int rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, d_bu, d_bi, d_bj, n, batch, first_step, n_steps, hyper, adam_step0,
                         d_step_loss, 1, nullptr, 1);
    if (rc != DRB_OK) return rc;
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_steps(p, st);
    if (rc != DRB_OK) return rc;
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

extern "C" int drb_mf_bpr_train_steps_fused_neg(float *d_P, float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F,
                                                const int32_t *d_bu, const int32_t *d_bi, const int64_t *d_row_ptr,
                                                const int32_t *d_col, uint64_t seed, int32_t *d_neg_out, int64_t n,
                                                int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *hyper,
                                                int64_t adam_step0, double *d_step_loss, int32_t sync_and_check,
                                                int64_t *nan_step, void *stream)
{
    DRB_REQUIRE(d_row_ptr && d_col, "train_steps_fused_neg: the user->item CSR is required");
    DRB_REQUIRE(hyper && hyper->loss < DRB_LOSS_CL, "train_steps_fused_neg: pair-wise losses only");
    StepParams p;
    // the negative plane is unused in this mode (bi stands in so that the TMA staging code stays uniform)
    int rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, d_bu, d_bi, d_bi, n, batch, first_step, n_steps, hyper, adam_step0,
                         d_step_loss, 1);
    if (rc != DRB_OK) return rc;
    if (n_steps == 0) return DRB_OK;
    p.neg_row_ptr = d_row_ptr;
    p.neg_col = d_col;
    p.neg_out = d_neg_out;
    p.neg_seed = seed;
    p.dense_hint = 1;   // phase 2 must not re-derive negatives: dense sweep only
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_steps(p, st);
    if (rc != DRB_OK) return rc;
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

extern "C" int drb_mf_bpr_loss(const float *d_P, const float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F,
                               const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t batch,
                               const drb_hyper *hyper, double *d_loss, void *stream)
{
    StepParams p;
    int rc = fill_params(p, (float *)d_P, (float *)d_Q, d_ws, U, I, F, d_bu, d_bi, d_bj, batch, batch, 0, 1, hyper, 0,
                         d_loss, 0);
    if (rc != DRB_OK) return rc;
    return launch_steps(p, (cudaStream_t)stream);
}

// ---- FM (daisy/model/FMRecommender.py:61-97): the MF step with first-order terms; d_bias = [u_bias (U), i_bias (I), bias_]
extern "C" size_t drb_fm_workspace_bytes(int32_t U, int32_t I, int32_t F, int32_t opt)
{
    return carve(nullptr, U, I, F, opt, nullptr, 1);
}

extern "C" int drb_fm_workspace_init(void *d_ws, int32_t U, int32_t I, int32_t F, int32_t opt, void *stream)
{
    DRB_REQUIRE(d_ws != nullptr && U > 0 && I > 0 && F > 0, "fm_workspace_init: bad arguments");
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, carve(nullptr, U, I, F, opt, nullptr, 1), (cudaStream_t)stream));
    return DRB_OK;
}

extern "C" int drb_fm_train_steps(float *d_P, float *d_Q, float *d_bias, void *d_ws, int32_t U, int32_t I, int32_t F,
                                  const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch,
                                  int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                                  int32_t apply, double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream)
{
    DRB_REQUIRE(d_bias != nullptr, "fm_train_steps: the bias vector is required");
    StepParams p;
    int rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, d_bu, d_bi, d_bj, n, batch, first_step, n_steps, hyper, adam_step0,
                         d_step_loss, apply ? 1 : 0, d_bias);
    if (rc != DRB_OK) return rc;
    if (n_steps == 0) return DRB_OK;
    DRB_REQUIRE(apply || n_steps == 1, "fm_train_steps: apply=0 evaluates the loss of ONE batch");
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_steps(p, st);
    if (rc != DRB_OK) return rc;
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

extern "C" int drb_mf_bpr_train_step_host(float *d_P, float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F,
                                          const int32_t *h_bu, const int32_t *h_bi, const int32_t *h_bj, int64_t batch,
                                          const drb_hyper *hyper, int64_t adam_step0, int32_t *d_stage, double *h_loss,
                                          void *stream)
{
    DRB_REQUIRE(h_bu && h_bi && h_bj && d_stage && h_loss && batch > 0, "train_step_host: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    size_t stride = (size_t)((batch + 3) / 4 * 4);  // keep each array 16-byte aligned for the TMA path
    size_t bytes = sizeof(int32_t) * (size_t)batch;
    DRB_CUDA(cudaMemcpyAsync(d_stage, h_bu, bytes, cudaMemcpyHostToDevice, st));
    DRB_CUDA(cudaMemcpyAsync(d_stage + stride, h_bi, bytes, cudaMemcpyHostToDevice, st));
    DRB_CUDA(cudaMemcpyAsync(d_stage + 2 * stride, h_bj, bytes, cudaMemcpyHostToDevice, st));
    double *d_loss = (double *)(d_stage + 3 * stride);
    StepParams p;
    int rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, d_stage, d_stage + stride, d_stage + 2 * stride, batch, batch, 0, 1,
                         hyper, adam_step0, d_loss, 1);
    if (rc != DRB_OK) return rc;
    rc = launch_steps(p, st);
    if (rc != DRB_OK) return rc;
    DRB_CUDA(cudaMemcpyAsync(h_loss, d_loss, sizeof(double), cudaMemcpyDeviceToHost, st));
    int64_t nan_step = -1;
    return check_nan(d_ws, st, &nan_step);
}

// Pipelined end-to-end steps from HOST index planes: the H2D copy of step s+1 (copy stream) overlaps the
// kernel of step s (compute stream); every step's loss is read back to the host asynchronously.
extern "C" int drb_mf_bpr_train_steps_host(float *d_P, float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F,
                                           const int32_t *h_bu, const int32_t *h_bi, const int32_t *h_bj, int64_t n,
                                           int64_t batch, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                                           int32_t *d_stage, double *d_loss, double *h_loss, int64_t *nan_step,
                                           void *stream)
{
    DRB_REQUIRE(h_bu && h_bi && h_bj && d_stage && d_loss && h_loss && batch > 0 && n_steps >= 0 && n >= 0,
                "train_steps_host: bad arguments");
    DRB_REQUIRE(n_steps == 0 || (n_steps - 1) * batch < n, "train_steps_host: %lld steps exceed %lld triples",
                (long long)n_steps, (long long)n);
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local cudaStream_t copy_st = nullptr;
    if (!copy_st) DRB_CUDA(cudaStreamCreateWithFlags(&copy_st, cudaStreamNonBlocking));
    cudaEvent_t ready[2], freed[2], start;
    for (int k = 0; k < 2; ++k) {
        DRB_CUDA(cudaEventCreateWithFlags(&ready[k], cudaEventDisableTiming));
        DRB_CUDA(cudaEventCreateWithFlags(&freed[k], cudaEventDisableTiming));
    }
    DRB_CUDA(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
    const size_t stride = (size_t)((batch + 3) / 4 * 4);
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(WsHeader), st));   // clear a stale NaN flag once; sticky afterwards
    DRB_CUDA(cudaEventRecord(start, st));
    DRB_CUDA(cudaStreamWaitEvent(copy_st, start, 0));            // staging slots may still be in use upstream
    int rc = DRB_OK;
    for (int64_t s = 0; s < n_steps && rc == DRB_OK; ++s) {
        const int slot = (int)(s & 1);
        int32_t *sb = d_stage + (size_t)slot * 3 * stride;
        const int64_t base = s * batch, nb = (n - base < batch) ? n - base : batch;
        const size_t bytes = sizeof(int32_t) * (size_t)nb;
        if (s >= 2) DRB_CUDA(cudaStreamWaitEvent(copy_st, freed[slot], 0));
        DRB_CUDA(cudaMemcpyAsync(sb, h_bu + base, bytes, cudaMemcpyHostToDevice, copy_st));
        DRB_CUDA(cudaMemcpyAsync(sb + stride, h_bi + base, bytes, cudaMemcpyHostToDevice, copy_st));
        DRB_CUDA(cudaMemcpyAsync(sb + 2 * stride, h_bj + base, bytes, cudaMemcpyHostToDevice, copy_st));
        DRB_CUDA(cudaEventRecord(ready[slot], copy_st));
        DRB_CUDA(cudaStreamWaitEvent(st, ready[slot], 0));
        StepParams p;
        rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, sb, sb + stride, sb + 2 * stride, nb, nb, 0, 1, hyper, adam_step0 + s,
                         d_loss + s, 1);
        if (rc == DRB_OK) rc = launch_steps(p, st, /*keep_status=*/true);
        if (rc != DRB_OK) break;
        DRB_CUDA(cudaEventRecord(freed[slot], st));
        DRB_CUDA(cudaMemcpyAsync(h_loss + s, d_loss + s, sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    int rc2 = (rc == DRB_OK) ? check_nan(d_ws, st, nan_step) : rc;
    cudaStreamSynchronize(copy_st);
    for (int k = 0; k < 2; ++k) {
        cudaEventDestroy(ready[k]);
        cudaEventDestroy(freed[k]);
    }
    cudaEventDestroy(start);
    return rc2;
}

extern "C" int drb_gather_triples(const int32_t *d_triples, const int64_t *d_perm, int64_t n, int32_t *d_bu,
                                  int32_t *d_bi, int32_t *d_bj, void *stream)
{
    DRB_REQUIRE(d_triples && d_bu && d_bi && d_bj && n >= 0, "gather_triples: bad arguments");
    if (n == 0) return DRB_OK;
    gather_triples_kernel<<<grid_size(n, 256), 256, 0, (cudaStream_t)stream>>>(d_triples, d_perm, n, d_bu, d_bi, d_bj);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_mf_workspace_layout(int32_t U, int32_t I, int32_t F, int32_t opt, int64_t *out8)
{
    DRB_REQUIRE(out8 && U > 0 && I > 0 && F > 0, "workspace_layout: bad arguments");
    Workspace w;
    carve((void *)(uintptr_t)256, U, I, F, opt, &w);   // fake non-null base: pointers become offsets + 256
    auto off = [](const void *p) { return (int64_t)((uintptr_t)p - 256); };
    out8[0] = off(&w.hdr->acc[0][0]);  out8[1] = 8 * sizeof(double);
    out8[2] = off(w.gQ);               out8[3] = (int64_t)sizeof(float) * I * F;
    out8[4] = off(w.cntI);             out8[5] = (int64_t)sizeof(unsigned long long) * I;
    out8[6] = off(w.gP);               out8[7] = off(w.cntU);
    return DRB_OK;
}

extern "C" int drb_mf_bpr_phase(float *d_P, float *d_Q, void *d_ws, int32_t U, int32_t I, int32_t F, const int32_t *d_bu,
                                const int32_t *d_bi, const int32_t *d_bj, int64_t begin, int64_t count, int32_t phase,
                                const drb_hyper *hyper, int64_t adam_step0, double *d_loss, void *stream)
{
    DRB_REQUIRE(phase == 1 || phase == 2, "mf_bpr_phase: phase must be 1 or 2");
    DRB_REQUIRE(begin >= 0 && count >= 0, "mf_bpr_phase: bad range");
    DRB_REQUIRE(hyper && hyper->loss < DRB_LOSS_CL, "mf_bpr_phase: the sharded step covers the pair-wise losses only");
    StepParams p;
    // count may be 0 on a rank (its users have no triple in this global batch): phases still run (loss, sweep)
    int rc = fill_params(p, d_P, d_Q, d_ws, U, I, F, d_bu + begin, d_bi + begin, d_bj + begin, count, count > 0 ? count : 1,
                         0, 1, hyper, adam_step0, d_loss, 1);
    if (rc != DRB_OK) return rc;
    p.phases = phase;
    p.dense_hint = 1;
    return launch_steps(p, (cudaStream_t)stream);
}

// ---- Item2Vec (daisy/model/Item2VecRecommender.py): the point-wise CL step on ONE shared item table, and the user rows
namespace drb {
// P[u] = sum of Q[i] over the user's sorted train row, for every user with a train item (:56-60); one warp per user,
// the row's items summed in order, lanes over the factors
__global__ void item2vec_user_embed_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ col,
                                           const float *__restrict__ Q, int U, int F, float *__restrict__ P)
{
    const int lane = threadIdx.x & 31;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long u = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < U; u += nw) {
        const long long b = row_ptr[u], e = row_ptr[u + 1];
        if (b == e) continue;           // not a key of train_ur: the row keeps its initial values
        for (int f = lane; f < F; f += 32) {
            float acc = 0.f;
            for (long long s = b; s < e; ++s) acc += __ldg(Q + (size_t)__ldg(col + s) * F + f);
            P[(size_t)u * F + f] = acc;
        }
    }
}
}  // namespace drb

extern "C" size_t drb_item2vec_workspace_bytes(int32_t I, int32_t F, int32_t opt)
{
    return carve(nullptr, 0, I, F, opt, nullptr);
}

extern "C" int drb_item2vec_workspace_init(void *d_ws, int32_t I, int32_t F, int32_t opt, void *stream)
{
    DRB_REQUIRE(d_ws != nullptr && I > 0 && F > 0, "item2vec_workspace_init: bad arguments");
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, carve(nullptr, 0, I, F, opt, nullptr), (cudaStream_t)stream));
    return DRB_OK;
}

extern "C" int drb_item2vec_train_steps(float *d_Q, void *d_ws, int32_t I, int32_t F, const int32_t *d_bt, const int32_t *d_bc,
                                        const int32_t *d_blabel, int64_t n, int64_t batch, int64_t first_step, int64_t n_steps,
                                        const drb_hyper *hyper, int64_t adam_step0, int32_t apply, double *d_step_loss,
                                        int32_t sync_and_check, int64_t *nan_step, void *stream)
{
    DRB_REQUIRE(hyper && hyper->loss == DRB_LOSS_CL, "item2vec_train_steps: the loss is BCEWithLogitsLoss (DRB_LOSS_CL)");
    DRB_REQUIRE(hyper->reg_1 == 0.f && hyper->reg_2 == 0.f, "item2vec_train_steps: Item2Vec has no regulariser");
    StepParams p;
    int rc = fill_params(p, d_Q, d_Q, d_ws, 0, I, F, d_bt, d_bc, d_blabel, n, batch, first_step, n_steps, hyper, adam_step0,
                         d_step_loss, apply ? 1 : 0, nullptr, 0, 1);
    if (rc != DRB_OK) return rc;
    if (n_steps == 0) return DRB_OK;
    DRB_REQUIRE(apply || n_steps == 1, "item2vec_train_steps: apply=0 evaluates the loss of ONE batch");
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_steps(p, st);
    if (rc != DRB_OK) return rc;
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

extern "C" int drb_item2vec_user_embed(const int64_t *d_row_ptr, const int32_t *d_col, const float *d_Q, int32_t U, int32_t F,
                                       float *d_P, void *stream)
{
    DRB_REQUIRE(d_row_ptr && d_col && d_Q && d_P && U >= 0 && F > 0, "item2vec_user_embed: bad arguments");
    if (U == 0) return DRB_OK;
    item2vec_user_embed_kernel<<<grid_size((long long)U * 32, 256), 256, 0, (cudaStream_t)stream>>>(d_row_ptr, d_col, d_Q, U,
                                                                                                   F, d_P);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}
