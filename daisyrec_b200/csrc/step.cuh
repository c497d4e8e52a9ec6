// step.cuh -- shared declarations of the BPR step kernel (mf_bpr.cu), reused by lightgcn.cu.
#pragma once
#include "common.cuh"

namespace drb {

struct WsHeader {
    unsigned long long barrier;  // grid barrier ticket counter          } reset before every phase-1 launch
    double acc[2][8];            // [parity][bpr, l1u, l1i, l1j, s2u, s2i, s2j, g(bias_)]  }
    long long nan_step;          // step whose loss was NaN               } sticky in split (multi-GPU) mode
    int status;
    int pad[13];
};
constexpr size_t kHdrResetBytes = sizeof(unsigned long long) + sizeof(double) * 16;
static_assert(sizeof(WsHeader) <= 256, "header must fit its slot");

struct Workspace {
    WsHeader *hdr = nullptr;
    float *gP = nullptr, *gQ = nullptr;
    unsigned *cntU = nullptr;
    unsigned long long *cntI = nullptr;
    float *mP = nullptr, *vP = nullptr, *mQ = nullptr, *vQ = nullptr;
    // FM's first-order terms (FMRecommender.py:46-49): gradient accumulator and optimiser state of the packed
    // [u_bias (U), i_bias (I), bias_ (1)] vector; nullptr for plain MF
    float *gB = nullptr, *mB = nullptr, *vB = nullptr;
    // deterministic accumulation (opt-in): phase 1 adds fixed-point int64 images of every contribution (integer addition is
    // associative: the sums do not depend on the order the atomics land in), converted to fp32 once before phase 2
    long long *gP64 = nullptr, *gQ64 = nullptr, *accfx = nullptr;   // table-shaped accumulators + [8] loss / norm sums
};

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

inline size_t carve(void *base, int U, int I, int F, int opt, Workspace *w, int fm = 0, int det = 0)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align256(bytes);
        return p;
    };
    Workspace t;
    t.hdr = (WsHeader *)take(256);
    t.gP = (float *)take(sizeof(float) * (size_t)U * F);
    t.gQ = (float *)take(sizeof(float) * (size_t)I * F);
    t.cntU = (unsigned *)take(sizeof(unsigned) * (size_t)U);
    t.cntI = (unsigned long long *)take(sizeof(unsigned long long) * (size_t)I);
    if (opt != DRB_OPT_SGD) {  // Adam: m and v; Adagrad / RMSprop: one state table each, in the m slot
        t.mP = (float *)take(sizeof(float) * (size_t)U * F);
        if (opt == DRB_OPT_ADAM) t.vP = (float *)take(sizeof(float) * (size_t)U * F);
        t.mQ = (float *)take(sizeof(float) * (size_t)I * F);
        if (opt == DRB_OPT_ADAM) t.vQ = (float *)take(sizeof(float) * (size_t)I * F);
    }
    if (fm) {   // appended, so the MF part of the layout (drb_mf_workspace_layout) is the same with and without biases
        const size_t nb = (size_t)U + I + 1;
        t.gB = (float *)take(sizeof(float) * nb);
        if (opt != DRB_OPT_SGD) t.mB = (float *)take(sizeof(float) * nb);
        if (opt == DRB_OPT_ADAM) t.vB = (float *)take(sizeof(float) * nb);
    }
    if (det) {  // appended after everything else: the other layouts do not move
        t.gP64 = (long long *)take(sizeof(long long) * (size_t)U * F);
        t.gQ64 = (long long *)take(sizeof(long long) * (size_t)I * F);
        t.accfx = (long long *)take(sizeof(long long) * 8);
    }
    if (w) *w = t;
    return off;
}

struct StepParams {
    float *P = nullptr, *Q = nullptr;
    Workspace ws;
    const int32_t *bu = nullptr, *bi = nullptr, *bj = nullptr;
    long long n = 0, batch = 0, first_step = 0, n_steps = 0;
    int U = 0, I = 0, F = 0, tile = 0;   // tile: set by the launcher
    float lr = 0.f, reg1 = 0.f, reg2 = 0.f;
    int opt = DRB_OPT_SGD;
    float beta1 = 0.f, beta2 = 0.f, eps = 0.f;
    long long adam_step0 = 0;
    double *step_loss = nullptr;
    int apply = 1;
    int phases = 3;        // bit 0: phase 1 (accumulate), bit 1: phase 2 (apply); 3 = fused persistent steps
    int dense_hint = -1;   // -1 auto, 0 claim, 1 dense sweep (multi-GPU: always dense, counters are global)
    // LightGCN: scores come from the propagated tables P,Q while the regulariser norms use the ego tables
    const float *Pn = nullptr, *Qn = nullptr;   // ego (norm) tables; nullptr = same as P,Q
    float gscale = 1.f;    // factor applied to the accumulated gradient in phase 2 (1/(L+1) for LightGCN)
    int dense_grad = 0;    // 1: every row has a gradient (propagated), not only the rows a triple touched
    // NeuMF: the item-side regulariser counts the negative occurrences 2x (GMF table) or 0x (MLP table)
    float neg_mult = 1.f;  // multiplier of the negative-occurrence count in the regulariser gradient
    int keep_counts = 0;   // 1: leave the row counters untouched (another table pair still needs them)
    // Fused negative sampling (throughput mode, NOT the reference's per-user-once table): when neg_row_ptr != nullptr the
    // negative of triple t of step s is drawn inside phase 1: k = Philox(seed; t, step) scaled to [0, I - deg(u)), then
    // the k-th item outside the user's sorted CSR row (same complement distribution as sampler.py:86, fresh every step).
    const int64_t *neg_row_ptr = nullptr;
    const int32_t *neg_col = nullptr;
    int32_t *neg_out = nullptr;   // optional: the drawn negatives are written here (aligned with bu/bi) for inspection
    unsigned long long neg_seed = 0;
    int loss = DRB_LOSS_BPR;      // DRB_LOSS_BPR / _HL / _TL (pair-wise criterion, AbstractRecommender.py:79-93)
    // FM (FMRecommender.py:61-68): pred += (u_bias[u] + i_bias[item]) + bias_; bias = packed [U + I + 1]; nullptr = MF
    float *bias = nullptr;
    // deterministic accumulation: run-to-run bitwise reproducible steps (fixed-point int64 atomics, see Workspace); single GPU,
    // fused persistent launch only
    int det = 0;
    // Item2Vec (Item2VecRecommender.py:48-52): both rows of a triple come from ONE table.  The launcher passes U = 0, P = Q and
    // ws.gP = ws.gQ; the kernel then counts the target row in cntI and claims it as an item row.  GEN instantiation only.
    int shared = 0;
    // multi-GPU persistent mode: step s trains local triples [step_offsets[s], step_offsets[s+1]) (device array; the union
    // of the ranks' ranges is the global batch s).  nullptr = uniform batches of `batch` triples.
    const long long *step_offsets = nullptr;
};

inline void copy_hyper(StepParams &p, const drb_hyper *h)
{
    p.lr = h->lr; p.reg1 = h->reg_1; p.reg2 = h->reg_2; p.opt = h->opt;
    p.beta1 = h->beta1; p.beta2 = h->beta2; p.eps = h->eps;
}

// One BPR step of the split-phase trainers (LightGCN, NGCF, NFM, NeuMF): a single step over the nb triples at bu/bi/bj with a
// dense phase-2 sweep.  The caller sets the tables, the workspace, the phases and whatever else its model needs.
inline StepParams split_step(const drb_hyper *h, int U, int I, const int32_t *bu, const int32_t *bi, const int32_t *bj,
                             long long nb, long long adam_step, double *step_loss)
{
    StepParams p;
    copy_hyper(p, h);
    p.bu = bu; p.bi = bi; p.bj = bj;
    p.n = p.batch = nb; p.first_step = 0; p.n_steps = 1;
    p.U = U; p.I = I;
    p.adam_step0 = adam_step;
    p.step_loss = step_loss;
    p.dense_hint = 1;
    p.loss = DRB_LOSS_BPR;
    return p;
}

int fill_params(StepParams &p, float *P, float *Q, void *d_ws, int U, int I, int F, const int32_t *bu, const int32_t *bi,
                const int32_t *bj, long long n, long long batch, long long first, long long nsteps, const drb_hyper *h,
                long long adam_step0, double *d_step_loss, int apply, float *d_bias = nullptr, int det = 0,
                int shared = 0);
int launch_steps(StepParams &p, cudaStream_t st, bool keep_status = false);
int check_nan(void *d_ws, cudaStream_t st, int64_t *nan_step);

}  // namespace drb
