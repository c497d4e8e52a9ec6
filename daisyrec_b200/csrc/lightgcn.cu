// lightgcn.cu -- LightGCN + BPR on the B200 path (SURVEY 8(a) row a15).
//
// Stands behind daisy/model/LightGCNRecommender.py:
//   forward   :117-129   E_l = A_hat E_{l-1} (torch.sparse.mm, :122), mean over the L+1 layers
//   calc_loss :131-169   BPR on the PROPAGATED rows, un-squared L1/Frobenius regulariser on the EGO rows
//   backward + optimizer.step (AbstractRecommender.py:125-126; Adam by default, LightGCNRecommender.py:59)
//   rank / full_rank / predict :171-211 on the cached propagated tables (drb_mf_rank & co. on E_mean)
//
// Design.  E_0 = cat(P, Q) is ONE contiguous [(U+I), F] fp32 table.  The reference runs 2L sparse-dense
// products per step through autograd (L forward, L backward); here both directions are the same kernel,
// because E_mean = 1/(L+1) sum_l A^l E_0 with A symmetric gives dL/dE_0 = 1/(L+1) sum_l A^l (dL/dE_mean):
//   forward : S = E_0;  X_l = A X_{l-1};  S += X_l;          E_mean = S/(L+1)
//   phase 1 : the MF step kernel (mf_bpr.cu) on (E_mean_user, E_mean_item) -> G = dL/dE_mean (RED.ADD.F32x4),
//             loss + ego-row norms + row counters
//   backward: S' = G;   T_l = A T_{l-1};  S' += T_l
//   phase 2 : the MF dense sweep on E_0 with gradient gscale * S' + count * regulariser -> SGD / dense Adam
//
// SpMM kernel: CSR rows are cut into segments of <= kSegLen edges (popular items have 10^5 neighbours);
// a lane group (W = F/4 lanes) owns a segment: 128-bit gathers of neighbour rows (4 edges in flight),
// sequential fmaf accumulation in ascending-column order; single-segment rows are written with plain
// stores (deterministic), multi-segment rows are combined with RED.ADD.F32x4.  HBM/L2-bound:
// algorithmic bytes per product = nnzA*(8 + 4F) + n*4F (SURVEY 8(d)).
#include "step.cuh"
#include "spmm.cuh"

namespace drb {

constexpr int kSpmmThreads = 256;
constexpr int kSegLen = 256;

struct LgcnWs {
    WsHeader *hdr;
    float *Em, *Xa, *Xb, *G, *Gs;
    unsigned *cntU;
    unsigned long long *cntI;
    float *m, *v;
};

static size_t carve_lgcn(void *base, int U, int I, int F, int opt, LgcnWs *w)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align256(bytes);
        return p;
    };
    const size_t tab = sizeof(float) * ((size_t)U + I) * F;
    LgcnWs t;
    t.hdr = (WsHeader *)take(256);
    t.Em = (float *)take(tab);
    t.Xa = (float *)take(tab);
    t.Xb = (float *)take(tab);
    t.G = (float *)take(tab);
    t.Gs = (float *)take(tab);
    t.cntU = (unsigned *)take(sizeof(unsigned) * (size_t)U);
    t.cntI = (unsigned long long *)take(sizeof(unsigned long long) * (size_t)I);
    t.m = t.v = nullptr;
    if (opt == DRB_OPT_ADAM) {
        t.m = (float *)take(tab);
        t.v = (float *)take(tab);
    }
    if (w) *w = t;
    return off;
}


// Y[r] (+)= sum_e val[e] * X[col[e]]  over the segment's edges;  S[r] += the same (layer-sum accumulator)
template <int VEC, int W, int NCH>
__global__ void __launch_bounds__(kSpmmThreads) spmm_seg_kernel(Adj a, const float *__restrict__ X, float *__restrict__ Y,
                                                                float *__restrict__ S, int F)
{
    constexpr int GPW = 32 / W, GROUPS = (kSpmmThreads / 32) * GPW, E = 4;
    const int lane = threadIdx.x & 31, gl = lane % W;
    const int group = (threadIdx.x >> 5) * GPW + lane / W;
    const int chunks = F / VEC;
    for (long long k = (long long)blockIdx.x * GROUPS + group; k < a.nseg; k += (long long)gridDim.x * GROUPS) {
        const int r = a.seg_row[k];
        const long long b = a.seg_ptr[k], e = a.seg_ptr[k + 1];
        Row<VEC, W, NCH> acc;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
            for (int q = 0; q < VEC; ++q) acc.c[ch].v[q] = 0.f;
        // main loop: whole groups of E edges, no bounds checks (a full segment is 256 edges = 64 iterations)
        long long e0 = b;
        for (; e0 + E <= e; e0 += E) {
            float vv[E];
            Row<VEC, W, NCH> x[E];
#pragma unroll
            for (int q = 0; q < E; ++q) {
                const int cq = __ldg(a.col + e0 + q);
                vv[q] = __ldg(a.val + e0 + q);
                x[q] = load_row<VEC, W, NCH>(X + (size_t)cq * F, gl, chunks, true);
            }
#pragma unroll
            for (int q = 0; q < E; ++q)
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
                    for (int z = 0; z < VEC; ++z) acc.c[ch].v[z] = fmaf(vv[q], x[q].c[ch].v[z], acc.c[ch].v[z]);
        }
        // tail: fewer than E edges left, same ascending-column accumulation order
        for (; e0 < e; ++e0) {
            const int cq = __ldg(a.col + e0);
            const float v1 = __ldg(a.val + e0);
            const Row<VEC, W, NCH> x1 = load_row<VEC, W, NCH>(X + (size_t)cq * F, gl, chunks, true);
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
                for (int z = 0; z < VEC; ++z) acc.c[ch].v[z] = fmaf(v1, x1.c[ch].v[z], acc.c[ch].v[z]);
        }
        const bool multi = (a.row_ptr[r + 1] - a.row_ptr[r]) != (e - b);
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            int c = gl + ch * W;
            if (c >= chunks) continue;
            float *yp = Y + (size_t)r * F + c * VEC, *sp = S ? S + (size_t)r * F + c * VEC : nullptr;
            if (!multi) {
                st_row<VEC>(yp, acc.c[ch]);
                if (sp) {
                    Vec<VEC> s = ld_row<VEC>(sp);
#pragma unroll
                    for (int z = 0; z < VEC; ++z) s.v[z] += acc.c[ch].v[z];
                    st_row<VEC>(sp, s);
                }
            } else {
                red_row<VEC>(yp, acc.c[ch]);
                if (sp) red_row<VEC>(sp, acc.c[ch]);
            }
        }
    }
}

__global__ void scale_kernel(float *__restrict__ x, long long n4, float s)
{
    float4 *p = reinterpret_cast<float4 *>(x);
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += (long long)gridDim.x * blockDim.x) {
        float4 v = p[k];
        v.x *= s; v.y *= s; v.z *= s; v.w *= s;
        p[k] = v;
    }
}
__global__ void scale_tail_kernel(float *__restrict__ x, long long from, long long n, float s)
{
    for (long long k = from + (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x)
        x[k] *= s;
}

typedef void (*SpmmKernel)(Adj, const float *, float *, float *, int);
template <int VEC>
static SpmmKernel pick_spmm_v(int W, int NCH)
{
#define DRB_CASE(w, n) \
    if (W == w && NCH == n) return spmm_seg_kernel<VEC, w, n>;
    DRB_CASE(1, 1) DRB_CASE(2, 1) DRB_CASE(4, 1) DRB_CASE(8, 1) DRB_CASE(16, 1) DRB_CASE(32, 1)
    DRB_CASE(32, 2) DRB_CASE(32, 4) DRB_CASE(32, 8)
#undef DRB_CASE
    return nullptr;
}

int launch_spmm(const Adj &a, const float *X, float *Y, float *S, int F, cudaStream_t st)
{
    RowGeom g = row_geom(F);
    SpmmKernel k = g.vec == 4 ? pick_spmm_v<4>(g.width, g.nch) : g.vec == 2 ? pick_spmm_v<2>(g.width, g.nch)
                                                                           : pick_spmm_v<1>(g.width, g.nch);
    DRB_REQUIRE(k != nullptr, "unsupported factors=%d", F);
    DRB_CUDA(cudaMemsetAsync(Y, 0, sizeof(float) * (size_t)a.n * F, st));   // zero-degree rows + RED targets
    if (a.nseg == 0) return DRB_OK;
    long long groups = (kSpmmThreads / 32) * (32 / g.width);
    long long blocks = (a.nseg + groups - 1) / groups, cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    k<<<(int)blocks, kSpmmThreads, 0, st>>>(a, X, Y, S, F);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

// S = X0; for l = 1..L: T = A T; S += T.   Leaves sum_l A^l X0 in S (NOT yet divided by L+1).
static int propagate_sum(const Adj &a, const float *X0, float *S, float *Xa, float *Xb, int F, int L, cudaStream_t st)
{
    DRB_CUDA(cudaMemcpyAsync(S, X0, sizeof(float) * (size_t)a.n * F, cudaMemcpyDeviceToDevice, st));
    const float *prev = X0;
    for (int l = 0; l < L; ++l) {
        float *y = (l & 1) ? Xb : Xa;
        int rc = launch_spmm(a, prev, y, S, F, st);
        if (rc != DRB_OK) return rc;
        prev = y;
    }
    return DRB_OK;
}

static int scale_table(float *x, long long n, float s, cudaStream_t st)
{
    long long n4 = n / 4;
    if (n4 > 0) scale_kernel<<<grid_size(n4, 256), 256, 0, st>>>(x, n4, s);
    if (n4 * 4 < n) scale_tail_kernel<<<1, 32, 0, st>>>(x, n4 * 4, n, s);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

}  // namespace drb

using namespace drb;

extern "C" int64_t drb_lgcn_segment_count(const int64_t *h_row_ptr, int64_t n)
{
    if (!h_row_ptr || n < 0) return -1;
    int64_t k = 0;
    for (int64_t r = 0; r < n; ++r) k += (h_row_ptr[r + 1] - h_row_ptr[r] + kSegLen - 1) / kSegLen;
    return k;
}

extern "C" int drb_lgcn_segments(const int64_t *h_row_ptr, int64_t n, int32_t *h_seg_row, int64_t *h_seg_ptr)
{
    DRB_REQUIRE(h_row_ptr && h_seg_row && h_seg_ptr && n >= 0, "lgcn_segments: bad arguments");
    int64_t k = 0;
    for (int64_t r = 0; r < n; ++r)
        for (int64_t b = h_row_ptr[r]; b < h_row_ptr[r + 1]; b += kSegLen) {
            h_seg_row[k] = (int32_t)r;
            h_seg_ptr[k] = b;
            ++k;
        }
    h_seg_ptr[k] = h_row_ptr[n];
    return DRB_OK;
}

extern "C" size_t drb_lgcn_workspace_bytes(int32_t U, int32_t I, int32_t F, int32_t opt)
{
    return carve_lgcn(nullptr, U, I, F, opt, nullptr);
}

extern "C" int drb_lgcn_workspace_init(void *d_ws, int32_t U, int32_t I, int32_t F, int32_t opt, void *stream)
{
    DRB_REQUIRE(d_ws && U > 0 && I > 0 && F > 0, "lgcn_workspace_init: bad arguments");
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, carve_lgcn(nullptr, U, I, F, opt, nullptr), (cudaStream_t)stream));
    return DRB_OK;
}

// forward(): d_Em[(U+I),F] = mean_l A^l E0     (LightGCNRecommender.py:117-129)
extern "C" int drb_lgcn_propagate(const float *d_E0, void *d_ws, int32_t U, int32_t I, int32_t F, int32_t L,
                                  const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                                  const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, float *d_Em,
                                  void *stream)
{
    DRB_REQUIRE(d_E0 && d_ws && d_row_ptr && d_Em && L >= 0 && U > 0 && I > 0 && F > 0, "lgcn_propagate: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    LgcnWs w;
    carve_lgcn(d_ws, U, I, F, DRB_OPT_SGD, &w);
    const Adj a{d_row_ptr, d_col, d_val, d_seg_row, d_seg_ptr, nseg, (long long)U + I};
    int rc = propagate_sum(a, d_E0, d_Em, w.Xa, w.Xb, F, L, st);
    if (rc != DRB_OK) return rc;
    return scale_table(d_Em, ((long long)U + I) * F, 1.f / (float)(L + 1), st);
}

// n_steps synchronous LightGCN+BPR steps (apply != 0) or the loss of one batch (apply == 0, n_steps == 1).
extern "C" int drb_lgcn_bpr_train_steps(float *d_E0, void *d_ws, int32_t U, int32_t I, int32_t F, int32_t L,
                                        const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                                        const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg,
                                        const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n,
                                        int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *h,
                                        int64_t adam_step0, int32_t apply, double *d_step_loss, int32_t sync_and_check,
                                        int64_t *nan_step, void *stream)
{
    DRB_REQUIRE(d_E0 && d_ws && d_row_ptr && d_bu && d_bi && d_bj && h && d_step_loss, "lgcn_train_steps: null argument");
    DRB_REQUIRE(U > 0 && I > 0 && F > 0 && L >= 0 && batch > 0 && n_steps >= 0, "lgcn_train_steps: bad sizes");
    DRB_REQUIRE(n_steps == 0 || (first_step + n_steps - 1) * batch < n, "lgcn_train_steps: steps exceed %lld triples",
                (long long)n);
    DRB_REQUIRE(h->opt == DRB_OPT_SGD || h->opt == DRB_OPT_ADAM, "unknown optimizer id %d", h->opt);
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    LgcnWs w;
    carve_lgcn(d_ws, U, I, F, h->opt, &w);
    const long long nn = (long long)U + I;
    const Adj a{d_row_ptr, d_col, d_val, d_seg_row, d_seg_ptr, nseg, nn};
    const size_t tab = sizeof(float) * (size_t)nn * F;
    const float inv = 1.f / (float)(L + 1);
    DRB_CUDA(cudaMemsetAsync(w.hdr, 0, sizeof(WsHeader), st));   // clear a stale NaN flag; sticky within the call
    for (int64_t s = 0; s < n_steps; ++s) {
        const int64_t base = (first_step + s) * batch, nb = (n - base < batch) ? n - base : batch;
        // forward propagation -> E_mean
        int rc = propagate_sum(a, d_E0, w.Em, w.Xa, w.Xb, F, L, st);
        if (rc == DRB_OK) rc = scale_table(w.Em, nn * F, inv, st);
        if (rc != DRB_OK) return rc;
        // phase 1 on the propagated tables (scores) + ego tables (norms): G = dL/dE_mean
        StepParams p = split_step(h, U, I, d_bu + base, d_bi + base, d_bj + base, nb, adam_step0 + s, d_step_loss + s);
        p.P = w.Em; p.Q = w.Em + (size_t)U * F; p.F = F;
        p.ws.hdr = w.hdr; p.ws.gP = w.G; p.ws.gQ = w.G + (size_t)U * F; p.ws.cntU = w.cntU; p.ws.cntI = w.cntI;
        p.ws.mP = w.m; p.ws.vP = w.v; p.ws.mQ = w.m ? w.m + (size_t)U * F : nullptr; p.ws.vQ = w.v ? w.v + (size_t)U * F : nullptr;
        p.Pn = d_E0; p.Qn = d_E0 + (size_t)U * F;
        p.dense_grad = 1;
        p.apply = apply ? 1 : 0;
        p.phases = apply ? 1 : 3;                                // loss only: both phases in one launch, no update
        if (!apply) return launch_steps(p, st, /*keep_status=*/true);
        DRB_CUDA(cudaMemsetAsync(w.G, 0, tab, st));
        rc = launch_steps(p, st, true);
        if (rc != DRB_OK) return rc;
        // backward propagation of the gradient: Gs = sum_l A^l G
        rc = propagate_sum(a, w.G, w.Gs, w.Xa, w.Xb, F, L, st);
        if (rc != DRB_OK) return rc;
        // phase 2 on the ego table with gradient Gs/(L+1) + regulariser
        p.P = d_E0; p.Q = d_E0 + (size_t)U * F;
        p.ws.gP = w.Gs; p.ws.gQ = w.Gs + (size_t)U * F;
        p.Pn = nullptr; p.Qn = nullptr;
        p.gscale = inv;
        p.phases = 2;
        rc = launch_steps(p, st, true);
        if (rc != DRB_OK) return rc;
    }
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}
