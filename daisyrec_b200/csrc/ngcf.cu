// ngcf.cu -- NGCF + BPR on the B200 path (SURVEY 8(f) rank 4).
//
// Stands behind daisy/model/NGCFRecommender.py (node_dropout = mess_dropout = 0; the reference's dropout masks come from
// torch's RNG, and its message dropout is even active at rank() time, :164):
//   BiGNN.forward :51-59     X = A_hat E;  Y = Linear1(E + X) + Linear2(X * E)
//   NGCF.forward  :157-172   E_{l+1} = normalize(LeakyReLU_0.2(Y_l)) row-wise;  representation = cat(E_0 .. E_L, dim=1)
//   calc_loss     :174-205   BPR on the concatenated rows, un-squared L1 / Frobenius regulariser on the EGO rows
//   backward + optimizer.step (AbstractRecommender.py:125-126; Adam by default, NGCFRecommender.py:113)
//   rank / full_rank / predict :207-252 = dot products of the concatenated rows (drb_mf_rank & co. on the representation)
//
// One step is host-sequenced out of kernels that already exist plus four row-wise ones:
//   per layer   spmm_seg_kernel (lightgcn.cu) -> ngcf_mix_kernel [S | T] = [E + X | X * E] -> two GEMMs (neumf.cu dispatcher)
//               -> ngcf_act_kernel (bias, LeakyReLU, row norm, write E_{l+1} and its block of the representation)
//   scores      phase 1 of the MF step kernel on the [n, C] representation (C = sum of layer widths), ego tables for the norms
//   per layer, backwards   ngcf_act_bwd_kernel (normalize + LeakyReLU backward) -> bias column sums, two weight-gradient
//               GEMMs, two input-gradient GEMMs -> ngcf_mix_bwd_kernel (dE, dX) -> spmm (A_hat symmetric) -> add
//   update      phase 2 of the MF kernel on the ego table (dense gradient + counter-weighted regulariser, SGD / Adam),
//               dense_update (neumf.cu) on the flat layer block.
// Parameter block W (flat fp32, module registration order :106-108 / :46-47): per layer W1 [out, in], b1 [out], W2 [out, in],
// b2 [out].  HBM-bound like LightGCN: every step streams the [n, width] activations of every layer a handful of times.
#include "gemm.cuh"
#include "spmm.cuh"
#include "step.cuh"

namespace drb {

constexpr int kNgcfMaxL = 8;

struct NgcfDims {
    int U, I, L, C;
    long long n;
    int d[kNgcfMaxL + 1], off[kNgcfMaxL + 2];
    long long w_off[kNgcfMaxL], nW;
    int dmax;
};

static bool ngcf_dims(NgcfDims &q, int U, int I, const int32_t *dims, int L)
{
    if (U <= 0 || I <= 0 || !dims || L < 1 || L > kNgcfMaxL) return false;
    q.U = U; q.I = I; q.L = L; q.n = (long long)U + I;
    int C = 0, dmax = 0;
    long long o = 0;
    for (int l = 0; l <= L; ++l) {
        if (dims[l] <= 0 || dims[l] > 256) return false;                            // the GEMM tile covers N <= 256
        q.d[l] = dims[l];
        q.off[l] = C;
        C += dims[l];
        if (dims[l] > dmax) dmax = dims[l];
    }
    q.off[L + 1] = C;
    q.C = C; q.dmax = dmax;
    for (int l = 0; l < L; ++l) { q.w_off[l] = o; o += 2 * ((long long)dims[l] * dims[l + 1] + dims[l + 1]); }
    q.nW = o;
    return true;
}

struct NgcfWs {
    WsHeader *hdr;
    float *ALL, *G;                    // [n, C] representation and its gradient (phase-1 accumulators)
    float *E[kNgcfMaxL + 1];           // E_1 .. E_L   ([n, d_l]; E[0] = the ego table, not in the workspace)
    float *X[kNgcfMaxL], *Y[kNgcfMaxL];   // X_l = A E_l [n, d_l], Y_l pre-activation [n, d_{l+1}]
    float *rn[kNgcfMaxL];              // max(||Z row||, 1e-12)
    float *ST, *Y1, *Y2, *dY, *dS, *dT, *dX, *dEa, *dEb, *AdX;   // scratch, widest layer
    float *gE, *gW;                    // ego gradient [n, F], layer-block gradient
    double *scratch;                   // [8] phase 2 writes its own (MF-ordered) loss here; the real one comes from finalize
    unsigned *cntU;
    unsigned long long *cntI;
    float *mE, *vE, *mW, *vW;
};

static size_t carve_ngcf(void *base, const NgcfDims &q, int opt, NgcfWs *w)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align256(bytes);
        return p;
    };
    NgcfWs t;
    const size_t n = (size_t)q.n;
    t.hdr = (WsHeader *)take(256);
    t.ALL = (float *)take(sizeof(float) * n * q.C);
    t.G = (float *)take(sizeof(float) * n * q.C);
    t.E[0] = nullptr;
    for (int l = 0; l < q.L; ++l) {
        t.E[l + 1] = (float *)take(sizeof(float) * n * q.d[l + 1]);
        t.X[l] = (float *)take(sizeof(float) * n * q.d[l]);
        t.Y[l] = (float *)take(sizeof(float) * n * q.d[l + 1]);
        t.rn[l] = (float *)take(sizeof(float) * n);
    }
    const size_t wide = sizeof(float) * n * q.dmax;
    t.ST = (float *)take(2 * wide);
    t.Y1 = (float *)take(wide); t.Y2 = (float *)take(wide); t.dY = (float *)take(wide);
    t.dS = (float *)take(wide); t.dT = (float *)take(wide); t.dX = (float *)take(wide);
    t.dEa = (float *)take(wide); t.dEb = (float *)take(wide); t.AdX = (float *)take(wide);
    t.gE = (float *)take(sizeof(float) * n * q.d[0]);
    t.gW = (float *)take(sizeof(float) * (size_t)q.nW);
    t.scratch = (double *)take(sizeof(double) * 8);
    t.cntU = (unsigned *)take(sizeof(unsigned) * (size_t)q.U);
    t.cntI = (unsigned long long *)take(sizeof(unsigned long long) * (size_t)q.I);
    t.mE = t.vE = t.mW = t.vW = nullptr;
    if (opt == DRB_OPT_ADAM) {
        t.mE = (float *)take(sizeof(float) * n * q.d[0]); t.vE = (float *)take(sizeof(float) * n * q.d[0]);
        t.mW = (float *)take(sizeof(float) * (size_t)q.nW); t.vW = (float *)take(sizeof(float) * (size_t)q.nW);
    }
    if (w) *w = t;
    return off;
}

// scalar forms of the two mix kernels for layer widths that are not multiples of 4
__global__ void ngcf_mix_scalar_kernel(const float *__restrict__ E, const float *__restrict__ X, long long n, int d,
                                       float *__restrict__ ST)
{
    const long long total = n * d;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / d;
        const int c = (int)(k - r * d);
        const float e = __ldcg(E + k), x = X[k];
        ST[(size_t)r * 2 * d + c] = e + x;
        ST[(size_t)r * 2 * d + d + c] = x * e;
    }
}
__global__ void ngcf_mix_bwd_scalar_kernel(const float *__restrict__ dS, const float *__restrict__ dT, const float *__restrict__ E,
                                           const float *__restrict__ X, long long total, float *__restrict__ dEl,
                                           float *__restrict__ dX)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const float s = dS[k], t = dT[k];
        dEl[k] = fmaf(t, X[k], s);
        dX[k] = fmaf(t, __ldcg(E + k), s);
    }
}

// ST[r] = [E[r] + X[r] | X[r] * E[r]]   (BiGNN.forward :54-57), one thread per float4
__global__ void ngcf_mix_kernel(const float *__restrict__ E, const float *__restrict__ X, long long n, int d, float *__restrict__ ST)
{
    const int d4 = d / 4;
    const long long total = n * d4;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / d4;
        const int c = (int)(k - r * d4);
        const float4 e = __ldcg(reinterpret_cast<const float4 *>(E) + k), x = __ldcg(reinterpret_cast<const float4 *>(X) + k);
        float4 *o = reinterpret_cast<float4 *>(ST + (size_t)r * 2 * d);
        o[c] = make_float4(e.x + x.x, e.y + x.y, e.z + x.z, e.w + x.w);
        o[d4 + c] = make_float4(x.x * e.x, x.y * e.y, x.z * e.z, x.w * e.w);
    }
}

// one warp per row: y = (Y1 + b1) + (Y2 + b2) (:59), z = LeakyReLU_0.2(y), rn = max(||z||_2, 1e-12), N = z / rn (F.normalize :165)
// keep (optional): the mask nn.Dropout(mess_dropout) draws over this layer's [n, d] output (:164), bytes; z *= keep ? scale : 0
__global__ void __launch_bounds__(256) ngcf_act_kernel(const float *__restrict__ Y1, const float *__restrict__ Y2,
                                                       const float *__restrict__ b1, const float *__restrict__ b2, long long n,
                                                       int d, float *__restrict__ Y, float *__restrict__ rn, float *__restrict__ N,
                                                       float *__restrict__ ALL, int C, int coff, const uint8_t *__restrict__ keep,
                                                       float scale)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < n; r += nw) {
        double ss = 0.0;
        for (int o = lane; o < d; o += 32) {
            const float y = (Y1[r * d + o] + b1[o]) + (Y2[r * d + o] + b2[o]);
            float z = y > 0.f ? y : 0.2f * y;
            if (keep) z = z * (keep[r * d + o] ? scale : 0.f);
            Y[r * d + o] = y;
            ss += (double)(z * z);
        }
        ss = warp_sum(ss);
        double nr = sqrt(ss);
        if (nr < 1e-12) nr = 1e-12;
        if (lane == 0) rn[r] = (float)nr;
        for (int o = lane; o < d; o += 32) {
            const float y = Y[r * d + o];
            float z = y > 0.f ? y : 0.2f * y;
            if (keep) z = z * (keep[r * d + o] ? scale : 0.f);
            const float v = (float)((double)z / nr);
            N[r * d + o] = v;
            ALL[r * C + coff + o] = v;
        }
    }
}

// ALL[:, 0:F] = E_0
__global__ void ngcf_copy_block_kernel(const float *__restrict__ E, long long n, int d, float *__restrict__ ALL, int C, int coff)
{
    const long long total = n * d;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / d;
        ALL[r * C + coff + (int)(k - r * d)] = E[k];
    }
}

// one warp per row: dN = G[:, block] (+ dE from the layer above);  dz = (dN - N <N, dN>) / rn  (clamped rows: dN / rn);
// dY = dz * LeakyReLU'(y)
__global__ void __launch_bounds__(256) ngcf_act_bwd_kernel(const float *__restrict__ G, int C, int coff,
                                                           const float *__restrict__ dE, const float *__restrict__ N,
                                                           const float *__restrict__ Y, const float *__restrict__ rn,
                                                           long long n, int d, float *__restrict__ dY,
                                                           const uint8_t *__restrict__ keep, float scale)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < n; r += nw) {
        double dot = 0.0;
        for (int o = lane; o < d; o += 32) {
            const double dn = (double)G[r * C + coff + o] + (dE ? (double)dE[r * d + o] : 0.0);
            dot += dn * (double)N[r * d + o];
        }
        dot = warp_sum(dot);
        const double nr = (double)rn[r];
        for (int o = lane; o < d; o += 32) {
            const double dn = (double)G[r * C + coff + o] + (dE ? (double)dE[r * d + o] : 0.0);
            const double dz = (nr > 1e-12) ? (dn - (double)N[r * d + o] * dot) / nr : dn / nr;
            float dzf = (float)dz;
            if (keep) dzf = dzf * (keep[r * d + o] ? scale : 0.f);        // Dropout backward
            dY[r * d + o] = dzf * (Y[r * d + o] > 0.f ? 1.f : 0.2f);
        }
    }
}

// dEl = dS + dT * X (through E + X and X * E, E side);  dX = dS + dT * E (X side)
__global__ void ngcf_mix_bwd_kernel(const float *__restrict__ dS, const float *__restrict__ dT, const float *__restrict__ E,
                                    const float *__restrict__ X, long long n4, float *__restrict__ dEl, float *__restrict__ dX)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += (long long)gridDim.x * blockDim.x) {
        const float4 s = reinterpret_cast<const float4 *>(dS)[k], t = reinterpret_cast<const float4 *>(dT)[k];
        const float4 e = __ldcg(reinterpret_cast<const float4 *>(E) + k), x = reinterpret_cast<const float4 *>(X)[k];
        reinterpret_cast<float4 *>(dEl)[k] = make_float4(fmaf(t.x, x.x, s.x), fmaf(t.y, x.y, s.y), fmaf(t.z, x.z, s.z), fmaf(t.w, x.w, s.w));
        reinterpret_cast<float4 *>(dX)[k] = make_float4(fmaf(t.x, e.x, s.x), fmaf(t.y, e.y, s.y), fmaf(t.z, e.z, s.z), fmaf(t.w, e.w, s.w));
    }
}

// out = a + b (+ c[:, coff : coff+d] of a [n, C] matrix when c != nullptr)
__global__ void ngcf_add_kernel(const float *a, const float *__restrict__ b, const float *__restrict__ c, int C,
                                int coff, long long n, int d, float *out)   // out may alias a (in-place accumulate)
{
    const long long total = n * d;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        float v = (a ? a[k] : 0.f) + (b ? b[k] : 0.f);
        if (c) { const long long r = k / d; v += c[r * C + coff + (int)(k - r * d)]; }
        out[k] = v;
    }
}

// The regulariser norms of the batch's EGO rows (F wide; the score rows of phase 1 are C wide, so phase 1 runs with the
// regulariser switched off and these six sums are added to its accumulators here): acc[1..3] L1 of (u, i, j) rows,
// acc[4..6] their squared sums.  One warp per triple, fp64 block reduction.
__global__ void __launch_bounds__(256) ngcf_norms_kernel(const float *__restrict__ E0, int U, int F, const int32_t *__restrict__ bu,
                                                         const int32_t *__restrict__ bi, const int32_t *__restrict__ bj,
                                                         long long B, double *__restrict__ acc)
{
    __shared__ double s_acc[6];
    if (threadIdx.x < 6) s_acc[threadIdx.x] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    float l1[3] = {0.f, 0.f, 0.f}, s2[3] = {0.f, 0.f, 0.f};
    for (long long t = warp; t < B; t += nw) {
        const float *rows[3] = {E0 + (size_t)bu[t] * F, E0 + ((size_t)U + bi[t]) * F, E0 + ((size_t)U + bj[t]) * F};
#pragma unroll
        for (int k = 0; k < 3; ++k)
            for (int f = lane; f < F; f += 32) {
                const float v = __ldcg(rows[k] + f);
                l1[k] += fabsf(v);
                s2[k] = fmaf(v, v, s2[k]);
            }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double a = warp_sum((double)l1[k]), b = warp_sum((double)s2[k]);
        if (lane == 0) { atomicAdd(&s_acc[k], a); atomicAdd(&s_acc[3 + k], b); }
    }
    __syncthreads();
    if (threadIdx.x < 6 && s_acc[threadIdx.x] != 0.0) atomicAdd(acc + 1 + threadIdx.x, s_acc[threadIdx.x]);
}

// fp32 loss in the reference's order (NGCFRecommender.py:196-198) from phase 1's accumulators; NaN -> sticky status
__global__ void ngcf_finalize_kernel(WsHeader *hdr, float reg1, float reg2, double *__restrict__ loss_out, long long step)
{
    const double *a = hdr->acc[0];   // bpr, l1u, l1i, l1j, s2u, s2i, s2j
    float loss = (float)a[0];
    loss += reg1 * (((float)a[1] + (float)a[2]) + (float)a[3]);
    loss += reg2 * (((float)sqrt(a[4]) + (float)sqrt(a[5])) + (float)sqrt(a[6]));
    *loss_out = (double)loss;
    if (isnan(loss)) { hdr->status = DRB_ERR_NAN_LOSS; hdr->nan_step = step; }
}

// keep: masks of the L layers concatenated ([n, d[1]], [n, d[2]], ...), or nullptr
static int ngcf_forward(const NgcfDims &q, const NgcfWs &w, const Adj &adj, const float *E0, const float *W, int dtype,
                        cudaStream_t st, const uint8_t *keep = nullptr, float scale = 1.f)
{
    const long long n = q.n;
    ngcf_copy_block_kernel<<<grid_size(n * q.d[0], 256), 256, 0, st>>>(E0, n, q.d[0], w.ALL, q.C, 0);
    DRB_CUDA(cudaGetLastError());
    const float *E = E0;
    for (int l = 0; l < q.L; ++l) {
        const int in = q.d[l], out = q.d[l + 1];
        const float *W1 = W + q.w_off[l], *b1 = W1 + (size_t)in * out, *W2 = b1 + out, *b2 = W2 + (size_t)in * out;
        int rc = launch_spmm(adj, E, w.X[l], nullptr, in, st);
        if (rc != DRB_OK) return rc;
        if (in % 4 == 0) ngcf_mix_kernel<<<grid_size(n * (in / 4), 256), 256, 0, st>>>(E, w.X[l], n, in, w.ST);
        else ngcf_mix_scalar_kernel<<<grid_size(n * in, 256), 256, 0, st>>>(E, w.X[l], n, in, w.ST);
        DRB_CUDA(cudaGetLastError());
        rc = gemm_nt(dtype, n, out, in, w.ST, 2 * in, W1, in, w.Y1, out, st);
        if (rc == DRB_OK) rc = gemm_nt(dtype, n, out, in, w.ST + in, 2 * in, W2, in, w.Y2, out, st);
        if (rc != DRB_OK) return rc;
        ngcf_act_kernel<<<grid_size(n * 32, 256), 256, 0, st>>>(w.Y1, w.Y2, b1, b2, n, out, w.Y[l], w.rn[l], w.E[l + 1], w.ALL,
                                                                q.C, q.off[l + 1], keep, scale);
        DRB_CUDA(cudaGetLastError());
        if (keep) keep += (size_t)n * out;
        E = w.E[l + 1];
    }
    return DRB_OK;
}

}  // namespace drb

using namespace drb;

extern "C" int64_t drb_ngcf_param_count(const int32_t *dims, int32_t L)
{
    NgcfDims q;
    if (!ngcf_dims(q, 1, 1, dims, L)) return -1;
    return q.nW;
}

extern "C" size_t drb_ngcf_workspace_bytes(int32_t U, int32_t I, const int32_t *dims, int32_t L, int32_t opt)
{
    NgcfDims q;
    if (!ngcf_dims(q, U, I, dims, L)) return 0;
    return carve_ngcf(nullptr, q, opt, nullptr);
}

extern "C" int drb_ngcf_workspace_init(void *d_ws, int32_t U, int32_t I, const int32_t *dims, int32_t L, int32_t opt, void *stream)
{
    NgcfDims q;
    DRB_REQUIRE(d_ws && ngcf_dims(q, U, I, dims, L), "ngcf_workspace_init: bad arguments (layer widths 1..256, 1 <= layers <= 8)");
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, carve_ngcf(nullptr, q, opt, nullptr), (cudaStream_t)stream));
    return DRB_OK;
}

// NGCF.forward: d_out [n, C] = cat(E_0 .. E_L, dim=1), with nn.Dropout(mess_dropout) active when d_keep != NULL (:164; the
// reference's module is always in training mode, rank() included).  d_keep: the masks torch draws, one per layer over its
// [n, width] output, as bytes, layers concatenated.
extern "C" int drb_ngcf_forward(const float *d_E0, const float *d_W, void *d_ws, int32_t U, int32_t I, const int32_t *dims,
                                int32_t L, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                                const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, int32_t tower_dtype,
                                const uint8_t *d_keep, float dropout, float *d_out, void *stream)
{
    NgcfDims q;
    DRB_REQUIRE(d_keep == nullptr || (dropout > 0.f && dropout < 1.f), "ngcf: dropout masks need 0 < mess_dropout < 1");
    DRB_REQUIRE(d_E0 && d_W && d_ws && d_row_ptr && d_out && ngcf_dims(q, U, I, dims, L), "ngcf_forward: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    NgcfWs w;
    carve_ngcf(d_ws, q, DRB_OPT_SGD, &w);
    const Adj adj{d_row_ptr, d_col, d_val, d_seg_row, d_seg_ptr, nseg, q.n};
    int rc = ngcf_forward(q, w, adj, d_E0, d_W, tower_dtype, st, d_keep, d_keep ? 1.0f / (float)(1.0 - (double)dropout) : 1.f);
    if (rc != DRB_OK) return rc;
    DRB_CUDA(cudaMemcpyAsync(d_out, w.ALL, sizeof(float) * (size_t)q.n * q.C, cudaMemcpyDeviceToDevice, st));
    return DRB_OK;
}

// n_steps synchronous NGCF + BPR steps (apply != 0) or the loss of one batch (apply == 0), with the message dropout of :164
// active when d_keep != NULL (reference default mess_dropout 0.1).  d_keep: per step the masks of the one forward() a step runs
// (layers concatenated, bytes), steps concatenated.
extern "C" int drb_ngcf_bpr_train_steps(float *d_E0, float *d_W, void *d_ws, int32_t U, int32_t I, const int32_t *dims, int32_t L,
                                        const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                                        const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, const int32_t *d_bu,
                                        const int32_t *d_bi, const int32_t *d_bj, int64_t n_triples, int64_t batch,
                                        int64_t first_step, int64_t n_steps, const drb_hyper *h, int64_t adam_step0,
                                        int32_t apply, int32_t tower_dtype, const uint8_t *d_keep, float dropout,
                                        double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream)
{
    NgcfDims q;
    DRB_REQUIRE(d_keep == nullptr || (dropout > 0.f && dropout < 1.f), "ngcf: dropout masks need 0 < mess_dropout < 1");
    const float drop_scale = d_keep ? 1.0f / (float)(1.0 - (double)dropout) : 1.f;
    DRB_REQUIRE(d_E0 && d_W && d_ws && d_row_ptr && d_bu && d_bi && d_bj && h && d_step_loss, "ngcf_train_steps: null argument");
    DRB_REQUIRE(ngcf_dims(q, U, I, dims, L), "ngcf_train_steps: bad layer widths (1..256, 1 <= layers <= 8)");
    DRB_REQUIRE(batch > 0 && n_steps >= 0 && (n_steps == 0 || (first_step + n_steps - 1) * batch < n_triples),
                "ngcf_train_steps: steps exceed %lld triples", (long long)n_triples);
    DRB_REQUIRE(h->opt == DRB_OPT_SGD || h->opt == DRB_OPT_ADAM, "ngcf: SGD and Adam only (optimizer id %d)", h->opt);
    DRB_REQUIRE(h->loss == DRB_LOSS_BPR, "ngcf: BPR only");
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    NgcfWs w;
    carve_ngcf(d_ws, q, h->opt, &w);
    const Adj adj{d_row_ptr, d_col, d_val, d_seg_row, d_seg_ptr, nseg, q.n};
    const long long n = q.n;
    const int F = q.d[0], C = q.C;
    DRB_CUDA(cudaMemsetAsync(w.hdr, 0, sizeof(WsHeader), st));
    for (int64_t s = 0; s < n_steps; ++s) {
        const int64_t base = (first_step + s) * batch, nb = (n_triples - base < batch) ? n_triples - base : batch;
        size_t keep_per_step = 0;
        for (int l = 0; l < q.L; ++l) keep_per_step += (size_t)n * q.d[l + 1];
        const uint8_t *keep = d_keep ? d_keep + (size_t)s * keep_per_step : nullptr;
        int rc = ngcf_forward(q, w, adj, d_E0, d_W, tower_dtype, st, keep, drop_scale);
        if (rc != DRB_OK) return rc;
        // phase 1: scores on the concatenated representation, norms on the ego rows, G = dL / d(representation)
        StepParams p = split_step(h, U, I, d_bu + base, d_bi + base, d_bj + base, nb, adam_step0 + s, d_step_loss + s);
        p.P = w.ALL; p.Q = w.ALL + (size_t)U * C; p.F = C;
        p.ws.hdr = w.hdr; p.ws.gP = w.G; p.ws.gQ = w.G + (size_t)U * C; p.ws.cntU = w.cntU; p.ws.cntI = w.cntI;
        p.reg1 = 0.f; p.reg2 = 0.f;                      // the ego rows are F wide, the score rows C wide: norms come from ngcf_norms_kernel
        p.dense_grad = 1;
        p.apply = apply ? 1 : 0;
        p.phases = 1;
        if (apply) DRB_CUDA(cudaMemsetAsync(w.G, 0, sizeof(float) * (size_t)n * C, st));
        rc = launch_steps(p, st, true);                  // resets the header accumulators, then accumulates the BPR sum
        if (rc != DRB_OK) return rc;
        if (h->reg_1 != 0.f || h->reg_2 != 0.f) {
            ngcf_norms_kernel<<<grid_size(nb * 32, 256), 256, 0, st>>>(d_E0, U, F, p.bu, p.bi, p.bj, nb, w.hdr->acc[0]);
            DRB_CUDA(cudaGetLastError());
        }
        ngcf_finalize_kernel<<<1, 1, 0, st>>>(w.hdr, h->reg_1, h->reg_2, d_step_loss + s, first_step + s);
        DRB_CUDA(cudaGetLastError());
        if (!apply) break;
        // layers, backwards
        float *dE = nullptr;
        for (int l = q.L - 1; l >= 0; --l) {
            const int in = q.d[l], out = q.d[l + 1];
            const float *El = l == 0 ? d_E0 : w.E[l];
            const float *W1 = d_W + q.w_off[l], *W2 = W1 + (size_t)in * out + out;
            float *gW1 = w.gW + q.w_off[l], *gb1 = gW1 + (size_t)in * out, *gW2 = gb1 + out, *gb2 = gW2 + (size_t)in * out;
            const uint8_t *keep_l = keep;
            if (keep_l) for (int k = 0; k < l; ++k) keep_l += (size_t)n * q.d[k + 1];
            ngcf_act_bwd_kernel<<<grid_size(n * 32, 256), 256, 0, st>>>(w.G, C, q.off[l + 1], dE, w.E[l + 1], w.Y[l], w.rn[l], n, out,
                                                                        w.dY, keep_l, drop_scale);
            DRB_CUDA(cudaGetLastError());
            rc = colsum_acc(w.dY, n, out, gb1, st);
            if (rc == DRB_OK) rc = colsum_acc(w.dY, n, out, gb2, st);
            if (in % 4 == 0) ngcf_mix_kernel<<<grid_size(n * (in / 4), 256), 256, 0, st>>>(El, w.X[l], n, in, w.ST);   // [S | T] again
                                                                                           else ngcf_mix_scalar_kernel<<<grid_size(n * in, 256), 256, 0, st>>>(El, w.X[l], n, in, w.ST);
            DRB_CUDA(cudaGetLastError());
            // gW1 [out, in] += dY^T S,  gW2 += dY^T T
            if (rc == DRB_OK) rc = gemm_tn_acc_t(tower_dtype, in, out, (int)n, w.ST, 2 * in, w.dY, out, gW1, in, st);
            if (rc == DRB_OK) rc = gemm_tn_acc_t(tower_dtype, in, out, (int)n, w.ST + in, 2 * in, w.dY, out, gW2, in, st);
            // dS = dY W1, dT = dY W2
            if (rc == DRB_OK) rc = gemm_nn(tower_dtype, n, in, out, w.dY, out, W1, in, w.dS, in, st);
            if (rc == DRB_OK) rc = gemm_nn(tower_dtype, n, in, out, w.dY, out, W2, in, w.dT, in, st);
            if (rc != DRB_OK) return rc;
            float *dEl = (dE == w.dEa) ? w.dEb : w.dEa;
            if (in % 4 == 0)
                ngcf_mix_bwd_kernel<<<grid_size(n * in / 4, 256), 256, 0, st>>>(w.dS, w.dT, El, w.X[l], n * in / 4, dEl, w.dX);
            else
                ngcf_mix_bwd_scalar_kernel<<<grid_size(n * in, 256), 256, 0, st>>>(w.dS, w.dT, El, w.X[l], n * in, dEl, w.dX);
            DRB_CUDA(cudaGetLastError());
            rc = launch_spmm(adj, w.dX, w.AdX, nullptr, in, st);                                       // A_hat symmetric
            if (rc != DRB_OK) return rc;
            if (l > 0) {
                ngcf_add_kernel<<<grid_size(n * in, 256), 256, 0, st>>>(dEl, w.AdX, nullptr, 0, 0, n, in, dEl);
            } else {   // gradient of the ego table: block 0 of G + the chain through layer 0
                ngcf_add_kernel<<<grid_size(n * in, 256), 256, 0, st>>>(dEl, w.AdX, w.G, C, 0, n, in, w.gE);
            }
            DRB_CUDA(cudaGetLastError());
            dE = dEl;
        }
        // phase 2 on the ego table: dense gradient gE + counter-weighted regulariser, SGD / Adam
        p.P = d_E0; p.Q = d_E0 + (size_t)U * F; p.F = F;
        p.ws.gP = w.gE; p.ws.gQ = w.gE + (size_t)U * F;
        p.ws.mP = w.mE; p.ws.vP = w.vE; p.ws.mQ = w.mE ? w.mE + (size_t)U * F : nullptr; p.ws.vQ = w.vE ? w.vE + (size_t)U * F : nullptr;
        p.reg1 = h->reg_1; p.reg2 = h->reg_2;
        p.step_loss = w.scratch;                           // the real loss was written by ngcf_finalize_kernel
        p.phases = 2;
        rc = launch_steps(p, st, true);
        if (rc == DRB_OK) rc = dense_update(d_W, w.gW, w.mW, w.vW, q.nW, h, adam_step0 + s, w.hdr, st);
        if (rc != DRB_OK) return rc;
    }
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}
