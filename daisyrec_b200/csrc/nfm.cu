// nfm.cu -- NFM + BPR on the B200 path (SURVEY 8(f) rank 4).
//
// Stands behind daisy/model/NFMRecommender.py (dropout = 0; the reference's masks come from torch's RNG):
//   forward   :110-123   e = P[u] * Q[item] -> [BatchNorm1d] -> L x { Linear(F, F) -> [BatchNorm1d] -> relu|sigmoid|tanh }
//                        -> fm = h + (u_bias[u] + i_bias[item] + bias_) broadcast over the F columns (:120) -> pred = <wp, fm>
//   calc_loss :125-151   two forward calls (pos, then neg): every BatchNorm uses the statistics of ITS call (biased variance,
//                        eps 1e-5) and moves its running statistics twice per step (momentum 0.1, unbiased variance);
//                        BPR(sum) + the FM-style regulariser on the factor rows
//   backward + optimizer.step (AbstractRecommender.py:125-126; SGD by default, NFMRecommender.py:51)
//   rank / full_rank / predict :153-209: the same forward under model.eval() (running statistics)
//
// A step on a batch of B triples works on R = 2B rows (pos rows [0,B), neg rows [B,2B)); BatchNorm statistics are taken per
// half.  It is host-sequenced out of the tower GEMM dispatcher (neumf.cu), the MF dense sweep (phase 2 of mf_bpr.cu) for the
// factor tables, and the row / column kernels below.  Parameter block N (flat fp32, module registration order :64-90):
// [gamma0, beta0] (FM_layers' BatchNorm, if batch_norm), per layer W [F,F], b [F], [gamma, beta], then wp [F].
// Running statistics Rs: per BatchNorm mean [F], var [F].  bias = packed [u_bias (U), i_bias (I), bias_].
#include "gemm.cuh"
#include "step.cuh"

namespace drb {

constexpr int kNfmMaxL = 8;
constexpr float kBnEps = 1e-5f;

struct NfmDims {
    int U, I, F, L, bn, act;
    long long o_bn0, oW[kNfmMaxL], oBN[kNfmMaxL], o_wp, nN, nR;
};

static bool nfm_dims(NfmDims &d, int U, int I, int F, int L, int bn, int act)
{
    if (U <= 0 || I <= 0 || F <= 0 || F > 256 || L < 0 || L > kNfmMaxL || act < 0 || act > 2) return false;
    d.U = U; d.I = I; d.F = F; d.L = L; d.bn = bn ? 1 : 0; d.act = act;
    long long o = 0;
    d.o_bn0 = 0;
    if (bn) o += 2 * F;
    for (int l = 0; l < L; ++l) {
        d.oW[l] = o; o += (long long)F * F + F;
        d.oBN[l] = o; if (bn) o += 2 * F;
    }
    d.o_wp = o; o += F;
    d.nN = o;
    d.nR = bn ? (long long)(1 + L) * 2 * F : 0;
    return true;
}

struct NfmWs {
    WsHeader *hdr;
    float *gP, *gQ, *gB, *gN;                 // gradient accumulators: tables, packed bias, parameter block
    unsigned *cntU;
    unsigned long long *cntI;
    float *mP, *vP, *mQ, *vQ, *mB, *vB, *mN, *vN;
    double *stats;                            // [2 halves][4][F] column sums scratch of the BatchNorm kernels
    float *bnm;                               // per BatchNorm and half: mean [F], inv_std [F]   ((1+L) x 2 x 2F)
    float *pred, *coef;                       // [R]
    float *e, *xh0, *h0;                      // [R,F] product, BN0 xhat, FM_layers output
    float *zpre[kNfmMaxL], *xh[kNfmMaxL], *z[kNfmMaxL], *h[kNfmMaxL];
    float *fm, *dh, *tmp;
    double *scratch;
};

static size_t carve_nfm(void *base, const NfmDims &d, int opt, long long max_rows, NfmWs *w)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align256(bytes);
        return p;
    };
    NfmWs t;
    const size_t F = (size_t)d.F, nb = (size_t)d.U + d.I + 1, act = sizeof(float) * (size_t)max_rows * F;
    t.hdr = (WsHeader *)take(256);
    t.gP = (float *)take(sizeof(float) * d.U * F); t.gQ = (float *)take(sizeof(float) * d.I * F);
    t.gB = (float *)take(sizeof(float) * nb); t.gN = (float *)take(sizeof(float) * (size_t)d.nN);
    t.cntU = (unsigned *)take(sizeof(unsigned) * (size_t)d.U);
    t.cntI = (unsigned long long *)take(sizeof(unsigned long long) * (size_t)d.I);
    t.mP = t.vP = t.mQ = t.vQ = t.mB = t.vB = t.mN = t.vN = nullptr;
    if (opt == DRB_OPT_ADAM) {
        t.mP = (float *)take(sizeof(float) * d.U * F); t.vP = (float *)take(sizeof(float) * d.U * F);
        t.mQ = (float *)take(sizeof(float) * d.I * F); t.vQ = (float *)take(sizeof(float) * d.I * F);
        t.mB = (float *)take(sizeof(float) * nb); t.vB = (float *)take(sizeof(float) * nb);
        t.mN = (float *)take(sizeof(float) * (size_t)d.nN); t.vN = (float *)take(sizeof(float) * (size_t)d.nN);
    }
    t.stats = (double *)take(sizeof(double) * 2 * 4 * F);
    t.bnm = (float *)take(sizeof(float) * (size_t)(1 + d.L) * 2 * 2 * F);
    t.scratch = (double *)take(sizeof(double) * 8);
    size_t head = off;                        // everything above is zeroed by workspace_init
    t.pred = (float *)take(sizeof(float) * (size_t)max_rows); t.coef = (float *)take(sizeof(float) * (size_t)max_rows);
    t.e = (float *)take(act); t.xh0 = (float *)take(act); t.h0 = (float *)take(act);
    for (int l = 0; l < kNfmMaxL; ++l) {
        if (l < d.L) {
            t.zpre[l] = (float *)take(act); t.xh[l] = (float *)take(act); t.z[l] = (float *)take(act); t.h[l] = (float *)take(act);
        } else {
            t.zpre[l] = t.xh[l] = t.z[l] = t.h[l] = nullptr;
        }
    }
    t.fm = (float *)take(act); t.dh = (float *)take(act); t.tmp = (float *)take(act);
    if (w) { *w = t; w->scratch = t.scratch; }
    (void)head;
    return off;
}

static size_t nfm_head_bytes(const NfmDims &d, int opt)
{
    NfmWs w;
    carve_nfm((void *)(uintptr_t)256, d, opt, 1, &w);
    return (size_t)((uintptr_t)w.pred - 256);
}

__device__ __forceinline__ float nfm_act(int act, float z)
{
    if (act == 0) return z > 0.f ? z : 0.f;
    if (act == 1) return 1.f / (1.f + expf(-z));
    return tanhf(z);
}
__device__ __forceinline__ float nfm_act_grad(int act, float z, float h)
{
    if (act == 0) return z > 0.f ? 1.f : 0.f;
    if (act == 1) return h * (1.f - h);
    return 1.f - h * h;
}

// e[r, :] = P[u_r] * Q[item_r]; training rows [0,B) use bi, [B,2B) use bj (users / items given explicitly for inference)
__global__ void nfm_product_kernel(const float *__restrict__ P, const float *__restrict__ Q, const int32_t *__restrict__ bu,
                                   const int32_t *__restrict__ bi, const int32_t *__restrict__ bj, long long B, long long R, int F,
                                   float *__restrict__ e)
{
    const long long total = R * F;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / F;
        const int f = (int)(k - r * F);
        const long long t = r < B ? r : r - B;
        const int item = r < B ? bi[t] : bj[t];
        e[k] = __ldcg(P + (size_t)bu[t] * F + f) * __ldcg(Q + (size_t)item * F + f);
    }
}

// column sums over the rows of each half: out[half][0][f] = sum x, [1] = sum (x - mean)^2 when `mean` is given (second pass)
// grid.y = half; each CTA reduces a slab of rows into shared memory, then one fp64 atomic per column
__global__ void __launch_bounds__(256) nfm_colstat_kernel(const float *__restrict__ x, const float *__restrict__ y, long long B,
                                                          int F, const float *__restrict__ mean2F, int mode,
                                                          double *__restrict__ out)
{
    // mode 0: out[h][0] += sum x                      mode 1: out[h][1] += sum (x - mean)^2
    // mode 2: out[h][2] += sum x * 1 (dy), out[h][3] += sum x * y (dy * xhat)   (BatchNorm backward)
    __shared__ double s_a[256], s_b[256];
    const int half = blockIdx.y;
    const int tn = threadIdx.x % F, tr = threadIdx.x / F, rows_per_pass = 256 / F > 0 ? 256 / F : 1;
    double a = 0.0, b = 0.0;
    if (tr < rows_per_pass && threadIdx.x < rows_per_pass * F) {
        const float m = mode == 1 ? mean2F[half * 2 * F + tn] : 0.f;
        for (long long r = (long long)blockIdx.x * rows_per_pass + tr; r < B; r += (long long)gridDim.x * rows_per_pass) {
            const long long k = (half * B + r) * F + tn;
            const float v = x[k];
            if (mode == 0) a += (double)v;
            else if (mode == 1) { const double dd = (double)v - (double)m; a += dd * dd; }
            else { a += (double)v; b += (double)v * (double)y[k]; }
        }
    }
    s_a[threadIdx.x] = a; s_b[threadIdx.x] = b;
    __syncthreads();
    if (threadIdx.x < F) {
        double ta = 0.0, tb = 0.0;
        for (int q = 0; q < rows_per_pass; ++q) { ta += s_a[q * F + threadIdx.x]; tb += s_b[q * F + threadIdx.x]; }
        double *o = out + (size_t)half * 4 * F;
        if (mode == 0) atomicAdd(o + threadIdx.x, ta);
        else if (mode == 1) atomicAdd(o + F + threadIdx.x, ta);
        else { atomicAdd(o + 2 * F + threadIdx.x, ta); atomicAdd(o + 3 * F + threadIdx.x, tb); }
    }
}

// after pass 0: mean[half][f] (fp32, as the reference rounds it);  after pass 1: inv_std + the running statistics
__global__ void nfm_bn_finish_kernel(const double *__restrict__ stats, long long B, int F, int pass, float *__restrict__ bnm,
                                     float *__restrict__ rm, float *__restrict__ rv)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    if (pass == 0) {
        for (int h = 0; h < 2; ++h) bnm[h * 2 * F + f] = (float)(stats[(size_t)h * 4 * F + f] / (double)B);
    } else {
        float m_run = rm[f], v_run = rv[f];
        for (int h = 0; h < 2; ++h) {                      // the pos call updates the running statistics first, then the neg call
            const double ss = stats[(size_t)h * 4 * F + F + f];
            const float mean = bnm[h * 2 * F + f];
            const float var = (float)(ss / (double)B);
            const float unbiased = B > 1 ? (float)(ss / (double)(B - 1)) : var;
            m_run = (1.f - 0.1f) * m_run + 0.1f * mean;
            v_run = (1.f - 0.1f) * v_run + 0.1f * unbiased;
            bnm[h * 2 * F + F + f] = 1.f / sqrtf(var + kBnEps);
        }
        rm[f] = m_run; rv[f] = v_run;
    }
}

// y = (x - mean) * inv_std * gamma + beta, xhat kept for the backward pass (train: per-half statistics; eval: running ones)
__global__ void nfm_bn_apply_kernel(const float *__restrict__ x, long long B, long long R, int F, const float *__restrict__ bnm,
                                    const float *__restrict__ rm, const float *__restrict__ rv, const float *__restrict__ gamma,
                                    const float *__restrict__ beta, int train, float *__restrict__ xhat, float *__restrict__ y)
{
    const long long total = R * F;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / F;
        const int f = (int)(k - r * F);
        float mean, is;
        if (train) {
            const int h = r < B ? 0 : 1;
            mean = bnm[h * 2 * F + f];
            is = bnm[h * 2 * F + F + f];
        } else {
            mean = rm[f];
            is = 1.f / sqrtf(rv[f] + kBnEps);
        }
        const float xh = (x[k] - mean) * is;
        if (xhat) xhat[k] = xh;
        y[k] = xh * gamma[f] + beta[f];
    }
}

// zpre += b (Linear bias), in place; without BatchNorm also z = zpre
__global__ void nfm_bias_kernel(float *__restrict__ zpre, const float *__restrict__ b, long long total, int F, float *__restrict__ z)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const float v = zpre[k] + b[(int)(k % F)];
        zpre[k] = v;
        if (z) z[k] = v;
    }
}

__global__ void nfm_act_kernel(const float *__restrict__ z, long long total, int act, float *__restrict__ h)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x)
        h[k] = nfm_act(act, z[k]);
}

// nn.Dropout with the caller's masks (NFMRecommender.py:67,:88): x *= keep ? 1/(1-p) : 0, in place.  keep is laid out as torch
// drew it: [forward call (pos, neg)][site][B][F] bytes; rows [0,B) belong to the positive call, [B,2B) to the negative one.
__device__ __forceinline__ float nfm_keep_factor(const uint8_t *__restrict__ keep, long long k, long long B, int F, int site,
                                                 int nsites, float scale)
{
    const long long r = k / F;
    const int f = (int)(k - r * F);
    const long long pass = r >= B ? 1 : 0, t = r - pass * B;
    return keep[((pass * nsites + site) * B + t) * F + f] ? scale : 0.f;
}
__global__ void nfm_dropout_kernel(float *__restrict__ x, const uint8_t *__restrict__ keep, long long B, long long total, int F,
                                   int site, int nsites, float scale)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x)
        x[k] = x[k] * nfm_keep_factor(keep, k, B, F, site, nsites, scale);
}

// one warp per row: fm = h + ((u_bias + i_bias) + bias_), pred = <fm, wp>   (rows given by (bu, bi|bj) or by explicit pairs)
__global__ void __launch_bounds__(256) nfm_head_kernel(const float *__restrict__ hin, const float *__restrict__ bias, int U, int I,
                                                       const int32_t *__restrict__ bu, const int32_t *__restrict__ bi,
                                                       const int32_t *__restrict__ bj, long long B, long long R, int F,
                                                       const float *__restrict__ wp, float *__restrict__ fm, float *__restrict__ pred)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < R; r += nw) {
        const long long t = r < B ? r : r - B;
        const int item = r < B ? bi[t] : bj[t];
        const float bsum = (bias[bu[t]] + bias[U + item]) + bias[U + I];          // :120
        double acc = 0.0;
        for (int f = lane; f < F; f += 32) {
            const float v = hin[r * F + f] + bsum;
            if (fm) fm[r * F + f] = v;
            acc += (double)(v * wp[f]);
        }
        acc = warp_sum(acc);
        if (lane == 0) pred[r] = (float)acc;
    }
}

// per triple: BPR coefficient for both rows, loss, factor-row norms, row counters
__global__ void __launch_bounds__(256) nfm_pair_kernel(const float *__restrict__ pred, const float *__restrict__ P,
                                                       const float *__restrict__ Q, const int32_t *__restrict__ bu,
                                                       const int32_t *__restrict__ bi, const int32_t *__restrict__ bj, long long B,
                                                       int F, int has_reg, int apply, float *__restrict__ coef,
                                                       unsigned *__restrict__ cntU, unsigned long long *__restrict__ cntI,
                                                       double *__restrict__ acc)
{
    __shared__ double s_acc[7];
    if (threadIdx.x < 7) s_acc[threadIdx.x] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    float loss = 0.f, l1[3] = {0.f, 0.f, 0.f}, s2[3] = {0.f, 0.f, 0.f};
    for (long long t = warp; t < B; t += nw) {
        const float x = pred[t] - pred[B + t];
        const float sg = 1.f / (1.f + expf(-x));
        const float c = -(sg * (1.f - sg)) / (1e-10f + sg);
        if (lane == 0) {
            loss += -logf(1e-10f + sg);
            coef[t] = c;
            coef[B + t] = -c;
            if (apply) {
                red_add_u32(cntU + bu[t], 1u);
                red_add_u64(cntI + bi[t], 1ull);
                red_add_u64(cntI + bj[t], 1ull << 32);
            }
        }
        if (has_reg) {
            const float *rows[3] = {P + (size_t)bu[t] * F, Q + (size_t)bi[t] * F, Q + (size_t)bj[t] * F};
#pragma unroll
            for (int k = 0; k < 3; ++k)
                for (int f = lane; f < F; f += 32) {
                    const float v = __ldcg(rows[k] + f);
                    l1[k] += fabsf(v);
                    s2[k] = fmaf(v, v, s2[k]);
                }
        }
    }
    double a = warp_sum((double)loss);
    if (lane == 0) atomicAdd(&s_acc[0], a);
    if (has_reg) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double u1 = warp_sum((double)l1[k]), u2 = warp_sum((double)s2[k]);
            if (lane == 0) { atomicAdd(&s_acc[1 + k], u1); atomicAdd(&s_acc[4 + k], u2); }
        }
    }
    __syncthreads();
    if (threadIdx.x < 7 && s_acc[threadIdx.x] != 0.0) atomicAdd(acc + threadIdx.x, s_acc[threadIdx.x]);
}

// loss in the reference's order (:141-149) from acc = {bpr, l1u, l1i, l1j, s2u, s2i, s2j}; NaN -> sticky status
__global__ void nfm_finalize_kernel(WsHeader *hdr, float reg1, float reg2, double *__restrict__ loss_out, long long step)
{
    const double *a = hdr->acc[0];
    float loss = (float)a[0];
    loss += reg1 * ((float)a[2] + (float)a[3]);
    loss += reg2 * ((float)sqrt(a[5]) + (float)sqrt(a[6]));
    loss += reg1 * (float)a[1];
    loss += reg2 * (float)sqrt(a[4]);
    *loss_out = (double)loss;
    if (isnan(loss)) { hdr->status = DRB_ERR_NAN_LOSS; hdr->nan_step = step; }
}

// One warp per TRIPLE (its pos row t and neg row B + t): dh = dpred * wp;  gwp += sum dpred * fm;  first-order terms:
// gbias[U + i] += bs_pos, gbias[U + j] += bs_neg, and the user / global terms take bs_pos + bs_neg of the SAME triple -- for BPR
// dpred_neg = -dpred_pos, so that sum is exactly 0, as it is in the reference (its two embedding backward passes add the same
// numbers with opposite signs in the same order); adding the halves separately would leave cancellation noise that Adam
// turns into +-lr steps.
__global__ void __launch_bounds__(256) nfm_head_bwd_kernel(const float *__restrict__ coef, const float *__restrict__ fm,
                                                           const float *__restrict__ wp, int U, int I,
                                                           const int32_t *__restrict__ bu, const int32_t *__restrict__ bi,
                                                           const int32_t *__restrict__ bj, long long B, long long R, int F,
                                                           float *__restrict__ dh, float *__restrict__ gwp, float *__restrict__ gB)
{
    extern __shared__ float s_gwp[];
    for (int k = threadIdx.x; k < F; k += blockDim.x) s_gwp[k] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    float b0 = 0.f;
    for (long long t = warp; t < B; t += nw) {
        const float dp = coef[t], dn = coef[B + t];
        float bsp = 0.f, bsn = 0.f;
        for (int f = lane; f < F; f += 32) {
            const float w = wp[f];
            const float d1 = dp * w, d2 = dn * w;
            dh[t * F + f] = d1;
            dh[(B + t) * F + f] = d2;
            bsp += d1;
            bsn += d2;
            atomicAdd(&s_gwp[f], dp * fm[t * F + f] + dn * fm[(B + t) * F + f]);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            bsp += __shfl_xor_sync(0xffffffffu, bsp, off);
            bsn += __shfl_xor_sync(0xffffffffu, bsn, off);
        }
        if (lane == 0) {
            const float both = bsp + bsn;
            if (both != 0.f) atomicAdd(gB + bu[t], both);
            atomicAdd(gB + U + bi[t], bsp);
            atomicAdd(gB + U + bj[t], bsn);
            b0 += both;
        }
    }
    if (lane == 0 && b0 != 0.f) atomicAdd(gB + U + I, b0);
    __syncthreads();
    for (int k = threadIdx.x; k < F; k += blockDim.x)
        if (s_gwp[k] != 0.f) atomicAdd(gwp + k, s_gwp[k]);
    (void)R;
}

// tmp = dh * act'(z, h)
__global__ void nfm_act_bwd_kernel(const float *__restrict__ dh, const float *__restrict__ z, const float *__restrict__ h,
                                   long long total, int act, float *__restrict__ out)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x)
        out[k] = dh[k] * nfm_act_grad(act, z[k], h[k]);
}
// the same behind a Dropout: tmp = (dh * keep factor) * act'(z, act(z))  (h holds the dropped activations, so act(z) is redone)
__global__ void nfm_act_bwd_drop_kernel(const float *__restrict__ dh, const float *__restrict__ z, const uint8_t *__restrict__ keep,
                                        long long B, long long total, int F, int site, int nsites, float scale, int act,
                                        float *__restrict__ out)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const float zz = z[k];
        out[k] = (dh[k] * nfm_keep_factor(keep, k, B, F, site, nsites, scale)) * nfm_act_grad(act, zz, nfm_act(act, zz));
    }
}

// BatchNorm backward (per half): dx = inv_std / B * (B dxh - sum(dxh) - xhat sum(dxh xhat)), dxh = dy gamma;
// dgamma += sum dy xhat, dbeta += sum dy (both halves).  stats[h][2] = sum dy, [3] = sum dy xhat.
__global__ void nfm_bn_bwd_kernel(const float *__restrict__ dy, const float *__restrict__ xhat, const double *__restrict__ stats,
                                  const float *__restrict__ bnm, const float *__restrict__ gamma, long long B, long long R, int F,
                                  float *__restrict__ dx)
{
    const long long total = R * F;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / F;
        const int f = (int)(k - r * F);
        const int h = r < B ? 0 : 1;
        const double g = (double)gamma[f];
        const double s1 = stats[(size_t)h * 4 * F + 2 * F + f] * g, s2 = stats[(size_t)h * 4 * F + 3 * F + f] * g;
        const double dxh = (double)dy[k] * g;
        dx[k] = (float)((double)bnm[h * 2 * F + F + f] / (double)B * ((double)B * dxh - s1 - (double)xhat[k] * s2));
    }
}
__global__ void nfm_bn_param_grad_kernel(const double *__restrict__ stats, int F, float *__restrict__ ggamma, float *__restrict__ gbeta)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    ggamma[f] += (float)(stats[3 * F + f] + stats[(size_t)4 * F + 3 * F + f]);
    gbeta[f] += (float)(stats[2 * F + f] + stats[(size_t)4 * F + 2 * F + f]);
}

// gP[u] += dh * Q[item], gQ[item] += dh * P[u]
__global__ void nfm_scatter_kernel(const float *__restrict__ dh, const float *__restrict__ P, const float *__restrict__ Q,
                                   const int32_t *__restrict__ bu, const int32_t *__restrict__ bi, const int32_t *__restrict__ bj,
                                   long long B, long long R, int F, float *__restrict__ gP, float *__restrict__ gQ)
{
    const long long total = R * F;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long r = k / F;
        const int f = (int)(k - r * F);
        const long long t = r < B ? r : r - B;
        const int u = bu[t], item = r < B ? bi[t] : bj[t];
        const float d = dh[k];
        atomicAdd(gP + (size_t)u * F + f, d * __ldcg(Q + (size_t)item * F + f));
        atomicAdd(gQ + (size_t)item * F + f, d * __ldcg(P + (size_t)u * F + f));
    }
}

// BatchNorm over the rows of x (two halves of B rows); statistics into w.bnm[slot], running statistics updated
static int nfm_bn_train(const NfmDims &d, const NfmWs &w, int slot, const float *x, long long B, const float *gamma,
                        const float *beta, float *rm, float *rv, float *xhat, float *y, cudaStream_t st)
{
    const int F = d.F;
    float *bnm = w.bnm + (size_t)slot * 4 * F;
    DRB_CUDA(cudaMemsetAsync(w.stats, 0, sizeof(double) * 8 * F, st));
    const int rows_per_pass = 256 / F > 0 ? 256 / F : 1;
    long long blocks = (B + rows_per_pass * 8 - 1) / (rows_per_pass * 8), cap = (long long)sm_count() * 4;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    dim3 grid((unsigned)blocks, 2);
    nfm_colstat_kernel<<<grid, 256, 0, st>>>(x, nullptr, B, F, nullptr, 0, w.stats);
    nfm_bn_finish_kernel<<<(F + 63) / 64, 64, 0, st>>>(w.stats, B, F, 0, bnm, rm, rv);
    nfm_colstat_kernel<<<grid, 256, 0, st>>>(x, nullptr, B, F, bnm, 1, w.stats);
    nfm_bn_finish_kernel<<<(F + 63) / 64, 64, 0, st>>>(w.stats, B, F, 1, bnm, rm, rv);
    nfm_bn_apply_kernel<<<grid_size(2 * B * F, 256), 256, 0, st>>>(x, B, 2 * B, F, bnm, rm, rv, gamma, beta, 1, xhat, y);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

static int nfm_bn_backward(const NfmDims &d, const NfmWs &w, int slot, const float *dy, const float *xhat, long long B,
                           const float *gamma, float *ggamma, float *gbeta, float *dx, cudaStream_t st)
{
    const int F = d.F;
    const float *bnm = w.bnm + (size_t)slot * 4 * F;
    DRB_CUDA(cudaMemsetAsync(w.stats, 0, sizeof(double) * 8 * F, st));
    const int rows_per_pass = 256 / F > 0 ? 256 / F : 1;
    long long blocks = (B + rows_per_pass * 8 - 1) / (rows_per_pass * 8), cap = (long long)sm_count() * 4;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    dim3 grid((unsigned)blocks, 2);
    nfm_colstat_kernel<<<grid, 256, 0, st>>>(dy, xhat, B, F, nullptr, 2, w.stats);
    nfm_bn_param_grad_kernel<<<(F + 63) / 64, 64, 0, st>>>(w.stats, F, ggamma, gbeta);
    nfm_bn_bwd_kernel<<<grid_size(2 * B * F, 256), 256, 0, st>>>(dy, xhat, w.stats, bnm, gamma, B, 2 * B, F, dx);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

}  // namespace drb

using namespace drb;

extern "C" int64_t drb_nfm_param_count(int32_t F, int32_t L, int32_t batch_norm)
{
    NfmDims d;
    if (!nfm_dims(d, 1, 1, F, L, batch_norm, 0)) return -1;
    return d.nN;
}

extern "C" size_t drb_nfm_workspace_bytes(int32_t U, int32_t I, int32_t F, int32_t L, int32_t batch_norm, int32_t opt,
                                          int64_t max_rows)
{
    NfmDims d;
    if (!nfm_dims(d, U, I, F, L, batch_norm, 0) || max_rows < 2) return 0;
    return carve_nfm(nullptr, d, opt, max_rows, nullptr);
}

extern "C" int drb_nfm_workspace_init(void *d_ws, int32_t U, int32_t I, int32_t F, int32_t L, int32_t batch_norm, int32_t opt,
                                      int64_t max_rows, void *stream)
{
    NfmDims d;
    DRB_REQUIRE(d_ws && nfm_dims(d, U, I, F, L, batch_norm, 0) && max_rows >= 2, "nfm_workspace_init: bad arguments");
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, nfm_head_bytes(d, opt), (cudaStream_t)stream));
    return DRB_OK;
}

// n_steps synchronous NFM + BPR steps (apply != 0) or the loss of one batch (apply == 0: like calc_loss under train(), the
// BatchNorm running statistics still move).  act: 0 relu, 1 sigmoid, 2 tanh.
// With d_keep != NULL nn.Dropout is active (dropout = config['dropout'] > 0, the reference default 0.5).  d_keep: the masks
// torch's Dropout modules draw, as bytes (0 / 1), for the n_steps steps in order: per step [forward call: pos, neg][site:
// FM_layers' Dropout, then the one behind each activation][batch][F] (the caller draws them on torch's CPU generator in exactly
// that order; a ragged last batch uses its own row count).  Every step must hold `batch` triples when n_steps > 1.
extern "C" int drb_nfm_bpr_train_steps(float *d_P, float *d_Q, float *d_bias, float *d_N, float *d_Rs, void *d_ws, int32_t U,
                                       int32_t I, int32_t F, int32_t L, int32_t batch_norm, int32_t act, int64_t max_rows,
                                       const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch,
                                       int64_t first_step, int64_t n_steps, const drb_hyper *h, int64_t adam_step0, int32_t apply,
                                       int32_t tower_dtype, const uint8_t *d_keep, float dropout, double *d_step_loss,
                                       int32_t sync_and_check, int64_t *nan_step, void *stream)
{
    NfmDims d;
    DRB_REQUIRE(d_keep == nullptr || (dropout > 0.f && dropout < 1.f), "nfm: dropout masks need 0 < dropout < 1");
    DRB_REQUIRE(d_keep == nullptr || n_steps <= 1 || (first_step + n_steps) * batch <= n,
                "nfm: with dropout masks every step of a multi-step call must be a full batch");
    const int nsites = 1 + L;
    const float drop_scale = d_keep ? 1.0f / (float)(1.0 - (double)dropout) : 1.f;
    DRB_REQUIRE(d_P && d_Q && d_bias && d_N && d_ws && d_bu && d_bi && d_bj && h && d_step_loss, "nfm_train_steps: null argument");
    DRB_REQUIRE(nfm_dims(d, U, I, F, L, batch_norm, act), "nfm_train_steps: bad dims (factors <= 256, 0 <= num_layers <= 8, act 0..2)");
    DRB_REQUIRE(!batch_norm || d_Rs, "nfm_train_steps: batch_norm needs the running-statistics block");
    DRB_REQUIRE(batch > 0 && 2 * batch <= max_rows, "nfm: batch %lld needs 2*batch <= max_rows=%lld", (long long)batch, (long long)max_rows);
    DRB_REQUIRE(n_steps == 0 || (first_step + n_steps - 1) * batch < n, "nfm: steps exceed %lld triples", (long long)n);
    DRB_REQUIRE(h->opt == DRB_OPT_SGD || h->opt == DRB_OPT_ADAM, "nfm: SGD and Adam only (optimizer id %d)", h->opt);
    DRB_REQUIRE(h->loss == DRB_LOSS_BPR, "nfm: BPR only");
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    NfmWs w;
    carve_nfm(d_ws, d, h->opt, max_rows, &w);
    const int has_reg = (h->reg_1 != 0.f) || (h->reg_2 != 0.f);
    const float *wp = d_N + d.o_wp;
    DRB_CUDA(cudaMemsetAsync(w.hdr, 0, sizeof(WsHeader), st));
    for (int64_t s = 0; s < n_steps; ++s) {
        const int64_t base = (first_step + s) * batch, B = (n - base < batch) ? n - base : batch;
        const long long R = 2 * B, tot = R * F;
        const int32_t *bu = d_bu + base, *bi = d_bi + base, *bj = d_bj + base;
        const uint8_t *keep = d_keep ? d_keep + (size_t)s * 2 * nsites * (size_t)batch * F : nullptr;   // this step's masks
        int rc = DRB_OK;
        // ---- forward (both calls at once; BatchNorm statistics per half)
        nfm_product_kernel<<<grid_size(tot, 256), 256, 0, st>>>(d_P, d_Q, bu, bi, bj, B, R, F, w.e);
        DRB_CUDA(cudaGetLastError());
        float *h_fm = w.e;                                                // output of FM_layers
        if (d.bn) {
            rc = nfm_bn_train(d, w, 0, w.e, B, d_N + d.o_bn0, d_N + d.o_bn0 + F, d_Rs, d_Rs + F, w.xh0, w.h0, st);
            if (rc != DRB_OK) return rc;
            h_fm = w.h0;
        }
        if (keep) {
            nfm_dropout_kernel<<<grid_size(tot, 256), 256, 0, st>>>(h_fm, keep, B, tot, F, 0, nsites, drop_scale);
            DRB_CUDA(cudaGetLastError());
        }
        const float *hin = h_fm;
        for (int l = 0; l < L; ++l) {
            const float *W = d_N + d.oW[l], *b = W + (size_t)F * F;
            rc = gemm_nt(tower_dtype, R, F, F, hin, F, W, F, w.zpre[l], F, st);
            if (rc != DRB_OK) return rc;
            nfm_bias_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.zpre[l], b, tot, F, d.bn ? nullptr : w.z[l]);
            DRB_CUDA(cudaGetLastError());
            if (d.bn) {
                rc = nfm_bn_train(d, w, 1 + l, w.zpre[l], B, d_N + d.oBN[l], d_N + d.oBN[l] + F, d_Rs + (size_t)(1 + l) * 2 * F,
                                  d_Rs + (size_t)(1 + l) * 2 * F + F, w.xh[l], w.z[l], st);
                if (rc != DRB_OK) return rc;
            }
            nfm_act_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.z[l], tot, d.act, w.h[l]);
            DRB_CUDA(cudaGetLastError());
            if (keep) {
                nfm_dropout_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.h[l], keep, B, tot, F, 1 + l, nsites, drop_scale);
                DRB_CUDA(cudaGetLastError());
            }
            hin = w.h[l];
        }
        nfm_head_kernel<<<grid_size(R * 32, 256), 256, 0, st>>>(hin, d_bias, U, I, bu, bi, bj, B, R, F, wp, w.fm, w.pred);
        DRB_CUDA(cudaMemsetAsync(w.hdr, 0, kHdrResetBytes, st));
        nfm_pair_kernel<<<grid_size(B * 32, 256), 256, 0, st>>>(w.pred, d_P, d_Q, bu, bi, bj, B, F, has_reg, apply ? 1 : 0, w.coef,
                                                                w.cntU, w.cntI, w.hdr->acc[0]);
        nfm_finalize_kernel<<<1, 1, 0, st>>>(w.hdr, h->reg_1, h->reg_2, d_step_loss + s, first_step + s);
        DRB_CUDA(cudaGetLastError());
        if (!apply) break;
        // ---- backward
        nfm_head_bwd_kernel<<<grid_size(B * 32, 256), 256, sizeof(float) * F, st>>>(w.coef, w.fm, wp, U, I, bu, bi, bj, B, R, F, w.dh,
                                                                                    w.gN + d.o_wp, w.gB);
        DRB_CUDA(cudaGetLastError());
        for (int l = L - 1; l >= 0; --l) {
            const float *W = d_N + d.oW[l];
            const float *hprev = l == 0 ? (d.bn ? w.h0 : w.e) : w.h[l - 1];
            float *gW = w.gN + d.oW[l], *gb = gW + (size_t)F * F;
            if (keep)
                nfm_act_bwd_drop_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.dh, w.z[l], keep, B, tot, F, 1 + l, nsites, drop_scale,
                                                                             d.act, w.tmp);
            else
                nfm_act_bwd_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.dh, w.z[l], w.h[l], tot, d.act, w.tmp);   // d act input
                                                                        DRB_CUDA(cudaGetLastError());
            float *dz = w.tmp;                                            // d Linear output
            if (d.bn) {
                rc = nfm_bn_backward(d, w, 1 + l, w.tmp, w.xh[l], B, d_N + d.oBN[l], w.gN + d.oBN[l], w.gN + d.oBN[l] + F, w.dh, st);
                if (rc != DRB_OK) return rc;
                dz = w.dh;
            }
            rc = colsum_acc(dz, R, F, gb, st);
            if (rc == DRB_OK) rc = gemm_tn_acc_t(tower_dtype, F, F, (int)R, hprev, F, dz, F, gW, F, st);   // gW [out,in] += dz^T h_in
            float *dprev = dz == w.tmp ? w.dh : w.tmp;
            if (rc == DRB_OK) rc = gemm_nn(tower_dtype, R, F, F, dz, F, W, F, dprev, F, st);               // d h_in = dz W
            if (rc != DRB_OK) return rc;
            if (dprev != w.dh) DRB_CUDA(cudaMemcpyAsync(w.dh, dprev, sizeof(float) * (size_t)tot, cudaMemcpyDeviceToDevice, st));
        }
        if (keep) {                                                       // backward of FM_layers' Dropout
            nfm_dropout_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.dh, keep, B, tot, F, 0, nsites, drop_scale);
            DRB_CUDA(cudaGetLastError());
        }
        if (d.bn) {
            rc = nfm_bn_backward(d, w, 0, w.dh, w.xh0, B, d_N + d.o_bn0, w.gN + d.o_bn0, w.gN + d.o_bn0 + F, w.tmp, st);
            if (rc != DRB_OK) return rc;
            DRB_CUDA(cudaMemcpyAsync(w.dh, w.tmp, sizeof(float) * (size_t)tot, cudaMemcpyDeviceToDevice, st));
        }
        nfm_scatter_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.dh, d_P, d_Q, bu, bi, bj, B, R, F, w.gP, w.gQ);
        DRB_CUDA(cudaGetLastError());
        // ---- update: factor tables through the MF dense sweep (counter-weighted regulariser), the rest densely
        StepParams p = split_step(h, U, I, bu, bi, bj, B, adam_step0 + s, w.scratch);
        p.P = d_P; p.Q = d_Q; p.F = F;
        p.ws.hdr = w.hdr; p.ws.gP = w.gP; p.ws.gQ = w.gQ; p.ws.cntU = w.cntU; p.ws.cntI = w.cntI;
        p.ws.mP = w.mP; p.ws.vP = w.vP; p.ws.mQ = w.mQ; p.ws.vQ = w.vQ;
        p.phases = 2;
        rc = launch_steps(p, st, true);
        if (rc == DRB_OK) rc = dense_update(d_bias, w.gB, w.mB, w.vB, (long long)U + I + 1, h, adam_step0 + s, w.hdr, st);
        if (rc == DRB_OK) rc = dense_update(d_N, w.gN, w.mN, w.vN, d.nN, h, adam_step0 + s, w.hdr, st);
        if (rc != DRB_OK) return rc;
    }
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

// eval-mode scores of (d_u[k], d_i[k]) pairs: forward() under model.eval() (rank / full_rank / predict, :153-209)
extern "C" int drb_nfm_scores(const float *d_P, const float *d_Q, const float *d_bias, const float *d_N, const float *d_Rs,
                              void *d_ws, int32_t U, int32_t I, int32_t F, int32_t L, int32_t batch_norm, int32_t act, int32_t opt,
                              int64_t max_rows, const int32_t *d_u, const int32_t *d_i, int64_t n, int32_t tower_dtype,
                              float *d_scores, void *stream)
{
    NfmDims d;
    DRB_REQUIRE(d_P && d_Q && d_bias && d_N && d_ws && d_u && d_i && d_scores && n >= 0, "nfm_scores: null argument");
    DRB_REQUIRE(nfm_dims(d, U, I, F, L, batch_norm, act) && max_rows >= 2, "nfm_scores: bad dims");
    DRB_REQUIRE(!batch_norm || d_Rs, "nfm_scores: batch_norm needs the running-statistics block");
    cudaStream_t st = (cudaStream_t)stream;
    NfmWs w;
    carve_nfm(d_ws, d, opt, max_rows, &w);
    const float *wp = d_N + d.o_wp;
    for (long long row0 = 0; row0 < n; row0 += max_rows) {
        const long long rows = n - row0 < max_rows ? n - row0 : max_rows, tot = rows * F;
        const int32_t *uu = d_u + row0, *ii = d_i + row0;
        // "B = rows": every row is a 'pos' row of the product / head kernels
        nfm_product_kernel<<<grid_size(tot, 256), 256, 0, st>>>(d_P, d_Q, uu, ii, ii, rows, rows, F, w.e);
        const float *hin = w.e;
        if (d.bn) {
            nfm_bn_apply_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.e, rows, rows, F, nullptr, d_Rs, d_Rs + F, d_N + d.o_bn0,
                                                                     d_N + d.o_bn0 + F, 0, nullptr, w.h0);
            hin = w.h0;
        }
        for (int l = 0; l < L; ++l) {
            const float *W = d_N + d.oW[l], *b = W + (size_t)F * F;
            int rc = gemm_nt(tower_dtype, rows, F, F, hin, F, W, F, w.zpre[l], F, st);
            if (rc != DRB_OK) return rc;
            nfm_bias_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.zpre[l], b, tot, F, d.bn ? nullptr : w.z[l]);
            if (d.bn)
                nfm_bn_apply_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.zpre[l], rows, rows, F, nullptr,
                                                                         d_Rs + (size_t)(1 + l) * 2 * F, d_Rs + (size_t)(1 + l) * 2 * F + F,
                                                                         d_N + d.oBN[l], d_N + d.oBN[l] + F, 0, nullptr, w.z[l]);
            nfm_act_kernel<<<grid_size(tot, 256), 256, 0, st>>>(w.z[l], tot, d.act, w.h[l]);
            hin = w.h[l];
        }
        nfm_head_kernel<<<grid_size(rows * 32, 256), 256, 0, st>>>(hin, d_bias, U, I, uu, ii, ii, rows, rows, F, wp, nullptr,
                                                                   d_scores + row0);
        DRB_CUDA(cudaGetLastError());
    }
    return DRB_OK;
}
